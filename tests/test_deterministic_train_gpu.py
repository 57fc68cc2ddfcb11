"""Deterministic mode, training step: the tcgen05 weight gradients and the single-launch BatchNorm kernels in their
fixed-order forms return the same bytes call after call -- also while other work runs on another stream -- agree with
the default forms to within reordering and with float64, and a module-path UNetSCN training step in a tensor-core
mode is bit-reproducible.  Inputs are nuScenes-shaped scans (several points per voxel for the whole step)."""
import hashlib
import warnings

import pytest
import torch

from mm2d3d_b200 import _lib, synth
from mm2d3d_b200 import functional as F
from mm2d3d_b200._lib import check, lib, ptr
from tests.test_deterministic_gpu import _det, _launches, _same_bytes
from tests.test_gpu_parity import DEV, TOL, _no_device_error, rel_err

pytestmark = pytest.mark.gpu

DET = _lib.DETERMINISTIC
PAIRS = [(16, 16), (32, 16), (64, 32), (96, 48), (160, 80), (192, 96)]


@pytest.fixture(scope="module")
def meta():
    from mm2d3d_b200.metadata import Metadata
    locs, _ = synth.make_batch("nuscenes", batch=2, seed0=7)
    return Metadata(torch.from_numpy(locs).to(DEV), 4096, 2, plans=True)


def _tables(meta, kind):
    """(table for the C ABI, float64 weight gradient of fp64 operands [n_in, ci] / [n_out, co])."""
    t, _, _ = F.conv_tables(meta, kind, 4096 if kind != "up" else 2048, plans=True)

    def ref(x, g):
        x, g = x.double(), g.double()
        out = torch.zeros(t.K, x.shape[1], g.shape[1], dtype=torch.float64, device=DEV)
        if kind == "smc":
            tbl = meta.nbr_table(4096).long()
        elif kind == "down":
            tbl = meta.down_tables(4096)[2].long()
        else:
            parent, off, _ = meta.down_tables(4096)
            tbl = torch.where(off.long()[:, None] == torch.arange(8, device=DEV)[None], parent.long()[:, None], -1)
        for k in range(t.K):
            idx = tbl[:, k]
            xg = x[idx.clamp(min=0)] * (idx >= 0)[:, None]
            out[k] = xg.t() @ g
        return out
    return t, ref


def _operand(t, mode):
    if mode == "tf32":
        return F._tf32(t)
    return F._planes(t, mode == "bf16")


def _wgrad(t, x, g, ci, co, mode, acc, flags, out=None, stream=None):
    m = _lib.MODES[mode]
    dw = out if out is not None else torch.zeros(t.K, ci, co, device=DEV)
    wsb = lib.mm3d_conv_wgrad_workspace_bytes(t.n_out, ci, co, t.K, m, flags)
    ws = torch.empty(max(wsb, 1), dtype=torch.uint8, device=DEV)
    s = stream if stream is not None else _lib.stream_ptr()
    check(lib.mm3d_conv_wgrad_ex(ptr(x), t.n_in, ci, ptr(g), t.n_out, co, ptr(dw), t.K, t.tbl, t.stride, t.onehot,
                                 t.plan, t.plan_cap, acc, m, ptr(ws) if wsb else None, wsb, s, flags), "wgrad_ex")
    return dw, ws


@pytest.mark.parametrize("mode", ["tf32", "tf32x3", "bf16"])
@pytest.mark.parametrize("kind", ["smc", "down", "up"])
def test_wgrad_deterministic(meta, kind, mode, monkeypatch):
    t, ref = _tables(meta, kind)
    gen = torch.Generator(device=DEV).manual_seed(3)
    side = torch.cuda.Stream(device=DEV)
    for ci, co in PAIRS:
        x = torch.randn(t.n_in, ci, device=DEV, generator=gen)
        g = torch.randn(t.n_out, co, device=DEV, generator=gen)
        xo, go = _operand(x, mode), _operand(g, mode)
        init = torch.randn(t.K, ci, co, device=DEV, generator=gen)
        want = ref(x, g)
        for acc in (0, 1):
            runs = [_wgrad(t, xo, go, ci, co, mode, acc, DET, out=init.clone())[0] for _ in range(3)]
            # the same while a default weight gradient of the same shape occupies the SMs from another stream
            busy = torch.zeros(t.K, ci, co, device=DEV)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                _wgrad(t, xo, go, ci, co, mode, 0, 0, out=busy, stream=side.cuda_stream)
            runs.append(_wgrad(t, xo, go, ci, co, mode, acc, DET, out=init.clone())[0])
            torch.cuda.synchronize()
            assert _same_bytes(*runs), (kind, mode, ci, co, acc)
            default = _wgrad(t, xo, go, ci, co, mode, acc, 0, out=init.clone())[0]
            # (tf32x3: each of its three launches' sums is rounded to FP32 before it is added, a coarser fixed order)
            bar = 1e-5 if mode == "tf32x3" else 1e-6
            assert rel_err(runs[0], default) < bar, (kind, mode, ci, co, acc, rel_err(runs[0], default))
            full = want + (init.double() if acc else 0)
            assert rel_err(runs[0], full) < TOL[mode], (kind, mode, ci, co, acc, rel_err(runs[0], full))
        # several launches over pieces of the tile list (smc only: the other tables are short)
        if kind == "smc":
            one = _wgrad(t, xo, go, ci, co, mode, 0, DET)[0]
            monkeypatch.setenv("MM3D_WGRAD_MAX_LOCAL", "4")
            many = [_wgrad(t, xo, go, ci, co, mode, 0, DET)[0] for _ in range(2)]
            monkeypatch.delenv("MM3D_WGRAD_MAX_LOCAL")
            assert _same_bytes(*many)
            # (each piece's sum is rounded to FP32 before it is added: another fixed order than one launch's)
            assert rel_err(many[0], one) < 1e-5 and rel_err(many[0], want) < TOL[mode]
    _no_device_error()


def test_wgrad_deterministic_refuses_simt_paths(meta):
    t, _ = _tables(meta, "smc")
    x, g = torch.randn(t.n_in, 16, device=DEV), torch.randn(t.n_out, 16, device=DEV)
    assert lib.mm3d_conv_wgrad_workspace_bytes(t.n_out, 16, 16, 27, _lib.MODE_FP32, DET) == 0
    dw = torch.empty(27, 16, 16, device=DEV)
    rc = lib.mm3d_conv_wgrad_ex(ptr(x), t.n_in, 16, ptr(g), t.n_out, 16, ptr(dw), 27, t.tbl, t.stride, None, t.plan,
                                t.plan_cap, 0, _lib.MODE_FP32, None, 0, _lib.stream_ptr(), DET)
    assert rc == 4 and b"deterministic" in lib.mm3d_last_error()
    x3 = torch.randn(t.n_in, 3, device=DEV)
    rc = lib.mm3d_conv_wgrad_ex(ptr(x3), t.n_in, 3, ptr(g), t.n_out, 16, ptr(dw), 27, t.tbl, t.stride, None, t.plan,
                                t.plan_cap, 0, _lib.MODE_TF32, None, 0, _lib.stream_ptr(), DET)
    assert rc == 4


def _bn(x, gamma, beta, rm, rv, dy, training, flags):
    n, c = x.shape
    y, dx = torch.empty_like(x), torch.empty_like(x)
    save, dgb = torch.empty(2, c, device=DEV), torch.empty(2, c, device=DEV)
    ws = torch.empty(lib.mm3d_bnrelu_workspace_bytes_ex(c, flags), dtype=torch.uint8, device=DEV)
    sp = _lib.stream_ptr()
    check(lib.mm3d_bnrelu_fwd_ex(ptr(x), ptr(y), n, c, ptr(gamma), ptr(beta), ptr(rm), ptr(rv), ptr(save[0]),
                                 ptr(save[1]), 1e-4, 0.9, 0.0, training, ptr(ws), ws.numel(), sp, flags), "bn_fwd_ex")
    check(lib.mm3d_bnrelu_bwd_ex(ptr(x), ptr(dy), ptr(dx), n, c, ptr(gamma), ptr(beta), ptr(save[0]), ptr(save[1]),
                                 ptr(dgb[0]), ptr(dgb[1]), 0.0, training, ptr(ws), ws.numel(), sp, flags), "bn_bwd_ex")
    return y, save, rm, rv, dx, dgb


def _bn_ref(x, gamma, beta, rm, rv, dy, training):
    """float64 BatchNorm + ReLU (biased batch variance, SparseConvNet's momentum) and its gradients."""
    x, gamma, beta, dy = (t.double().requires_grad_(True) for t in (x, gamma, beta, dy))
    n = x.shape[0]
    if training:
        mean, var = x.mean(0), x.var(0, unbiased=False)
        rm = 0.9 * rm.double() + 0.1 * mean.detach()
        rv = 0.9 * rv.double() + 0.1 * var.detach() * n / max(n - 1, 1)
    else:
        mean, var = rm.double(), rv.double()
    y = torch.relu((x - mean) / torch.sqrt(var + 1e-4) * gamma + beta)
    dx, dg, db = torch.autograd.grad(y, (x, gamma, beta), dy.detach())
    return y.detach(), rm, rv, dx, dg, db


@pytest.mark.parametrize("n,c", [(238_000, 16), (100_003, 96), (3561, 112), (150, 64)])
def test_bnrelu_deterministic(n, c):
    gen = torch.Generator(device=DEV).manual_seed(n + c)
    x = torch.randn(n, c, device=DEV, generator=gen) * 2 + 0.5
    dy = torch.randn(n, c, device=DEV, generator=gen)
    gamma, beta = 1 + 0.2 * torch.randn(c, device=DEV, generator=gen), 0.1 * torch.randn(c, device=DEV, generator=gen)
    rm0, rv0 = 0.1 * torch.randn(c, device=DEV, generator=gen), torch.rand(c, device=DEV, generator=gen) + 0.5
    # (a weight gradient on another stream: the BatchNorm grid's CTAs start late, its barrier still completes)
    from mm2d3d_b200.metadata import Metadata
    side = torch.cuda.Stream(device=DEV)
    locs, _ = synth.make_batch("nuscenes", batch=1, seed0=1)
    m = Metadata(torch.from_numpy(locs).to(DEV), 4096, 1, plans=True)
    t, _ = _tables(m, "smc")
    xb, gb = F._tf32(torch.randn(t.n_in, 64, device=DEV)), F._tf32(torch.randn(t.n_out, 64, device=DEV))
    for training in (1, 0):
        outs = []
        for i in range(4):
            if i == 3:
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side):
                    _wgrad(t, xb, gb, 64, 64, "tf32", 0, 0, stream=side.cuda_stream)
            outs.append(_bn(x, gamma, beta, rm0.clone(), rv0.clone(), dy, training, DET))
        torch.cuda.synchronize()
        for j in range(6):
            assert _same_bytes(*[o[j] for o in outs]), (n, c, training, j)
        d = _bn(x, gamma, beta, rm0.clone(), rv0.clone(), dy, training, 0)
        y, save, rm, rv, dx, dgb = outs[0]
        for a, b in zip(outs[0], d):
            assert rel_err(a, b) < 1e-6, (n, c, training)
        ry, rrm, rrv, rdx, rdg, rdb = _bn_ref(x, gamma, beta, rm0, rv0, dy, training)
        for a, b in ((y, ry), (rm, rrm), (rv, rrv), (dx, rdx), (dgb[0], rdg), (dgb[1], rdb)):
            assert rel_err(a, b) < 1e-4, (n, c, training, rel_err(a, b))
    _no_device_error()


def _digest(*ts):
    h = hashlib.sha256()
    for t in ts:
        h.update(t.detach().contiguous().cpu().numpy().tobytes())
    return h.hexdigest()


@pytest.mark.parametrize("mode", ["tf32", "tf32x3", "bf16"])
@pytest.mark.parametrize("reps", [1, 2])
def test_unetscn_module_path_step_is_reproducible(mode, reps):
    from mm2d3d_b200 import scn
    from mm2d3d_b200.unet import UNetSCN
    locs, feats = synth.make_batch("nuscenes", batch=2, seed0=11)
    locs = locs.copy()
    locs[:, :3] //= 2  # several points per voxel
    coords, x0 = torch.from_numpy(locs).to(DEV), torch.from_numpy(feats).to(DEV)
    torch.manual_seed(0)
    net = UNetSCN(in_channels=3, block_reps=reps).to(DEV)
    net.fused = False
    state = {k: v.clone() for k, v in net.state_dict().items()}
    g = torch.randn(len(locs), 16, device=DEV, generator=torch.Generator(device=DEV).manual_seed(1))
    prev = scn.get_conv_mode()

    def step():
        net.load_state_dict(state)
        net.zero_grad(set_to_none=True)
        x = x0.clone().requires_grad_(True)
        out = net([coords, x])
        out.backward(g)
        grads = [p.grad for p in net.parameters()]
        assert all(gr is not None for gr in grads)
        bufs = list(net.buffers())  # the BatchNorm running statistics
        return _digest(out, x.grad, *grads, *bufs)

    try:
        scn.set_conv_mode(mode)
        with _det(True), warnings.catch_warnings(record=True) as rec:
            warnings.simplefilter("always")
            a, b = step(), step()
        assert not [w for w in rec if "no deterministic form" in str(w.message)], [str(w.message) for w in rec]
        assert a == b
    finally:
        scn.set_conv_mode(prev)
    _no_device_error()


def test_mode_off_launches_and_allocates_as_before(meta):
    """With the mode off, the module path's weight gradient and BatchNorm launch what the original entry points
    launch, and no slab-sized scratch is requested."""
    t, _ = _tables(meta, "smc")
    x, w = torch.randn(t.n_in, 32, device=DEV), torch.randn(27, 1, 32, 16, device=DEV) * 0.2
    bx, dy = torch.randn(5000, 32, device=DEV), torch.randn(5000, 32, device=DEV)
    gamma, beta = torch.ones(32, device=DEV), torch.zeros(32, device=DEV)

    def count(fn):
        torch.cuda.synchronize()
        k0 = _launches()
        fn()
        torch.cuda.synchronize()
        return _launches() - k0

    with _det(False):
        F._scratch.clear()
        ww = w.clone().requires_grad_(True)
        y = F.TableConvFn.apply(x, ww, meta, "smc", 4096, "tf32")
        g = torch.randn_like(y)
        module_wgrad = count(lambda: torch.autograd.grad(y, ww, g))  # d_out rounding + weight gradient
        b = bx.clone().requires_grad_(True)
        module_bn = count(lambda: torch.autograd.grad(F.BatchNormReLUFn.apply(b, gamma, beta, torch.zeros(32, device=DEV),
                                                                              torch.ones(32, device=DEV), 1e-4, 0.9, 0.0,
                                                                              True), b, dy))
        scratch_off = max(buf.numel() for buf in F._scratch.values())
    xo, go = F._tf32(x), F._tf32(g)
    dw = torch.empty(27, 32, 16, device=DEV)
    orig_wgrad = count(lambda: check(lib.mm3d_conv_wgrad(ptr(xo), t.n_in, 32, ptr(go), t.n_out, 16, ptr(dw), 27, t.tbl,
                                                         t.stride, None, t.plan, t.plan_cap, 0, _lib.MODE_TF32, None, 0,
                                                         _lib.stream_ptr())))
    orig_bn = count(lambda: _bn(bx, gamma, beta, torch.zeros(32, device=DEV), torch.ones(32, device=DEV), dy, 1, 0))
    assert module_wgrad == 1 + orig_wgrad
    assert module_bn == orig_bn == 2
    assert scratch_off < lib.mm3d_conv_wgrad_workspace_bytes(t.n_out, 32, 16, 27, _lib.MODE_TF32, DET)
    with _det(True):
        ww = w.clone().requires_grad_(True)
        y = F.TableConvFn.apply(x, ww, meta, "smc", 4096, "tf32")
        assert count(lambda: torch.autograd.grad(y, ww, g)) == module_wgrad + 1  # + the slab reduction
    _no_device_error()
