"""UNetSCN block topologies beyond the reference configuration (block_reps > 1, residual blocks) through the
whole-network executor, and the K = 1 NetworkInNetwork convolution underneath the residual blocks.

Configurations: (block_reps, residual) in C = {(2, VGG), (1, residual), (2, residual)}; the reference
configuration (1, VGG) must issue exactly what it issued before the topology entry points existed.
"""
import copy

import numpy as np
import pytest
import torch

from mm2d3d_b200 import synth
from oracle import scn_cpu
from tests.test_gpu_parity import (DEV, TOL, _bn_modules, _freeze_gates, _no_device_error, rel_err,
                                   rel_l2)

pytestmark = pytest.mark.gpu

CONFIGS = [(2, False), (1, True), (2, True)]
MODES = ["fp32", "tf32", "tf32x3", "bf16"]


def _ids(cfg):
    return f"reps{cfg[0]}-{'res' if cfg[1] else 'vgg'}"


# ------------------------------------------------------------------------------ per op: NetworkInNetwork
def _identity_plan(n):
    """Row plan of the identity table tbl[0][j] = j, built by the library's own plan builder."""
    from mm2d3d_b200 import _lib
    from mm2d3d_b200._lib import check, lib
    tbl = torch.arange(max(n, 1), dtype=torch.int32, device=DEV)
    n_dev = torch.tensor([n], dtype=torch.int32, device=DEV)
    nbytes = lib.mm3d_plan_bytes(n, 1)
    plan = torch.empty(nbytes, dtype=torch.uint8, device=DEV)
    check(lib.mm3d_build_plan(tbl.data_ptr(), n, None, n_dev.data_ptr(), n, 1, plan.data_ptr(), nbytes,
                              _lib.stream_ptr()), "mm3d_build_plan")
    return tbl, n_dev, plan


def _operand(t, m):
    from mm2d3d_b200 import _lib
    from mm2d3d_b200 import functional as F
    if m in (_lib.MODE_TF32X3, _lib.MODE_BF16):
        return F._planes(t, m == _lib.MODE_BF16)
    return F._tf32(t) if m == _lib.MODE_TF32 else t.contiguous()


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("c_in,c_out", [(32, 16), (64, 32), (96, 48), (224, 112)])
def test_nin_as_k1_convolution(c_in, c_out, mode):
    """NetworkInNetwork (features @ W, W [c_in, c_out]) as a K = 1 rule-table convolution over the identity table:
    forward, dgrad (transposed weight image) and wgrad against a float64 matmul, at the per-op bars.  224 input
    channels take the weight-gradient kernel's two-M-block path."""
    from mm2d3d_b200 import _lib
    from mm2d3d_b200._lib import check, lib
    from mm2d3d_b200 import functional as F
    m = _lib.MODES[mode]
    torch.manual_seed(c_in + m)
    for n in (1, 127, 128, 129, 180_000):
        x = torch.randn(n, c_in, device=DEV)
        w = torch.randn(c_in, c_out, device=DEV) / c_in ** 0.5
        g = torch.randn(n, c_out, device=DEV)
        tbl, _, plan = _identity_plan(n)
        stream = _lib.stream_ptr()
        ws = F.scratch(lib.mm3d_conv_workspace_bytes(n, n, c_in, c_out, 1, m), x.device)
        xo, go = _operand(x, m), _operand(g, m)
        y = torch.empty(n, c_out, device=DEV)
        check(lib.mm3d_conv_fwd(xo.data_ptr(), n, c_in, y.data_ptr(), n, c_out, w.data_ptr(), 1, tbl.data_ptr(), n, None,
                                plan.data_ptr(), n, 0, m, ws.data_ptr(), ws.numel(), stream), "nin fwd")
        dx = torch.empty(n, c_in, device=DEV)
        check(lib.mm3d_conv_fwd(go.data_ptr(), n, c_out, dx.data_ptr(), n, c_in, w.data_ptr(), 1, tbl.data_ptr(), n, None,
                                plan.data_ptr(), n, _lib.CONV_TRANSPOSE_W, m, ws.data_ptr(), ws.numel(), stream),
              "nin dgrad")
        x64, w64, g64 = x.double(), w.double(), g.double()
        tol = TOL[mode]
        assert rel_err(y, x64 @ w64) < tol, (n, "fwd", rel_err(y, x64 @ w64))
        assert rel_err(dx, g64 @ w64.t()) < tol, (n, "dgrad", rel_err(dx, g64 @ w64.t()))
        if m == _lib.MODE_FP32 and c_in > 192:
            continue  # (the FP32 SIMT weight gradient takes up to 192 input channels)
        dw = torch.empty(c_in, c_out, device=DEV)
        check(lib.mm3d_conv_wgrad(xo.data_ptr(), n, c_in, go.data_ptr(), n, c_out, dw.data_ptr(), 1, tbl.data_ptr(), n,
                                  None, plan.data_ptr(), n, 0, m, ws.data_ptr(), ws.numel(), stream), "nin wgrad")
        assert rel_err(dw, x64.t() @ g64) < tol, (n, "wgrad", rel_err(dw, x64.t() @ g64))
    _no_device_error()


# ------------------------------------------------------------------------------ fused executor vs module path
class _NinThroughLibrary(torch.autograd.Function):
    """features @ W as the library's K = 1 convolution over an identity row plan (forward, dgrad, wgrad), with the
    operands in the mode's operand form: the executor's NetworkInNetwork arithmetic, called module by module."""

    @staticmethod
    def forward(ctx, x, w, mode):
        from mm2d3d_b200 import _lib
        from mm2d3d_b200 import functional as F
        from mm2d3d_b200._lib import check, lib
        m = _lib.MODES[mode]
        n, c_in, c_out = x.shape[0], x.shape[1], w.shape[1]
        tbl, _, plan = _identity_plan(n)
        xo, w = _operand(x.contiguous(), m), w.contiguous()
        ws = F.scratch(lib.mm3d_conv_workspace_bytes(n, n, c_in, c_out, 1, m), x.device)
        y = torch.empty(n, c_out, device=x.device)
        check(lib.mm3d_conv_fwd(xo.data_ptr(), n, c_in, y.data_ptr(), n, c_out, w.data_ptr(), 1, tbl.data_ptr(), n, None,
                                plan.data_ptr(), n, 0, m, ws.data_ptr(), ws.numel(), _lib.stream_ptr()), "nin fwd")
        ctx.save_for_backward(xo, w, tbl, plan)
        ctx.m = m
        return y

    @staticmethod
    def backward(ctx, g):
        from mm2d3d_b200 import _lib
        from mm2d3d_b200 import functional as F
        from mm2d3d_b200._lib import check, lib
        xo, w, tbl, plan = ctx.saved_tensors
        m = ctx.m
        n, c_in, c_out = g.shape[0], w.shape[0], w.shape[1]
        go = _operand(g.contiguous(), m)
        ws = F.scratch(lib.mm3d_conv_workspace_bytes(n, n, c_in, c_out, 1, m), g.device)
        dx = torch.empty(n, c_in, device=g.device)
        dw = torch.empty(c_in, c_out, device=g.device)
        check(lib.mm3d_conv_fwd(go.data_ptr(), n, c_out, dx.data_ptr(), n, c_in, w.data_ptr(), 1, tbl.data_ptr(), n, None,
                                plan.data_ptr(), n, _lib.CONV_TRANSPOSE_W, m, ws.data_ptr(), ws.numel(), _lib.stream_ptr()),
              "nin dgrad")
        check(lib.mm3d_conv_wgrad(xo.data_ptr(), n, c_in, go.data_ptr(), n, c_out, dw.data_ptr(), 1, tbl.data_ptr(), n,
                                  None, plan.data_ptr(), n, 0, m, ws.data_ptr(), ws.numel(), _lib.stream_ptr()), "nin wgrad")
        return dx, dw, None


def _nin_through_library(net, mode):
    """Module path with the executor's NetworkInNetwork arithmetic (the module path's own is an FP32 torch matmul).
    Otherwise the two paths differ in the last bits of every shortcut output, which in the tensor-core modes moves
    later TF32 / BF16 roundings by a whole unit and flips ReLU gates of the randomly initialised network: the
    free-running gradients would then compare two different arithmetics, not the executor's wiring."""
    import types

    import mm2d3d_b200.scn as scn
    for mod in net.modules():
        if isinstance(mod, scn.NetworkInNetwork):
            def fwd(self, x):
                y = _NinThroughLibrary.apply(x.features, self.weight, mode)
                return scn.SparseConvNetTensor(y, x.metadata, x.spatial_size)
            mod.forward = types.MethodType(fwd, mod)


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("cfg", CONFIGS, ids=_ids)
def test_variant_fused_matches_module_path(cfg, mode):
    """Every configuration runs as one native call per direction and agrees with the module-by-module path: output,
    every gradient, the BatchNorm buffers and eval mode, at the tolerances of test_fused_executor_matches_module_path.
    (The module path's NetworkInNetwork runs here as the library's K = 1 convolution, as in the executor.)"""
    import mm2d3d_b200.scn as scn
    from mm2d3d_b200 import executor
    from mm2d3d_b200.unet import UNetSCN
    reps, res = cfg
    torch.manual_seed(9)
    locs, feats = synth.make_batch("nuscenes", batch=2, seed0=5)
    coords, feats = torch.from_numpy(locs).to(DEV), torch.from_numpy(feats).to(DEV)
    net_a = UNetSCN(in_channels=3, block_reps=reps, residual_blocks=res).to(DEV)
    assert executor.fusable(net_a)
    net_b = copy.deepcopy(net_a)
    net_b.fused = False
    _nin_through_library(net_b, mode)
    net_c = copy.deepcopy(net_b)  # (the module path a second time: its run-to-run spread)
    g = torch.randn(locs.shape[0], 16, device=DEV)
    scn.set_conv_mode(mode)
    try:
        res_ = []
        for net in (net_a, net_b, net_c):
            x = feats.clone().requires_grad_(True)
            out = net([coords, x])
            if net is net_a:
                assert out.grad_fn is not None and type(out.grad_fn).__name__ == "UNetSCNFnBackward"
            grads = torch.autograd.grad(out, [x] + list(net.parameters()), g)
            res_.append((out, grads, [b.clone() for b in net.buffers()]))
        _no_device_error()
        tol = {"tf32": 1e-3, "bf16": 1e-2}.get(mode, 1e-5)
        assert rel_err(res_[0][0], res_[1][0]) < tol, rel_err(res_[0][0], res_[1][0])
        names = ["feats"] + [k for k, _ in net_a.named_parameters()]
        # FP32 summation order varies run to run (atomics); a ReLU gate it flips moves gradients of this deep
        # network by O(1e-2), in the module path against itself too: the bar is 2e-2 or 3 x that spread
        errs = [(name, rel_l2(a, b), rel_l2(b2, b)) for name, a, b, b2 in zip(names, res_[0][1], res_[1][1], res_[2][1])]
        print(f"\n[{mode}] {_ids(cfg)}: forward {rel_err(res_[0][0], res_[1][0]):.2e}, worst gradient rel-L2 "
              f"{max(e for _, e, _ in errs):.2e} ({max(errs, key=lambda t: t[1])[0]}), module path against itself "
              f"{max(n for _, _, n in errs):.2e}")
        for name, e, noise in errs:
            assert e < max(2e-2, 3 * noise), (name, e, noise)
        for a, b in zip(res_[0][2], res_[1][2]):
            assert rel_err(a, b) < tol
        net_a.eval(); net_b.eval()
        with torch.no_grad():
            assert rel_err(net_a([coords, feats]), net_b([coords, feats])) < tol
    finally:
        scn.set_conv_mode("fp32")


# ------------------------------------------------------------------------------ against the FP64 oracle
def test_residual_reps2_one_scan_against_oracle():
    """(2, residual), m = 16, 7 planes, one nuScenes-shaped scan: the fused FP32 executor against the FP64 oracle,
    free running.  Forward within 1e-4.  The gradients of this ~100-layer BN/ReLU network are decided by ReLU gates
    that the (run-to-run varying) summation order of the BatchNorm statistics flips: per tensor they land anywhere
    from 1e-6 to a few 1e-3 from FP64, in the module-by-module path just the same (both are printed), so they are
    held to the free-running FP32 bar of test_product_arm_dumps_the_last_timed_step, 2e-2 rel-L2.  The per-tensor
    1e-4 bar with the gates frozen is test_residual_reps2_gradients_with_frozen_gates."""
    from mm2d3d_b200.unet import UNetSCN
    torch.manual_seed(5)
    locs, feats = synth.make_batch("nuscenes", batch=1, seed0=3)
    coords, feats = torch.from_numpy(locs), torch.from_numpy(feats)
    net_ref = UNetSCN(in_channels=3, block_reps=2, residual_blocks=True, backend=scn_cpu)
    runs, g = {}, None
    for tag, ref, dt in (("f64", copy.deepcopy(net_ref).double(), torch.float64), ("f32", net_ref, torch.float32)):
        xr = feats.clone().to(dt).requires_grad_(True)
        out_r = ref([coords, xr])
        if g is None:
            g = torch.randn_like(out_r)
        pr = dict(ref.named_parameters())
        runs[tag] = (out_r, dict(zip(["feats"] + list(pr), torch.autograd.grad(out_r, [xr] + list(pr.values()), g.to(dt)))))
    names = list(runs["f64"][1])
    gpu = {}
    for tag in ("fused", "module"):
        net = UNetSCN(in_channels=3, block_reps=2, residual_blocks=True).to(DEV)
        net.load_state_dict(net_ref.state_dict())
        net.fused = tag == "fused"
        x = feats.clone().to(DEV).requires_grad_(True)
        out = net([coords.to(DEV), x])
        p = dict(net.named_parameters())
        gpu[tag] = (out, torch.autograd.grad(out, [x] + [p[k] for k in names[1:]], g.float().to(DEV)))
    _no_device_error()
    e_out = rel_err(gpu["fused"][0], runs["f64"][0])
    print(f"\n(2, residual) FP32 executor vs FP64 oracle: forward max-abs-rel {e_out:.2e}")
    assert e_out < TOL["fp32"], ("forward", e_out)
    for name, a, b in zip(names, gpu["fused"][1], gpu["module"][1]):
        ref64 = runs["f64"][1][name]
        e, e_mod, e_cpu = rel_l2(a, ref64), rel_l2(b, ref64), rel_l2(runs["f32"][1][name], ref64)
        print(f"  d {name:60s} fused {e:.2e}  module path {e_mod:.2e}  FP32 CPU oracle {e_cpu:.2e}")
        assert e <= 2e-2, (name, e, e_mod, e_cpu)


@pytest.mark.parametrize("mode", MODES)
def test_residual_reps2_gradients_with_frozen_gates(mode):
    """test_unetscn_gradients_with_frozen_gates for (2, residual): BatchNorm statistics and ReLU gates of the FP64
    oracle's forward frozen in both networks, so the chain of convolutions (and the identity / NetworkInNetwork
    shortcuts between them) is compared per tensor, rel-L2 and max-abs-rel, against FP64.  Bars: FP32 and TF32x3
    1e-4, TF32 1e-2; BF16 is held to 1e-1 and its achieved figures are printed."""
    import mm2d3d_b200.scn as scn
    from mm2d3d_b200.unet import UNetSCN
    torch.manual_seed(8)
    locs, feats = synth.make_batch("nuscenes", batch=1, seed0=6)
    coords, feats = torch.from_numpy(locs), torch.from_numpy(feats)
    net_ref = UNetSCN(in_channels=3, block_reps=2, residual_blocks=True, backend=scn_cpu)
    with torch.no_grad():
        for m in _bn_modules(net_ref):
            m.weight.add_(0.2 * torch.randn_like(m.weight))
            m.bias.add_(0.1 * torch.randn_like(m.bias))
    net = UNetSCN(in_channels=3, block_reps=2, residual_blocks=True).to(DEV)
    net.load_state_dict(net_ref.state_dict())
    net.fused = False  # (the frozen gates replace the BatchNorm modules' forward)
    net64 = copy.deepcopy(net_ref).double()
    records, hooks = [], []

    def hook(mod, inp, out):
        x = inp[0].features.detach()
        mean, var = x.mean(0), x.var(0, unbiased=False)
        records.append((mean, 1.0 / torch.sqrt(var + mod.eps), (out.features.detach() > 0).to(x.dtype)))
    for m in _bn_modules(net64):
        hooks.append(m.register_forward_hook(hook))
    with torch.no_grad():
        out_true = net64([coords, feats.double()])
    for h in hooks:
        h.remove()
    assert len(records) == len(_bn_modules(net64))
    _freeze_gates(net64, records, "cpu", torch.float64, scn_cpu.SparseConvNetTensor)
    _freeze_gates(net, records, DEV, torch.float32, scn.SparseConvNetTensor)
    x64 = feats.double().requires_grad_(True)
    out64 = net64([coords, x64])
    assert rel_err(out64, out_true) < 1e-12
    g = torch.randn_like(out64)
    p64 = dict(net64.named_parameters())
    names = ["feats"] + list(p64)
    g64 = dict(zip(names, torch.autograd.grad(out64, [x64] + list(p64.values()), g)))
    scn.set_conv_mode(mode)
    try:
        x = feats.clone().to(DEV).requires_grad_(True)
        out = net([coords.to(DEV), x])
        p = dict(net.named_parameters())
        gg = torch.autograd.grad(out, [x] + [p[k] for k in names[1:]], g.float().to(DEV))
    finally:
        scn.set_conv_mode("fp32")
    _no_device_error()
    # BF16 (unit round-off 2^-9): the (2, residual) chain has ~80 convolutions against the reference configuration's
    # 27, and its achieved figures (printed; B200: rel-L2 <= 4.7e-2, max-abs-rel <= 7e-2) are held to 1e-1
    tol = 1e-1 if mode == "bf16" else TOL[mode]
    e_out = rel_err(out, out64)
    rows = [(name, rel_l2(a, g64[name]), rel_err(a, g64[name])) for name, a in zip(names, gg)]
    print(f"\n[{mode}] (2, residual) frozen-gate parity vs FP64 oracle: forward max-abs-rel {e_out:.2e}, "
          f"worst gradient rel-L2 {max(r[1] for r in rows):.2e}, max-abs-rel {max(r[2] for r in rows):.2e}")
    for name, e2, em in rows:
        print(f"[{mode}]   d {name:52s} rel-L2 {e2:.2e}  max-abs-rel {em:.2e}")
    assert e_out < tol, ("forward", e_out)
    for name, e2, em in rows:
        assert e2 <= tol and em <= tol, (mode, name, e2, em)


# ------------------------------------------------------------------------------ reference configuration
def _unique_batch(seed0, batch=2, div=16):
    locs, feats = synth.make_batch("nuscenes", batch=batch, seed0=seed0)
    locs[:, :3] //= div
    locs, first = np.unique(locs, axis=0, return_index=True)  # one point per voxel: no order-dependent float atomics
    return torch.from_numpy(locs).to(DEV), torch.from_numpy(feats[first]).to(DEV)


class _ReferenceEntryPoints:
    """The executor's library handle with the mm3d_unet_topo_* calls routed to the reference-configuration entry
    points that predate them (which must only ever see block_reps = 1, VGG)."""

    def __init__(self, lib):
        self._lib = lib

    def __getattr__(self, name):
        return getattr(self._lib, name)

    def mm3d_unet_topo_act_bytes(self, in_ch, m, L, reps, res, *rest):
        assert (reps, res) == (1, 0)
        return self._lib.mm3d_unet_act_bytes(in_ch, m, L, *rest)

    def mm3d_unet_topo_bwd_bytes(self, in_ch, m, L, reps, res, *rest):
        assert (reps, res) == (1, 0)
        return self._lib.mm3d_unet_bwd_bytes(in_ch, m, L, *rest)

    def mm3d_unet_topo_scratch_bytes(self, in_ch, m, L, reps, res, mode):
        assert (reps, res) == (1, 0)
        return self._lib.mm3d_unet_scratch_bytes(in_ch, m, L, mode)

    def mm3d_unet_topo_forward(self, in_ch, m, L, reps, res, *rest):
        assert (reps, res) == (1, 0)
        return self._lib.mm3d_unet_forward(in_ch, m, L, *rest)

    def mm3d_unet_topo_backward(self, in_ch, m, L, reps, res, *rest):
        assert (reps, res) == (1, 0)
        return self._lib.mm3d_unet_backward(in_ch, m, L, *rest)


@pytest.mark.parametrize("mode", ["tf32", "fp32"])
def test_reference_config_old_and_new_entry_points_agree(monkeypatch, mode):
    """block_reps = 1, VGG: the topology entry points and the original ones give bit-identical forward output and
    d_feats (one point per voxel: no order-dependent atomics on that path in TF32 mode; FP32 within 1e-6) and launch
    the same number of kernels per training step."""
    import mm2d3d_b200.scn as scn
    from mm2d3d_b200 import _lib, executor
    from mm2d3d_b200.unet import UNetSCN
    torch.manual_seed(4)
    net = UNetSCN(in_channels=3).to(DEV)
    coords, feats = _unique_batch(21)
    g = torch.randn(coords.shape[0], 16, device=DEV)
    scn.set_conv_mode(mode)
    try:
        def step(prep):
            x = feats.clone().requires_grad_(True)
            torch.cuda.synchronize()
            n0 = _lib.lib.mm3d_kernel_launches()
            out = net([prep, x])
            (gx,) = torch.autograd.grad(out, [x], g)
            torch.cuda.synchronize()
            return out.detach().clone(), gx.clone(), _lib.lib.mm3d_kernel_launches() - n0

        prep = [net.prepare(coords, wait=True) for _ in range(4)]
        runs = {}
        for rnd in range(2):  # alternating, twice: the launch counts are the same every step
            runs.setdefault("new", []).append(step(prep[2 * rnd]))
            with monkeypatch.context() as mp:
                mp.setattr(executor, "lib", _ReferenceEntryPoints(_lib.lib))
                runs.setdefault("old", []).append(step(prep[2 * rnd + 1]))
    finally:
        scn.set_conv_mode("fp32")
    _no_device_error()
    for (o_new, gx_new, l_new), (o_old, gx_old, l_old) in zip(runs["new"], runs["old"]):
        assert l_new == l_old and l_new > 0, (l_new, l_old)
        if mode == "tf32":
            assert torch.equal(o_new, o_old) and torch.equal(gx_new, gx_old)
        else:
            assert rel_err(o_new, o_old) < 1e-6 and rel_err(gx_new, gx_old) < 1e-6
    print(f"[{mode}] reference configuration: {runs['new'][0][2]} launches per training step (both entry points)")


# ------------------------------------------------------------------------------ structure reuse, frozen weights
def test_residual_prepared_structure_on_side_stream_matches_inline():
    """UNetSCN.prepare() works for a residual network: structure built one step ahead on another stream gives the
    same bits as the inline build (TF32: no atomics on the forward / d_feats path with one point per voxel)."""
    import mm2d3d_b200.scn as scn
    from mm2d3d_b200.unet import UNetSCN
    torch.manual_seed(3)
    net = UNetSCN(in_channels=3, m=16, block_reps=2, residual_blocks=True, num_planes=4, full_scale=256).to(DEV)
    batches = [_unique_batch(40 + 2 * r) for r in range(3)]
    nin = next(m for m in net.modules() if isinstance(m, scn.NetworkInNetwork))
    scn.set_conv_mode("tf32")
    try:
        def run(prep_of):
            outs = []
            for i in range(5):
                locs, feats = batches[i % 3]
                x = feats.clone().requires_grad_(True)
                net.zero_grad(set_to_none=True)
                out = net([prep_of(i, locs), x])
                out.square().sum().backward()
                outs.append((out.detach().clone(), x.grad.clone(), nin.weight.grad.clone()))
            torch.cuda.synchronize()
            return outs

        inline = run(lambda i, locs: locs)
        side = torch.cuda.Stream(device=DEV, priority=-1)
        ahead = {}

        def prep_of(i, locs):
            if i not in ahead:
                with torch.cuda.stream(side):
                    ahead[i] = net.prepare(locs)
            cur = ahead.pop(i)
            with torch.cuda.stream(side):
                ahead[i + 1] = net.prepare(batches[(i + 1) % 3][0])
            return cur

        piped = run(prep_of)
    finally:
        scn.set_conv_mode("fp32")
    _no_device_error()
    for step, ((a, b, c), (d, e, f)) in enumerate(zip(inline, piped)):
        assert torch.equal(a, d) and torch.equal(b, e), step
        assert float((c - f).abs().max()) <= 1e-5 * float(c.abs().max()), step


def test_residual_frozen_nin_weight():
    """A frozen NetworkInNetwork weight (requires_grad=False) gets no gradient; every other gradient is unchanged."""
    from mm2d3d_b200 import scn as scn_mod
    from mm2d3d_b200.unet import UNetSCN
    torch.manual_seed(12)
    net = UNetSCN(in_channels=3, m=16, block_reps=2, residual_blocks=True, num_planes=4, full_scale=256).to(DEV)
    coords, feats = _unique_batch(60)
    nins = [m for m in net.modules() if isinstance(m, scn_mod.NetworkInNetwork)]
    assert len(nins) == 3  # the first post block of every level but the deepest
    scn_mod.set_conv_mode("tf32")
    try:
        def grads():
            net.zero_grad(set_to_none=True)
            x = feats.clone().requires_grad_(True)
            net([coords, x]).square().sum().backward()
            return x.grad.clone(), {k: (p.grad.clone() if p.grad is not None else None) for k, p in net.named_parameters()}

        gx0, g0 = grads()
        nins[0].weight.requires_grad_(False)
        gx1, g1 = grads()
    finally:
        nins[0].weight.requires_grad_(True)
        scn_mod.set_conv_mode("fp32")
    _no_device_error()
    frozen = [k for k, p in net.named_parameters() if p is nins[0].weight]
    assert g1[frozen[0]] is None
    assert torch.equal(gx0, gx1)
    for k in g0:
        if k != frozen[0]:
            assert float((g0[k] - g1[k]).abs().max()) <= 1e-5 * float(g0[k].abs().max()) + 1e-30, k
