"""Deterministic mode of the whole-network executor (net.fused = True, the default): a fused UNetSCN training step in
the tf32, tf32x3 and bf16 modes gives the same bytes on every run -- outputs, input and parameter gradients, running
statistics, with and without the RGB mask, from coordinates or from a structure prepared on a side stream, with or
without the weight-gradient side stream, and in a fresh process -- and stays within the usual bars of the default
step and of the module path.  Inputs are nuScenes-shaped scans with several points per voxel."""
import copy
import os
import subprocess
import sys
import warnings

import numpy as np
import pytest
import torch

from mm2d3d_b200 import _lib, synth
from mm2d3d_b200 import functional as F
from mm2d3d_b200._lib import check, lib, ptr
from tests.test_deterministic_gpu import _det, _launches, _same_bytes
from tests.test_deterministic_train_gpu import _digest
from tests.test_gpu_parity import DEV, _no_device_error, rel_err, rel_l2

pytestmark = pytest.mark.gpu

DET = _lib.DETERMINISTIC
MODES = ["tf32", "tf32x3", "bf16"]
TOL = {"tf32": 1e-3, "bf16": 1e-2, "tf32x3": 1e-5}  # the bars of test_fused_executor_matches_module_path
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class _conv_mode:
    def __init__(self, mode):
        self.mode = mode

    def __enter__(self):
        from mm2d3d_b200 import scn
        self.prev = scn.get_conv_mode()
        scn.set_conv_mode(self.mode)

    def __exit__(self, *a):
        from mm2d3d_b200 import scn
        scn.set_conv_mode(self.prev)


def _batch():
    locs, feats = synth.make_batch("nuscenes", batch=2, seed0=11)
    locs = locs.copy()
    locs[:, :3] //= 2  # several points per voxel
    return torch.from_numpy(locs).to(DEV), torch.from_numpy(feats).to(DEV)


def _net(reps=1, res=False, fused=True):
    from mm2d3d_b200.unet import UNetSCN
    torch.manual_seed(0)
    net = UNetSCN(in_channels=3, block_reps=reps, residual_blocks=res).to(DEV)
    net.fused = fused
    mask = torch.nn.Linear(3, 1).to(DEV)
    return net, mask, copy.deepcopy(net.state_dict()), copy.deepcopy(mask.state_dict())


def _step(net, mask, state, mstate, inp, x0, g, use_mask=False):
    """One training step from the saved state: (digest, [output, d_x, parameter gradients, running statistics])."""
    net.load_state_dict(state)
    mask.load_state_dict(mstate)
    net.zero_grad(set_to_none=True)
    mask.zero_grad(set_to_none=True)
    x = x0.clone().requires_grad_(True)
    out = net([inp, x], rgb_mask=mask if use_mask else None)
    out.backward(g)
    ts = [out, x.grad] + [p.grad for p in net.parameters()] + [b.clone() for b in net.buffers()]
    if use_mask:
        ts += [mask.weight.grad, mask.bias.grad]
    assert all(t is not None for t in ts)
    return _digest(*ts), ts


def _grad(n):
    return torch.randn(n, 16, device=DEV, generator=torch.Generator(device=DEV).manual_seed(1))


def _no_warning(rec):
    assert not [w for w in rec if "no deterministic form" in str(w.message)], [str(w.message) for w in rec]


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("reps,res", [(1, False), (2, False), (1, True), (2, True)])
def test_fused_step_is_reproducible(mode, reps, res):
    coords, x0 = _batch()
    net, mask, state, mstate = _net(reps, res)
    g = _grad(len(coords))
    with _conv_mode(mode), _det(True), warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter("always")
        a, _ = _step(net, mask, state, mstate, coords, x0, g)
        b, _ = _step(net, mask, state, mstate, coords, x0, g)
    _no_warning(rec)
    assert a == b, (mode, reps, res)
    _no_device_error()


@pytest.mark.parametrize("mode", MODES)
def test_fused_step_with_mask_is_reproducible(mode):
    coords, x0 = _batch()
    net, mask, state, mstate = _net()
    g = _grad(len(coords))
    with _conv_mode(mode), _det(True), warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter("always")
        a, _ = _step(net, mask, state, mstate, coords, x0, g, use_mask=True)
        b, _ = _step(net, mask, state, mstate, coords, x0, g, use_mask=True)
    _no_warning(rec)
    assert a == b, mode
    _no_device_error()


@pytest.mark.parametrize("mode", MODES)
def test_prepared_structures_give_the_coordinate_digest(mode):
    """prepare(coords) and prepare_points(raw points), each built on a side stream with the mode on (the point lists
    are then built there too, before the row counts are known), give the coordinate input's bytes."""
    from mm2d3d_b200.augment import scale_points
    scans = [synth.raycast_points("nuscenes", seed) for seed in (5, 6)]
    offs = np.concatenate([[0], np.cumsum([len(p) for p in scans])]).astype(np.int64)
    pts = torch.from_numpy(np.concatenate(scans, 0)).to(DEV)
    rot = np.stack([np.eye(3, dtype=np.float32)] * 2)
    coords, keep, _, _ = scale_points(pts, offs, rot, None, 20.0, 4096)
    assert bool(keep.all())
    x0 = torch.rand(len(coords), 3, device=DEV, generator=torch.Generator(device=DEV).manual_seed(2))
    net, mask, state, mstate = _net()
    g = _grad(len(coords))
    with _conv_mode(mode), _det(True), warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter("always")
        want, _ = _step(net, mask, state, mstate, coords, x0, g, use_mask=True)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            prep_c = net.prepare(coords)
            prep_p = net.prepare_points(pts, offs, rot, None, 20.0)
        assert prep_c.meta._point_csr is not None and prep_p.meta._point_csr is not None
        assert prep_p.kept() is None
        got_c, _ = _step(net, mask, state, mstate, prep_c, x0, g, use_mask=True)
        got_p, _ = _step(net, mask, state, mstate, prep_p, x0, g, use_mask=True)
    _no_warning(rec)
    assert got_c == want and got_p == want, mode
    _no_device_error()


def test_no_dependence_on_the_side_stream():
    coords, x0 = _batch()
    net, mask, state, mstate = _net(2, True)
    g = _grad(len(coords))
    with _conv_mode("tf32"), _det(True):
        a, _ = _step(net, mask, state, mstate, coords, x0, g, use_mask=True)
        prev = os.environ.get("MM3D_NO_SIDE_STREAM")
        os.environ["MM3D_NO_SIDE_STREAM"] = "1"
        try:
            b, _ = _step(net, mask, state, mstate, coords, x0, g, use_mask=True)
        finally:
            if prev is None:
                del os.environ["MM3D_NO_SIDE_STREAM"]
            else:
                os.environ["MM3D_NO_SIDE_STREAM"] = prev
    assert a == b
    _no_device_error()


def _reference_digest():
    """The digest of one deterministic tf32 step of the reference topology (also run in a fresh process)."""
    coords, x0 = _batch()
    net, mask, state, mstate = _net()
    with _conv_mode("tf32"), _det(True):
        d, _ = _step(net, mask, state, mstate, coords, x0, _grad(len(coords)), use_mask=True)
    return d


def test_same_digest_in_a_fresh_process():
    here = _reference_digest()
    r = subprocess.run([sys.executable, "-c", "from tests.test_deterministic_exec_gpu import _reference_digest as f; "
                        "print('DIGEST', f())"], cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    there = [line.split()[1] for line in r.stdout.splitlines() if line.startswith("DIGEST ")]
    assert there == [here]


@pytest.mark.parametrize("mode", MODES)
def test_deterministic_step_is_accurate(mode):
    """Fused deterministic against fused default and against module-path deterministic: the bars of
    test_fused_executor_matches_module_path."""
    coords, x0 = _batch()
    net, mask, state, mstate = _net()
    g = _grad(len(coords))
    n_par = len(list(net.parameters()))
    with _conv_mode(mode):
        with _det(True):
            _, det = _step(net, mask, state, mstate, coords, x0, g)
        with _det(False):
            _, dflt = _step(net, mask, state, mstate, coords, x0, g)
        net.fused = False
        try:
            with _det(True):
                _, mod = _step(net, mask, state, mstate, coords, x0, g)
        finally:
            net.fused = True
    for other in (dflt, mod):
        assert rel_err(det[0], other[0]) < TOL[mode]
        for a, b in zip(det[1:2 + n_par], other[1:2 + n_par]):
            assert rel_l2(a, b) < 2e-2
        for a, b in zip(det[2 + n_par:], other[2 + n_par:]):
            assert rel_err(a, b) < TOL[mode]
    _no_device_error()


@pytest.mark.parametrize("mode", ["fp32", "tf32"])
def test_mode_off_launches_and_scratch_unchanged(mode):
    """With the mode off the fused step makes the calls it made before: the same launch count before and after a
    deterministic step, and the scratch the flags-0 query asks for."""
    coords, x0 = _batch()
    net, mask, state, mstate = _net()
    g = _grad(len(coords))
    in_ch, m, L = 3, 16, net._num_planes

    def count(det):
        with _det(det):
            torch.cuda.synchronize()
            k0 = _launches()
            _step(net, mask, state, mstate, coords, x0, g)
            torch.cuda.synchronize()
            return _launches() - k0

    with _conv_mode(mode):
        F._scratch.clear()
        off = count(False)
        key = (torch.device(DEV).type, torch.device(DEV).index)
        assert F._scratch[key].numel() == max(lib.mm3d_unet_topo_scratch_bytes(in_ch, m, L, 1, 0, _lib.MODES[mode]), 1 << 20)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            on = count(True)
        assert count(False) == off
        assert on > off
    _no_device_error()


# ------------------------------------------------------------------------------ the two new kernels against FP64
def _masked_ref(x, wb, p2v, cnt, n_vox, d_vox):
    """FP64 restatement of the masked InputLayer (mean) and its backward."""
    x, wb, d_vox = x.double(), wb.double(), d_vox.double()
    p2v = p2v.long()
    s = torch.sigmoid(x @ wb[:3] + wb[3])
    c = cnt.double()[p2v][:, None]
    out = torch.zeros(n_vox, 3, dtype=torch.float64, device=DEV).index_add_(0, p2v, x * s[:, None] / c)
    gg = d_vox[p2v] / c
    t = (gg * x).sum(1) * s * (1 - s)
    d_feats = gg * s[:, None] + t[:, None] * wb[:3][None]
    d_wb = torch.cat([(t[:, None] * x).sum(0), t.sum()[None]])
    return out, s, d_feats, d_wb


@pytest.mark.parametrize("coarse", [False, True])
def test_masked_input_kernels_against_fp64(coarse):
    from mm2d3d_b200.metadata import Metadata
    locs, _ = synth.make_batch("nuscenes", batch=2, seed0=3)
    locs = locs.copy()
    if coarse:
        locs[:, :3] //= 8  # many points per voxel
    meta = Metadata(torch.from_numpy(locs).to(DEV), 4096, 1)
    n, nv = meta.n_points, meta.n_voxels
    gen = torch.Generator(device=DEV).manual_seed(4)
    x = torch.rand(n, 3, device=DEV, generator=gen)
    wb = torch.tensor([0.7, -1.1, 0.4, 0.2], device=DEV)
    d_vox = torch.randn(nv, 3, device=DEV, generator=gen)
    start, pts = meta.point_csr()
    st = _lib.stream_ptr()

    def fwd_csr():
        out, s = torch.empty(nv, 3, device=DEV), torch.empty(n, device=DEV)
        check(lib.mm3d_input_masked_fwd_csr(ptr(x), ptr(start), ptr(pts), nv, 3, 4, ptr(wb), ptr(out), ptr(s), st))
        return out, s

    def fwd_atomic():
        out, s = torch.empty(nv, 3, device=DEV), torch.empty(n, device=DEV)
        check(lib.mm3d_input_masked_fwd(ptr(x), meta.p2v_ptr, meta.npts_ptr, n, nv, 3, 4, ptr(wb), ptr(out), ptr(s), st))
        return out, s

    def bwd(s, flags):
        d_feats, d_wb = torch.empty(n, 3, device=DEV), torch.empty(4, device=DEV)
        ws = torch.empty(4 * _lib.DET_CTAS, dtype=torch.float64, device=DEV)
        check(lib.mm3d_input_masked_bwd_ex(ptr(d_vox), ptr(x), ptr(s), meta.p2v_ptr, meta.npts_ptr, n, 3, 4, ptr(wb),
                                           ptr(d_feats), ptr(d_wb), ptr(ws), ws.numel() * 8, st, flags))
        return d_feats, d_wb

    outs = [fwd_csr() for _ in range(3)]
    ref_out, ref_s = fwd_atomic()
    s = outs[0][1]
    grads = [bwd(s, DET) for _ in range(3)]
    ref_grads = bwd(s, 0)
    torch.cuda.synchronize()
    _no_device_error()
    for j in range(2):
        assert _same_bytes(*[o[j] for o in outs]) and _same_bytes(*[gr[j] for gr in grads])
    out, s = outs[0]
    d_feats, d_wb = grads[0]
    assert torch.equal(s, ref_s)  # the same gate arithmetic
    assert rel_err(out, ref_out) < 1e-6
    assert rel_err(d_feats, ref_grads[0]) < 1e-6 and rel_err(d_wb, ref_grads[1]) < 1e-6
    single = meta.npts()[:nv] == 1
    assert bool(single.any())
    assert _same_bytes(out[single], ref_out[single])  # a voxel of one point: the atomic form's bits
    r_out, r_s, r_df, r_dwb = _masked_ref(x, wb, meta.p2v()[:n], meta.npts()[:nv], nv, d_vox)
    assert rel_err(out, r_out) < 1e-5 and rel_err(s, r_s) < 1e-5
    assert rel_err(d_feats, r_df) < 1e-5 and rel_err(d_wb, r_dwb) < 1e-5
