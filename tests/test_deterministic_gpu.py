"""Deterministic mode on the GPU: the group-by builders equal the numpy statement, and every op in its deterministic
form returns the same bytes call after call, agrees with the default form to within reordering and with float64.
Inputs include duplicate-heavy voxels and pixels: nuScenes-shaped scans and the same scans coarsened 8x."""
import numpy as np
import pytest
import torch

from mm2d3d_b200 import _lib, synth
from mm2d3d_b200._lib import check, lib, ptr
from tests.test_deterministic_cpu import groupby_reference
from tests.test_gpu_parity import DEV, _no_device_error, rel_err

pytestmark = pytest.mark.gpu


def _same_bytes(*ts):
    a = ts[0].detach().cpu().contiguous().view(torch.uint8)
    return all(torch.equal(a, t.detach().cpu().contiguous().view(torch.uint8)) for t in ts[1:])


def _launches():
    return lib.mm3d_kernel_launches()


class _det:
    """Deterministic mode on (True) or off inside a block; restores the previous setting."""

    def __init__(self, flag):
        self.flag = flag

    def __enter__(self):
        from mm2d3d_b200 import functional as F
        self.prev = F.DETERMINISTIC
        F.DETERMINISTIC = self.flag

    def __exit__(self, *a):
        from mm2d3d_b200 import functional as F
        F.DETERMINISTIC = self.prev


@pytest.fixture(scope="module", params=["scan", "coarse"])
def scan(request):
    locs, feats = synth.make_batch("nuscenes", batch=2, seed0=3)
    if request.param == "coarse":
        locs = locs.copy()
        locs[:, :3] //= 8  # many points per voxel
    from mm2d3d_b200.metadata import Metadata
    meta = Metadata(torch.from_numpy(locs).to(DEV), 4096, 1)
    return meta, torch.from_numpy(feats).to(DEV)


# ------------------------------------------------------------------------------ group-by builders
def test_point_csr_equals_stable_argsort(scan):
    meta, _ = scan
    start, pts = meta.point_csr()
    _no_device_error()
    p2v = meta.p2v().cpu().numpy()
    rs, rp = groupby_reference(p2v, meta.n_voxels)
    assert np.array_equal(start.cpu().numpy(), rs)
    assert np.array_equal(pts[:meta.n_points].cpu().numpy(), rp)
    if meta.npts().max().item() > 1:
        assert (np.diff(rs) > 1).any()


def _img_indices(window, n=(9000, 7000)):
    return synth.make_img_indices(list(n), height=60, width=90, seed=1, window=window)


@pytest.mark.parametrize("window", [None, 6])
def test_lift_csr_equals_stable_argsort(window):
    from mm2d3d_b200.functional import lift_csr
    from mm2d3d_b200.lift import LiftIndices
    B, H, W = 2, 60, 90
    ii = _img_indices(window)
    ii[0][::7] -= np.array([H, W])  # negative indices, normalised like torch indexing
    li = LiftIndices(ii, DEV)
    start, ent = lift_csr(li.idx, None, li.offsets, B, H, W)
    _no_device_error()
    cat = np.concatenate(ii, 0) % np.array([H, W])
    b = np.repeat(np.arange(B), [len(x) for x in ii])
    rs, re = groupby_reference((b * H + cat[:, 0]) * W + cat[:, 1], B * H * W)
    assert np.array_equal(start.cpu().numpy(), rs) and np.array_equal(ent[:len(re)].cpu().numpy(), re)
    # bilinear: (point, tap) entries 4 p + q, taps outside the map or of weight zero dropped
    rng = np.random.default_rng(2)
    uv = [rng.uniform(-1.5, [H + 0.5, W + 0.5], (n, 2)).astype(np.float32) for n in (3000, 2000)]
    uv[1][:200] = np.round(uv[1][:200])  # integer coordinates: three zero-weight taps
    uvd = torch.from_numpy(np.concatenate(uv, 0)).to(DEV)
    offs = torch.tensor([0, 3000, 5000], dtype=torch.int64, device=DEV)
    start, ent = lift_csr(None, uvd, offs, B, H, W)
    u = np.concatenate(uv, 0).astype(np.float64)
    bb = np.repeat(np.arange(B), [3000, 2000])
    r0, c0 = np.floor(u[:, 0]), np.floor(u[:, 1])
    fr, fc = u[:, 0] - r0, u[:, 1] - c0
    keys = np.full((len(u), 4), -1, np.int64)
    for q in range(4):
        rr, cc = r0 + (q >> 1), c0 + (q & 1)
        w = (fr if q >> 1 else 1 - fr) * (fc if q & 1 else 1 - fc)
        ok = (rr >= 0) & (rr < H) & (cc >= 0) & (cc < W) & (w != 0)
        keys[ok, q] = ((bb * H + rr) * W + cc)[ok].astype(np.int64)
    rs, re = groupby_reference(keys.reshape(-1), B * H * W)
    assert np.array_equal(start.cpu().numpy(), rs) and np.array_equal(ent[:len(re)].cpu().numpy(), re)


# ------------------------------------------------------------------------------ InputLayer / OutputLayer
@pytest.mark.parametrize("c,mode", [(3, 4), (3, 3), (16, 3)])
def test_input_output_layers(scan, c, mode):
    from mm2d3d_b200 import functional as F
    meta, feats = scan
    torch.manual_seed(0)
    x = feats if c == 3 else torch.rand(meta.n_points, c, device=DEV)
    g = torch.randn(meta.n_points, c, device=DEV)

    def run():
        xi = x.clone().requires_grad_(True)
        v = F.InputLayerFn.apply(xi, meta, mode)
        o = F.OutputLayerFn.apply(v, meta)
        (gv,) = torch.autograd.grad(o, v, g)
        return v.detach(), gv

    with _det(True):
        runs = [run() for _ in range(3)]
    with _det(False):
        v0, gv0 = run()
    _no_device_error()
    assert _same_bytes(*[r[0] for r in runs]) and _same_bytes(*[r[1] for r in runs])
    v, gv = runs[0]
    # (voxels of hundreds of points in the coarsened scans: FP32 sums in two orders)
    assert rel_err(v, v0) <= 1e-5 and rel_err(gv, gv0) <= 1e-5
    # float64
    p2v = meta.p2v().long()
    cnt = torch.bincount(p2v, minlength=meta.n_voxels).double()
    v64 = torch.zeros(meta.n_voxels, c, dtype=torch.float64, device=DEV).index_add_(0, p2v, x.double())
    if mode == 4:
        v64 /= cnt[:, None]
    g64 = torch.zeros(meta.n_voxels, c, dtype=torch.float64, device=DEV).index_add_(0, p2v, g.double())
    assert rel_err(v, v64) < 1e-5 and rel_err(gv, g64) < 1e-5
    # one point per voxel: the deterministic InputLayer forward gives the default path's bits
    one = (cnt[p2v] == 1).nonzero().squeeze(1)
    rows = p2v[one]
    assert torch.equal(v[rows], v0[rows])


# ------------------------------------------------------------------------------ lift
_EPS = {torch.float32: 2.0 ** -23, torch.float16: 2.0 ** -10, torch.bfloat16: 2.0 ** -7}


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.bfloat16])
@pytest.mark.parametrize("channels_last", [False, True])
@pytest.mark.parametrize("bilinear", [False, True])
def test_lift_backward(dtype, channels_last, bilinear):
    from mm2d3d_b200.lift import lift2d, lift2d_bilinear
    B, C, H, W = 2, 24, 60, 90
    ii = _img_indices(6)  # duplicate-heavy: every point in a 6x6 window
    rng = np.random.default_rng(5)
    uv = [x.astype(np.float32) + rng.uniform(-0.5, 0.5, x.shape).astype(np.float32) for x in ii]
    fmap = torch.randn(B, C, H, W, device=DEV).to(dtype)
    if channels_last:
        fmap = fmap.contiguous(memory_format=torch.channels_last)
    n = sum(len(x) for x in ii)
    g = torch.randn(n, C, device=DEV).to(dtype)

    def run():
        f = fmap.clone().requires_grad_(True)
        out = lift2d_bilinear(f, uv) if bilinear else lift2d(f, ii)
        (gf,) = torch.autograd.grad(out, f, g)
        return gf

    with _det(True):
        gs = [run() for _ in range(3)]
    with _det(False):
        g0 = run()
    _no_device_error()
    assert _same_bytes(*gs)
    assert gs[0].is_contiguous(memory_format=torch.channels_last) == channels_last
    # float64 reference by index_add over the flattened NHWC pixels
    gd = g.double()
    ref = torch.zeros(B * H * W, C, dtype=torch.float64, device=DEV)
    bidx = torch.from_numpy(np.repeat(np.arange(B), [len(x) for x in ii])).to(DEV)
    if bilinear:
        u = torch.from_numpy(np.concatenate(uv, 0)).to(DEV).double()
        r0, c0 = u[:, 0].floor(), u[:, 1].floor()
        fr, fc = u[:, 0] - r0, u[:, 1] - c0
        for q in range(4):
            rr, cc = r0 + (q >> 1), c0 + (q & 1)
            w = (fr if q >> 1 else 1 - fr) * (fc if q & 1 else 1 - fc)
            ok = (rr >= 0) & (rr < H) & (cc >= 0) & (cc < W)
            key = ((bidx * H + rr.long()) * W + cc.long())[ok]
            ref.index_add_(0, key, gd[ok] * w[ok, None])
    else:
        cat = torch.from_numpy(np.concatenate(ii, 0)).to(DEV)
        ref.index_add_(0, (bidx * H + cat[:, 0]) * W + cat[:, 1], gd)
    ref = ref.view(B, H, W, C).permute(0, 3, 1, 2)
    got = gs[0].double()
    if dtype == torch.float32:
        assert rel_err(got, ref) < 1e-5 and rel_err(got, g0) <= 1e-5
    else:  # one rounding of the float64 sum (plus the FP32 accumulation's own few ulps)
        tol = _EPS[dtype] * ref.abs() + 1e-6 * ref.abs().max()
        assert ((got - ref).abs() <= tol).all()


# ------------------------------------------------------------------------------ rgb_mask, KL, heads3d
def test_rgb_mask_kl_heads3d():
    from mm2d3d_b200.heads import cross_modal_kl, heads3d, rgb_mask
    torch.manual_seed(1)
    n, c, f, C = 300_000, 3, 16, 10
    x = torch.rand(n, c, device=DEV)
    wm, bm = torch.randn(1, c, device=DEV), torch.randn(1, device=DEV)
    feat = torch.randn(n, f, device=DEV)
    w1, b1, w2, b2 = (torch.randn(C, f, device=DEV) * 0.3, torch.randn(C, device=DEV), torch.randn(C, f, device=DEV) * 0.3,
                      torch.randn(C, device=DEV))
    tgt = torch.randn(n, C, device=DEV)
    gy, g1, g2 = torch.randn(n, c, device=DEV), torch.randn(n, C, device=DEV), torch.randn(n, C, device=DEV)

    def run(dbl=False):
        cast = (lambda t: t.double()) if dbl else (lambda t: t)
        ps = [cast(t).clone().requires_grad_(True) for t in (x, wm, bm, feat, w1, b1, w2, b2)]
        if dbl:  # float64 statement of the three ops
            y = ps[0] * torch.sigmoid(ps[0] @ ps[1].t() + ps[2])
            l1, l2 = ps[3] @ ps[4].t() + ps[5], ps[3] @ ps[6].t() + ps[7]
            q = torch.softmax(tgt.double(), 1)
            kl = (q * (torch.log_softmax(tgt.double(), 1) - torch.log_softmax(l2, 1))).sum(1).mean()
            kl2 = kl
        else:
            y = rgb_mask(*ps[:3])
            l1, l2, kl = heads3d(ps[3], *ps[4:], target=tgt)
            kl2 = cross_modal_kl(l2.detach(), tgt)
        tot = (y * cast(gy)).sum() + (l1 * cast(g1)).sum() + (l2 * cast(g2)).sum() + 3.0 * kl
        grads = torch.autograd.grad(tot, ps[1:])
        return [kl.detach().reshape(1), kl2.detach().reshape(1)] + list(grads)

    with _det(True):
        runs = [run() for _ in range(3)]
    with _det(False):
        r0 = run()
    r64 = run(dbl=True)
    _no_device_error()
    for i in range(len(runs[0])):
        assert _same_bytes(*[r[i] for r in runs]), i
        assert rel_err(runs[0][i], r0[i]) <= 1e-6, i
        assert rel_err(runs[0][i], r64[i]) < 1e-4, i


# ------------------------------------------------------------------------------ the default path is unchanged
def test_ex_twins_with_zero_flags_match_the_original_entry_points():
    torch.manual_seed(2)
    n, c, f, C = 100_000, 3, 16, 10
    x, s, dy = torch.rand(n, c, device=DEV), torch.rand(n, device=DEV), torch.randn(n, c, device=DEV)
    w = torch.randn(c, device=DEV)
    feat, tgt = torch.randn(n, f, device=DEV), torch.randn(n, C, device=DEV)
    w1, b1, w2, b2 = torch.randn(C, f, device=DEV), torch.randn(C, device=DEV), torch.randn(C, f, device=DEV), torch.randn(C, device=DEV)
    d1, d2, dl = torch.randn(n, C, device=DEV), torch.randn(n, C, device=DEV), torch.ones(1, device=DEV)
    ws = torch.empty(1 << 16, dtype=torch.float64, device=DEV)
    sp = _lib.stream_ptr()

    def calls(ex):
        out = [torch.empty(k, device=DEV) for k in (n * c, c, 1, 1, n * C, n * C, 1, n * f, C * f, C, C * f, C)]
        dx, dw, db, kl, l1, l2, hl, dfe, dw1, db1, dw2, db2 = out
        tail = (0,) if ex else ()
        sfx = "_ex" if ex else ""
        torch.cuda.synchronize()
        k0 = _launches()
        check(getattr(lib, "mm3d_rgb_mask_bwd" + sfx)(ptr(x), ptr(s), ptr(dy), n, c, ptr(w), ptr(dx), ptr(dw), ptr(db),
                                                       ptr(ws), ws.numel() * 8, sp, *tail))
        check(getattr(lib, "mm3d_kl_logits_fwd" + sfx)(ptr(d1), ptr(tgt), n, C, ptr(kl), ptr(ws), ws.numel() * 8, sp, *tail))
        check(getattr(lib, "mm3d_heads3d_fwd" + sfx)(ptr(feat), n, f, C, ptr(w1), ptr(b1), ptr(w2), ptr(b2), ptr(tgt), ptr(l1),
                                                      ptr(l2), ptr(hl), ptr(ws), ws.numel() * 8, sp, *tail))
        check(getattr(lib, "mm3d_heads3d_bwd" + sfx)(ptr(feat), n, f, C, ptr(w1), ptr(w2), ptr(b2), ptr(tgt), ptr(d1), ptr(d2),
                                                      ptr(dl), ptr(dfe), ptr(dw1), ptr(db1), ptr(dw2), ptr(db2), ptr(ws),
                                                      ws.numel() * 8, sp, *tail))
        torch.cuda.synchronize()
        return out, _launches() - k0

    a, na = calls(False)
    b, nb = calls(True)
    _no_device_error()
    assert na == nb
    # (the FP64 atomics of the default path may land in another order between the two calls: compare with the
    # tolerance of that reordering; the element-wise outputs are exact)
    for i, (p, q) in enumerate(zip(a, b)):
        if i in (0, 4, 5, 7):
            assert torch.equal(p, q), i
        else:
            assert rel_err(p, q) <= 1e-6, i


def test_default_mode_is_unchanged():
    """With the switch off, the InputLayer forward, the OutputLayer backward and the lift backward launch what the
    original entry points launch and give their results, and no deterministic list is built."""
    from mm2d3d_b200 import functional as F
    from mm2d3d_b200.lift import LiftIndices, lift2d
    from mm2d3d_b200.metadata import Metadata
    locs, feats = synth.make_batch("nuscenes", batch=2, seed0=4)
    locs[:, :3] //= 4  # several points per voxel
    meta = Metadata(torch.from_numpy(locs).to(DEV), 4096, 1)  # fresh: no list cached by another test
    x = torch.from_numpy(feats).to(DEV).requires_grad_(True)
    sp = _lib.stream_ptr()

    def counted(fn):
        torch.cuda.synchronize()
        k0 = _launches()
        out = fn()
        torch.cuda.synchronize()
        return out, _launches() - k0

    with _det(False):
        v, nv = counted(lambda: F.InputLayerFn.apply(x, meta, 4))
        o = F.OutputLayerFn.apply(v, meta)
        g = torch.randn_like(o)
        (gv,), ngv = counted(lambda: torch.autograd.grad(o, v, g))
        B, C, H, W = 2, 16, 60, 90
        li = LiftIndices([np.stack([np.arange(n) % H, np.arange(n) // H], 1) for n in (5000, 4000)], DEV)  # one point per pixel
        fmap = torch.randn(B, C, H, W, device=DEV, requires_grad=True)
        out = lift2d(fmap, li)
        gl = torch.randn_like(out)
        (gf,), ngf = counted(lambda: torch.autograd.grad(out, fmap, gl))
    v_ref, nv_ref = counted(lambda: check(lib.mm3d_input_fwd(ptr(x), meta.p2v_ptr, meta.npts_ptr, meta.n_points,
                                                             meta.n_voxels, 3, 4, ptr(torch.empty_like(v)), sp)))
    gv_ref = torch.empty_like(gv)
    _, ngv_ref = counted(lambda: check(lib.mm3d_output_bwd(ptr(g), meta.p2v_ptr, meta.n_points, meta.n_voxels, 3,
                                                           ptr(gv_ref), sp)))
    gf_ref = torch.zeros_like(gf)
    _, ngf_ref = counted(lambda: check(lib.mm3d_lift2d_bwd(ptr(gl), 0, B, C, H, W, *gf_ref.stride(), ptr(li.idx),
                                                           ptr(li.offsets), li.n, ptr(gf_ref), sp)))
    _no_device_error()
    assert (nv, ngv, ngf) == (nv_ref, ngv_ref, ngf_ref) == (1, 1, 1)
    assert meta._point_csr is None and not li._pixel_lists
    # (the default OutputLayer backward adds with float atomics: equal to within their reordering)
    assert rel_err(gv, gv_ref) <= 1e-6
    assert torch.equal(gf, gf_ref)  # one point per pixel: no reordering


def test_long_segments():
    """Every point in one pixel: the builder's long-segment sort (heapsort) orders 200 000 entries."""
    from mm2d3d_b200.functional import lift_csr
    from mm2d3d_b200.lift import LiftIndices, lift2d
    n, C = 200_000, 8
    li = LiftIndices([np.full((n, 2), 3, np.int64)], DEV)
    start, ent = lift_csr(li.idx, None, li.offsets, 1, 8, 8)
    _no_device_error()
    assert start[27].item() == 0 and start[28].item() == n
    assert torch.equal(ent.cpu(), torch.arange(n, dtype=torch.int32))
    fmap = torch.randn(1, C, 8, 8, device=DEV, requires_grad=True)
    g = torch.randn(n, C, device=DEV)
    with _det(True):
        gs = [torch.autograd.grad(lift2d(fmap, li), fmap, g)[0] for _ in range(2)]
    assert _same_bytes(*gs)
    # one FP32 sum of 2e5 terms: ~sqrt(n) * 2^-24 of the terms' scale off float64, i.e. ~1e-5 of the total here
    assert rel_err(gs[0][0, :, 3, 3], g.double().sum(0)) < 1e-4


def test_uncovered_ops_warn_in_deterministic_mode():
    """Ops without a deterministic form say so while the mode is on, and stay silent while it is off."""
    import warnings
    from mm2d3d_b200.unet import UNetSCN
    locs, feats = synth.make_batch("nuscenes", batch=1, seed0=5)
    keep = np.random.default_rng(0).random(len(locs)) < 0.2
    coords, x = torch.from_numpy(locs[keep]).to(DEV), torch.from_numpy(feats[keep]).to(DEV)
    for fused in (True, False):
        net = UNetSCN(in_channels=3).to(DEV)
        net.fused = fused
        for flag in (False, True):
            with _det(flag), warnings.catch_warnings(record=True) as rec:
                warnings.simplefilter("always")
                net([coords, x]).sum().backward()
            msgs = [str(w.message) for w in rec if "no deterministic form" in str(w.message)]
            assert bool(msgs) == flag, (fused, flag, msgs)
    _no_device_error()


def test_torch_flag_turns_it_on():
    from mm2d3d_b200 import scn
    from mm2d3d_b200.lift import lift2d
    prev = torch.are_deterministic_algorithms_enabled()
    fmap = torch.randn(2, 16, 60, 90, device=DEV)
    ii = _img_indices(4)
    g = torch.randn(sum(len(x) for x in ii), 16, device=DEV)

    def run():
        f = fmap.clone().requires_grad_(True)
        (gf,) = torch.autograd.grad(lift2d(f, ii), f, g)
        return gf

    with _det(None):
        try:
            torch.use_deterministic_algorithms(True, warn_only=True)
            assert scn.get_deterministic()
            torch.cuda.synchronize()
            k0 = _launches()
            a = run()
            torch.cuda.synchronize()
            k1 = _launches()
            b = run()
        finally:
            torch.use_deterministic_algorithms(prev)
    _no_device_error()
    assert _same_bytes(a, b)
    assert k1 - k0 > 2  # fwd + the pixel-list build + the segmented backward
