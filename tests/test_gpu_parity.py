"""Parity of the CUDA path (through the C ABI) against the CPU oracle on the same seeded inputs.

Bars (BASELINE.json north_star): voxel ids / level coordinates / rule tables BIT-EXACT;
FP32-mode activations and gradients within 1e-4 relative error (max-abs error over max-abs
reference, per tensor); TF32 / BF16 tensor-core modes within 1e-2.
"""
import os

import numpy as np
import pytest
import torch

from oracle import lift_oracle, scn_cpu
from oracle import scn_oracle as O
from mm2d3d_b200 import synth

pytestmark = pytest.mark.gpu

G = os.path.join(os.path.dirname(__file__), "golden")
DEV = "cuda:0"

TOL = {"fp32": 1e-4, "tf32": 1e-2, "bf16": 1e-2, "tf32x3": 1e-4}


def rel_err(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    denom = b.abs().max().item()
    return (a - b).abs().max().item() / (denom if denom > 0 else 1.0)


def _scn():
    import mm2d3d_b200.scn as scn
    return scn


def _meta(coords, spatial, levels):
    from mm2d3d_b200.metadata import Metadata
    return Metadata(torch.from_numpy(coords).to(DEV), spatial, levels)


def _cloud(seed, n=400, b=3, span=40, origin=100):
    rng = np.random.default_rng(seed)
    pts = []
    for s in range(b):
        u = rng.integers(0, span, (n, 2))
        z = (u[:, 0] // 3 + rng.integers(0, 2, n)) % span
        pts.append(np.concatenate([np.stack([u[:, 0], u[:, 1], z], 1) + origin, np.full((n, 1), s)], 1))
    return np.concatenate(pts, 0).astype(np.int64)


# ------------------------------------------------------------------------------ structure
def _check_structure(coords, spatial, levels):
    ref = O.Metadata(coords, spatial)
    meta = _meta(coords, spatial, levels)
    assert np.array_equal(meta.p2v().cpu().numpy(), ref.p2v)
    assert np.array_equal(meta.npts().cpu().numpy(), ref.npts)
    s = spatial
    for lvl in range(levels):
        assert np.array_equal(meta.coords_at(s).cpu().numpy(), ref.coords_at(s)), f"coords level {lvl}"
        assert np.array_equal(meta.nbr_table(s).cpu().numpy(), ref.nbr(s)), f"nbr level {lvl}"
        if lvl + 1 < levels:
            parent, off, child = meta.down_tables(s)
            rp, ro, nc = ref.down(s)
            assert np.array_equal(parent.cpu().numpy(), rp)
            assert np.array_equal(off.cpu().numpy(), ro)
            assert np.array_equal(child.cpu().numpy(), O.child_table(rp, ro, nc))
        s //= 2
    return meta, ref


def test_structure_a10_known_answer():
    locs = np.array([(1, 1, 1, 0), (2, 1, 1, 0), (1, 1, 1, 0), (5, 5, 5, 0), (1, 1, 1, 1), (4, 5, 5, 0)], dtype=np.int64)
    meta, _ = _check_structure(locs, 4096, 2)
    assert meta.p2v().tolist() == [0, 1, 0, 2, 3, 4]
    assert meta.coords_at(2048).tolist() == [[0, 0, 0, 0], [1, 0, 0, 0], [2, 2, 2, 0], [0, 0, 0, 1]]


def test_structure_golden_fixture():
    z = np.load(os.path.join(G, "structure_small.npz"))
    meta = _meta(z["coords"], 4096, 4)
    assert np.array_equal(meta.p2v().cpu().numpy(), z["p2v"])
    s = 4096
    for lvl in range(4):
        assert np.array_equal(meta.coords_at(s).cpu().numpy(), z[f"coords_l{lvl}"])
        assert np.array_equal(meta.nbr_table(s).cpu().numpy(), z[f"nbr_l{lvl}"])
        if lvl < 3:
            parent, off, child = meta.down_tables(s)
            assert np.array_equal(parent.cpu().numpy(), z[f"parent_l{lvl}"])
            assert np.array_equal(child.cpu().numpy(), z[f"child_l{lvl}"])
        s //= 2


@pytest.mark.parametrize("seed", [0, 1])
def test_structure_random_clouds(seed):
    _check_structure(_cloud(seed), 4096, 5)


def test_structure_edge_cases():
    # empty input
    meta = _meta(np.zeros((0, 4), np.int64), 16, 3)
    assert meta.n_voxels == 0 and meta.level(8).n == 0
    # single point; all points identical; borders of the grid (no wrap-around neighbours)
    _check_structure(np.array([[3, 3, 3, 0]], dtype=np.int64), 16, 3)
    _check_structure(np.array([[7, 7, 7, 2]] * 50, dtype=np.int64), 16, 4)
    _check_structure(np.array([[0, 0, 0, 0], [15, 15, 15, 0], [0, 0, 15, 0], [15, 0, 0, 1]], dtype=np.int64), 16, 4)
    # lazily built level (not part of the pre-built pyramid)
    coords = _cloud(4)
    ref = O.Metadata(coords, 4096)
    meta = _meta(coords, 4096, 1)
    parent, off, child = meta.down_tables(4096)
    rp, ro, nc = ref.down(4096)
    assert np.array_equal(parent.cpu().numpy(), rp) and np.array_equal(child.cpu().numpy(), O.child_table(rp, ro, nc))
    assert np.array_equal(meta.nbr_table(2048).cpu().numpy(), ref.nbr(2048))
    # out-of-range coordinates raise
    with pytest.raises(ValueError):
        _meta(np.array([[16, 0, 0, 0]], dtype=np.int64), 16, 1)
    with pytest.raises(ValueError):
        _meta(np.array([[0, -1, 0, 0]], dtype=np.int64), 16, 1)


def test_structure_nuscenes_scan_all_levels():
    """One full synthetic nuScenes-shaped scan (~34k points), all 7 levels, bit-exact."""
    locs, _ = synth.make_batch("nuscenes", batch=2, seed0=0)
    _check_structure(locs, 4096, 7)


def test_structure_full_batch_properties():
    """Batch-8 (BASELINE config 2) -- size-independent invariants instead of the CPU oracle."""
    locs, _ = synth.make_batch("nuscenes", batch=8, seed0=0)
    meta = _meta(locs, 4096, 7)
    p2v = meta.p2v().long()
    assert int(meta.npts().sum()) == locs.shape[0]
    assert int(p2v.max()) + 1 == meta.n_voxels
    # first-occurrence numbering: the running maximum of p2v grows by at most one per point
    cm = torch.cummax(p2v, 0).values
    assert int((cm[1:] - cm[:-1]).max()) <= 1 and int(p2v[0]) == 0
    # every point's voxel coordinate equals the point's coordinate
    vc = meta.coords_at(4096)
    assert torch.equal(vc[p2v], torch.from_numpy(locs).to(DEV))
    s, prev = 4096, None
    for lvl in range(7):
        lv = meta.level(s)
        if prev is not None:
            assert lv.n <= prev
        prev = lv.n
        t = meta.nbr_table(s).long()
        n = t.shape[0]
        assert torch.equal(t[:, 13], torch.arange(n, device=DEV))
        # symmetry: nbr[j][k] == i  <=>  nbr[i][26-k] == j
        for k in (0, 4, 10, 12):
            j = torch.nonzero(t[:, k] >= 0).squeeze(1)
            assert torch.equal(t[t[j, k], 26 - k], j)
        if lvl < 6:
            parent, off, child = meta.down_tables(s)
            f = torch.arange(n, device=DEV)
            assert torch.equal(child[parent.long(), off.long()].long(), f)
            assert torch.equal(meta.coords_at(s // 2)[parent.long()][:, :3], meta.coords_at(s)[:, :3] >> 1)
        s //= 2


def _natural_table(meta, kind, spatial):
    if kind == "smc":
        return meta.nbr_table(spatial).cpu().numpy()
    parent, off, child = meta.down_tables(spatial)
    if kind == "down":
        return child.cpu().numpy()
    parent, off = parent.cpu().numpy(), off.cpu().numpy()
    t = np.full((parent.shape[0], 8), -1, np.int32)
    t[np.arange(parent.shape[0]), off] = parent
    return t


@pytest.mark.parametrize("kind", ["smc", "down", "up"])
@pytest.mark.parametrize("shape,batch", [("cloud", 0), ("nuscenes", 2)])
def test_row_plan(kind, shape, batch):
    """Row plans (csrc/plan.cu) are integer work: the permutation covers every row exactly once, the
    permuted table equals the natural table under it, the tile masks are exact -- and ordering rows by
    neighbour mask leaves fewer non-empty (tile, offset) blocks than the natural order."""
    coords = _cloud(5, n=900, b=3, span=30) if shape == "cloud" else synth.make_batch("nuscenes", batch=batch)[0]
    meta = _meta(coords, 4096, 2)
    nat = _natural_table(meta, kind, 4096)  # [rows, K]
    n, K = nat.shape
    perm, mask, tbl, order = (t.cpu().numpy() for t in meta.plan_tensors(kind, 4096))
    # padding (-1) only at the end of the last tile; 2^3 tables are sorted inside chunks of 8192 consecutive rows, 3^3
    # tables with more than one chunk are pre-ordered globally (plan.cu), so their rows may leave their chunk
    T = (n + 127) // 128
    p = perm[:T * 128]
    assert np.array_equal(np.sort(p[p >= 0]), np.arange(n))
    assert np.all(p[:n] >= 0) and np.all(p[n:] == -1)
    if kind != "smc":
        for c0 in range(0, n, 8192):
            seg = p[c0:min(c0 + 8192, n)]
            assert seg.min() >= c0 and seg.max() < c0 + 8192
    want = np.full((K, T * 128), -1, np.int32)
    want[:, :n] = nat[p[:n]].T
    assert np.array_equal(tbl[:, :T * 128], want)
    blocks = (want.reshape(K, T, 128) >= 0).any(2)  # [K, T]
    want_mask = (blocks.astype(np.int64) << np.arange(K)[:, None]).sum(0)
    want_mask[want_mask == 0] = 1
    assert np.array_equal(mask[:T].astype(np.int64) & 0xFFFFFFFF, want_mask)
    # tile order: every tile once, by descending number of non-empty offsets, ties in tile order
    pc = blocks.sum(0)
    pc[pc == 0] = 1
    assert np.array_equal(order[:T], np.argsort(-pc, kind="stable"))
    if shape == "nuscenes":
        natural = np.full((K, T * 128), -1, np.int32)
        natural[:, :n] = nat.T
        nat_blocks = (natural.reshape(K, T, 128) >= 0).any(2).sum()
        assert blocks.sum() < (0.7 if kind != "down" else 0.95) * nat_blocks, (kind, blocks.sum(), nat_blocks)
    # deterministic: a second build gives the same plan
    meta2 = _meta(coords, 4096, 2)
    perm2, mask2, tbl2, _ = (t.cpu().numpy() for t in meta2.plan_tensors(kind, 4096))
    assert np.array_equal(perm2[:T * 128], p) and np.array_equal(mask2[:T], mask[:T])


def test_row_plan_global_preorder(monkeypatch):
    """3^3 tables with more than one chunk of 8192 rows are pre-ordered globally before the chunk sort (plan.cu):
    fewer non-empty (tile, offset) blocks than the chunk-only order, the same plan on every build, and convolution
    results that do not depend on the order (up to the FP32 summation order inside a row)."""
    from mm2d3d_b200 import functional as F
    coords = synth.make_batch("nuscenes", batch=2)[0]

    def build():
        meta = _meta(coords, 4096, 2)
        perm, mask, tbl, order = (t.cpu().numpy() for t in meta.plan_tensors("smc", 4096))
        return meta, perm, mask

    def blocks(mask, n):
        m = mask[:(n + 127) // 128].astype(np.int64) & 0xFFFFFFFF
        return int(sum(((m >> k) & 1).sum() for k in range(27)))

    meta_a, perm_a, mask_a = build()
    n = meta_a.nbr_table(4096).shape[0]
    assert n > 3 * 8192
    meta_a2, perm_a2, mask_a2 = build()
    T = (n + 127) // 128  # (the buffers are sized for a capacity: what lies behind the last tile is not written)
    assert np.array_equal(perm_a[:T * 128], perm_a2[:T * 128]) and np.array_equal(mask_a[:T], mask_a2[:T])  # deterministic
    monkeypatch.setenv("MM3D_PLAN_NO_PREORDER", "1")
    meta_b, perm_b, mask_b = build()
    monkeypatch.delenv("MM3D_PLAN_NO_PREORDER")
    assert blocks(mask_a, n) < 0.9 * blocks(mask_b, n), (blocks(mask_a, n), blocks(mask_b, n))
    torch.manual_seed(3)
    x = torch.randn(n, 32, device=DEV)
    w = torch.randn(27, 1, 32, 48, device=DEV) / 32 ** 0.5
    ya = F.TableConvFn.apply(x, w, meta_a, "smc", 4096, "tf32")
    yb = F.TableConvFn.apply(x, w, meta_b, "smc", 4096, "tf32")
    assert rel_err(ya, yb) < 1e-5
    _no_device_error()


# ------------------------------------------------------------------------------ single ops
def test_io_layers():
    from mm2d3d_b200 import functional as F
    coords = _cloud(7, n=500, b=2, span=12)
    ref = O.Metadata(coords, 4096)
    meta = _meta(coords, 4096, 1)
    torch.manual_seed(0)
    for c, mode in ((3, 4), (1, 4), (16, 3)):
        feats = torch.randn(coords.shape[0], c)
        x_ref = feats.clone().requires_grad_(True)
        x = feats.to(DEV).requires_grad_(True)
        v_ref = O.input_layer(ref, x_ref, mode)
        v = F.InputLayerFn.apply(x, meta, mode)
        assert rel_err(v, v_ref) < 1e-6
        o_ref = O.output_layer(ref, v_ref)
        o = F.OutputLayerFn.apply(v, meta)
        assert rel_err(o, o_ref) < 1e-6
        g = torch.randn_like(o_ref)
        (gx_ref,) = torch.autograd.grad(o_ref, x_ref, g)
        (gx,) = torch.autograd.grad(o, x, g.to(DEV))
        assert rel_err(gx, gx_ref) < 1e-5


CONV_SHAPES = [(3, 16), (16, 16), (32, 16), (48, 48), (64, 96), (112, 112), (192, 96), (20, 7)]


def _no_device_error():
    from mm2d3d_b200 import _lib
    torch.cuda.synchronize()
    assert _lib.lib.mm3d_take_device_error() == 0, "a kernel reported a pipeline time-out"


@pytest.mark.parametrize("mode", ["fp32", "tf32", "tf32x3", "bf16"])
@pytest.mark.parametrize("kind", ["smc", "down", "up"])
def test_conv_fwd_bwd(kind, mode):
    from mm2d3d_b200 import functional as F
    coords = _cloud(11, n=700, b=2, span=24)
    ref = O.Metadata(coords, 4096)
    meta = _meta(coords, 4096, 2)
    torch.manual_seed(1)
    for c_in, c_out in CONV_SHAPES:
        K = 27 if kind == "smc" else 8
        if kind == "up":
            n_in = ref.down(4096)[2]
            spatial_in = 2048
        else:
            n_in = ref.npts.shape[0]
            spatial_in = 4096
        xr = torch.randn(n_in, c_in, requires_grad=True)
        wr = (torch.randn(K, 1, c_in, c_out) / (c_in ** 0.5)).requires_grad_(True)
        if kind == "smc":
            yr = O.submanifold_conv(ref, 4096, xr, wr)
        elif kind == "down":
            yr = O.conv_down(ref, 4096, xr, wr)
        else:
            yr = O.deconv_up(ref, 4096, xr, wr)
        x = xr.detach().to(DEV).requires_grad_(True)
        w = wr.detach().to(DEV).requires_grad_(True)
        y = F.TableConvFn.apply(x, w, meta, kind, spatial_in, mode)
        assert y.shape == yr.shape
        tol = TOL[mode]
        assert rel_err(y, yr) < tol, (kind, c_in, c_out, "fwd", rel_err(y, yr))
        g = torch.randn_like(yr)
        gxr, gwr = torch.autograd.grad(yr, (xr, wr), g)
        gx, gw = torch.autograd.grad(y, (x, w), g.to(DEV))
        assert rel_err(gx, gxr) < tol, (kind, c_in, c_out, "dgrad", rel_err(gx, gxr))
        assert rel_err(gw, gwr) < tol, (kind, c_in, c_out, "wgrad", rel_err(gw, gwr))
    _no_device_error()


@pytest.mark.parametrize("c", [16, 48, 112, 192, 6])
def test_bnrelu(c):
    from mm2d3d_b200 import functional as F
    torch.manual_seed(2)
    for n, leak, training in ((1000, 0.0, True), (37, 0.333, True), (500, 0.0, False), (1, 0.0, True)):
        xr = (torch.randn(n, c) * 2 + 0.5).requires_grad_(True)
        gr = (1 + 0.2 * torch.randn(c)).requires_grad_(True)
        br = (0.1 * torch.randn(c)).requires_grad_(True)
        rm_r, rv_r = torch.randn(c) * 0.1, torch.rand(c) + 0.5
        rm, rv = rm_r.clone().to(DEV), rv_r.clone().to(DEV)
        yr = O.batchnorm_relu(xr, gr, br, rm_r, rv_r, 1e-4, 0.9, training, leak)
        x = xr.detach().to(DEV).requires_grad_(True)
        g_ = gr.detach().to(DEV).requires_grad_(True)
        b_ = br.detach().to(DEV).requires_grad_(True)
        y = F.BatchNormReLUFn.apply(x, g_, b_, rm, rv, 1e-4, 0.9, leak, training)
        assert rel_err(y, yr) < 1e-4
        if n > 1:
            assert rel_err(rm, rm_r) < 1e-5 and rel_err(rv, rv_r) < 1e-5
        go = torch.randn_like(yr)
        ref_grads = torch.autograd.grad(yr, (xr, gr, br), go)
        grads = torch.autograd.grad(y, (x, g_, b_), go.to(DEV))
        if n > 1:
            for a, b in zip(grads, ref_grads):
                assert rel_err(a, b) < 1e-4


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.bfloat16])
def test_lift2d_reference_fixture(dtype):
    """lift_ref.npz comes from the reference's own L2G_classifier_2D (tests/golden/make_golden.py)."""
    from mm2d3d_b200.lift import LiftIndices, lift2d
    z = np.load(os.path.join(G, "lift_ref.npz"))
    offs = np.concatenate([[0], np.cumsum(z["counts"])])
    idx = [z["idx"][offs[i]:offs[i + 1]] for i in range(len(z["counts"]))]
    fmap = torch.from_numpy(z["fmap"]).to(DEV, dtype).requires_grad_(True)
    out = lift2d(fmap, idx)
    want = torch.from_numpy(z["lifted"]).to(dtype)
    assert torch.equal(out.detach().cpu(), want)  # a gather is exact in every dtype
    (g,) = torch.autograd.grad(out, fmap, torch.from_numpy(z["grad_out"]).to(DEV, dtype))
    tol = 1e-6 if dtype == torch.float32 else 2e-2
    assert rel_err(g, torch.from_numpy(z["grad_fmap"])) < tol
    # pre-uploaded indices give the same result
    li = LiftIndices(idx, DEV)
    assert torch.equal(lift2d(fmap, li), out)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_lift2d_channels_last_map(dtype):
    """A channels-last map (what cuDNN produces for the 2D network) is gathered in place through its strides; results
    and gradients equal those of the contiguous map, and the gradient comes back in the map's memory format."""
    from mm2d3d_b200.lift import lift2d
    torch.manual_seed(4)
    fmap = torch.randn(3, 6, 45, 80, device=DEV).to(dtype)
    idx = synth.make_img_indices([700, 0, 300], 45, 80, seed=3)
    a = fmap.clone().requires_grad_(True)
    b = fmap.clone().contiguous(memory_format=torch.channels_last).requires_grad_(True)
    ra, rb = lift2d(a, idx), lift2d(b, idx)
    assert torch.equal(ra, rb)
    assert torch.equal(ra.detach().cpu(), lift_oracle.lift2d(fmap.cpu(), idx))
    g = torch.randn_like(ra)
    (ga,) = torch.autograd.grad(ra, a, g)
    (gb,) = torch.autograd.grad(rb, b, g)
    assert gb.is_contiguous(memory_format=torch.channels_last)
    assert rel_err(gb, ga) < (1e-6 if dtype == torch.float32 else 2e-2)


def test_lift2d_benchmark_shape():
    from mm2d3d_b200.lift import lift2d
    torch.manual_seed(3)
    fmap = torch.randn(8, 6, 225, 400)
    idx = synth.make_img_indices([3000] * 8, seed=1)
    idx[3] = synth.make_img_indices([3000], seed=2, window=50)[0]  # duplicate-heavy sample
    a = fmap.clone().requires_grad_(True)
    b = fmap.clone().to(DEV).requires_grad_(True)
    ra = lift_oracle.lift2d(a, idx)
    rb = lift2d(b, idx)
    assert torch.equal(rb.detach().cpu(), ra.detach())
    g = torch.randn_like(ra)
    (ga,) = torch.autograd.grad(ra, a, g)
    (gb,) = torch.autograd.grad(rb, b, g.to(DEV))
    assert rel_err(gb, ga) < 1e-6


@pytest.mark.parametrize("dtype,channels_last", [(torch.float32, False), (torch.float32, True), (torch.bfloat16, True)])
def test_lift2d_bilinear_matches_oracle_and_grid_sample(dtype, channels_last):
    """Bilinear lift (an extension of the reference's integer gather; floating-point kernel, FP32 arithmetic): against
    the four-tap oracle, which tests/test_oracle.py pins to F.grid_sample, and against torch's own CUDA grid_sample;
    bar 1e-5 in FP32 (bf16: the output rounding, 1e-2).  Gradient of the map against autograd of the oracle."""
    import torch.nn.functional as F
    from mm2d3d_b200.lift import lift2d, lift2d_bilinear
    torch.manual_seed(9)
    B, C, H, W = 3, 8, 45, 80
    fmap = torch.randn(B, C, H, W, device=DEV).to(dtype)
    if channels_last:
        fmap = fmap.contiguous(memory_format=torch.channels_last)
    rng = np.random.default_rng(2)
    coords = [np.stack([rng.uniform(-1.5, H + 0.5, n), rng.uniform(-1.5, W + 0.5, n)], 1).astype(np.float32) for n in (900, 0, 400)]
    coords[0][:6] = [[0, 0], [H - 1, W - 1], [3, 4], [H - 1, 2.5], [-1, -1], [H, W]]
    x = fmap.clone().requires_grad_(True)
    out = lift2d_bilinear(x, coords)
    xr = fmap.detach().cpu().float().contiguous().requires_grad_(True)
    want = lift_oracle.lift2d_bilinear(xr, coords)
    tol = 1e-5 if dtype == torch.float32 else 1e-2
    assert out.dtype == dtype and rel_err(out, want) < tol
    if dtype == torch.float32:
        for i, rc in enumerate(coords):
            if len(rc) == 0:
                continue
            rc = torch.from_numpy(rc).to(DEV)
            grid = torch.stack([2 * rc[:, 1] / (W - 1) - 1, 2 * rc[:, 0] / (H - 1) - 1], 1)[None, :, None, :]
            ref = F.grid_sample(fmap[i:i + 1], grid, mode="bilinear", padding_mode="zeros", align_corners=True)[0, :, :, 0].t()
            lo = sum(len(c) for c in coords[:i])
            assert rel_err(out[lo:lo + len(rc)], ref) < 1e-5
    g = torch.randn(out.shape, device=DEV).to(dtype)
    (gx,) = torch.autograd.grad(out, x, g)
    (gr,) = torch.autograd.grad(want, xr, g.cpu().float())
    assert gx.is_contiguous(memory_format=torch.channels_last if channels_last else torch.contiguous_format)
    assert rel_err(gx, gr) < (1e-5 if dtype == torch.float32 else 3e-2)
    # at integer pixels the blend degenerates to the reference's gather, bit for bit
    ints = synth.make_img_indices([500, 0, 300], H, W, seed=5)
    assert torch.equal(lift2d_bilinear(fmap, [a.astype(np.float32) for a in ints]), lift2d(fmap, ints))


# ------------------------------------------------------------------------------ whole network
def rel_l2(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return ((a - b).norm() / max(b.norm().item(), 1e-300)).item()


def _run_pair(net_ref32, net, coords, feats, tol):
    """Whole-network parity.  Truth = the oracle in FLOAT64.  The forward output must be within
    `tol` (max-abs relative).  Gradients of a randomly initialised 60-layer BN/ReLU network are
    ill-conditioned in FP32 -- the FP32 CPU oracle itself is ~3e-3 (relative L2) away from its own
    FP64 run -- so the gradient bar is: per tensor, relative-L2 error <= max(tol, 3 x the FP32 CPU
    oracle's error on that tensor).  The per-op tests above hold the strict per-op tolerance."""
    import copy
    net_ref64 = copy.deepcopy(net_ref32).double()
    g = None
    runs = {}
    for tag, ref, dt in (("f64", net_ref64, torch.float64), ("f32", net_ref32, torch.float32)):
        xr = feats.clone().to(dt).requires_grad_(True)
        out_r = ref([coords, xr])
        if g is None:
            g = torch.randn_like(out_r)
        pr = dict(ref.named_parameters())
        gr = torch.autograd.grad(out_r, [xr] + list(pr.values()), g.to(dt))
        runs[tag] = (out_r, dict(zip(["feats"] + list(pr), gr)))
    x = feats.clone().to(DEV).requires_grad_(True)
    out = net([coords.to(DEV), x])
    out64, g64 = runs["f64"]
    _, g32 = runs["f32"]
    assert out.shape == out64.shape
    assert rel_err(out, out64) < tol, ("forward", rel_err(out, out64))
    p = dict(net.named_parameters())
    names = list(g64)
    gg = torch.autograd.grad(out, [x] + [p[k] for k in names[1:]], g.float().to(DEV))
    worst = (0.0, "")
    for name, a in zip(names, gg):
        e_gpu, e_cpu = rel_l2(a, g64[name]), rel_l2(g32[name], g64[name])
        worst = max(worst, (e_gpu / max(e_cpu, 1e-12), name))
        assert e_gpu <= max(tol, 3 * e_cpu), (name, e_gpu, e_cpu)
    for (k, a), (_, b) in zip(net.named_buffers(), net_ref64.named_buffers()):
        assert rel_err(a, b) < max(tol, 1e-4), k
    return worst


def test_unet_small_golden_fixture():
    from mm2d3d_b200.unet import UNetSCN
    z = np.load(os.path.join(G, "unet_small.npz"))
    net = UNetSCN(in_channels=3, m=4, num_planes=4, full_scale=64).to(DEV)
    sd = {k[len("param:"):]: torch.from_numpy(z[k]).float() for k in z.files if k.startswith("param:")}
    net.load_state_dict(sd, strict=False)
    x = torch.from_numpy(z["feats"]).to(DEV).requires_grad_(True)
    out = net([torch.from_numpy(z["coords"]).to(DEV), x])
    assert rel_err(out, torch.from_numpy(z["out"])) < 1e-4
    params = dict(net.named_parameters())
    grads = torch.autograd.grad(out, [x] + list(params.values()), torch.from_numpy(z["grad_out"]).float().to(DEV))
    assert rel_err(grads[0], torch.from_numpy(z["grad_feats"])) < 5e-4
    for (name, _), g in zip(params.items(), grads[1:]):
        assert rel_err(g, torch.from_numpy(z["grad:" + name])) < 5e-4, name
    for name, b in net.named_buffers():
        assert rel_err(b, torch.from_numpy(z["buffer_after:" + name])) < 1e-4, name


def test_unetscn_full_config_one_scan():
    """BASELINE config 1: UNetSCN(m=16, 7 planes, full_scale 4096) on one nuScenes-shaped scan."""
    from mm2d3d_b200.unet import UNetSCN
    torch.manual_seed(5)
    locs, feats = synth.make_batch("nuscenes", batch=1, seed0=3)
    net_ref = UNetSCN(in_channels=3, backend=scn_cpu)
    net = UNetSCN(in_channels=3).to(DEV)
    net.load_state_dict(net_ref.state_dict())
    worst = _run_pair(net_ref, net, torch.from_numpy(locs), torch.from_numpy(feats), TOL["fp32"])
    print("worst gradient error relative to the FP32 CPU oracle's own error", worst)


def _emulate_tf32_convs():
    """Context manager: the CPU oracle's convolutions with both operands of forward, dgrad AND wgrad rounded
    to TF32 (round-to-nearest, ties away), FP32 accumulate -- the arithmetic of the tcgen05 TF32 mode (activations
    and gradients are rounded where they are produced, weights inside the kernels)."""
    import contextlib

    def rna(t):
        return ((t.contiguous().view(torch.int32) + 0x1000) & ~0x1FFF).view(torch.float32)

    class Emul(torch.autograd.Function):
        @staticmethod
        def forward(ctx, x, w, fn):
            ctx.fn = fn
            ctx.save_for_backward(x, w)
            with torch.no_grad():
                return fn(rna(x), rna(w))

        @staticmethod
        def backward(ctx, g):
            x, w = ctx.saved_tensors
            with torch.enable_grad():
                xx = x.detach().requires_grad_(True)
                (gx,) = torch.autograd.grad(ctx.fn(xx, rna(w.detach())), xx, rna(g))
                ww = w.detach().requires_grad_(True)
                (gw,) = torch.autograd.grad(ctx.fn(rna(x.detach()), ww), ww, rna(g))
            return gx, gw, None

    @contextlib.contextmanager
    def cm():
        orig = (O.submanifold_conv, O.conv_down, O.deconv_up)

        def wrap(f):
            def g(meta, s, x, w):
                if x.dtype != torch.float32 or x.shape[1] % 4:
                    return f(meta, s, x, w)
                return Emul.apply(x, w, lambda a, b: f(meta, s, a, b))
            return g
        O.submanifold_conv, O.conv_down, O.deconv_up = (wrap(f) for f in orig)
        try:
            yield
        finally:
            O.submanifold_conv, O.conv_down, O.deconv_up = orig
    return cm()


def test_unetscn_full_config_tf32():
    """Same network in the tcgen05 TF32 mode.  Forward: 1e-2 (north_star) against the FP64 oracle.
    Whole-network GRADIENTS of the FREE-RUNNING network (ReLU gates and batch statistics recomputed from
    the perturbed activations) are dominated by gate flips: the CPU oracle with its convolution operands
    rounded to TF32 is itself several 1e-2 (relative L2) away from FP64 on this randomly initialised
    60-layer BN/ReLU network, so here the kernels are held to: no worse than 2x the error of that
    TF32-emulating oracle, per tensor, and gradient direction preserved (cosine > 0.97).  north_star's
    1e-2 on gradients is held directly, per tensor, by test_unetscn_gradients_with_frozen_gates (gates and
    statistics pinned to the FP64 oracle's) and per op by test_conv_fwd_bwd / test_tf32_edge_sizes."""
    import copy

    import mm2d3d_b200.scn as scn
    from mm2d3d_b200.unet import UNetSCN
    torch.manual_seed(6)
    locs, feats = synth.make_batch("nuscenes", batch=1, seed0=4)
    coords, feats = torch.from_numpy(locs), torch.from_numpy(feats)
    net_ref = UNetSCN(in_channels=3, backend=scn_cpu)
    net = UNetSCN(in_channels=3).to(DEV)
    net.load_state_dict(net_ref.state_dict())
    net64 = copy.deepcopy(net_ref).double()

    def run(ref, dt, g=None):
        xr = feats.clone().to(dt).requires_grad_(True)
        out = ref([coords, xr])
        g = torch.randn_like(out) if g is None else g.to(dt)
        pr = dict(ref.named_parameters())
        gr = torch.autograd.grad(out, [xr] + list(pr.values()), g)
        return out, dict(zip(["feats"] + list(pr), gr)), g

    out64, g64, g = run(net64, torch.float64)
    with _emulate_tf32_convs():
        _, gemu, _ = run(net_ref, torch.float32, g)
    scn.set_conv_mode("tf32")
    try:
        x = feats.clone().to(DEV).requires_grad_(True)
        out = net([coords.to(DEV), x])
        p = dict(net.named_parameters())
        names = list(g64)
        gg = torch.autograd.grad(out, [x] + [p[k] for k in names[1:]], g.float().to(DEV))
    finally:
        scn.set_conv_mode("fp32")
    _no_device_error()
    assert rel_err(out, out64) < TOL["tf32"], ("forward", rel_err(out, out64))
    worst = 0.0
    for name, a in zip(names, gg):
        e_gpu, e_emu = rel_l2(a, g64[name]), rel_l2(gemu[name], g64[name])
        a64, b64 = a.detach().double().cpu().flatten(), g64[name].flatten()
        cos = float(torch.dot(a64, b64) / (a64.norm() * b64.norm()).clamp_min(1e-300))
        worst = max(worst, e_gpu)
        print(f"[tf32 free-running] d {name:44s} rel-L2 {e_gpu:.2e} (TF32-emulating CPU oracle {e_emu:.2e})  cosine {cos:.5f}")
        assert e_gpu <= max(TOL["tf32"], 2.0 * e_emu), (name, e_gpu, e_emu)
        assert cos > 0.97, (name, cos)
    print("worst whole-network gradient rel-L2 error in TF32 mode (free-running gates and statistics)", worst)


def test_module_surface_matches_reference_usage():
    """The call pattern of 3d_net/scn_unet.py:129-143 (its only 'test'): b=2, n=100 random coords."""
    from mm2d3d_b200.unet import UNetSCN
    b, n = 2, 100
    coords = torch.randint(4096, [b, n, 3])
    batch_idxs = torch.arange(b).reshape(b, 1, 1).repeat(1, n, 1)
    coords = torch.cat([coords, batch_idxs], 2).reshape(-1, 4)
    feats = torch.rand(b * n, 3)
    net = UNetSCN(3).cuda()
    out = net([coords, feats.cuda()])  # coords stay on the CPU as in the reference
    assert out.shape == (200, 16) and out.is_cuda
    # eval mode uses running statistics and does not touch them
    net.eval()
    before = net.layer4.running_mean.clone()
    net([coords, feats.cuda()])
    assert torch.equal(before, net.layer4.running_mean)
    # autocast does not change the 3D branch (FP32 inside, SURVEY A.11)
    net.train()
    with torch.autocast("cuda", dtype=torch.float16):
        out16 = net([coords, feats.cuda()])
    assert out16.dtype == torch.float32


def _line_cloud(n_vox, seed):
    """`n_vox` distinct voxels along a jagged line (every voxel has neighbours, some have children siblings)."""
    rng = np.random.default_rng(seed)
    x = np.arange(n_vox) // 3 + 10
    y = (np.arange(n_vox) % 3) + 20 + (rng.integers(0, 2, n_vox) * (np.arange(n_vox) % 7 == 0))
    z = np.full(n_vox, 30) + (np.arange(n_vox) % 3 == 2)
    c = np.stack([x, y, z, np.zeros(n_vox, np.int64)], 1).astype(np.int64)
    return np.unique(c, axis=0)


@pytest.mark.parametrize("n_vox", [1, 2, 127, 128, 129, 1000, 8191, 8192, 8193, 20000])
def test_tf32_edge_sizes(n_vox):
    """Row counts around the tile (128) and plan-chunk (8192) boundaries, single rows, ragged tails: the
    tensor-core kernels (plans, block-sparse K, wgrad groups) against the FP32 kernels, all three layer types."""
    from mm2d3d_b200 import functional as F
    coords = _line_cloud(n_vox, n_vox)
    assert coords[:, 0].max() < 8192
    meta = _meta(coords, 8192, 2)
    torch.manual_seed(n_vox)
    for kind, c_in, c_out in (("smc", 16, 32), ("smc", 96, 48), ("down", 32, 48), ("up", 48, 32)):
        spatial_in = 4096 if kind == "up" else 8192
        fwd_t, _, _ = F.conv_tables(meta, kind, spatial_in)
        x = torch.randn(fwd_t.n_in, c_in, device=DEV)
        w = torch.randn(fwd_t.K, 1, c_in, c_out, device=DEV) / (c_in ** 0.5)
        g = torch.randn(fwd_t.n_out, c_out, device=DEV)
        res = {}
        for mode in ("fp32", "tf32"):
            xx, ww = x.clone().requires_grad_(True), w.clone().requires_grad_(True)
            y = F.TableConvFn.apply(xx, ww, meta, kind, spatial_in, mode)
            gx, gw = torch.autograd.grad(y, (xx, ww), g)
            res[mode] = (y, gx, gw)
        for a, b, what in zip(res["tf32"], res["fp32"], ("fwd", "dgrad", "wgrad")):
            assert rel_err(a, b) < 1e-2, (n_vox, kind, what, rel_err(a, b))
    _no_device_error()


def test_tf32_forward_is_bit_reproducible():
    """Forward and dgrad of the tensor-core path do not depend on run-to-run scheduling (no atomics, fixed
    accumulation order per output row)."""
    from mm2d3d_b200 import functional as F
    locs, _ = synth.make_batch("nuscenes", batch=2, seed0=3)
    torch.manual_seed(5)
    outs = []
    for _ in range(2):
        meta = _meta(locs, 4096, 2)
        t, _, _ = F.conv_tables(meta, "smc", 4096)
        g = torch.Generator(device=DEV).manual_seed(1)
        x = torch.randn(t.n_in, 32, device=DEV, generator=g).requires_grad_(True)
        w = torch.randn(27, 1, 32, 48, device=DEV, generator=g)
        y = F.TableConvFn.apply(x, w, meta, "smc", 4096, "tf32")
        gx, = torch.autograd.grad(y, x, torch.ones_like(y))
        outs.append((y.detach().clone(), gx.clone()))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])


@pytest.mark.parametrize("kind,c_in,c_out", [("smc", 16, 16), ("smc", 64, 32), ("down", 16, 32), ("up", 32, 16)])
def test_tf32_matches_fp32_kernels_at_bench_size(kind, c_in, c_out):
    """Batch-8 nuScenes-shaped structure (BASELINE configs[1] size, ~238k rows, 1860 tiles): every
    persistent CTA of the tcgen05 kernels walks several tiles (ring wrap-around, double-buffered
    accumulators, G-buffer reuse).  The CPU oracle is too slow here, so the FP32 SIMT kernels --
    themselves pinned against the oracle at small sizes -- are the reference; bar 1e-2."""
    from mm2d3d_b200 import functional as F
    locs, _ = synth.make_batch("nuscenes", batch=8, seed0=0)
    meta = _meta(locs, 4096, 2)
    fwd_t, _, _ = F.conv_tables(meta, kind, 2048 if kind == "up" else 4096)
    torch.manual_seed(3)
    K = fwd_t.K
    x = torch.randn(fwd_t.n_in, c_in, device=DEV)
    w = torch.randn(K, 1, c_in, c_out, device=DEV) / (c_in ** 0.5)
    g = torch.randn(fwd_t.n_out, c_out, device=DEV)
    res = {}
    for mode in ("fp32", "tf32"):
        xx, ww = x.clone().requires_grad_(True), w.clone().requires_grad_(True)
        y = F.TableConvFn.apply(xx, ww, meta, kind, 2048 if kind == "up" else 4096, mode)
        gx, gw = torch.autograd.grad(y, (xx, ww), g)
        res[mode] = (y, gx, gw)
    for a, b, what in zip(res["tf32"], res["fp32"], ("fwd", "dgrad", "wgrad")):
        assert rel_err(a, b) < 1e-2, (kind, c_in, c_out, what, rel_err(a, b))
    _no_device_error()


@pytest.mark.parametrize("mode", ["fp32", "tf32", "tf32x3", "bf16"])
def test_fused_executor_matches_module_path(mode):
    """UNetSCN.forward defaults to the native whole-network executor (csrc/unet_exec.cu); it issues
    the same kernels as the module-by-module path, so outputs, every gradient and the BN running
    statistics must agree to FP32 round-off (BN / wgrad reductions use atomics)."""
    import copy

    import mm2d3d_b200.scn as scn
    from mm2d3d_b200.unet import UNetSCN
    torch.manual_seed(9)
    locs, feats = synth.make_batch("nuscenes", batch=2, seed0=5)
    coords, feats = torch.from_numpy(locs).to(DEV), torch.from_numpy(feats).to(DEV)
    net_a = UNetSCN(in_channels=3).to(DEV)
    net_b = copy.deepcopy(net_a)
    net_b.fused = False
    g = torch.randn(locs.shape[0], 16, device=DEV)
    scn.set_conv_mode(mode)
    try:
        res = []
        for net in (net_a, net_b):
            x = feats.clone().requires_grad_(True)
            out = net([coords, x])
            grads = torch.autograd.grad(out, [x] + list(net.parameters()), g)
            res.append((out, grads, [b.clone() for b in net.buffers()]))
    finally:
        scn.set_conv_mode("fp32")
    _no_device_error()
    # (a last-bit difference of an FP32 value can move its TF32 / BF16 rounding by a whole unit of that format)
    tol = {"tf32": 1e-3, "bf16": 1e-2}.get(mode, 1e-5)
    assert rel_err(res[0][0], res[1][0]) < tol
    for a, b in zip(res[0][1], res[1][1]):
        assert rel_l2(a, b) < 2e-2  # same kernels; atomic reduction order noise, amplified by the deep BN/ReLU net
    for a, b in zip(res[0][2], res[1][2]):
        assert rel_err(a, b) < tol
    # eval mode through the executor
    net_a.eval(); net_b.eval()
    with torch.no_grad():
        assert rel_err(net_a([coords, feats]), net_b([coords, feats])) < tol


# ------------------------------------------------------------------------------ points -> voxel coordinates
def test_scale_points_reference_fixture():
    """mm3d_scale_points against tests/golden/augment_ref.npz, which the reference's own augment_and_scale_3d +
    integer cast + range filter produced (make_golden.py).  Integer work: min_value, the no-augmentation sample
    and everything downstream of the rotation are bit-exact; the rotation itself is a float32 BLAS dot product in
    the reference whose rounding numpy does not pin, so for augmented samples a coordinate may differ by one voxel
    where the float value sits on an integer boundary -- at most 1e-4 of the points, never by more than 1."""
    from mm2d3d_b200.augment import scale_points
    z = np.load(os.path.join(G, "augment_ref.npz"))
    pts = torch.from_numpy(z["points"]).to(DEV)
    offs = z["offsets"]
    u = z["u"] * z["transl"][:, None]  # samples without translation: zero draws = zero offset
    for full_scale, want_c, want_k, transl_u in ((int(z["full_scale"]), z["coords"], z["keep"], u),
                                                  (int(z["small_full_scale"]), z["coords_small"], z["keep_small"], None)):
        coords, keep, mn, off = scale_points(pts, offs, z["rot"], transl_u, float(z["scale"]), full_scale)
        coords, keep = coords.cpu().numpy(), keep.cpu().numpy()
        assert np.array_equal(coords[:, 3], np.repeat(np.arange(len(offs) - 1), np.diff(offs)))
        for i in range(len(offs) - 1):
            sl = slice(offs[i], offs[i + 1])
            d = np.abs(coords[sl, :3] - want_c[sl])
            identity = np.array_equal(z["rot"][i], np.eye(3, dtype=np.float32))
            if identity:
                assert d.max() == 0 and np.array_equal(keep[sl], want_k[sl])
                assert np.array_equal(mn[i].cpu().numpy(), z["min_value"][i])
            else:
                assert d.max() <= 1 and (d > 0).any(1).mean() <= 1e-4, (i, d.max(), (d > 0).any(1).mean())
                assert (keep[sl] != want_k[sl]).mean() <= 1e-4
                assert np.allclose(mn[i].cpu().numpy(), z["min_value"][i], rtol=1e-6, atol=1e-3)
            if transl_u is not None:
                assert np.allclose(off[i].cpu().numpy(), z["offset"][i], rtol=1e-6, atol=1e-3)
    # the filtered coordinates feed InputLayer directly
    meta = _meta(coords[keep], 4096, 2)
    ref = O.Metadata(coords[keep], 4096)
    assert np.array_equal(meta.p2v().cpu().numpy(), ref.p2v)


def _same_structure(a, b, levels, spatial):
    """Two Metadata objects hold bit-identical structures (point map, rows, tables of every level)."""
    assert a.n_points == b.n_points and a.n_voxels == b.n_voxels
    assert torch.equal(a.p2v(), b.p2v()) and torch.equal(a.npts(), b.npts())
    s = spatial
    for l in range(levels):
        assert torch.equal(a.coords_at(s), b.coords_at(s))
        assert torch.equal(a.nbr_table(s), b.nbr_table(s))
        if l + 1 < levels:
            for x, y in zip(a.down_tables(s), b.down_tables(s)):
                assert torch.equal(x, y)
        s //= 2


def test_voxelize_points_matches_scale_then_voxelize():
    """mm3d_voxelize_points (SURVEY 8(f).1: raw float points straight into the voxel hash) against the two-step path
    it replaces, mm3d_scale_points -> coords[keep] -> mm3d_voxelize, itself pinned by the reference-produced fixture
    above.  Integer work: every output is bit-exact -- point -> voxel map, voxel rows of all levels, 3^3 and 2^3
    tables, min_value / offset by-products; and when points fall outside the receptive field (the small grid of the
    fixture), the keep mask and the structure of the survivors."""
    from mm2d3d_b200.augment import scale_points, voxelize_points
    from mm2d3d_b200.metadata import Metadata
    z = np.load(os.path.join(G, "augment_ref.npz"))
    pts = torch.from_numpy(z["points"]).to(DEV)
    offs = z["offsets"]
    u = z["u"] * z["transl"][:, None]
    for full_scale, transl_u, levels in ((int(z["full_scale"]), u, 4), (int(z["small_full_scale"]), None, 3)):
        coords, keep, mn, off = scale_points(pts, offs, z["rot"], transl_u, float(z["scale"]), full_scale)
        ref = Metadata(coords[keep], full_scale, levels)
        ps = voxelize_points(pts, offs, z["rot"], transl_u, float(z["scale"]), full_scale, prebuild_levels=levels)
        meta, kept = ps.resolve()
        if bool(keep.all()):
            assert kept is None and not meta.dropped
        else:
            assert kept is not None and torch.equal(kept, keep)
        assert torch.equal(ps.min_value, mn) and torch.equal(ps.offset, off)
        _same_structure(meta, ref, levels, full_scale)
    assert not bool(keep.all()), "the fixture's small grid must drop points (exercises the rebuild)"
    # full nuScenes-shaped batch, all 7 levels, deferred synchronisation, with and without augmentation
    from mm2d3d_b200.augment import draw_augmentation
    scans = [synth.raycast_points("nuscenes", seed) for seed in range(3)]
    offs = np.concatenate([[0], np.cumsum([len(p) for p in scans])]).astype(np.int64)
    pts = torch.from_numpy(np.concatenate(scans, 0)).to(DEV)
    rng = np.random.RandomState(7)
    draws = [draw_augmentation(noisy_rot=0.03, flip_y=0.5, rot_z=6.2831, transl=True, rng=rng) for _ in scans]
    for rot, tu in ((np.stack([np.eye(3, dtype=np.float32)] * 3), None),
                    (np.stack([d[0] for d in draws]), np.stack([d[1] for d in draws]))):
        coords, keep, mn, off = scale_points(pts, offs, rot, tu, 20.0, 4096)
        assert bool(keep.all())
        ref = Metadata(coords, 4096, 7)
        ps = voxelize_points(pts, offs, rot, tu, 20.0, 4096, prebuild_levels=7, plans=True, defer_sync=True)
        meta, kept = ps.resolve()
        assert kept is None
        assert torch.equal(ps.min_value, mn) and torch.equal(ps.offset, off)
        _same_structure(meta, ref, 7, 4096)
        if tu is None:  # without augmentation: the synthetic generator's own (float64, numpy) transform
            want = np.concatenate([np.concatenate([synth.scan_coords("nuscenes", s), np.full((len(scans[s]), 1), s)], 1)
                                   for s in range(3)])
            differ = (np.abs(coords.cpu().numpy() - want).max(1) > 0).mean()
            assert differ < 5e-3, differ  # (float32 vs float64 arithmetic at integer boundaries)
    _no_device_error()


def test_unetscn_prepare_points_equals_coordinate_input():
    """UNetSCN.prepare_points(raw points) -> forward([prepared, feats]) equals forward([coords, feats]) with the
    coordinates of the two-step path: same structure bits, same kernels (FP32 mode: only the float atomics of the
    InputLayer's duplicate points differ in order; TF32 mode: rounding amplifies that, bars as in
    test_fused_executor_matches_module_path)."""
    from mm2d3d_b200 import scn as scn_mod
    from mm2d3d_b200.augment import scale_points
    from mm2d3d_b200.unet import UNetSCN
    torch.manual_seed(11)
    net = UNetSCN(in_channels=3, m=16, num_planes=5, full_scale=4096).to(DEV)
    scans = [synth.raycast_points("nuscenes", seed) for seed in (5, 6)]
    offs = np.concatenate([[0], np.cumsum([len(p) for p in scans])]).astype(np.int64)
    pts = torch.from_numpy(np.concatenate(scans, 0)).to(DEV)
    rot = np.stack([np.eye(3, dtype=np.float32)] * 2)
    coords, keep, _, _ = scale_points(pts, offs, rot, None, 20.0, 4096)
    assert bool(keep.all())
    # features are a function of the voxel: the InputLayer's float atomics then add equal values, whose sum does not
    # depend on their order -- the data path is reproducible and the two runs can be held to tight bars
    feats = ((coords[:, :3].double() * torch.tensor([0.37, 0.11, 0.73], dtype=torch.float64, device=DEV)) % 1.0).float()
    try:
        for mode, tol_out, tol_grad in (("fp32", 1e-5, 1e-4), ("tf32", 1e-3, 2e-2)):
            scn_mod.set_conv_mode(mode)
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                prep = net.prepare_points(pts, offs, rot, None, 20.0)
            assert prep.kept() is None
            outs = []
            for x0 in (prep, coords):
                x = feats.clone().requires_grad_(True)
                out = net([x0, x])
                (g,) = torch.autograd.grad(out.square().sum(), x)
                outs.append((out.detach(), g))
            e_out, e_grad = rel_err(outs[0][0], outs[1][0]), rel_l2(outs[0][1], outs[1][1])
            print(f"\n[prepare_points vs coordinates, {mode}] forward max-abs-rel {e_out:.2e}, d_feats rel-L2 {e_grad:.2e}")
            assert e_out < tol_out and e_grad < tol_grad, (mode, e_out, e_grad)
        scn_mod.set_conv_mode("fp32")
        # a receptive field the scans do not fit into: the handle reports the survivors and serves the rebuilt structure
        small = UNetSCN(in_channels=3, m=16, num_planes=3, full_scale=1024).to(DEV)
        prep = small.prepare_points(pts, offs, rot, None, 20.0)
        k = prep.kept()
        c2, keep2, _, _ = scale_points(pts, offs, rot, None, 20.0, 1024)
        assert k is not None and torch.equal(k, keep2) and 0 < int(k.sum()) < len(k)
        with torch.no_grad():
            a = small([prep, feats[k]])
            b = small([c2[keep2], feats[keep2]])
        assert rel_err(a, b) < 1e-5
    finally:
        scn_mod.set_conv_mode("fp32")
    _no_device_error()


@pytest.mark.parametrize("sizes", [[4000, 3000], [0, 17], [1], [20000, 20000, 1, 0]])
def test_rasterize_points_matches_numpy_assignment(sizes):
    """Sparse depth / 2D label maps (nuscenes_dataloader.py:274-278): bit-exact, including which of several points on one
    pixel wins, and consistent with the loaders' horizontal flip; RGB point features (:364-367) through lift2d."""
    from mm2d3d_b200.lift import LiftIndices, lift2d, rasterize_points
    from oracle import raster_oracle
    rng = np.random.default_rng(5)
    H, W = 45, 80                                  # small map -> many duplicate pixels
    idx = [np.stack([rng.integers(0, H, n), rng.integers(0, W, n)], 1).astype(np.int64) for n in sizes]
    depth = [rng.uniform(0.5, 60.0, n).astype(np.float32) for n in sizes]
    label = [rng.integers(0, 10, n).astype(np.float32) for n in sizes]
    li = LiftIndices(idx, DEV)
    d = rasterize_points(li, torch.from_numpy(np.concatenate(depth)).to(DEV), H, W, 0.0).cpu().numpy()
    l = rasterize_points(li, torch.from_numpy(np.concatenate(label)).to(DEV), H, W, -100.0).cpu().numpy()
    for b in range(len(sizes)):
        want_d = raster_oracle.rasterize(idx[b], depth[b], H, W, 0.0)
        want_l = raster_oracle.rasterize(idx[b], label[b], H, W, -100.0)
        assert np.array_equal(d[b], want_d.astype(np.float32))
        assert np.array_equal(l[b], want_l.astype(np.float32))
    # flip: rasterising the flipped indices equals flipping the maps
    fl = [raster_oracle.fliplr(ix, [], W)[0] for ix in idx]
    d_f = rasterize_points(fl, torch.from_numpy(np.concatenate(depth)).to(DEV), H, W, 0.0).cpu().numpy()
    assert np.array_equal(d_f, d[:, :, ::-1])
    # RGB features of the points = the lift of the image
    img = rng.random((len(sizes), 3, H, W)).astype(np.float32)
    got = lift2d(torch.from_numpy(img).to(DEV), li).cpu().numpy()
    want = np.concatenate([raster_oracle.rgb_feats(img[b], idx[b]) for b in range(len(sizes))], 0)
    assert np.array_equal(got, want)


def test_prepared_structure_on_side_stream_matches_inline():
    """UNetSCN.prepare(): structure built one step ahead on another stream gives the same bits as the inline build,
    over several steps with rotating batches (exercises allocator reuse across the two streams)."""
    from mm2d3d_b200.unet import UNetSCN
    from mm2d3d_b200 import scn as scn_mod
    torch.manual_seed(3)
    net = UNetSCN(in_channels=3, m=16, num_planes=4, full_scale=256).to(DEV)
    batches = []
    for r in range(3):
        locs, feats = synth.make_batch("nuscenes", batch=2, seed0=40 + 2 * r)
        locs[:, :3] //= 16
        # one point per voxel: the Input/OutputLayer sums over duplicate points are float atomics (order-dependent
        # rounding, which TF32 rounding and ReLU gates amplify); without duplicates the TF32 data path is bit-reproducible
        locs, first = np.unique(locs, axis=0, return_index=True)
        batches.append((torch.from_numpy(locs).to(DEV), torch.from_numpy(feats[first]).to(DEV)))
    for mode in ("tf32", "fp32"):
        scn_mod.set_conv_mode(mode)
        try:
            def run(prep_of):
                outs = []
                for i in range(7):
                    locs, feats = batches[i % 3]
                    x = feats.clone().requires_grad_(True)
                    net.zero_grad(set_to_none=True)
                    out = net([prep_of(i, locs), x])
                    out.square().sum().backward()
                    outs.append((out.detach().clone(), x.grad.clone(), net.layer2.weight.grad.clone()))
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
                with torch.cuda.stream(side):  # next step's structure while this one is being enqueued
                    ahead[i + 1] = net.prepare(batches[(i + 1) % 3][0])
                return cur

            piped = run(prep_of)
            for step, ((a, b, c), (d, e, f)) in enumerate(zip(inline, piped)):
                if mode == "tf32":
                    # forward and d_feats have no atomics in this mode: identical bits
                    assert torch.equal(a, d) and torch.equal(b, e), (mode, step)
                    assert float((c - f).abs().max()) <= 1e-5 * float(c.abs().max()), (mode, step)
                else:
                    # the FP32 kernels accumulate with atomics (order-dependent rounding, amplified by ReLU gates)
                    assert float((a - d).abs().max()) <= 1e-4 * float(a.abs().max()), (mode, step)
                    assert float((b - e).abs().max()) <= 5e-3 * float(b.abs().max()), (mode, step)
                    assert float((c - f).abs().max()) <= 5e-3 * float(c.abs().max()), (mode, step)
            stale = ahead.popitem()[1]
            scn_mod.set_conv_mode("tf32" if mode == "fp32" else "fp32")
            with pytest.raises(ValueError):  # a structure prepared for another convolution mode is refused
                net([stale, batches[1][1]])
        finally:
            scn_mod.set_conv_mode("fp32")


@pytest.mark.parametrize("ci", [32, 64])  # 32: the two-ring kernel of the narrow layers, 64: the general one
def test_tf32_wgrad_in_several_launches(monkeypatch, ci):
    """Row counts whose per-CTA tile list does not fit in shared memory are processed in several launches over
    pieces of the plan's tile order (happens from ~300 k rows at 192 channels); forced here at 20 k rows."""
    from mm2d3d_b200 import _lib
    from mm2d3d_b200 import functional as F
    from mm2d3d_b200.metadata import Metadata
    locs, _ = synth.make_batch("nuscenes", batch=1, seed0=3)
    meta = Metadata(torch.from_numpy(locs).to(DEV), 4096, 1, plans=True)
    t, _, _ = F.conv_tables(meta, "smc", 4096, plans=True)
    n, co = t.n_out, 48
    torch.manual_seed(1)
    x, dout = torch.randn(n, ci, device=DEV), torch.randn(n, co, device=DEV)
    lib, sp = _lib.lib, _lib.stream_ptr()

    def wgrad(mode):
        dw = torch.empty(27, 1, ci, co, device=DEV)
        m = _lib.MODES[mode]
        plan, cap = (t.plan, t.plan_cap) if mode == "tf32" else (None, 0)
        _lib.check(lib.mm3d_conv_wgrad(x.data_ptr(), n, ci, dout.data_ptr(), n, co, dw.data_ptr(), 27, t.tbl, t.stride, None,
                                       plan, cap, 0, m, None, 0, sp))
        torch.cuda.synchronize()
        return dw

    ref = wgrad("fp32")
    one = wgrad("tf32")
    monkeypatch.setenv("MM3D_WGRAD_MAX_LOCAL", "4")
    many = wgrad("tf32")
    assert lib.mm3d_take_device_error() == 0
    scale = float(ref.abs().max())
    assert float((one - ref).abs().max()) < 1e-2 * scale
    assert float((many - ref).abs().max()) < 1e-2 * scale
    assert float((many - one).abs().max()) < 1e-5 * scale  # same products, different accumulation order


def test_heads_reference_fixture():
    """RGB-mask prologue and cross-modal KL term (SURVEY 8(f).3) against tests/golden/heads_ref.npz, which the
    reference's Net3DSeg.forward / torch lines produced: forward 1e-6, gradients 1e-5 relative to the tensor scale."""
    from mm2d3d_b200.heads import cross_modal_kl, rgb_mask
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "heads_ref.npz"))
    dev = lambda k: torch.from_numpy(z[k]).to(DEV)
    x, w, b = dev("feats").requires_grad_(True), dev("w").requires_grad_(True), dev("b").requires_grad_(True)
    y = rgb_mask(x, w, b)
    assert float((y.detach().cpu() - torch.from_numpy(z["masked"])).abs().max()) < 1e-6
    y.backward(dev("g"))
    for got, key in ((x.grad, "dx"), (w.grad, "dw"), (b.grad, "db")):
        want = torch.from_numpy(z[key])
        assert got.shape == want.shape
        assert float((got.cpu() - want).abs().max()) <= 1e-5 * max(float(want.abs().max()), 1.0), key
    pred = dev("pred").requires_grad_(True)
    loss = cross_modal_kl(pred, dev("target"))
    assert abs(float(loss.detach()) - float(z["loss"])) <= 1e-6 * abs(float(z["loss"]))
    (2.5 * loss).backward()
    want = 2.5 * torch.from_numpy(z["dpred"])
    assert float((pred.grad.cpu() - want).abs().max()) <= 1e-5 * float(want.abs().max())
    # a data tensor that does not need a gradient, larger batch, odd sizes
    x2 = torch.rand(100003, 3, device=DEV)
    y2 = rgb_mask(x2, w.detach(), b.detach())
    ref = x2 * torch.sigmoid(x2 @ w.detach().t() + b.detach())
    assert float((y2 - ref).abs().max()) < 1e-6


def test_heads3d_reference_fixture():
    """The fused 3D heads (two Linear(16 -> classes) + the 3D cross-modal term in one pass, SURVEY 8(f).3) against
    tests/golden/heads3d_ref.npz, whose logits the reference's own Net3DSeg.forward produced: forward 1e-6, gradients
    1e-5 relative to the tensor scale; also without a target, without a feature gradient and on a large odd batch."""
    from mm2d3d_b200.heads import heads3d
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "heads3d_ref.npz"))
    dev = lambda k: torch.from_numpy(z[k]).to(DEV)
    feat = dev("feat").requires_grad_(True)
    w1, b1, w2, b2 = (dev(k).requires_grad_(True) for k in ("w1", "b1", "w2", "b2"))
    l1, l2, loss = heads3d(feat, w1, b1, w2, b2, dev("target"))
    assert float((l1.detach().cpu() - torch.from_numpy(z["logit1"])).abs().max()) < 1e-5
    assert float((l2.detach().cpu() - torch.from_numpy(z["logit2"])).abs().max()) < 1e-5
    assert abs(float(loss.detach()) - float(z["loss"])) <= 1e-6 * abs(float(z["loss"]))
    ((l1 * dev("g1")).sum() + (l2 * dev("g2")).sum() + float(z["lam"]) * loss).backward()
    for got, key in ((feat.grad, "d_feat"), (w1.grad, "d_w1"), (b1.grad, "d_b1"), (w2.grad, "d_w2"), (b2.grad, "d_b2")):
        want = torch.from_numpy(z[key])
        assert got.shape == want.shape, key
        assert float((got.cpu() - want).abs().max()) <= 1e-5 * max(float(want.abs().max()), 1.0), key
    # no target (inference), features that are data, a large odd row count and 10 classes vs plain torch
    torch.manual_seed(5)
    n, f, C = 100003, 16, 10
    x = torch.randn(n, f, device=DEV)
    lin1, lin2 = torch.nn.Linear(f, C).to(DEV), torch.nn.Linear(f, C).to(DEV)
    a1, a2, zero = heads3d(x, lin1.weight, lin1.bias, lin2.weight, lin2.bias)
    assert float((a1 - lin1(x)).detach().abs().max()) < 1e-5 and float((a2 - lin2(x)).detach().abs().max()) < 1e-5 and float(zero.detach()) == 0.0
    tgt = torch.randn(n, C, device=DEV)
    a1, a2, kl = heads3d(x, lin1.weight, lin1.bias, lin2.weight, lin2.bias, tgt)
    want_kl = torch.nn.functional.kl_div(torch.log_softmax(lin2(x), 1), torch.softmax(tgt, 1), reduction="none").sum(1).mean()
    assert abs(float(kl.detach()) - float(want_kl.detach())) < 1e-5 * abs(float(want_kl.detach()))
    g = torch.randn(n, C, device=DEV)
    got = torch.autograd.grad((a1 * g).sum() + kl, [lin1.weight, lin1.bias, lin2.weight, lin2.bias])
    want = torch.autograd.grad((lin1(x) * g).sum() + want_kl, [lin1.weight, lin1.bias, lin2.weight, lin2.bias])
    for a, b in zip(got, want):
        assert float((a - b).abs().max()) <= 2e-5 * max(float(b.abs().max()), 1.0)


@pytest.mark.parametrize("mode", ["fp32", "tf32"])
def test_unetscn_with_folded_rgb_mask(mode):
    """``net(x, rgb_mask=linear)`` (the RGB-mask prologue of Net3DSeg.forward folded into the executor's InputLayer,
    SURVEY 8(f).3) against the prologue as its own op followed by the plain network: same outputs, feature gradient,
    mask gradients and parameter gradients; also when the features are data and on the module-by-module path."""
    import copy

    import mm2d3d_b200.scn as scn
    from mm2d3d_b200.heads import rgb_mask
    from mm2d3d_b200.unet import UNetSCN
    torch.manual_seed(12)
    locs, feats = synth.make_batch("nuscenes", batch=2, seed0=9)
    locs, first = np.unique(locs, axis=0, return_index=True)  # one point per voxel: no float atomics in the I/O layers
    coords, feats = torch.from_numpy(locs).to(DEV), torch.from_numpy(feats[first]).to(DEV)
    net = UNetSCN(in_channels=3, m=16, num_planes=5, full_scale=4096).to(DEV)
    lin = torch.nn.Linear(3, 1).to(DEV)
    g = torch.randn(locs.shape[0], 16, device=DEV)
    scn.set_conv_mode(mode)
    try:
        xa = feats.clone().requires_grad_(True)
        pa = [lin.weight, lin.bias] + list(net.parameters())
        ya = net([coords, xa], rgb_mask=lin)
        ga = torch.autograd.grad(ya, [xa] + pa, g)
        xb = feats.clone().requires_grad_(True)
        yb = net([coords, rgb_mask(xb, lin.weight, lin.bias)])
        gb = torch.autograd.grad(yb, [xb] + pa, g)
        # features as data: only the mask and the network get gradients
        yc = net([coords, feats], rgb_mask=(lin.weight, lin.bias))
        gc = torch.autograd.grad(yc, pa, g)
        # module-by-module path
        net2 = copy.deepcopy(net)
        net2.fused = False
        yd = net2([coords, feats], rgb_mask=lin)
    finally:
        scn.set_conv_mode("fp32")
    _no_device_error()
    tol = 1e-5 if mode == "fp32" else 2e-3
    assert rel_err(ya, yb) < tol and rel_err(yc, yb) < tol and rel_err(yd, yb) < tol
    for a, b in zip(ga, gb):
        assert rel_l2(a, b) < 10 * tol
    for a, b in zip(gc, gb[1:]):
        assert rel_l2(a, b) < 10 * tol


# ------------------------------------------------------------------------------ whole network, frozen gates
def _bn_modules(net):
    return [m for m in net.modules() if type(m).__name__ in ("BatchNormLeakyReLU", "BatchNormReLU")]


def _freeze_gates(net, records, device, dtype, tensor_cls):
    """Replace every BatchNorm+ReLU of `net` by the FROZEN map  y = gate * ((x - mean) * invstd * weight + bias)
    with (mean, invstd, gate) taken from `records` (one per BN module, module order) as constants.  The network
    becomes piecewise linear with fixed pieces: no ReLU-gate flips, no gradient through the batch statistics."""
    import types
    for m, (mean, invstd, gate) in zip(_bn_modules(net), records):
        mean_d, invstd_d, gate_d = mean.to(device, dtype), invstd.to(device, dtype), gate.to(device, dtype)

        def fwd(self, x, mean_d=mean_d, invstd_d=invstd_d, gate_d=gate_d):
            y = ((x.features - mean_d) * (invstd_d * self.weight) + self.bias) * gate_d
            return tensor_cls(y, x.metadata, x.spatial_size)
        m.forward = types.MethodType(fwd, m)


@pytest.mark.parametrize("mode", ["fp32", "tf32", "tf32x3", "bf16"])
def test_unetscn_gradients_with_frozen_gates(mode):
    """north_star's tolerance on whole-network GRADIENTS, stated per tensor and held directly: 1e-4 (FP32 mode) /
    1e-2 (TF32 mode), relative L2 AND max-abs-relative, against the FP64 oracle.

    The free-running network cannot show this: one ReLU gate that flips under a 1e-3 perturbation changes its
    gradient entry by O(1), and with batch statistics in the loop the FP32 CPU oracle itself is ~3e-3 away from
    its FP64 run (test_unetscn_full_config_*).  Here the ReLU gates and the BatchNorm statistics of all 26
    BatchNorm layers are taken from the FP64 oracle's forward and frozen in BOTH networks, so what is compared is
    the chain of 27 sparse convolutions (forward, dgrad, wgrad), InputLayer and OutputLayer -- every kernel the
    arithmetic mode touches -- over the whole depth of the network with its error accumulation, module by module
    through the C ABI.  (The BatchNorm kernels are held to 1e-4 per op in test_bnrelu; the executor is tied to
    this module path in test_fused_executor_matches_module_path.)"""
    import copy

    import mm2d3d_b200.scn as scn
    from mm2d3d_b200.unet import UNetSCN
    torch.manual_seed(8)
    locs, feats = synth.make_batch("nuscenes", batch=1, seed0=6)
    coords, feats = torch.from_numpy(locs), torch.from_numpy(feats)
    net_ref = UNetSCN(in_channels=3, backend=scn_cpu)
    with torch.no_grad():  # non-trivial affine parameters
        for m in _bn_modules(net_ref):
            m.weight.add_(0.2 * torch.randn_like(m.weight))
            m.bias.add_(0.1 * torch.randn_like(m.bias))
    net = UNetSCN(in_channels=3).to(DEV)
    net.load_state_dict(net_ref.state_dict())
    net.fused = False
    net64 = copy.deepcopy(net_ref).double()

    # 1) true FP64 forward: record statistics and gates of every BatchNorm layer
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
    assert len(records) == 26

    # 2) the frozen function in FP64 on the oracle (reference) and on the GPU in `mode`
    _freeze_gates(net64, records, "cpu", torch.float64, scn_cpu.SparseConvNetTensor)
    _freeze_gates(net, records, DEV, torch.float32, scn.SparseConvNetTensor)
    x64 = feats.double().requires_grad_(True)
    out64 = net64([coords, x64])
    assert rel_err(out64, out_true) < 1e-12  # same statistics and gates: the frozen forward IS the true forward
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
    # BF16 operands carry 8 mantissa bits (unit round-off 2^-9, four times TF32's 2^-11): the per-op bar of 1e-2 holds
    # (test_conv_fwd_bwd); over the 27-convolution chain the achieved whole-network figures are printed (B200, this
    # input: forward 1.0e-2, gradients rel-L2 <= 2.4e-2, max-abs-rel <= 3.2e-2) and held to 5e-2
    tol = 5e-2 if mode == "bf16" else TOL[mode]
    e_out = rel_err(out, out64)
    assert e_out < tol, ("forward", e_out)
    rows, worst = [], (0.0, 0.0, "")
    for name, a in zip(names, gg):
        e2, em = rel_l2(a, g64[name]), rel_err(a, g64[name])
        rows.append((name, e2, em))
        worst = max(worst, (max(e2, em), e2, name))
    print(f"\n[{mode}] frozen-gate whole-network parity vs FP64 oracle: forward max-abs-rel {e_out:.2e}")
    for name, e2, em in rows:
        print(f"[{mode}]   d {name:44s} rel-L2 {e2:.2e}  max-abs-rel {em:.2e}")
    for name, e2, em in rows:
        assert e2 <= tol and em <= tol, (mode, name, e2, em)


def test_frozen_parameters_backward():
    """Gradient w.r.t. the features through a network whose parameters (all, or only BatchNorm / only the
    convolutions) are frozen: the executor receives NULL gradient pointers for those slots (ADVICE r1)."""
    from mm2d3d_b200 import scn as scn_mod
    from mm2d3d_b200.unet import UNetSCN
    torch.manual_seed(4)
    net = UNetSCN(in_channels=3, m=16, num_planes=4, full_scale=256).to(DEV)
    locs, feats = synth.make_batch("nuscenes", batch=2, seed0=8)
    locs[:, :3] //= 16
    # one point per voxel: no float atomics in the I/O layers, so the TF32 data path is bit-reproducible and the
    # comparison below is not blurred by run-to-run noise amplified through the ReLU gates
    locs, first = np.unique(locs, axis=0, return_index=True)
    coords, feats = torch.from_numpy(locs).to(DEV), torch.from_numpy(feats[first]).to(DEV)
    g = torch.randn(locs.shape[0], 16, device=DEV)
    for mode in ("fp32", "tf32"):
        scn_mod.set_conv_mode(mode)
        try:
            net.requires_grad_(True)
            x = feats.clone().requires_grad_(True)
            full = torch.autograd.grad(net([coords, x]), [x] + list(net.parameters()), g)
            named = list(dict(net.named_parameters()))
            for frozen in ("all", "bn", "conv"):
                for k, p_ in net.named_parameters():
                    is_bn = p_.dim() == 1
                    p_.requires_grad_(not (frozen == "all" or (frozen == "bn") == is_bn))
                live = [p_ for p_ in net.parameters() if p_.requires_grad]
                x2 = feats.clone().requires_grad_(True)
                got = torch.autograd.grad(net([coords, x2]), [x2] + live, g)
                torch.cuda.synchronize()
                # same kernels as the all-trainable run.  TF32 mode: forward and dgrad have no atomics -> identical
                # d_feats; FP32 mode: the SIMT kernels accumulate with atomics (order-dependent rounding, amplified by
                # the free-running BatchNorm/ReLU stack)
                if mode == "tf32":
                    assert torch.equal(got[0], full[0]), (mode, frozen, rel_l2(got[0], full[0]))
                else:
                    assert rel_l2(got[0], full[0]) < 5e-3, (mode, frozen, rel_l2(got[0], full[0]))
                want = {k: full[1 + i] for i, k in enumerate(named)}
                name_of = {id(v): k for k, v in net.named_parameters()}
                for p_, a in zip(live, got[1:]):
                    bar = 1e-4 if mode == "tf32" else 5e-3
                    assert rel_l2(a, want[name_of[id(p_)]]) < bar, (mode, frozen, name_of[id(p_)])
        finally:
            scn_mod.set_conv_mode("fp32")
            net.requires_grad_(True)
    _no_device_error()


class _ForeignUNet(torch.nn.Module):
    """A host network assembled from the raw ``scn.*`` surface the way the reference's 3d_net/scn_unet.py:90-126 does
    (five members layer1..layer5 called in sequence, InputLayer with its default prebuild of ONE level) -- i.e. NOT
    mm2d3d_b200.unet.UNetSCN, so neither the whole-network executor nor the pre-built pyramid is involved and every
    coarser level is built lazily by the first layer that needs it.  The reference file itself is not part of this
    repository; tests/test_oracle.py and tests/test_cabi.py pin UNetSCN's module tree to the one SURVEY.md Appendix B
    records for it (tests/golden/unetscn_tree.json)."""

    def __init__(self, scn, in_channels, m, num_planes, full_scale):
        super().__init__()
        from mm2d3d_b200.unet import build_unet
        self.layer1 = scn.InputLayer(3, full_scale, mode=4)
        self.layer2 = scn.SubmanifoldConvolution(3, in_channels, m, 3, False)
        self.layer3 = build_unet(scn, 1, [(i + 1) * m for i in range(num_planes)], False)
        self.layer4 = scn.BatchNormReLU(m)
        self.layer5 = scn.OutputLayer(3)

    def forward(self, x):
        for layer in (self.layer1, self.layer2, self.layer3, self.layer4, self.layer5):
            x = layer(x)
        return x


@pytest.mark.parametrize("mode", ["fp32", "tf32"])
def test_raw_scn_surface_forward_backward(mode):
    """INTEGRATION.md option A on the GPU: forward AND backward of a network built from the raw scn.* modules
    (reference call pattern, lazily built levels, coordinates left on the CPU) against the oracle."""
    import mm2d3d_b200.scn as scn
    torch.manual_seed(12)
    kw = dict(in_channels=3, m=16, num_planes=5, full_scale=4096)
    ref = _ForeignUNet(scn_cpu, **kw)
    net = _ForeignUNet(scn, **kw).to(DEV)
    net.load_state_dict(ref.state_dict())
    locs, feats = synth.make_batch("nuscenes", batch=2, seed0=9)
    keep = np.random.default_rng(1).random(locs.shape[0]) < 0.3
    coords, feats = torch.from_numpy(locs[keep]), torch.from_numpy(feats[keep])
    ref64 = __import__("copy").deepcopy(ref).double()
    x64 = feats.double().requires_grad_(True)
    out64 = ref64([coords, x64])
    g = torch.randn_like(out64)
    p64 = dict(ref64.named_parameters())
    g64 = torch.autograd.grad(out64, [x64] + list(p64.values()), g)
    scn.set_conv_mode(mode)
    try:
        x = feats.clone().to(DEV).requires_grad_(True)
        out = net([coords, x])  # coords stay on the CPU as in scn_unet.py:131-137
        gg = torch.autograd.grad(out, [x] + list(net.parameters()), g.float().to(DEV))
    finally:
        scn.set_conv_mode("fp32")
    _no_device_error()
    assert rel_err(out, out64) < TOL[mode]
    # free-running BatchNorm/ReLU: gradients are compared by direction and size (see the frozen-gate test for the bar)
    for (name, _), a, b in zip([("feats", None)] + list(p64.items()), gg, g64):
        assert rel_l2(a, b) < (2e-2 if mode == "fp32" else 0.3), (name, rel_l2(a, b))
    for (k, a), (_, b) in zip(net.named_buffers(), ref64.named_buffers()):
        assert rel_err(a, b) < max(TOL[mode], 1e-4), k


def test_unetscn_semantickitti_shaped_scan():
    """BASELINE configs[3] shape: one SemanticKITTI-shaped scan (~120 k points) through the whole network, FP32
    mode against the oracle (forward 1e-4; gradients relative to the FP32 CPU oracle's own error, as for nuScenes),
    then the TF32 executor against the FP32 one on the same scan (forward 1e-2)."""
    import mm2d3d_b200.scn as scn
    from mm2d3d_b200.unet import UNetSCN
    torch.manual_seed(15)
    locs, feats = synth.make_batch("semantickitti", batch=1, seed0=2)
    assert locs.shape[0] > 90_000
    net_ref = UNetSCN(in_channels=3, backend=scn_cpu)
    net = UNetSCN(in_channels=3).to(DEV)
    net.load_state_dict(net_ref.state_dict())
    import copy
    coords, fe = torch.from_numpy(locs), torch.from_numpy(feats)
    net64 = copy.deepcopy(net_ref).double()
    x64 = fe.double().requires_grad_(True)
    out64 = net64([coords, x64])
    g = torch.randn_like(out64)
    p64 = dict(net64.named_parameters())
    g64 = torch.autograd.grad(out64, [x64] + list(p64.values()), g)
    x = fe.clone().to(DEV).requires_grad_(True)
    out = net([coords.to(DEV), x])
    gg = torch.autograd.grad(out, [x] + list(net.parameters()), g.float().to(DEV))
    assert rel_err(out, out64) < TOL["fp32"], rel_err(out, out64)
    # free-running ReLU gates and batch statistics: the FP32 SIMT kernels accumulate with atomics, and a gate that
    # flips on that noise changes its gradient entry by O(1); run to run the worst tensor moves between ~1e-3 and
    # ~6e-3 -- gradients are held to 2e-2 relative L2 here, the strict 1e-4 is held with frozen gates
    # (test_unetscn_gradients_with_frozen_gates) and per op
    worst = max((rel_l2(a, b), n) for a, b, n in zip(gg, g64, ["feats"] + list(p64)))
    print("SemanticKITTI-shaped scan, FP32 mode: forward", rel_err(out, out64), "worst gradient rel-L2", worst)
    assert worst[0] < 2e-2, worst
    c, f = torch.from_numpy(locs).to(DEV), torch.from_numpy(feats).to(DEV)
    with torch.no_grad():
        net.eval()
        a = net([c, f])
        scn.set_conv_mode("tf32")
        try:
            b = net([c, f])
        finally:
            scn.set_conv_mode("fp32")
    _no_device_error()
    assert rel_err(b, a) < TOL["tf32"]


def test_lift2d_out_of_image_index_raises():
    from mm2d3d_b200 import _lib
    from mm2d3d_b200.functional import Lift2DFn
    from mm2d3d_b200.lift import LiftIndices, lift2d
    fmap = torch.randn(2, 4, 10, 12, device=DEV)
    good = [np.array([[0, 0], [9, 11], [-1, -12]]), np.array([[3, 4]])]
    assert lift2d(fmap, good).shape == (4, 4)
    for bad in ([np.array([[10, 0]]), np.array([[0, 0]])], [np.array([[0, 0]]), np.array([[0, 12]])],
                [np.array([[-11, 0]]), np.array([[0, 0]])]):
        with pytest.raises(IndexError):  # synchronous, like the reference's advanced indexing (2d_net/model.py:131-137)
            lift2d(fmap, bad)
    # the kernels bound-check too (a caller of the C ABI gets a zero row and the sticky error bit, no wild access)
    li = LiftIndices([np.array([[0, 0], [10, 3]]), np.array([[2, 2]])], DEV)
    torch.cuda.synchronize()
    _lib.lib.mm3d_take_device_error()
    out = Lift2DFn.apply(fmap, li.idx, li.offsets)
    torch.cuda.synchronize()
    assert _lib.lib.mm3d_take_device_error() & 2
    assert float(out[1].abs().max()) == 0.0 and torch.equal(out[0], fmap[0, :, 0, 0])
