"""Pins the CPU oracle (no reference-owned test exists for the 3D path -- SURVEY.md 4.1):
known-answer micro-example (A.10), literal-loop vs vectorised structure, dense conv3d
equivalence (4.3), float64 gradcheck, and that the UNetSCN builder makes the module tree that
Appendix B specifies for the reference's ``scn_unet.py`` (golden/unetscn_tree.json)."""
import json
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import scn_cpu
from oracle import scn_oracle as O


def _rand_coords(rng, n, size, batch):
    c = rng.integers(0, size, (n, 3))
    b = np.sort(rng.integers(0, batch, (n, 1)), 0)
    return np.concatenate([c, b], 1).astype(np.int64)


# ---------------------------------------------------------------- A.10 known-answer test
A10_LOCS = np.array([(1, 1, 1, 0), (2, 1, 1, 0), (1, 1, 1, 0), (5, 5, 5, 0), (1, 1, 1, 1), (4, 5, 5, 0)])
A10_FEATS = np.array([(1, 0, 0), (0, 2, 0), (3, 0, 0), (0, 0, 4), (5, 5, 5), (0, 0, 8)], dtype=np.float32)


def _ruleset(tbl):
    return {k: sorted((int(tbl[j, k]), j) for j in range(tbl.shape[0]) if tbl[j, k] >= 0)
            for k in range(tbl.shape[1]) if (tbl[:, k] >= 0).any()}


def test_a10_known_answer():
    meta = O.Metadata(A10_LOCS, 4096)
    assert meta.p2v.tolist() == [0, 1, 0, 2, 3, 4]
    # (x,y,z,b) rows in first-occurrence order
    assert meta.coords_at(4096).tolist() == [[1, 1, 1, 0], [2, 1, 1, 0], [5, 5, 5, 0], [1, 1, 1, 1], [4, 5, 5, 0]]
    f = O.input_layer(meta, torch.from_numpy(A10_FEATS))
    assert f.tolist() == [[2, 0, 0], [0, 2, 0], [0, 0, 4], [5, 5, 5], [0, 0, 8]]
    assert _ruleset(meta.nbr(4096)) == {
        13: [(0, 0), (1, 1), (2, 2), (3, 3), (4, 4)], 22: [(1, 0), (2, 4)], 4: [(0, 1), (4, 2)]}
    parent, off, n1 = meta.down(4096)
    rules = {k: [(i, int(parent[i])) for i in range(5) if off[i] == k] for k in set(off.tolist())}
    assert rules == {7: [(0, 0), (2, 2), (3, 3)], 3: [(1, 1), (4, 2)]}
    assert n1 == 4
    assert meta.coords_at(2048).tolist() == [[0, 0, 0, 0], [1, 0, 0, 0], [2, 2, 2, 0], [0, 0, 0, 1]]
    assert _ruleset(meta.nbr(2048)) == {13: [(0, 0), (1, 1), (2, 2), (3, 3)], 22: [(1, 0)], 4: [(0, 1)]}


# ---------------------------------------------------------------- loops vs vectorised
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_structure_matches_literal_loops(seed):
    rng = np.random.default_rng(seed)
    coords = _rand_coords(rng, 400, 12, 3)
    ids_l, uniq_l = O.first_occurrence_ids_loop(O.pack_keys(coords))
    ids_v, uniq_v = O.first_occurrence_ids(O.pack_keys(coords))
    assert np.array_equal(ids_l, ids_v) and np.array_equal(uniq_l, uniq_v)
    _, vc, _ = O.voxelize(coords)
    assert np.array_equal(O.nbr_table(vc, 12), O.nbr_table_loop(vc, 12))
    tbl = O.nbr_table(vc, 12)
    # symmetry: nbr[j][k] == i  <=>  nbr[i][26-k] == j
    for j in range(tbl.shape[0]):
        for k in range(27):
            if tbl[j, k] >= 0:
                assert tbl[tbl[j, k], 26 - k] == j


def test_empty_and_single_point():
    meta = O.Metadata(np.zeros((0, 4), np.int64), 16)
    assert meta.p2v.shape == (0,) and meta.nbr(16).shape == (0, 27)
    meta = O.Metadata(np.array([[3, 3, 3, 0]]), 16)
    assert meta.nbr(16)[0].tolist() == [-1] * 13 + [0] + [-1] * 13
    # borders: neighbours outside [0, size) never match (no wrap-around through key packing)
    meta = O.Metadata(np.array([[0, 0, 0, 0], [15, 15, 15, 0], [0, 0, 15, 0]]), 16)
    assert (meta.nbr(16) >= 0).sum() == 3


# ---------------------------------------------------------------- dense equivalence (4.3)
def _dense(vc, feats, size, batch):
    d = torch.zeros(batch, feats.shape[1], size, size, size, dtype=feats.dtype)
    d[vc[:, 3], :, vc[:, 0], vc[:, 1], vc[:, 2]] = feats
    return d


def _sample(d, vc):
    return d[vc[:, 3], :, vc[:, 0], vc[:, 1], vc[:, 2]]


def test_dense_conv3d_equivalence():
    rng = np.random.default_rng(5)
    torch.manual_seed(5)
    S, B, Ci, Co = 16, 2, 5, 7
    coords = _rand_coords(rng, 900, S, B)
    meta = O.Metadata(coords, S)
    vc = torch.from_numpy(meta.coords_at(S))
    x = torch.randn(vc.shape[0], Ci, dtype=torch.float64, requires_grad=True)

    # submanifold 3^3: W[k, ci, co] <-> Wd[co, ci, dx, dy, dz], k = (dx*3+dy)*3+dz
    W = torch.randn(27, 1, Ci, Co, dtype=torch.float64, requires_grad=True)
    y = O.submanifold_conv(meta, S, x, W)
    Wd = W.reshape(3, 3, 3, Ci, Co).permute(4, 3, 0, 1, 2)
    yd = _sample(F.conv3d(_dense(vc, x, S, B), Wd, padding=1), vc)
    assert torch.allclose(y, yd, atol=1e-10)
    g = torch.randn_like(y)
    gx, gw = torch.autograd.grad(y, (x, W), g)
    gxd, gwd = torch.autograd.grad(yd, (x, W), g)
    assert torch.allclose(gx, gxd, atol=1e-10) and torch.allclose(gw, gwd, atol=1e-10)

    # convolution size 2 stride 2
    W2 = torch.randn(8, 1, Ci, Co, dtype=torch.float64, requires_grad=True)
    y2 = O.conv_down(meta, S, x, W2)
    vc1 = torch.from_numpy(meta.coords_at(S // 2))
    W2d = W2.reshape(2, 2, 2, Ci, Co).permute(4, 3, 0, 1, 2)
    dense2 = F.conv3d(_dense(vc, x, S, B), W2d, stride=2)
    assert torch.allclose(y2, _sample(dense2, vc1), atol=1e-10)
    # coarse active set == coarse sites with >= 1 active child
    occ = F.max_pool3d(_dense(vc, torch.ones(vc.shape[0], 1, dtype=torch.float64), S, B), 2)
    assert int(occ.sum()) == vc1.shape[0]

    # deconvolution size 2 stride 2 back onto the fine grid
    W3 = torch.randn(8, 1, Co, Ci, dtype=torch.float64, requires_grad=True)
    y3 = O.deconv_up(meta, S, y2, W3)
    W3d = W3.reshape(2, 2, 2, Co, Ci).permute(3, 4, 0, 1, 2)
    dense3 = F.conv_transpose3d(_dense(vc1, y2, S // 2, B), W3d, stride=2)
    assert torch.allclose(y3, _sample(dense3, vc), atol=1e-10)


def test_io_layers_and_bn():
    rng = np.random.default_rng(9)
    torch.manual_seed(9)
    coords = _rand_coords(rng, 500, 6, 2)
    meta = O.Metadata(coords, 6)
    feats = torch.randn(500, 4, dtype=torch.float64)
    v = O.input_layer(meta, feats)
    for j in (0, 3, v.shape[0] - 1):
        assert torch.allclose(v[j], feats[torch.from_numpy(meta.p2v == j)].mean(0))
    back = O.output_layer(meta, v)
    assert back.shape == feats.shape and torch.equal(back[7], v[meta.p2v[7]])

    x = torch.randn(300, 6, dtype=torch.float64) * 3 + 1
    g, b = torch.randn(6, dtype=torch.float64), torch.randn(6, dtype=torch.float64)
    rm, rv = torch.zeros(6, dtype=torch.float64), torch.ones(6, dtype=torch.float64)
    y = O.batchnorm_relu(x, g, b, rm, rv, eps=1e-4, momentum=0.9, training=True)
    rm2, rv2 = torch.zeros(6, dtype=torch.float64), torch.ones(6, dtype=torch.float64)
    yt = F.relu(F.batch_norm(x, rm2, rv2, g, b, training=True, momentum=0.1, eps=1e-4))
    assert torch.allclose(y, yt, atol=1e-12)
    assert torch.allclose(rm, rm2) and torch.allclose(rv, rv2)
    ye = O.batchnorm_relu(x, g, b, rm, rv, training=False)
    assert torch.allclose(ye, F.relu(F.batch_norm(x, rm, rv, g, b, training=False, eps=1e-4)))


def test_gradcheck_float64():
    rng = np.random.default_rng(3)
    torch.manual_seed(3)
    coords = _rand_coords(rng, 60, 4, 2)
    meta = O.Metadata(coords, 4)
    n0 = meta.npts.shape[0]
    x = torch.randn(n0, 3, dtype=torch.float64, requires_grad=True)
    W = torch.randn(27, 1, 3, 2, dtype=torch.float64, requires_grad=True)
    W2 = torch.randn(8, 1, 3, 2, dtype=torch.float64, requires_grad=True)
    W3 = torch.randn(8, 1, 2, 3, dtype=torch.float64, requires_grad=True)
    assert torch.autograd.gradcheck(lambda a, w: O.submanifold_conv(meta, 4, a, w), (x, W))
    assert torch.autograd.gradcheck(
        lambda a, w, v: O.deconv_up(meta, 4, O.conv_down(meta, 4, a, w), v), (x, W2, W3))
    f = torch.randn(60, 3, dtype=torch.float64, requires_grad=True)
    assert torch.autograd.gradcheck(lambda a: O.output_layer(meta, O.input_layer(meta, a)), (f,))


# ---------------------------------------------------------------- network level
def test_unetscn_parameter_tree():
    """Appendix B names/shapes; conv 2 685 712 + BN 3 808 parameters."""
    from mm2d3d_b200.unet import UNetSCN
    net = UNetSCN(in_channels=3, backend=scn_cpu)
    sd = net.state_dict()
    assert tuple(sd["layer2.weight"].shape) == (27, 1, 3, 16)
    assert tuple(sd["layer3.0.1.weight"].shape) == (27, 1, 16, 16)
    assert tuple(sd["layer3.1.1.1.weight"].shape) == (8, 1, 16, 32)
    assert tuple(sd["layer3.1.1.2.0.1.weight"].shape) == (27, 1, 32, 32)
    assert tuple(sd["layer3.1.1.4.weight"].shape) == (8, 1, 32, 16)
    assert tuple(sd["layer3.3.1.weight"].shape) == (27, 1, 32, 16)
    assert tuple(sd["layer3.3.0.running_mean"].shape) == (32,)
    assert sum(p.numel() for p in net.parameters()) == 2_689_520
    assert net.out_channels == 16 and net.in_channels == 3


def test_unetscn_tree_matches_spec_fixture():
    """Our builder on the oracle's ``scn`` surface makes the module tree that SURVEY.md Appendix B records for the
    reference's ``3d_net/scn_unet.py`` (golden/unetscn_tree.json: state_dict keys in order and their shapes, written
    out from that spec by make_golden.py, not produced by running the reference)."""
    from mm2d3d_b200.unet import UNetSCN
    with open(os.path.join(os.path.dirname(__file__), "golden", "unetscn_tree.json")) as f:
        ref = json.load(f)
    net = UNetSCN(in_channels=ref["in_channels"], m=ref["m"], num_planes=ref["num_planes"], backend=scn_cpu)
    assert [[k, list(v.shape)] for k, v in net.state_dict().items()] == ref["state_dict"]


def test_bilinear_lift_oracle_is_grid_sample():
    """The bilinear lift has no counterpart in the reference; its oracle (explicit four taps, zero outside the map) is
    pinned to torch's grid_sample (bilinear, zeros padding, align_corners=True) on CPU, including points on the border,
    outside the map and at integer pixels (where it equals the reference's integer gather)."""
    import torch.nn.functional as F
    from oracle import lift_oracle
    torch.manual_seed(0)
    B, C, H, W = 3, 5, 9, 14
    fmap = torch.randn(B, C, H, W)
    rng = np.random.default_rng(0)
    coords = [np.stack([rng.uniform(-1.5, H + 0.5, n), rng.uniform(-1.5, W + 0.5, n)], 1).astype(np.float32) for n in (40, 0, 25)]
    coords[0][:6] = [[0, 0], [H - 1, W - 1], [3, 4], [H - 1, 2.5], [-1, -1], [H, W]]
    got = lift_oracle.lift2d_bilinear(fmap, coords)
    want = []
    for i, rc in enumerate(coords):
        rc = torch.from_numpy(rc)
        grid = torch.stack([2 * rc[:, 1] / (W - 1) - 1, 2 * rc[:, 0] / (H - 1) - 1], 1)[None, :, None, :]  # (x, y)
        want.append(F.grid_sample(fmap[i:i + 1], grid, mode="bilinear", padding_mode="zeros", align_corners=True)[0, :, :, 0].t())
    want = torch.cat(want, 0)
    assert got.shape == want.shape == (65, C)
    assert (got - want).abs().max().item() < 1e-5
    ints = [np.stack([rng.integers(0, H, 30), rng.integers(0, W, 30)], 1) for _ in range(B)]
    assert torch.allclose(lift_oracle.lift2d_bilinear(fmap, [x.astype(np.float32) for x in ints]), lift_oracle.lift2d(fmap, ints))
