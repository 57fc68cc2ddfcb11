"""Grouped BatchNorm statistics (``UNetSCN.forward_groups``) without a GPU: the C ABI's new symbols, the grouped size
queries against the existing ones, argument validation, and the oracle the GPU tests compare with -- G separate
passes of the FP64 network, whose running statistics compose in group order."""
import ctypes as C
import os
import re

import pytest
import torch

from mm2d3d_b200 import _lib
from mm2d3d_b200._lib import lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW = ["mm3d_group_bounds", "mm3d_bnrelu_workspace_bytes_grouped", "mm3d_bnrelu_fwd_grouped", "mm3d_bnrelu_bwd_grouped",
       "mm3d_unet_topo_act_bytes_grouped", "mm3d_unet_topo_scratch_bytes_grouped", "mm3d_unet_topo_forward_grouped",
       "mm3d_unet_topo_backward_grouped"]
TOPOLOGIES = [(1, 0), (2, 0), (1, 1), (2, 1)]


def test_symbols_declared_exported_bound_and_abi_unchanged():
    header = open(os.path.join(ROOT, "include", "mm3d.h")).read()
    for name in NEW:
        assert re.search(rf"MM3D_API \w+ {name}\(", header), name
        assert hasattr(lib, name), name
        assert name in _lib.SIGNATURES, name
    assert lib.mm3d_abi_version() == 8 == _lib.ABI_VERSION
    assert re.search(r"#define MM3D_LEVEL_DESC_WORDS 10\b", header)
    assert re.search(rf"#define MM3D_BN_MAX_GROUPS {_lib.BN_MAX_GROUPS}\b", header)


def _desc(L, n0=50000):
    W = _lib.LEVEL_DESC_WORDS
    desc = (C.c_int64 * (W * L))()
    n = n0
    for l in range(L):
        desc[W * l] = n
        n = max(n // 3, 1)
    return desc


@pytest.mark.parametrize("reps,res", TOPOLOGIES)
@pytest.mark.parametrize("mode", [0, 1, 2, 3])
def test_one_group_queries_equal_the_existing_ones(reps, res, mode):
    L, m = 7, 16
    desc = _desc(L)
    assert lib.mm3d_unet_topo_act_bytes_grouped(3, m, L, reps, res, mode, desc, 60000, 1) == \
        lib.mm3d_unet_topo_act_bytes(3, m, L, reps, res, mode, desc, 60000)
    for flags in (0, _lib.DETERMINISTIC):
        assert lib.mm3d_unet_topo_scratch_bytes_grouped(3, m, L, reps, res, mode, flags, 1) == \
            lib.mm3d_unet_topo_scratch_bytes_ex(3, m, L, reps, res, mode, flags)
    for c in (16, 96, 259, 512):
        for flags in (0, _lib.DETERMINISTIC):
            assert lib.mm3d_bnrelu_workspace_bytes_grouped(c, 1, flags) == lib.mm3d_bnrelu_workspace_bytes_ex(c, flags)


def _bn_widths(L, m, reps, res):
    """Channels of every BatchNorm of the network (module-tree order), from the constructor's topology."""
    from mm2d3d_b200.unet import level_plan
    widths = []
    for lvl in level_plan([m * (i + 1) for i in range(L)], reps):
        for a, b in lvl["pre"] + lvl["post"]:
            widths += [a, b] if res else [a]
        if lvl["deeper"] is not None:
            widths += [lvl["planes"], lvl["deeper"]]
    return widths + [m]


@pytest.mark.parametrize("reps,res", TOPOLOGIES)
@pytest.mark.parametrize("G", [2, 3, 8])
def test_queries_grow_with_the_groups_only_by_the_statistics(reps, res, G):
    """act grows by the saved statistics (G - 1 more [2, C] rows per BatchNorm, each piece 256-byte aligned); the
    scratch buffer by the BatchNorm workspace (G times the accumulators); the backward temporaries not at all."""
    L, m, mode = 7, 16, 1
    desc = _desc(L)
    al = lambda x: (x + 255) // 256 * 256
    one = lib.mm3d_unet_topo_act_bytes(3, m, L, reps, res, mode, desc, 60000)
    grown = lib.mm3d_unet_topo_act_bytes_grouped(3, m, L, reps, res, mode, desc, 60000, G)
    want = sum(al(4 * 2 * G * c) - al(4 * 2 * c) for c in _bn_widths(L, m, reps, res))
    assert grown - one == want
    for flags in (0, _lib.DETERMINISTIC):
        s1 = lib.mm3d_unet_topo_scratch_bytes_ex(3, m, L, reps, res, mode, flags)
        sg = lib.mm3d_unet_topo_scratch_bytes_grouped(3, m, L, reps, res, mode, flags, G)
        # (the deterministic layout keeps the default BatchNorm workspace in front of its own)
        grow = sum(al(lib.mm3d_bnrelu_workspace_bytes_grouped(2 * m * L, G, f)) - al(lib.mm3d_bnrelu_workspace_bytes_ex(2 * m * L, f))
                   for f in {0, flags})
        assert sg - s1 == grow
        assert lib.mm3d_bnrelu_workspace_bytes_grouped(2 * m * L, G, flags) == \
            lib.mm3d_bnrelu_workspace_bytes_ex(2 * m * L * G, flags)


def test_argument_validation():
    assert lib.mm3d_bnrelu_workspace_bytes_grouped(16, 0, 0) == 0
    assert lib.mm3d_bnrelu_workspace_bytes_grouped(16, _lib.BN_MAX_GROUPS + 1, 0) == 0
    assert lib.mm3d_unet_topo_act_bytes_grouped(3, 16, 7, 1, 0, 1, _desc(7), 1000, 0) == 0
    assert lib.mm3d_unet_topo_scratch_bytes_grouped(3, 16, 7, 1, 0, 1, 0, _lib.BN_MAX_GROUPS + 1) == 0
    n = 100
    for G, bounds in [(0, [0, n]), (_lib.BN_MAX_GROUPS + 1, [0] * _lib.BN_MAX_GROUPS + [n, n]), (2, [1, 50, n]),
                      (2, [0, 50, n - 1]), (2, [0, 60, 50])]:
        b = (C.c_int64 * len(bounds))(*bounds)
        # (rejected before any CUDA call: NULL device pointers are never touched)
        assert lib.mm3d_bnrelu_fwd_grouped(None, None, n, 16, None, None, None, None, None, None, 1e-4, 0.9, 0.0, 1,
                                           None, 0, None, 0, G, b) == 1, (G, bounds)
        assert lib.mm3d_bnrelu_bwd_grouped(None, None, None, n, 16, None, None, None, None, None, None, 0.0, 1, None, 0,
                                           None, 0, G, b) == 1, (G, bounds)
    # the executor: groups without boundaries, and boundaries that do not end at a level's row count
    L = 7
    desc = _desc(L)
    g = _lib.UnetGroups(2, None)
    assert lib.mm3d_unet_topo_forward_grouped(3, 16, L, 1, 0, 1, 1, 1e-4, 0.9, desc, 1000, None, None, None, None, None,
                                              None, None, None, 0, None, 0, None, None, 0, C.byref(g)) == 1
    bad = (C.c_int64 * (3 * L))(*[v for l in range(L) for v in (0, 1, desc[_lib.LEVEL_DESC_WORDS * l] + 1)])
    g = _lib.UnetGroups(2, C.addressof(bad))
    assert lib.mm3d_unet_topo_forward_grouped(3, 16, L, 1, 0, 1, 1, 1e-4, 0.9, desc, 1000, None, None, None, None, None,
                                              None, None, None, 0, None, 0, None, None, 0, C.byref(g)) == 1
    assert "boundaries" in lib.mm3d_last_error().decode()


def test_forward_groups_rejects_bad_group_lists():
    from mm2d3d_b200.metadata import group_coords
    from mm2d3d_b200.unet import UNetSCN
    net = UNetSCN(in_channels=3, m=8, num_planes=3)
    c = torch.zeros(4, 4, dtype=torch.int64)
    f = torch.zeros(4, 3)
    with pytest.raises(ValueError, match="non-empty"):
        net.forward_groups([], [])
    with pytest.raises(ValueError, match="at most 8"):
        net.forward_groups([c] * 9, [f] * 9)
    with pytest.raises(ValueError, match="2 coordinate groups but 3"):
        net.forward_groups([c, c], [f, f, f])
    with pytest.raises(ValueError, match="at most"):
        group_coords([c] * 9)
    with pytest.raises(ValueError, match="non-empty"):
        group_coords([])


# ------------------------------------------------------------------------------ the oracle: G separate passes
def grouped_oracle(net, coords, feats, g_out, lin=None):
    """What ``forward_groups`` must equal: one forward + backward per group on `net` (any dtype), in group order, the
    running statistics evolving from pass to pass; outputs and feature gradients per group, parameter gradients
    summed over the groups.  `lin`: the RGB mask (``feats * sigmoid(lin(feats))`` in front of the network), whose
    gradients are summed too, as ``mask.weight`` / ``mask.bias``.  Returns (outs, feature grads, {name: summed grad},
    {name: buffer after the last pass})."""
    params = dict(net.named_parameters())
    if lin is not None:
        params.update({"mask." + k: v for k, v in lin.named_parameters()})
    outs, gx, total = [], [], {k: torch.zeros_like(p) for k, p in params.items()}
    for c, f, g in zip(coords, feats, g_out):
        x = f.clone().requires_grad_(True)
        out = net([c, x * torch.sigmoid(lin(x)) if lin is not None else x])
        grads = torch.autograd.grad(out, [x] + list(params.values()), g)
        outs.append(out.detach())
        gx.append(grads[0])
        for k, d in zip(params, grads[1:]):
            total[k] += d
    return outs, gx, total, {k: b.clone() for k, b in net.named_buffers()}


def test_oracle_running_statistics_compose_in_group_order():
    """The oracle's G passes against a direct statement of the contract: after the groups, every BatchNorm's running
    statistics are the momentum update applied once per group, in order, with that group's batch mean and unbiased
    variance (n_g / (n_g - 1))."""
    from oracle import scn_cpu
    from mm2d3d_b200.unet import UNetSCN
    from tests.test_exec_fp64_cpu import bn_modules
    torch.manual_seed(0)
    net = UNetSCN(in_channels=3, m=8, num_planes=3, full_scale=64, backend=scn_cpu).double()
    gen = torch.Generator().manual_seed(1)
    coords, feats = [], []
    for n, b in [(300, 2), (120, 1), (200, 3)]:
        c = torch.cat([torch.randint(0, 64, (n, 3), generator=gen), torch.randint(0, b, (n, 1), generator=gen)], 1)
        coords.append(c)
        feats.append(torch.randn(n, 3, generator=gen, dtype=torch.float64))
    bns = bn_modules(net)
    start = [(b.running_mean.clone(), b.running_var.clone()) for b in bns]
    # the inputs every BatchNorm sees, per group (one separate pass each)
    seen = [[] for _ in bns]
    hooks = [b.register_forward_hook(lambda mod, inp, out, i=i: seen[i].append(inp[0].features.detach().clone()))
             for i, b in enumerate(bns)]
    g_out = [torch.randn(c.shape[0], 8, generator=gen, dtype=torch.float64) for c in coords]
    outs, gx, grads, buffers = grouped_oracle(net, coords, feats, g_out)
    for h in hooks:
        h.remove()
    assert len(outs) == 3 and all(o.shape == (c.shape[0], 8) for o, c in zip(outs, coords))
    for i, b in enumerate(bns):
        mean, var = start[i]
        assert len(seen[i]) == 3
        for x in seen[i]:
            n = x.shape[0]
            mean = b.momentum * mean + (1 - b.momentum) * x.mean(0)
            var = b.momentum * var + (1 - b.momentum) * x.var(0, unbiased=False) * n / max(n - 1, 1)
        torch.testing.assert_close(b.running_mean, mean, rtol=1e-12, atol=1e-12)
        torch.testing.assert_close(b.running_var, var, rtol=1e-12, atol=1e-12)
