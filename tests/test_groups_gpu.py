"""Grouped BatchNorm statistics on the GPU: ``UNetSCN.forward_groups`` / ``prepare_groups`` against G separate passes of
the FP64 oracle, the grouped BatchNorm kernels against FP64, the groups' row layout at every level, and the
equivalences (one group = a plain call, eval mode = the groups change nothing, deterministic = the same bits)."""
import copy

import pytest
import torch

from mm2d3d_b200 import _lib, synth
from tests.test_exec_fp64_cpu import conditioned_net, mask_linear, output_grad, scan
from tests.test_exec_fp64_gpu import BAR, _settings
from tests.test_gpu_parity import DEV, _no_device_error, rel_err, rel_l2
from tests.test_groups_cpu import grouped_oracle

pytestmark = pytest.mark.gpu

MODES = ["fp32", "tf32", "tf32x3", "bf16"]


def _split_scan():
    """scan()'s two nuScenes-shaped scans as two groups, each with its batch column from 0."""
    coords, feats = scan()
    groups = []
    for b in (0, 1):
        sel = coords[:, 3] == b
        c = coords[sel].clone()
        c[:, 3] = 0
        groups.append((c, feats[sel].clone()))
    return [g[0] for g in groups], [g[1] for g in groups]


# ---------------------------------------------------------------------------------------------- row layout
def test_group_rows_are_contiguous_at_every_level():
    """Each group is one contiguous row range at every level, as long as its own structure's row count; the grouped
    structure's keys are the groups' keys one after the other (batch offset).  The second group lists its scans out of
    batch-index order."""
    from mm2d3d_b200.metadata import Metadata, group_coords
    locs, _ = synth.make_batch("nuscenes", batch=3, seed0=5)
    locs = torch.from_numpy(locs)
    a = locs[locs[:, 3] == 0]
    b = torch.cat([locs[locs[:, 3] == 2], locs[locs[:, 3] == 1]])  # scan 1 after scan 2
    b[:, 3] -= 1
    groups = [a.to(DEV), b.to(DEV), a[:1].to(DEV)]  # (and a group of one point)
    spatial, L = 4096, 7
    c, batch_start = group_coords(groups)
    meta = Metadata(c, spatial, L, defer_sync=True, batch_start=batch_start)
    bounds = meta.group_bounds()
    assert batch_start.tolist() == [0, 1, 3, 4]
    s = spatial
    for l in range(L):
        sep = [Metadata(g, spatial, L).coords_at(s) for g in groups]
        bl = bounds[l]
        assert bl[0] == 0 and bl[-1] == meta.level(s).n
        keys = meta.coords_at(s)
        for k, cs in enumerate(sep):
            assert bl[k + 1] - bl[k] == cs.shape[0], (l, k)
            got = keys[bl[k]:bl[k + 1]].clone()
            got[:, 3] -= batch_start[k]
            assert torch.equal(got, cs), (l, k)
        s //= 2
    _no_device_error()


# ---------------------------------------------------------------------------------------------- BatchNorm op
def _bn_case(c, sizes, seed):
    gen = torch.Generator().manual_seed(seed)
    n = sum(sizes)
    x = (torch.randn(n, c, generator=gen, dtype=torch.float64) * 2 + torch.randn(c, generator=gen, dtype=torch.float64))
    gamma = 1 + 0.2 * torch.randn(c, generator=gen, dtype=torch.float64)
    beta = torch.randn(c, generator=gen, dtype=torch.float64)
    dy = torch.randn(n, c, generator=gen, dtype=torch.float64)
    rm, rv = torch.randn(c, generator=gen, dtype=torch.float64), 1 + torch.rand(c, generator=gen, dtype=torch.float64)
    return x, gamma, beta, dy, rm, rv


def _bn_fp64(x, gamma, beta, dy, rm, rv, bounds, eps=1e-4, mom=0.9):
    """Grouped BatchNorm+ReLU forward / backward in FP64, one group after the other."""
    x = x.clone().requires_grad_(True)
    g = gamma.clone().requires_grad_(True)
    b = beta.clone().requires_grad_(True)
    ys = []
    rm, rv = rm.clone(), rv.clone()
    for lo, hi in zip(bounds[:-1], bounds[1:]):
        xs = x[lo:hi]
        n = hi - lo
        mean, var = xs.mean(0), xs.var(0, unbiased=False)
        ys.append(torch.relu((xs - mean) / torch.sqrt(var + eps) * g + b))
        rm = mom * rm + (1 - mom) * mean.detach()
        rv = mom * rv + (1 - mom) * var.detach() * n / max(n - 1, 1)
    y = torch.cat(ys)
    dx, dg, db = torch.autograd.grad(y, [x, g, b], dy)
    return y.detach(), dx, dg, db, rm, rv


def _bn_gpu(x, gamma, beta, dy, rm, rv, bounds, det=False):
    from mm2d3d_b200 import functional as F
    t = lambda v: v.float().to(DEV)
    rm_, rv_ = t(rm), t(rv)
    xg = t(x).requires_grad_(True)
    gg, bg = t(gamma).requires_grad_(True), t(beta).requires_grad_(True)
    prev = F.DETERMINISTIC
    F.DETERMINISTIC = det
    try:
        y = F.BatchNormReLUFn.apply(xg, gg, bg, rm_, rv_, 1e-4, 0.9, 0.0, True, tuple(bounds))
        dx, dg, db = torch.autograd.grad(y, [xg, gg, bg], t(dy))
    finally:
        F.DETERMINISTIC = prev
    return y.detach(), dx, dg, db, rm_, rv_


@pytest.mark.parametrize("c", [16, 96, 99, 259, 512])
@pytest.mark.parametrize("sizes", [(5000, 1), (1, 7000, 300), (40000, 30000)], ids=lambda s: "-".join(map(str, s)))
def test_grouped_bnrelu_against_fp64(c, sizes):
    x, gamma, beta, dy, rm, rv = _bn_case(c, sizes, seed=c + len(sizes))
    bounds = [0]
    for s in sizes:
        bounds.append(bounds[-1] + s)
    # no upstream gradient where the FP64 pre-activation lies within 1e-3 of the ReLU kink: FP32 round-off may flip
    # that gate, which moves dx there by O(1) without any error in the kernel (the gates still vary per row)
    for lo, hi in zip(bounds[:-1], bounds[1:]):
        xs = x[lo:hi]
        pre = (xs - xs.mean(0)) / torch.sqrt(xs.var(0, unbiased=False) + 1e-4) * gamma + beta
        dy[lo:hi][pre.abs() < 1e-3] = 0
    want = _bn_fp64(x, gamma, beta, dy, rm, rv, bounds)
    for det in (False, True):
        got = _bn_gpu(x, gamma, beta, dy, rm, rv, bounds, det)
        for name, g_, w in zip(["y", "dx", "d_gamma", "d_beta", "running_mean", "running_var"], got, want):
            e = rel_err(g_, w)
            assert e < 1e-4, (c, sizes, det, name, e)
        if det:
            again = _bn_gpu(x, gamma, beta, dy, rm, rv, bounds, det)
            assert all(torch.equal(a, b) for a, b in zip(got, again)), (c, sizes)
    _no_device_error()


# ---------------------------------------------------------------------------------------------- whole network
def _scans(batches):
    """Groups of nuScenes-shaped scans (batch sizes `batches`, each group's batch column from 0), coordinates halved
    like scan() so that voxels hold several points; "1+1" is scan()'s two scans as two groups."""
    if batches == (1, 1):
        return _split_scan()
    coords, feats = [], []
    for k, b in enumerate(batches):
        locs, f = synth.make_batch("nuscenes", batch=b, seed0=3 + 100 * k)
        locs[:, :3] //= 2
        coords.append(torch.from_numpy(locs))
        feats.append(torch.from_numpy(f))
    return coords, feats


def _oracle_groups(batches, reps, res, m, mask):
    """FP64 oracle of the grouped step: G separate passes of the conditioned network (and RGB mask)."""
    net, _ = conditioned_net(reps, res, m)
    lin = mask_linear() if mask else None
    state = copy.deepcopy(net.state_dict())
    mask_state = copy.deepcopy(lin.state_dict()) if mask else None
    coords, feats = _scans(batches)
    g = output_grad(sum(c.shape[0] for c in coords), m)
    g_out = list(g.split([c.shape[0] for c in coords]))
    net64 = copy.deepcopy(net).double()
    lin64 = copy.deepcopy(lin).double() if mask else None
    outs, gx, grads, buffers = grouped_oracle(net64, coords, [f.double() for f in feats], g_out, lin64)
    return {"state": state, "mask_state": mask_state, "coords": coords, "feats": feats, "g": g_out, "outs": outs,
            "gx": gx, "grads": grads, "buffers": buffers}


_CACHE = {}


def _oracle(batches=(1, 1), reps=1, res=False, m=16, mask=False):
    key = (batches, reps, res, m, mask)
    if key not in _CACHE:
        _CACHE[key] = _oracle_groups(*key)
    return _CACHE[key]


def _gpu_groups(ref, reps, res, mode, fused=True, prepared=False, m=16):
    """The grouped step on the GPU from the oracle's initial state.  `prepared`: the structure from prepare_groups
    (built before `fused` is applied, so the module path also runs from a prepared structure)."""
    from mm2d3d_b200.unet import UNetSCN
    net = UNetSCN(in_channels=3, m=m, block_reps=reps, residual_blocks=res).to(DEV)
    net.load_state_dict(ref["state"])
    params = dict(net.named_parameters())
    lin = None
    if ref["mask_state"] is not None:
        lin = torch.nn.Linear(3, 1).to(DEV)
        lin.load_state_dict(ref["mask_state"])
        params.update({"mask." + k: v for k, v in lin.named_parameters()})
    coords = [c.to(DEV) for c in ref["coords"]]
    xs = [f.to(DEV).requires_grad_(True) for f in ref["feats"]]
    with _settings(mode):
        src = net.prepare_groups(coords) if prepared else coords
        net.fused = fused
        outs = net.forward_groups(src, xs, rgb_mask=lin)
        # the outputs are views of one output: of the executor's, or of the module path's OutputLayer
        node = type(outs[0].grad_fn.next_functions[0][0]).__name__
        assert node == ("UNetSCNFnBackward" if fused else "OutputLayerFnBackward"), node
        torch.autograd.backward(outs, [g.float().to(DEV) for g in ref["g"]])
    _no_device_error()
    return params, net, outs, xs


def _separate_gpu(ref, reps, res, mode, m=16):
    """What the grouped step replaces, on the GPU: one plain call per group in group order, one backward of both,
    from the same initial state (parameter gradients sum in p.grad)."""
    from mm2d3d_b200.unet import UNetSCN
    net = UNetSCN(in_channels=3, m=m, block_reps=reps, residual_blocks=res).to(DEV)
    net.load_state_dict(ref["state"])
    params = dict(net.named_parameters())
    lin = None
    if ref["mask_state"] is not None:
        lin = torch.nn.Linear(3, 1).to(DEV)
        lin.load_state_dict(ref["mask_state"])
        params.update({"mask." + k: v for k, v in lin.named_parameters()})
    xs = [f.to(DEV).requires_grad_(True) for f in ref["feats"]]
    with _settings(mode):
        outs = [net([c.to(DEV), x], rgb_mask=lin) for c, x in zip(ref["coords"], xs)]
        torch.autograd.backward(outs, [g.float().to(DEV) for g in ref["g"]])
    _no_device_error()
    return params, net, outs, xs


def _rows(ref, params, net, outs, xs):
    rows = []
    for k in range(len(outs)):
        rows.append((f"out[{k}]", outs[k].detach(), ref["outs"][k]))
        rows.append((f"feats.grad[{k}]", xs[k].grad, ref["gx"][k]))
    rows += [(k, p.grad, ref["grads"][k]) for k, p in params.items()]
    rows += [(k, b, ref["buffers"][k]) for k, b in net.named_buffers()]
    assert len(rows) == 2 * len(outs) + len(ref["grads"]) + len(ref["buffers"])
    return {k: (rel_l2(a, b), rel_err(a, b)) for k, a, b in rows}


def _check_network(tag, ref, got, bar, separate):
    """Every tensor of the grouped step within `bar` of the FP64 oracle (rel-L2 and max-abs-rel), or, where the two
    separate calls it replaces are themselves further than `bar` from the oracle (TF32 / BF16 operand rounding at a few
    ReLU gates of a 16-scan batch), within 1.25 times their error.  Both sets of figures are printed."""
    g, s_ = _rows(ref, *got), _rows(ref, *separate)
    worst = max(g, key=lambda k: g[k][0])
    print(f"\n[{tag}] grouped vs FP64 oracle (G separate passes), bar {bar:.0e}: worst rel-L2 {g[worst][0]:.2e} "
          f"({worst}); the two separate calls: {s_[worst][0]:.2e}; worst grouped - separate difference of figures "
          f"{max(abs(g[k][0] - s_[k][0]) for k in g):.2e}")
    b = max(bar, 1e-4)
    failed = [(k, g[k], s_[k]) for k in g
              if not (g[k][0] <= max(b, 1.25 * s_[k][0]) and g[k][1] <= max(b, 1.25 * s_[k][1]))]
    beyond = [(k, g[k], s_[k]) for k in g if not (g[k][0] <= b and g[k][1] <= b)]
    if beyond:
        print(f"[{tag}] beyond the bar, with the separate calls' figures: {beyond}")
    assert not failed, (tag, failed)


# (groups' batch sizes, mode, fused, prepared, RGB mask): 8 + 8 scans with the mask in every mode, on both paths and
# from a prepared structure; the unequal 3 + 8 split
CASES = [((8, 8), mode, True, False, True) for mode in MODES]
CASES += [((8, 8), "tf32", True, True, True), ((8, 8), "fp32", False, False, True), ((8, 8), "bf16", False, True, True)]
CASES += [((3, 8), "tf32", True, False, False), ((3, 8), "fp32", False, False, False)]


def _case_id(c):
    batches, mode, fused, prepared, mask = c
    return (f"{batches[0]}+{batches[1]}-{mode}-{'fused' if fused else 'modules'}{'-prepared' if prepared else ''}"
            f"{'-mask' if mask else ''}")


@pytest.mark.parametrize("batches,mode,fused,prepared,mask", CASES, ids=[_case_id(c) for c in CASES])
def test_grouped_step_against_fp64(batches, mode, fused, prepared, mask):
    ref = _oracle(batches, mask=mask)
    got = _gpu_groups(ref, 1, False, mode, fused, prepared)
    _check_network(_case_id((batches, mode, fused, prepared, mask)), ref, got, BAR[mode],
                   _separate_gpu(ref, 1, False, mode))


@pytest.mark.parametrize("topo", [(2, False), (1, True)], ids=["reps2", "residual"])
def test_grouped_step_topologies(topo):
    ref = _oracle((1, 1), *topo)
    got = _gpu_groups(ref, *topo, "tf32")
    _check_network(f"tf32 {topo}", ref, got, BAR["tf32"], _separate_gpu(ref, *topo, "tf32"))


@pytest.mark.parametrize("mode", ["tf32", "tf32x3"])
def test_grouped_step_width_32(mode):
    """m = 32: the 512-thread BatchNorm (the joins' 448 channels) and the sliced decoder convolutions."""
    ref = _oracle((1, 1), m=32)
    got = _gpu_groups(ref, 1, False, mode, m=32)
    _check_network(f"{mode} m=32", ref, got, BAR[mode], _separate_gpu(ref, 1, False, mode, m=32))


# ---------------------------------------------------------------------------------------------- equivalences
def _net(m=16):
    from mm2d3d_b200.unet import UNetSCN
    torch.manual_seed(3)
    return UNetSCN(in_channels=3, m=m).to(DEV)


def test_one_group_is_a_plain_call():
    """(deterministic mode: the default kernels' atomics make two plain calls differ in the last bits already)"""
    coords, feats = _split_scan()
    c, f = coords[0].to(DEV), feats[0].to(DEV)
    g = torch.randn(c.shape[0], 16, device=DEV)
    results = []
    for grouped in (False, True):
        net = _net()
        with _settings("tf32", det=True):
            x = f.clone().requires_grad_(True)
            n0 = _lib.lib.mm3d_kernel_launches()
            out = net.forward_groups([c], [x])[0] if grouped else net([c, x])
            out.backward(g)
            torch.cuda.synchronize()
            launches = _lib.lib.mm3d_kernel_launches() - n0
        results.append((out.detach(), x.grad, [p.grad for p in net.parameters()], launches))
    a, b = results
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and all(torch.equal(p, q) for p, q in zip(a[2], b[2]))
    assert a[3] == b[3]


def test_eval_mode_groups_change_nothing():
    coords, feats = _split_scan()
    coords, feats = [c.to(DEV) for c in coords], [f.to(DEV) for f in feats]
    net = _net().eval()
    with _settings("bf16", det=True):  # (bit comparison: the InputLayer's point sums in a fixed order)
        with torch.no_grad():
            outs = net.forward_groups(coords, feats)
            for o, c, f in zip(outs, coords, feats):
                assert torch.equal(o, net([c, f]))
            assert outs[0].grad_fn is None
        xs = [f.clone().requires_grad_(True) for f in feats]
        outs = net.forward_groups(coords, xs)
        for o, c, f in zip(outs, coords, feats):
            assert torch.equal(o.detach(), net([c, f.clone().requires_grad_(True)]).detach())
        # a prepared structure of both groups: one eval forward over it, the same values up to rounding
        with torch.no_grad():
            outs_p = net.forward_groups(net.prepare_groups(coords), feats)
        for o, p_ in zip(outs, outs_p):
            assert rel_err(p_, o.detach()) < BAR["bf16"]
    _no_device_error()


@pytest.mark.parametrize("mode", ["tf32", "tf32x3", "bf16"])
def test_deterministic_grouped_step_is_bit_reproducible(mode):
    coords, feats = _split_scan()
    runs = []
    for _ in range(2):
        net = _net()
        cs, xs = [c.to(DEV) for c in coords], [f.to(DEV).requires_grad_(True) for f in feats]
        with _settings(mode, det=True):
            outs = net.forward_groups(cs, xs)
            torch.autograd.backward(outs, [torch.ones_like(o) for o in outs])
        runs.append([o.detach() for o in outs] + [x.grad for x in xs] + [p.grad for p in net.parameters()]
                    + [b.clone() for b in net.buffers()])
    assert all(torch.equal(a, b) for a, b in zip(*runs))
    # one flat gradient tensor: FlatGradAllReduce finds the common base
    import types
    from mm2d3d_b200.dp import FlatGradAllReduce
    assert FlatGradAllReduce._common_base(types.SimpleNamespace(params=list(net.parameters()))) is not None


def test_grouped_step_launches_fewer_kernels_than_two_calls():
    coords, feats = _split_scan()
    cs, fs = [c.to(DEV) for c in coords], [f.to(DEV) for f in feats]
    counts = []
    for grouped in (False, True):
        net = _net()
        with _settings("tf32"):
            for rep in range(2):  # (the second pass is counted: the first loads modules)
                xs = [f.clone().requires_grad_(True) for f in fs]
                torch.cuda.synchronize()
                n0 = _lib.lib.mm3d_kernel_launches()
                outs = net.forward_groups(cs, xs) if grouped else [net([c, x]) for c, x in zip(cs, xs)]
                torch.autograd.backward(outs, [torch.ones_like(o) for o in outs])
                torch.cuda.synchronize()
                n = _lib.lib.mm3d_kernel_launches() - n0
        counts.append(n)
    print(f"\nlibmm3d launches per step: two calls {counts[0]}, forward_groups {counts[1]}")
    assert counts[1] < counts[0]
