"""Inference forward of the whole-network executor (mm3d_unet_topo_infer) on the GPU: the same bytes as the existing
eval forward in every mode and block topology, dispatch, no side effects, launches and memory, the workspace
contract and prepared structures."""
import contextlib
import copy

import numpy as np
import pytest
import torch

from mm2d3d_b200 import synth
from tests.test_gpu_parity import DEV, _no_device_error

pytestmark = pytest.mark.gpu

MODES = ["fp32", "tf32", "tf32x3", "bf16"]
CONFIGS = [(1, False), (2, False), (1, True), (2, True)]
MM3D_ERR_WORKSPACE = 3
WS_BYTES = 17  # position of ws_bytes among mm3d_unet_topo_infer's arguments


@pytest.fixture
def every_mode(monkeypatch):
    """The inference path in every convolution mode (the executor takes it only where it measured faster)."""
    from mm2d3d_b200 import _lib, executor
    monkeypatch.setattr(executor, "INFER_MODES", frozenset(_lib.MODES.values()))


def _ids(cfg):
    return f"reps{cfg[0]}-{'res' if cfg[1] else 'vgg'}"


@contextlib.contextmanager
def _modes(conv="fp32", det=False):
    import mm2d3d_b200.scn as scn
    scn.set_conv_mode(conv)
    scn.set_deterministic(det)
    try:
        yield
    finally:
        scn.set_conv_mode("fp32")
        scn.set_deterministic(False)


def _batch(seed0, unique, batch=2, div=8):
    """nuScenes-shaped scans, coarsened; unique: one point per voxel (no order-dependent float atomics in the
    InputLayer), else several points per voxel (for the deterministic mode)."""
    locs, feats = synth.make_batch("nuscenes", batch=batch, seed0=seed0)
    locs[:, :3] //= div
    if unique:
        locs, first = np.unique(locs, axis=0, return_index=True)
        feats = feats[first]
    return torch.from_numpy(locs).to(DEV), torch.from_numpy(feats).to(DEV)


def _net(reps, res, m=16, seed=0):
    """An eval-mode network with non-trivial running statistics and BatchNorm affine parameters (both ReLU gate signs
    in every layer), and an RGB mask."""
    import mm2d3d_b200.scn as scn
    from mm2d3d_b200.unet import UNetSCN
    torch.manual_seed(seed)
    net = UNetSCN(in_channels=3, m=m, block_reps=reps, residual_blocks=res).to(DEV)
    with torch.no_grad():
        for mod in net.modules():
            if isinstance(mod, scn.BatchNormLeakyReLU):
                mod.weight.copy_(1 + 0.3 * torch.randn_like(mod.weight))
                mod.bias.copy_(0.2 * torch.randn_like(mod.bias))
                mod.running_mean.copy_(0.3 * torch.randn_like(mod.running_mean))
                mod.running_var.copy_(0.5 + torch.rand_like(mod.running_var))
    mask = torch.nn.Linear(3, 1).to(DEV)
    return net.eval(), mask


class _Spy:
    """The executor's library handle, counting calls of the inference entry point."""

    def __init__(self, lib, short=0):
        self._lib, self.short = lib, short
        self.calls, self.rc, self.launches = 0, None, None

    def __getattr__(self, name):
        return getattr(self._lib, name)

    def mm3d_unet_topo_infer(self, *args):
        args = list(args)
        args[WS_BYTES] -= self.short
        self.calls += 1
        n0 = self._lib.mm3d_kernel_launches()
        self.rc = self._lib.mm3d_unet_topo_infer(*args)
        self.launches = self._lib.mm3d_kernel_launches() - n0
        return self.rc


def _bits(t):
    return t.detach().contiguous().view(torch.int32).clone()


def _both(net, inp, mask=None):
    """(existing eval forward through the autograd function, inference forward), each as int32 bits."""
    old = net(inp, rgb_mask=mask)  # grad mode on, parameters require grad: UNetSCNFn
    assert old.requires_grad
    with torch.no_grad():
        new = net(inp, rgb_mask=mask)
    assert not new.requires_grad
    return _bits(old), _bits(new)


def _check_identity(net, mask, coords, feats, tag):
    for use_mask in (False, True):
        old, new = _both(net, [coords, feats], mask if use_mask else None)
        diff = int((old != new).sum())
        assert diff == 0, (tag, use_mask, diff, old.numel())
        neg = float((new.view(torch.float32) <= 0).float().mean())
        assert 0.0 < neg < 1.0, (tag, neg)  # (the head's gates: both signs)


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("cfg", CONFIGS, ids=_ids)
def test_inference_bytes_equal_eval_forward(cfg, mode, every_mode):
    """Byte equality with the existing eval forward, with and without the RGB mask: one point per voxel in the
    default mode, several points per voxel in the deterministic mode."""
    reps, res = cfg
    net, mask = _net(reps, res, seed=reps + 2 * res)
    with _modes(mode):
        _check_identity(net, mask, *_batch(3, unique=True), (mode, cfg, "default"))
    with _modes(mode, det=True):
        _check_identity(net, mask, *_batch(4, unique=False), (mode, cfg, "deterministic"))
    _no_device_error()


@pytest.mark.parametrize("mode", ["fp32", "tf32"])
@pytest.mark.parametrize("cfg", [(1, False), (1, True)], ids=_ids)
def test_inference_bytes_equal_with_m8(cfg, mode, every_mode):
    """m = 8: in tf32 the 8-, 24-, 40-channel layers run the SIMT kernel, the others tcgen05."""
    net, mask = _net(*cfg, m=8, seed=7)
    with _modes(mode):
        _check_identity(net, mask, *_batch(5, unique=True), (mode, cfg, "m8"))
    with _modes(mode, det=True):
        _check_identity(net, mask, *_batch(6, unique=False), (mode, cfg, "m8 deterministic"))
    _no_device_error()


def test_dispatch(monkeypatch):
    """Under no_grad / inference_mode in eval mode the inference entry point is called (bf16 mode; in tf32 only once
    the mode is listed in INFER_MODES); in training mode, or with a tensor that requires a gradient, it is not."""
    from mm2d3d_b200 import _lib, executor
    net, mask = _net(1, False)
    coords, feats = _batch(7, unique=True)
    for mode, listed in (("bf16", True), ("tf32", False), ("tf32", True)):
        with _modes(mode), monkeypatch.context() as mp:
            if listed:
                mp.setattr(executor, "INFER_MODES", executor.INFER_MODES | {_lib.MODES[mode]})
            want = 2 if mode in ("bf16",) or listed else 0
            for ctx in (torch.no_grad, torch.inference_mode):
                spy = _Spy(_lib.lib)
                mp.setattr(executor, "lib", spy)
                with ctx():
                    out = net([coords, feats])
                    out_m = net([coords, feats], rgb_mask=mask)
                assert spy.calls == want and not out.requires_grad and not out_m.requires_grad, (mode, listed, ctx)
            if not want:
                continue
            # frozen network, grad mode on: nothing requires a gradient -> inference
            spy = _Spy(_lib.lib)
            mp.setattr(executor, "lib", spy)
            for p in net.parameters():
                p.requires_grad_(False)
            out = net([coords, feats])
            assert spy.calls == 1 and not out.requires_grad
            out = net([coords, feats.clone().requires_grad_(True)])  # features need a gradient
            assert spy.calls == 1 and out.requires_grad
            for p in net.parameters():
                p.requires_grad_(True)
            net([coords, feats])  # eval, grad mode on, parameters require grad
            net.train()
            with torch.no_grad():
                net([coords, feats])  # training mode
            net.eval()
            assert spy.calls == 1
    _no_device_error()


def test_no_side_effects_and_following_training_step(every_mode):
    """Parameters and running statistics are byte-unchanged by an inference forward; a deterministic tf32 training
    step after one gives the bits of the step without it."""
    net_a, mask = _net(1, True)
    net_b = copy.deepcopy(net_a)
    coords, feats = _batch(8, unique=False)
    g = torch.randn(coords.shape[0], 16, device=DEV, generator=torch.Generator(device=DEV).manual_seed(1))
    before = [_bits(t) if t.dtype == torch.float32 else t.clone() for t in net_b.state_dict().values()]
    with _modes("tf32", det=True):
        with torch.no_grad():
            net_b([coords, feats], rgb_mask=mask)
        after = [_bits(t) if t.dtype == torch.float32 else t.clone() for t in net_b.state_dict().values()]
        assert all(torch.equal(a, b) for a, b in zip(before, after))
        res = []
        for net in (net_a, net_b):
            net.train()
            x = feats.clone().requires_grad_(True)
            out = net([coords, x], rgb_mask=mask)
            grads = torch.autograd.grad(out, [x] + list(net.parameters()), g)
            res.append([_bits(out)] + [_bits(t) for t in grads] + [_bits(b) for b in net.buffers() if b.dtype == torch.float32])
    assert all(torch.equal(a, b) for a, b in zip(*res))
    _no_device_error()


def _kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


@pytest.mark.parametrize("cfg", CONFIGS, ids=_ids)
def test_launches_and_memory(cfg, every_mode):
    """The inference forward issues no standalone BatchNorm and no join kernel, fewer launches than the existing eval
    forward, and allocates less memory at its peak (counts printed)."""
    from mm2d3d_b200 import _lib
    net, _ = _net(*cfg)
    coords, feats = _batch(9, unique=True, div=4)
    with _modes("tf32"):
        prep = net.prepare(coords, wait=True)
        stats = {}
        for arm in ("old", "infer", "old", "infer"):
            def run():
                if arm == "old":
                    return net([prep, feats]).detach()
                with torch.no_grad():
                    return net([prep, feats])
            torch.cuda.synchronize()
            base = torch.cuda.memory_allocated()
            torch.cuda.reset_peak_memory_stats()
            n0 = _lib.lib.mm3d_kernel_launches()
            out = run()
            torch.cuda.synchronize()
            stats[arm] = (_lib.lib.mm3d_kernel_launches() - n0, torch.cuda.max_memory_allocated() - base)
            del out

        def infer():
            with torch.no_grad():
                net([prep, feats])
        names = _kernels(infer)
    bad = [k for k in names if ("k_bn_" in k and "k_bn_scales" not in k) or "k_concat2" in k or "k_copy_cols" in k]
    print(f"\n{_ids(cfg)} tf32: launches per forward eval {stats['old'][0]} -> inference {stats['infer'][0]}, peak "
          f"allocated {stats['old'][1] / 2**20:.1f} -> {stats['infer'][1] / 2**20:.1f} MiB; inference kernels: "
          f"{sorted(set(names))}")
    assert not bad, bad
    assert stats["infer"][0] < stats["old"][0]
    assert stats["infer"][1] < stats["old"][1]
    _no_device_error()


@pytest.mark.parametrize("mode", ["tf32", "bf16"])
@pytest.mark.parametrize("cfg", [(1, False), (2, True)], ids=_ids)
def test_workspace_query_is_exact(monkeypatch, cfg, mode, every_mode):
    from mm2d3d_b200 import _lib, executor
    net, _ = _net(*cfg)
    coords, feats = _batch(10, unique=True)
    with _modes(mode):
        for short in (1, 0):
            spy = _Spy(_lib.lib, short)
            with monkeypatch.context() as mp, torch.no_grad():
                mp.setattr(executor, "lib", spy)
                if short:
                    with pytest.raises(_lib.Mm3dError, match="inference workspace too small"):
                        net([coords, feats])
                else:
                    net([coords, feats])
            torch.cuda.synchronize()
            if short:
                assert spy.rc == MM3D_ERR_WORKSPACE and spy.launches == 0, (spy.rc, spy.launches)
            else:
                assert spy.rc == 0 and spy.launches > 0, (spy.rc, spy.launches)
    _no_device_error()


@pytest.mark.parametrize("det", [False, True], ids=["default", "deterministic"])
def test_prepared_structures_on_side_stream(det, every_mode):
    """prepare(coords) and prepare_points(raw points), built on a side stream, give the coordinate input's bytes."""
    from mm2d3d_b200.augment import scale_points
    scans = [synth.raycast_points("nuscenes", seed) for seed in (5, 6)]
    offs = np.concatenate([[0], np.cumsum([len(p) for p in scans])]).astype(np.int64)
    pts = torch.from_numpy(np.concatenate(scans, 0)).to(DEV)
    rot = np.stack([np.eye(3, dtype=np.float32)] * 2)
    coords, keep, _, _ = scale_points(pts, offs, rot, None, 20.0, 4096)
    assert bool(keep.all())
    net, mask = _net(2, True)
    with _modes("tf32", det=det), torch.no_grad():
        # (several points per voxel: the default mode's InputLayer sums in atomic order, so there one point per voxel)
        x = torch.rand(len(coords), 3, device=DEV, generator=torch.Generator(device=DEV).manual_seed(2))
        if not det:
            _, first = np.unique(coords.cpu().numpy(), axis=0, return_index=True)
            sel = torch.from_numpy(np.sort(first)).to(DEV)
            pts, coords, x = pts[sel], coords[sel], x[sel]
            offs = np.array([0, int((sel < offs[1]).sum()), len(sel)], dtype=np.int64)
        want = _bits(net([coords, x], rgb_mask=mask))
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            prep_c = net.prepare(coords)
            prep_p = net.prepare_points(pts, offs, rot, None, 20.0)
        assert prep_p.kept() is None
        got_c = _bits(net([prep_c, x], rgb_mask=mask))
        got_p = _bits(net([prep_p, x], rgb_mask=mask))
    assert torch.equal(got_c, want) and torch.equal(got_p, want)
    _no_device_error()
