"""The whole-network executor (``UNetSCN.forward`` with ``fused = True``, csrc/unet_exec.cu) against the FP64 oracle,
per tensor, at the per-op bars: 1e-4 in the fp32 and tf32x3 modes, 1e-2 in tf32, 5e-2 in bf16 (two exceptions with
their evidence in `_bar`) -- relative L2 AND max-abs-relative, for the output, the input gradient, every parameter
gradient (and the RGB mask's) and the running statistics after the step (there max(bar, 1e-4)).

The network runs free: batch statistics in the loop, real ReLU gates, the executor's own code.  What makes the FP64
comparison meaningful is the open-gate conditioning of test_exec_fp64_cpu.py (BatchNorm biases +-8, far from the
ReLU kink), so FP32 and TF32 round-off flip no gate (BF16: see `_bar`); its self-check fails loudly if a change to the inputs or the init breaks it.
The gates are then constant per channel, so per-row gating under round-off is not what this file tests: that stays
with test_bnrelu, test_bnrelu_deterministic and the frozen-gate module-path tests.

Covered: training steps of every block topology in every mode (tensor-core modes also in deterministic mode),
eval-mode backward (the executor's frozen-statistics branches, with the running statistics set to the FP64 batch
statistics of the same input), two steps with an in-place SGD update in between, the RGB mask folded into the
InputLayer, width m = 8 (tcgen05 layers mixed with SIMT fallbacks in the tf32 mode; refused in tf32x3 and bf16),
and the parameter-slot list after parameters or buffers are replaced by new objects.  The input is two
nuScenes-shaped scans with several points per voxel.  On a failed bar the module path's figures under the same
conditioning are printed beside the executor's: they tell an executor error from one shared with the per-op kernels.
"""
import re

import pytest
import torch

from mm2d3d_b200 import _lib, synth
from tests.test_exec_fp64_cpu import LR, Fp64Cache, compare, output_grad, scan
from tests.test_gpu_parity import DEV, _no_device_error, rel_err, rel_l2

pytestmark = pytest.mark.gpu

TOPOLOGIES = [(1, False), (2, False), (1, True), (2, True)]
MODES = ["fp32", "tf32", "tf32x3", "bf16"]
BAR = {"fp32": 1e-4, "tf32x3": 1e-4, "tf32": 1e-2, "bf16": 5e-2}


def _bar(mode, reps, res, training=True):
    """BAR[mode], with two bf16 exceptions (unit round-off 2^-9, four times TF32's).

    (2, residual): about 80 convolutions in a chain against the reference configuration's 27 -- the bar of
    test_residual_reps2_gradients_with_frozen_gates, 1e-1.

    (2, VGG) training step: 2e-1.  The conditioning leaves 3 pre-activations within 1e-2 of the ReLU kink in this
    network on this input, two of them in the BatchNorm layer3.2.1.2.4.0 and one in layer3.2.1.2.2.1.2.1.0 (levels 1
    and 2, 26k and 14k rows).  BF16 operands move the forward by ~2e-3 relative (~2e-2 absolute at |pre| ~ 8), enough
    to flip those gates, and in training a flipped row enters the channel's batch-statistics backward.  Printed
    figures (NVIDIA B200, 1000 W): executor rel-L2 6.3e-2 on layer3.2.1.2.2.1.2.1.0.weight, max-abs-rel 1.57e-1 on
    layer3.2.1.2.4.0.weight; the module path gives the same figures to three digits, and the CPU oracle with its
    convolution operands rounded to BF16 gives 6.5e-2 and 1.53e-1 on the same tensors.  So the error is BF16
    rounding at a gate, not the executor's; TF32 on the same network is 2.1e-3 / 2.6e-3, and the eval-mode
    backward in bf16 1.4e-2 / 2.1e-2."""
    if mode == "bf16" and (reps, res) == (2, True):
        return 1e-1
    if mode == "bf16" and (reps, res) == (2, False) and training:
        return 2e-1
    return BAR[mode]


def _ids(t):
    return f"{t[0]}-{'res' if t[1] else 'vgg'}"


@pytest.fixture(scope="module")
def fp64():
    return Fp64Cache()


class _settings:
    """Convolution mode and deterministic mode for the duration of a block."""

    def __init__(self, mode, det=False):
        self.mode, self.det = mode, det

    def __enter__(self):
        from mm2d3d_b200 import functional as F
        from mm2d3d_b200 import scn
        self.prev = (scn.get_conv_mode(), F.DETERMINISTIC)
        scn.set_conv_mode(self.mode)
        scn.set_deterministic(self.det)

    def __exit__(self, *a):
        from mm2d3d_b200 import scn
        scn.set_conv_mode(self.prev[0])
        scn.set_deterministic(self.prev[1])


def gpu_steps(ref, reps, res, mode, training=True, mask=False, steps=1, m=16, det=False, fused=True):
    """What oracle_run does, on the GPU: the network loaded with the reference's initial state, `steps` forward +
    backward passes with p -= LR * p.grad in between.  Asserts the executor ran when `fused`."""
    from mm2d3d_b200.unet import UNetSCN
    coords, feats = scan()
    coords, feats = coords.to(DEV), feats.to(DEV)
    g = output_grad(feats.shape[0], m).float().to(DEV)
    net = UNetSCN(in_channels=3, m=m, block_reps=reps, residual_blocks=res).to(DEV)
    net.load_state_dict(ref["state"])
    net.train(training)
    net.fused = fused
    params = dict(net.named_parameters())
    lin = None
    if mask:
        lin = torch.nn.Linear(3, 1).to(DEV)
        lin.load_state_dict(ref["mask_state"])
        params.update({"mask." + k: v for k, v in lin.named_parameters()})
    results = []
    with _settings(mode, det):
        for step in range(steps):
            if step:
                with torch.no_grad():
                    for p in params.values():
                        p -= LR * p.grad
            for p in params.values():
                p.grad = None
            x = feats.clone().requires_grad_(True)
            out = net([coords, x], rgb_mask=lin)
            if fused:
                assert type(out.grad_fn).__name__ == "UNetSCNFnBackward", type(out.grad_fn)
            out.backward(g)
            grads = {"feats": x.grad, **{k: p.grad for k, p in params.items()}}
            results.append({"out": out.detach(), "grads": grads,
                            "buffers": {k: b.clone() for k, b in net.named_buffers()}})
    _no_device_error()
    return results


def _rows(got, want, bar):
    """[(name, rel-L2, max-abs-rel, bar)] for the output, every gradient and every running buffer."""
    rows = [("out", rel_l2(got["out"], want["out"]), rel_err(got["out"], want["out"]), bar)]
    rows += [(k, e2, em, bar) for k, e2, em in compare(got["grads"], want["grads"])]
    rows += [(k, e2, em, max(bar, 1e-4)) for k, e2, em in compare(got["buffers"], want["buffers"])]
    return rows


def _summary(rows):
    w2 = max(rows[1:], key=lambda r: r[1])
    wm = max(rows[1:], key=lambda r: r[2])
    return (f"forward rel-L2 {rows[0][1]:.2e} max-abs-rel {rows[0][2]:.2e} | worst gradient/buffer rel-L2 {w2[1]:.2e} "
            f"({w2[0]}) | worst max-abs-rel {wm[2]:.2e} ({wm[0]})")


def check(tag, got, want, bar, module_path=None):
    """Hold every tensor of `got` to `bar` against the FP64 `want`; print the per-tensor table.  On a failure the
    module path's figures (`module_path()`: the same step with fused = False) are printed beside the executor's."""
    rows = _rows(got, want, bar)
    print(f"\n[{tag}] executor vs FP64 oracle (bar {bar:.0e}): {_summary(rows)}")
    for name, e2, em, b in rows:
        print(f"[{tag}]   {name:60s} rel-L2 {e2:.2e}  max-abs-rel {em:.2e}")
    failed = [(name, e2, em, b) for name, e2, em, b in rows if not (e2 <= b and em <= b)]
    if failed and module_path is not None:
        mrows = {r[0]: r for r in _rows(module_path(), want, bar)}
        print(f"[{tag}] FAILED; module path under the same conditioning: {_summary(list(mrows.values()))}")
        for name, e2, em, b in failed:
            print(f"[{tag}]   {name:60s} executor {e2:.2e} / {em:.2e}   module path {mrows[name][1]:.2e} / "
                  f"{mrows[name][2]:.2e}")
    assert not failed, (tag, failed)


# ---------------------------------------------------------------------------------------------- training step
TRAIN_CASES = [(t, mode, False) for t in TOPOLOGIES for mode in MODES]
TRAIN_CASES += [(t, mode, True) for t in [(1, False), (2, True)] for mode in ("tf32", "tf32x3", "bf16")]


@pytest.mark.parametrize("topo,mode,det", TRAIN_CASES,
                         ids=[f"{_ids(t)}-{mode}{'-det' if det else ''}" for t, mode, det in TRAIN_CASES])
def test_training_step_against_fp64(fp64, topo, mode, det):
    """One free-running training step through the executor: output, d_feats, every parameter gradient and the
    running statistics after the momentum update.  Deterministic mode runs the slab-reduced tcgen05 weight
    gradients, the fixed-order BatchNorm and the point-list InputLayer / OutputLayer: their own kernels."""
    reps, res = topo
    ref = fp64(reps, res)
    bar = _bar(mode, reps, res)
    got = gpu_steps(ref, reps, res, mode, det=det)[0]
    check(f"{mode}{' det' if det else ''} training {_ids(topo)}", got, ref["steps"][0], bar,
          lambda: gpu_steps(ref, reps, res, mode, det=det, fused=False)[0])


# ---------------------------------------------------------------------------------------------- eval backward
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("topo", TOPOLOGIES, ids=_ids)
def test_eval_backward_against_fp64(fp64, topo, mode):
    """Backward through the executor in eval mode (frozen statistics: frozen-BatchNorm fine-tuning, input gradients
    of a deployed network).  These are the executor's !training branches (the JoinTable materialised rather than
    read split); the running statistics must come out untouched."""
    reps, res = topo
    ref = fp64(reps, res, training=False)
    got = gpu_steps(ref, reps, res, mode, training=False)[0]
    check(f"{mode} eval {_ids(topo)}", got, ref["steps"][0], _bar(mode, reps, res, training=False),
          lambda: gpu_steps(ref, reps, res, mode, training=False, fused=False)[0])


# ---------------------------------------------------------------------------------------------- two steps
@pytest.mark.parametrize("mode", ["fp32", "tf32"])
def test_second_step_after_inplace_update_against_fp64(fp64, mode):
    """Step 1, p -= LR * p.grad in place on both sides, step 2: the second step and the running statistics after two
    momentum updates.  Anything the executor kept from the earlier call (weight images, temporaries, slots) shows."""
    ref = fp64(1, False, steps=2)
    got = gpu_steps(ref, 1, False, mode, steps=2)
    for step in range(2):
        check(f"{mode} step {step + 1} of 2", got[step], ref["steps"][step], BAR[mode],
              lambda: gpu_steps(ref, 1, False, mode, steps=2, fused=False)[step])


# ---------------------------------------------------------------------------------------------- RGB mask
@pytest.mark.parametrize("mode", ["fp32", "tf32"])
def test_masked_input_against_fp64(fp64, mode):
    """``net(x, rgb_mask=linear)``: the mask x * sigmoid(linear(x)) folded into the executor's InputLayer, against the
    FP64 oracle with the mask in front of it; the mask's weight and bias gradients included."""
    ref = fp64(1, False, mask=True)
    got = gpu_steps(ref, 1, False, mode, mask=True)[0]
    assert {"mask.weight", "mask.bias"} <= set(got["grads"])
    check(f"{mode} masked", got, ref["steps"][0], BAR[mode],
          lambda: gpu_steps(ref, 1, False, mode, mask=True, fused=False)[0])


# ---------------------------------------------------------------------------------------------- width m = 8
@pytest.mark.parametrize("mode", ["fp32", "tf32"])
def test_width_8_against_fp64(fp64, mode):
    """m = 8, planes 8 ... 56: in the tf32 mode the layers with c_in = 8, 24, 40, 56 run the SIMT kernels and the
    multiples of 16 the tcgen05 ones, inside one executor call."""
    ref = fp64(1, False, m=8)
    got = gpu_steps(ref, 1, False, mode, m=8)[0]
    check(f"{mode} m=8", got, ref["steps"][0], BAR[mode], lambda: gpu_steps(ref, 1, False, mode, m=8, fused=False)[0])


@pytest.mark.parametrize("mode", ["tf32x3", "bf16"])
def test_width_8_refused_in_split_modes(mode):
    """tf32x3 and bf16 have no SIMT form: a layer whose input width is not a multiple of 16 is refused with an error
    that names the width, and leaves no device error behind."""
    from mm2d3d_b200.unet import UNetSCN
    coords, feats = scan()
    net = UNetSCN(in_channels=3, m=8).to(DEV)
    with _settings(mode), pytest.raises(_lib.Mm3dError) as e:
        net([coords.to(DEV), feats.to(DEV)])
    print(f"\n[{mode}] m = 8 refused: {e.value}")
    assert re.search(r"\b(8|24|40|56)\b", str(e.value)), str(e.value)
    _no_device_error()


# ---------------------------------------------------------------------------------------------- slot list
@pytest.mark.parametrize("how", ["parameter", "buffer", "load_state_dict_assign"])
def test_replaced_tensors_reach_the_executor(how):
    """A parameter or buffer of an inner module replaced by a new object after the executor has run once: outputs,
    every gradient and the running statistics equal a freshly constructed network's with the same state (bit for
    bit: the deterministic tf32 step), and the new parameter gets its gradient."""
    from mm2d3d_b200.unet import UNetSCN

    def make():
        return UNetSCN(in_channels=3, m=16, block_reps=2, residual_blocks=True, num_planes=4, full_scale=256).to(DEV)
    locs, feats = synth.make_batch("nuscenes", batch=2, seed0=8)
    locs[:, :3] //= 16
    coords, feats = torch.from_numpy(locs).to(DEV), torch.from_numpy(feats).to(DEV)
    g = torch.randn(locs.shape[0], 16, generator=torch.Generator().manual_seed(3)).to(DEV)

    def step(net):
        net.zero_grad(set_to_none=True)
        x = feats.clone().requires_grad_(True)
        out = net([coords, x])
        assert type(out.grad_fn).__name__ == "UNetSCNFnBackward"
        out.backward(g)
        return out.detach(), x.grad, {k: p.grad for k, p in net.named_parameters()}

    torch.manual_seed(1)
    net = make()
    other = make()  # new values for the replaced tensors
    with _settings("tf32", det=True):
        step(net)  # the executor has run: the slot list is cached
        conv, bn = net.layer3[0][1][1], net.layer3[0][1][0]
        if how == "parameter":
            conv.weight = torch.nn.Parameter(other.layer3[0][1][1].weight.detach().clone())
            replaced = ["layer3.0.1.1.weight"]
        elif how == "buffer":
            bn.running_mean = other.layer3[0][1][0].running_mean.clone() + 0.5
            replaced = []
        else:
            sd = {k: v.clone() + 0.5 for k, v in other.state_dict().items() if k.startswith("layer3.0.1.")}
            net.load_state_dict(sd, strict=False, assign=True)
            replaced = [k for k in sd if k in dict(net.named_parameters())]
        fresh = make()
        fresh.load_state_dict(net.state_dict())
        got, want = step(net), step(fresh)
    assert replaced or how == "buffer"
    for k in replaced:
        assert got[2][k] is not None, k
    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])
    for k in want[2]:
        assert torch.equal(got[2][k], want[2][k]), k
    for (k, a), (_, b) in zip(net.named_buffers(), fresh.named_buffers()):
        assert torch.equal(a, b), k
