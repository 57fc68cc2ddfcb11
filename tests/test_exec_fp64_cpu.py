"""Open-gate conditioning of UNetSCN and its FP64 oracle, without a GPU.

Whole-network gradients of a randomly initialised BatchNorm/ReLU U-Net depend on ReLU gates that flip under
round-off, so they cannot be held to the per-op bars.  Conditioning removes that: every BatchNorm's bias is pushed
far from the ReLU kink (+8 on about 75 % of the channels, -8 on the rest, weight 1 + 0.2 randn), so almost no
pre-activation lies near zero while the network runs free (batch statistics in the loop).  This file holds the
conditioning, its self-check (how many BatchNorm pre-activations lie within 1e-2 of the kink), the cached FP64
oracle runs the executor is compared with in test_exec_fp64_gpu.py, and checks the premise of that comparison on
every CPU run: under the conditioning the FP32 oracle agrees with the FP64 oracle to FP32 round-off, per tensor.
It also checks that the executor's parameter-slot list follows parameters and buffers replaced by new objects.
"""
import copy

import pytest
import torch

from mm2d3d_b200 import synth
from oracle import scn_cpu
from tests.test_gpu_parity import rel_err, rel_l2

BIAS, OFF_FRAC, WEIGHT_SPREAD = 8.0, 0.25, 0.2
NEAR_KINK, MAX_NEAR_KINK = 1e-2, 16  # (measured on scan(): 1 to 7 entries of 7 M to 32 M, per configuration)
LR = 1e-4  # SGD step between the two steps of a two-step run


def bn_modules(net):
    return [m for m in net.modules() if type(m).__name__ in ("BatchNormLeakyReLU", "BatchNormReLU")]


def scan():
    """Two nuScenes-shaped scans (the batch index is part of the voxel keys), coordinates halved so that voxels hold
    several points (the InputLayer and OutputLayer reduce over point lists)."""
    locs, feats = synth.make_batch("nuscenes", batch=2, seed0=3)
    locs[:, :3] //= 2
    return torch.from_numpy(locs), torch.from_numpy(feats)


def condition(net, seed=2):
    """Open-gate conditioning of every BatchNorm(+ReLU) of `net` in place; convolution weights keep their init."""
    gen = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for bn in bn_modules(net):
            c = bn.weight.numel()
            bn.weight.copy_(1 + WEIGHT_SPREAD * torch.randn(c, generator=gen))
            bn.bias.copy_(torch.where(torch.rand(c, generator=gen) < OFF_FRAC, -BIAS, BIAS))
    return net


class BnProbe:
    """Forward hooks on every BatchNorm of an oracle network: the statistics each one normalised with (batch
    statistics with the biased variance in training, running statistics in eval) and how many of its
    pre-activations lie within NEAR_KINK of the ReLU kink."""

    def __init__(self, net):
        self.stats, self.near_kink, self.entries = [], 0, 0
        self.hooks = [m.register_forward_hook(self.hook) for m in bn_modules(net)]

    def hook(self, mod, inp, out):
        x = inp[0].features.detach()
        if mod.training:
            mean, var = x.mean(0), x.var(0, unbiased=False)
        else:
            mean, var = mod.running_mean.to(x.dtype), mod.running_var.to(x.dtype)
        pre = (x - mean) * torch.rsqrt(var + mod.eps) * mod.weight.detach() + mod.bias.detach()
        self.stats.append((mean, var))
        self.near_kink += int((pre.abs() < NEAR_KINK).sum())
        self.entries += pre.numel()

    def close(self):
        for h in self.hooks:
            h.remove()

    def check(self):
        assert self.near_kink <= MAX_NEAR_KINK, (
            f"open-gate conditioning broken: {self.near_kink} of {self.entries} BatchNorm pre-activations lie within "
            f"{NEAR_KINK} of the ReLU kink (at most {MAX_NEAR_KINK} expected); the FP64 comparisons would be flaky")


def conditioned_net(reps, res, m=16, seed=5):
    """The conditioned oracle network (FP32) and its self-check: an FP64 forward of `scan()` that asserts the gates
    are open and returns the number of pre-activations near the kink."""
    from mm2d3d_b200.unet import UNetSCN
    torch.manual_seed(seed)
    net = condition(UNetSCN(in_channels=3, m=m, block_reps=reps, residual_blocks=res, backend=scn_cpu))

    def self_check():
        net64 = copy.deepcopy(net).double()
        coords, feats = scan()
        probe = BnProbe(net64)
        with torch.no_grad():
            net64([coords, feats.double()])
        probe.close()
        probe.check()
        return probe.near_kink
    return net, self_check


def output_grad(n, m):
    return torch.randn(n, m, generator=torch.Generator().manual_seed(7), dtype=torch.float64)


def mask_linear():
    torch.manual_seed(11)
    return torch.nn.Linear(3, 1)


def oracle_run(reps, res, training=True, mask=False, steps=1, m=16, dtype=torch.float64):
    """Forward + backward of the conditioned oracle network in `dtype` on `scan()`, `steps` times with an in-place SGD
    step (p -= LR * p.grad) in between.  Eval (`training` False): the running statistics are first set to the
    FP64 batch statistics of the same input (biased variance) -- the frozen-statistics network.
    Returns {"state": the FP32 state dict to load into the network under test (before the first step),
    "mask_state": the mask Linear's (or None), "steps": per step {"out", "grads": {"feats", parameter names,
    "mask.weight", "mask.bias"}, "buffers": running statistics after the step}}."""
    net, _ = conditioned_net(reps, res, m)
    lin = mask_linear() if mask else None
    coords, feats = scan()
    if not training:  # running statistics := the FP64 batch statistics of this input
        net64 = copy.deepcopy(net).double()
        probe = BnProbe(net64)
        with torch.no_grad():
            net64([coords, feats.double()])
        probe.close()
        with torch.no_grad():
            for bn, (mean, var) in zip(bn_modules(net), probe.stats):
                bn.running_mean.copy_(mean)
                bn.running_var.copy_(var)
        net.eval()
    state = copy.deepcopy(net.state_dict())
    mask_state = copy.deepcopy(lin.state_dict()) if mask else None
    net = copy.deepcopy(net).to(dtype)
    lin = copy.deepcopy(lin).to(dtype) if mask else None
    params = dict(net.named_parameters())
    if mask:
        params.update({"mask." + k: v for k, v in lin.named_parameters()})
    g = output_grad(feats.shape[0], m).to(dtype)
    results = []
    for step in range(steps):
        if step:
            with torch.no_grad():
                for name, p in params.items():
                    p -= LR * results[-1]["grads"][name]
        x = feats.to(dtype).requires_grad_(True)
        x_in = x * torch.sigmoid(lin(x)) if mask else x
        probe = BnProbe(net)
        out = net([coords, x_in])
        probe.close()
        if dtype == torch.float64:
            probe.check()
        grads = torch.autograd.grad(out, [x] + list(params.values()), g)
        results.append({"out": out.detach(), "grads": dict(zip(["feats"] + list(params), grads)),
                        "buffers": {k: b.clone() for k, b in net.named_buffers()}})
    return {"state": state, "mask_state": mask_state, "steps": results}


class Fp64Cache:
    """FP64 oracle runs keyed by (topology, training, mask, steps): computed once, shared by every mode and by the
    deterministic on / off variants."""

    def __init__(self):
        self.runs = {}

    def __call__(self, reps, res, training=True, mask=False, steps=1, m=16):
        key = ((reps, res, m), training, mask, steps)
        if key not in self.runs:
            self.runs[key] = oracle_run(reps, res, training, mask, steps, m)
        return self.runs[key]


def compare(got, want, names=None):
    """[(name, rel-L2, max-abs-rel)] of the tensors `got[name]` against `want[name]`."""
    return [(k, rel_l2(got[k], want[k]), rel_err(got[k], want[k])) for k in (names or want)]


@pytest.fixture(scope="module")
def fp64():
    return Fp64Cache()


# ------------------------------------------------------------------------------------------------------------ tests
@pytest.mark.parametrize("reps,res", [(1, False), (2, True)])
def test_conditioning_opens_the_gates(reps, res):
    _, self_check = conditioned_net(reps, res)
    near = self_check()
    print(f"\n({reps}, {'residual' if res else 'VGG'}): {near} BatchNorm pre-activations within {NEAR_KINK} of the kink")


@pytest.mark.parametrize("training", [True, False])
@pytest.mark.parametrize("reps,res", [(1, False), (2, True)])
def test_fp32_oracle_matches_fp64_oracle_under_conditioning(fp64, reps, res, training):
    """The premise of test_exec_fp64_gpu.py: with open gates, FP32 arithmetic moves no tensor of a whole training step
    (output, input gradient, every parameter gradient, running statistics) by more than 2e-5 (measured 1.9e-6)."""
    want = fp64(reps, res, training)["steps"][0]
    got = oracle_run(reps, res, training, dtype=torch.float32)["steps"][0]
    rows = [("out", rel_l2(got["out"], want["out"]), rel_err(got["out"], want["out"]))]
    rows += compare(got["grads"], want["grads"]) + compare(got["buffers"], want["buffers"])
    worst = max(rows, key=lambda r: max(r[1], r[2]))
    print(f"\n({reps}, {res}, training={training}) FP32 vs FP64 oracle: worst {worst}")
    for name, e2, em in rows:
        assert e2 <= 2e-5 and em <= 2e-5, (name, e2, em)


def test_fp64_cache_is_computed_once(fp64):
    a = fp64(1, False)
    assert fp64(1, False) is a and fp64(1, False, training=False) is not a


def _slot_names(net):
    """The executor's slot list as parameter / buffer names (identity lookup)."""
    from mm2d3d_b200 import executor
    names = {id(t): k for k, t in list(net.named_parameters()) + list(net.named_buffers())}
    return [names[id(t)] for t in executor.collect_slots(net)]


@pytest.mark.parametrize("how", ["parameter", "buffer", "load_state_dict_assign"])
def test_slot_list_follows_replaced_tensors(how):
    """A parameter or buffer replaced by a new tensor object anywhere in the network is what the executor reads and
    writes the gradient of: the slot list is rebuilt from the modules on every call."""
    from mm2d3d_b200 import executor
    from mm2d3d_b200.unet import UNetSCN
    net = UNetSCN(in_channels=3, m=16, block_reps=2, residual_blocks=True, num_planes=4)
    before = executor.collect_slots(net)
    order = _slot_names(net)
    conv = net.layer3[0][1][1]  # an inner convolution: neither the first nor the last slot
    bn = net.layer3[0][1][0]
    if how == "parameter":
        old = [conv.weight]
        conv.weight = torch.nn.Parameter(conv.weight.detach().clone())
        new = [conv.weight]
    elif how == "buffer":
        old = [bn.running_mean]
        bn.running_mean = torch.zeros_like(bn.running_mean)
        new = [bn.running_mean]
    else:
        prefix = "layer3.0.1."  # the first residual body: a BatchNorm and a convolution, parameters and buffers
        sd = {k: v.clone() for k, v in net.state_dict().items() if k.startswith(prefix)}
        tensors = lambda: dict(list(net.named_parameters()) + list(net.named_buffers()))  # noqa: E731
        old = [tensors()[k] for k in sd]
        net.load_state_dict(sd, strict=False, assign=True)
        new = [tensors()[k] for k in sd]
    after = executor.collect_slots(net)
    assert _slot_names(net) == order
    assert all(any(t is s for s in after) for t in new)
    assert not any(t is s for t in old for s in after)
    assert sum(any(t is s for s in after) for t in before) == len(before) - len(old)
