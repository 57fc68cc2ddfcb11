"""Cost of the deterministic mode on the fused UNetSCN training step (the whole-network executor, net.fused = True).

Workload: batch-8 nuScenes-shaped scans (synth.make_batch), UNetSCN(in_channels=3) in its reference configuration,
forward + backward of a fixed upstream gradient, in each of tf32, tf32x3 and bf16.  Four arms per mode, in blocks of
--steps steps that alternate (--rounds times each, after a warm-up of every arm), timed with CUDA events:
  fused_default    net.fused = True, mode off
  fused_det        net.fused = True, scn.set_deterministic(True)
  fused_det_torch  net.fused = True, torch.use_deterministic_algorithms(True) -- the switch Lightning's
                   Trainer(deterministic=True) sets; torch then also fills every torch.empty with NaN
                   (torch.utils.deterministic.fill_uninitialized_memory), the executor's act / tmp buffers included
  module_det       net.fused = False, scn.set_deterministic(True) (the previous way to a reproducible step)
It prints ms/step and mm3d_kernel_launches per step of each arm, checks that two fused deterministic steps from the same
state give equal SHA-256 digests of the output, the input gradient, every parameter gradient and the running statistics
(and that the torch switch gives the same digest), and reads the GPU's name and power limit in the same run.

    python tools/deterministic_exec_bench.py --steps 5 --rounds 3 [--json OUT]
"""
import argparse
import json
import os
import sys
import warnings

import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from deterministic_step_bench import MODES, Step, digest, gpu_info, timed  # noqa: E402

from mm2d3d_b200 import functional as F  # noqa: E402
from mm2d3d_b200 import scn  # noqa: E402
from mm2d3d_b200._lib import lib  # noqa: E402

ARMS = ("fused_default", "fused_det", "fused_det_torch", "module_det")


def set_arm(step, arm):
    step.net.fused = arm != "module_det"
    torch.use_deterministic_algorithms(arm == "fused_det_torch", warn_only=True)
    F.DETERMINISTIC = {"fused_default": False, "fused_det": True, "fused_det_torch": None, "module_det": True}[arm]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("deterministic_exec_bench: needs a CUDA device")
    dev = torch.device("cuda:0")
    out = {"workload": "UNetSCN(in_channels=3), batch-8 nuScenes-shaped scans, training step (forward + backward)",
           **gpu_info(), "steps": {}}
    step = Step(dev)
    prev = scn.get_conv_mode()
    warnings.simplefilter("ignore")  # (warn_only: torch's own notes on ops outside this package)
    try:
        for mode in MODES:
            scn.set_conv_mode(mode)
            for arm in ARMS:  # warm-up of every arm
                set_arm(step, arm)
                step()
                step()
            times = {a: [] for a in ARMS}
            launches = {}
            for _ in range(args.rounds):
                for arm in ARMS:
                    set_arm(step, arm)
                    ms, k = timed(step, args.steps)
                    times[arm].append(ms)
                    launches[arm] = k
            set_arm(step, "fused_det")
            d1, d2 = digest(step(keep=True)), digest(step(keep=True))
            set_arm(step, "fused_det_torch")
            d3 = digest(step(keep=True))
            r = {"ms_per_step": {a: min(times[a]) for a in ARMS}, "ms_all_rounds": times, "launches_per_step": launches,
                 "fused_det_sha256_equal": d1 == d2, "torch_switch_same_sha256": d1 == d3, "fused_det_sha256": d1}
            out["steps"][mode] = r
            ms = r["ms_per_step"]
            print(f"{mode:7s} " + " | ".join(f"{a} {ms[a]:7.3f} ms {launches[a]:5.0f} launches" for a in ARMS) +
                  f" | det/default {ms['fused_det'] / ms['fused_default']:.3f}"
                  f" | sha256 equal: {d1 == d2}, torch switch same: {d1 == d3}", flush=True)
    finally:
        torch.use_deterministic_algorithms(False)
        F.DETERMINISTIC = None
        step.net.fused = True
        scn.set_conv_mode(prev)
    print(f"GPU: {out['gpu']}, power limit {out['power_limit']}")
    assert lib.mm3d_take_device_error() == 0
    if args.json:
        with open(args.json, "w") as f:
            json.dump(out, f, indent=1)
    if not all(v["fused_det_sha256_equal"] and v["torch_switch_same_sha256"] for v in out["steps"].values()):
        raise SystemExit("deterministic steps differ")


if __name__ == "__main__":
    main()
