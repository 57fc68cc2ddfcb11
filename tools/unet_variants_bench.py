"""Training-step time of UNetSCN's block topologies, fused executor vs module by module.

Workload: batch-8 nuScenes-shaped scans (synth.make_batch), TF32 mode, forward + backward of the 3D network with
the sparse structure prepared one step ahead on a second stream (as in bench.py).  The module-by-module path
cannot take a prepared structure: it builds its structure inside the step.  Per configuration
(block_reps, residual) it prints ms/step (CUDA events over the timed window, after warm-up) and kernel launches
per step (mm3d_kernel_launches); for the reference configuration it also times the original mm3d_unet_* entry
points against the topology ones, alternating in this process.  The GPU's name and power limit are read in the
same run.

    python tools/unet_variants_bench.py --steps 50 --warmup 10 [--json OUT]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from mm2d3d_b200 import _lib, executor, synth  # noqa: E402
from mm2d3d_b200 import scn  # noqa: E402
from mm2d3d_b200.unet import UNetSCN  # noqa: E402

CONFIGS = [(1, False), (2, False), (1, True), (2, True)]


class ReferenceEntryPoints:
    """The executor's library handle with the topology calls routed to the original reference-configuration ones."""

    def __init__(self, lib):
        self._lib = lib

    def __getattr__(self, name):
        return getattr(self._lib, name)

    def mm3d_unet_topo_act_bytes(self, a, b, c, reps, res, *rest):
        return self._lib.mm3d_unet_act_bytes(a, b, c, *rest)

    def mm3d_unet_topo_bwd_bytes(self, a, b, c, reps, res, *rest):
        return self._lib.mm3d_unet_bwd_bytes(a, b, c, *rest)

    def mm3d_unet_topo_scratch_bytes(self, a, b, c, reps, res, mode):
        return self._lib.mm3d_unet_scratch_bytes(a, b, c, mode)

    def mm3d_unet_topo_forward(self, a, b, c, reps, res, *rest):
        return self._lib.mm3d_unet_forward(a, b, c, *rest)

    def mm3d_unet_topo_backward(self, a, b, c, reps, res, *rest):
        return self._lib.mm3d_unet_backward(a, b, c, *rest)


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        info["power_limit_and_max_sm_clock"] = q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        info["power_limit_and_max_sm_clock"] = "unknown"
    return info


def time_steps(net, batches, steps, warmup, fused):
    dev = batches[0][0].device
    side = torch.cuda.Stream(device=dev)
    ahead = {}

    def prep(i):
        with torch.cuda.stream(side):
            ahead[i] = net.prepare(batches[i % len(batches)][0])

    def step(i):
        coords, feats = batches[i % len(batches)]
        if fused:
            if i not in ahead:
                prep(i)
            x = ahead.pop(i)
            prep(i + 1)
        else:
            x = coords
        net.zero_grad(set_to_none=True)
        out = net([x, feats])
        out.square().mean().backward()

    for i in range(warmup):
        step(i)
    torch.cuda.synchronize()
    l0 = _lib.lib.mm3d_kernel_launches()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for i in range(warmup, warmup + steps):
        step(i)
    t1.record()
    torch.cuda.synchronize()
    launches = (_lib.lib.mm3d_kernel_launches() - l0) / steps
    ahead.clear()
    return t0.elapsed_time(t1) / steps, launches


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3, help="alternating rounds of the old / new entry-point comparison")
    ap.add_argument("--json", help="also write the results to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("unet_variants_bench: needs a CUDA device")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    scn.set_conv_mode("tf32")
    batches = []
    for r in range(4):
        locs, feats = synth.make_batch("nuscenes", batch=8, seed0=100 + 8 * r)
        batches.append((torch.from_numpy(locs).to(dev), torch.from_numpy(feats).to(dev)))
    result = {**gpu_info(), "mode": "tf32", "batch": 8, "shape": "nuscenes", "steps": args.steps,
              "warmup": args.warmup, "points_per_batch": [int(b[0].shape[0]) for b in batches], "configs": []}
    print(f"# {result['gpu']}, power limit / max SM clock: {result['power_limit_and_max_sm_clock']}")
    print(f"# TF32, batch 8 nuScenes-shaped scans, {args.steps} timed steps after {args.warmup} warm-up steps")
    for reps, res in CONFIGS:
        torch.manual_seed(0)
        net = UNetSCN(in_channels=3, m=16, block_reps=reps, residual_blocks=res).to(dev)
        assert executor.fusable(net)
        row = {"block_reps": reps, "residual": res, "params": sum(p.numel() for p in net.parameters())}
        row["fused_ms"], row["fused_launches"] = time_steps(net, batches, args.steps, args.warmup, True)
        net.fused = False
        row["module_ms"], row["module_launches"] = time_steps(net, batches, args.steps, args.warmup, False)
        net.fused = True
        if (reps, res) == (1, False):  # original entry points vs the topology ones, alternating
            old, new = [], []
            real = executor.lib
            for _ in range(args.rounds):
                new.append(time_steps(net, batches, args.steps, args.warmup, True))
                executor.lib = ReferenceEntryPoints(real)
                try:
                    old.append(time_steps(net, batches, args.steps, args.warmup, True))
                finally:
                    executor.lib = real
            row["entry_points"] = {"topology_ms": [t for t, _ in new], "original_ms": [t for t, _ in old],
                                   "topology_launches": new[0][1], "original_launches": old[0][1]}
        result["configs"].append(row)
        name = f"block_reps={reps} {'residual' if res else 'VGG'}"
        print(f"{name:26s} fused {row['fused_ms']:7.2f} ms/step {row['fused_launches']:6.0f} launches | "
              f"module by module {row['module_ms']:7.2f} ms/step {row['module_launches']:6.0f} launches | "
              f"{row['module_ms'] / row['fused_ms']:.2f}x")
        if "entry_points" in row:
            e = row["entry_points"]
            print(f"{'':26s} entry points, alternating: topology " + " ".join(f"{t:.3f}" for t in e["topology_ms"]) +
                  " | original " + " ".join(f"{t:.3f}" for t in e["original_ms"]) +
                  f" ms/step; launches {e['topology_launches']:.0f} vs {e['original_launches']:.0f}")
        del net
        torch.cuda.empty_cache()
    if args.json:
        with open(args.json, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
