"""Wide UNetSCN on the GPU: UNetSCN(m = 32, 7 planes), batch-8 nuScenes-shaped scans, in every mode.

    python tools/wide_bench.py [--steps 20] [--warmup 5] [--out FILE]

Per mode: ms per training step (structure build + forward + backward, CUDA events over `steps` steps), kernel
launches per step, peak allocation; the same for the eval forward under no_grad; and the sliced layers' share of the
step: the decoder convolutions 320 -> 160 (level 4) and 384 -> 192 (level 5), whose input runs as two channel slices
(DESIGN.md section 5), timed one op at a time (forward, dgrad and wgrad through TableConvFn, CUDA events) on the same
batch's tables, against the step.  Prints one JSON object with the card's name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from mm2d3d_b200 import _lib, synth  # noqa: E402
from mm2d3d_b200 import functional as F  # noqa: E402
from mm2d3d_b200.metadata import Metadata  # noqa: E402

M, PLANES, SCALE = 32, 7, 4096
SLICED = [(4, 320, 160), (5, 384, 192)]  # (level, c_in, c_out) of the decoder convolutions with c_in > 256


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def timed(fn, steps, warmup):
    """(ms per call, launches per call, peak MiB) of fn() over `steps` calls after `warmup`."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    l0 = _lib.lib.mm3d_kernel_launches()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return (a.elapsed_time(b) / steps, (_lib.lib.mm3d_kernel_launches() - l0) / steps,
            torch.cuda.max_memory_allocated() / 2 ** 20)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "wide_bench.py measures on the GPU"
    import mm2d3d_b200.scn as scn
    from mm2d3d_b200.unet import UNetSCN
    dev = "cuda:0"
    locs, feats = synth.make_batch("nuscenes", batch=8, seed0=0)
    coords, x = torch.from_numpy(locs).to(dev), torch.from_numpy(feats).to(dev)
    g = torch.randn(x.shape[0], M, device=dev, generator=torch.Generator(dev).manual_seed(1))
    meta = Metadata(coords, SCALE, PLANES, plans=True)
    res = {"card": card(), "config": f"UNetSCN(in_channels=3, m={M}, num_planes={PLANES}, full_scale={SCALE}), "
           f"batch 8 nuscenes-shaped scans ({x.shape[0]} points)", "steps": args.steps, "warmup": args.warmup,
           "modes": {}}
    for mode in ("fp32", "tf32", "tf32x3", "bf16"):
        scn.set_conv_mode(mode)
        torch.manual_seed(0)
        net = UNetSCN(in_channels=3, m=M, num_planes=PLANES, full_scale=SCALE).to(dev)

        def step():
            for p in net.parameters():
                p.grad = None
            net([coords, x]).backward(g)

        net.train()
        ms, launches, peak = timed(step, args.steps, args.warmup)
        net.eval()

        def fwd():
            with torch.no_grad():
                net([coords, x])

        ems, elaunches, epeak = timed(fwd, args.steps, args.warmup)
        layers = {}
        for lvl, ci, co in SLICED:
            xi = torch.randn(meta.nbr(SCALE >> lvl).n, ci, device=dev).requires_grad_(True)
            w = (torch.randn(27, 1, ci, co, device=dev) / ci ** 0.5).requires_grad_(True)
            gy = torch.randn(xi.shape[0], co, device=dev)

            def op():
                y = F.TableConvFn.apply(xi, w, meta, "smc", SCALE >> lvl, mode)
                torch.autograd.grad(y, (xi, w), gy)

            layers[f"L{lvl} {ci}->{co} ({xi.shape[0]} rows)"] = round(timed(op, args.steps, args.warmup)[0], 4)
        res["modes"][mode] = {
            "train_ms_per_step": round(ms, 4), "train_launches_per_step": launches, "train_peak_mib": round(peak, 1),
            "eval_fwd_ms": round(ems, 4), "eval_fwd_launches": elaunches, "eval_fwd_peak_mib": round(epeak, 1),
            "sliced_layers_fwd_dgrad_wgrad_ms": layers,
            "sliced_layers_share_of_step": round(sum(layers.values()) / ms, 4),
        }
        del net
        torch.cuda.empty_cache()
    scn.set_conv_mode("fp32")
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
