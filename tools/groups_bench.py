"""Two-domain training step of MM2D3D: two UNetSCN calls + one backward against one ``forward_groups`` + one backward.

Workload: a source and a target batch of 8 nuScenes-shaped scans each (synth.make_batch, different seeds),
UNetSCN(in_channels=3) in its reference configuration, forward of both batches, one backward of the summed loss
(fixed upstream gradients), in every convolution mode.  Structures are built inline (coordinates passed to the call)
or, separately, prepared one step ahead on the current stream (``prepare`` / ``prepare_groups``).  The two arms
alternate in blocks of --steps steps, --rounds times each after a warm-up; each block is timed with CUDA events (ms per
step) and with the host clock up to the enqueue of the step's last kernel (host ms per step).  Also reported: libmm3d
launches per step and the peak allocation of a step.  The GPU's name and power limit are read in the same run.

    python tools/groups_bench.py --steps 10 --rounds 5 [--modes tf32,bf16] [--json OUT]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from mm2d3d_b200 import _lib, scn, synth  # noqa: E402
from mm2d3d_b200.unet import UNetSCN  # noqa: E402


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        info["power_limit"] = q[0] if q else "unknown"
    except Exception:  # noqa: BLE001
        info["power_limit"] = "unknown"
    return info


def batch(seed0):
    locs, feats = synth.make_batch("nuscenes", batch=8, seed0=seed0)
    return torch.from_numpy(locs).cuda(), torch.from_numpy(feats).cuda()


def make_step(net, data, grads, grouped, prepared):
    (cs, fs), (ct, ft) = data
    pending = {}

    def prep():
        if grouped:
            pending["p"] = net.prepare_groups([cs, ct])
        else:
            pending["p"] = (net.prepare(cs), net.prepare(ct))

    def step():
        xs, xt = fs.clone().requires_grad_(True), ft.clone().requires_grad_(True)
        for p in net.parameters():
            p.grad = None
        if prepared:
            src = pending["p"]
            prep()  # the next step's structures, enqueued ahead
        if grouped:
            outs = net.forward_groups(src if prepared else [cs, ct], [xs, xt])
        else:
            outs = [net([src[0] if prepared else cs, xs]), net([src[1] if prepared else ct, xt])]
        torch.autograd.backward(outs, grads)
    if prepared:
        prep()
    return step


def time_block(step, steps):
    torch.cuda.synchronize()
    n0 = _lib.lib.mm3d_kernel_launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(steps):
        step()
    host = (time.perf_counter() - t0) * 1e3 / steps
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps, host, (_lib.lib.mm3d_kernel_launches() - n0) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--modes", default="fp32,tf32,tf32x3,bf16")
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("groups_bench.py needs a CUDA device")
    out = {**gpu_info(), "workload": "8 + 8 nuScenes-shaped scans, UNetSCN(in_channels=3) reference configuration, "
                                     "forward of both + one backward", "steps": a.steps, "rounds": a.rounds, "results": []}
    data = (batch(0), batch(100))
    torch.manual_seed(0)
    net = UNetSCN(in_channels=3).cuda()
    grads = [torch.randn(data[0][1].shape[0], 16, device="cuda"), torch.randn(data[1][1].shape[0], 16, device="cuda")]
    for mode in a.modes.split(","):
        scn.set_conv_mode(mode)
        for prepared in (False, True):
            arms = {name: make_step(net, data, grads, grouped, prepared)
                    for name, grouped in (("two_calls", False), ("forward_groups", True))}
            res = {name: {"ms": [], "host_ms": [], "launches": None, "peak_mb": None} for name in arms}
            for name, step in arms.items():  # warm-up, launches and peak allocation
                for _ in range(3):
                    step()
                torch.cuda.synchronize()
                torch.cuda.reset_peak_memory_stats()
                base = torch.cuda.memory_allocated()
                _, _, launches = time_block(step, 1)
                res[name]["launches"] = launches
                res[name]["peak_mb"] = round((torch.cuda.max_memory_allocated() - base) / 2**20, 1)
            for _ in range(a.rounds):
                for name, step in arms.items():
                    ms, host, _ = time_block(step, a.steps)
                    res[name]["ms"].append(round(ms, 4))
                    res[name]["host_ms"].append(round(host, 4))
            for name in arms:
                r = res[name]
                r["median_ms"] = statistics.median(r["ms"])
                r["spread_ms"] = round(max(r["ms"]) - min(r["ms"]), 4)
                r["median_host_ms"] = statistics.median(r["host_ms"])
            row = {"mode": mode, "structures": "prepared" if prepared else "inline", **res}
            out["results"].append(row)
            print(f"{mode:7s} {row['structures']:8s} two calls {res['two_calls']['median_ms']:.3f} ms "
                  f"(spread {res['two_calls']['spread_ms']:.3f}, host {res['two_calls']['median_host_ms']:.3f}, "
                  f"{res['two_calls']['launches']:.0f} launches, peak {res['two_calls']['peak_mb']} MB) | forward_groups "
                  f"{res['forward_groups']['median_ms']:.3f} ms (spread {res['forward_groups']['spread_ms']:.3f}, host "
                  f"{res['forward_groups']['median_host_ms']:.3f}, {res['forward_groups']['launches']:.0f} launches, "
                  f"peak {res['forward_groups']['peak_mb']} MB)", flush=True)
    scn.set_conv_mode("fp32")
    print(f"GPU: {out['gpu']}, power limit {out['power_limit']}")
    if a.json:
        os.makedirs(os.path.dirname(os.path.abspath(a.json)), exist_ok=True)
        with open(a.json, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
