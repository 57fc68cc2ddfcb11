"""Eval forward of UNetSCN: the existing path (``net(x).detach()`` with grad mode on: UNetSCNFn, the training-form
forward) against the inference path (``torch.no_grad()``: mm3d_unet_topo_infer), on a batch of 8 nuScenes-shaped scans
from ``synth``, in every convolution mode.

    python tools/infer_bench.py [--rounds 5] [--iters 20] [--out FILE.json]

Per mode and arm: ms per forward (CUDA events around ``iters`` forwards, after a warm-up; the arms alternate for
``rounds`` rounds, the median round is reported), ``mm3d_kernel_launches`` per forward and peak allocated memory per
forward (above what was allocated before it).  Structures are prepared once (``net.prepare``) and reused; one more arm
of each path builds them from the coordinates in every forward.  The outputs of the two paths are checked byte-equal at
the timed size (in the deterministic mode: several points per voxel, and the default mode's InputLayer sums them in
atomic order, which changes the last bits from one forward to the next in either path).  Both paths are measured in
every mode, including those in which the executor does not dispatch to the inference path (executor.INFER_MODES).
Prints the GPU's name and power limit."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return f"nvidia-smi unavailable ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("infer_bench needs a CUDA device")
    import mm2d3d_b200.scn as scn
    from mm2d3d_b200 import _lib, executor, synth
    from mm2d3d_b200.unet import UNetSCN

    dev = "cuda:0"
    info = {"gpu": gpu_info(), "torch": torch.__version__, "batch": a.batch}
    print("GPU (name, power limit, max SM clock):", info["gpu"])
    locs, feats = synth.make_batch("nuscenes", batch=a.batch, seed0=0)
    coords, feats = torch.from_numpy(locs).to(dev), torch.from_numpy(feats).to(dev)
    info["points"] = int(coords.shape[0])
    torch.manual_seed(0)
    net = UNetSCN(in_channels=3).to(dev)
    with torch.no_grad():  # running statistics and affine parameters of a trained-looking network
        for mod in net.modules():
            if isinstance(mod, scn.BatchNormLeakyReLU):
                mod.weight.copy_(1 + 0.3 * torch.randn_like(mod.weight))
                mod.bias.copy_(0.2 * torch.randn_like(mod.bias))
                mod.running_mean.copy_(0.3 * torch.randn_like(mod.running_mean))
                mod.running_var.copy_(0.5 + torch.rand_like(mod.running_var))
    net.eval()
    executor.INFER_MODES = frozenset(_lib.MODES.values())  # (measure the inference path in every mode)
    results = []
    for mode in ("fp32", "tf32", "tf32x3", "bf16"):
        scn.set_conv_mode(mode)
        prep = net.prepare(coords, wait=True)
        arms = {
            "eval (UNetSCNFn), prepared": lambda: net([prep, feats]).detach(),
            "inference, prepared": lambda: _nograd(net, [prep, feats]),
            "eval (UNetSCNFn), builds structures": lambda: net([coords, feats]).detach(),
            "inference, builds structures": lambda: _nograd(net, [coords, feats]),
        }
        scn.set_deterministic(True)
        outs = {k: f().view(torch.int32).clone() for k, f in arms.items()}  # (warm-up too)
        scn.set_deterministic(False)
        equal = all(torch.equal(outs[k], outs["eval (UNetSCNFn), prepared"]) for k in outs)
        for f in arms.values():
            for _ in range(3):
                f()
        torch.cuda.synchronize()
        ms = {k: [] for k in arms}
        launches, peak = {}, {}
        for _ in range(a.rounds):
            for k, f in arms.items():
                start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                start.record()
                for _ in range(a.iters):
                    f()
                end.record()
                torch.cuda.synchronize()
                ms[k].append(start.elapsed_time(end) / a.iters)
        for k, f in arms.items():
            torch.cuda.synchronize()
            base = torch.cuda.memory_allocated()
            torch.cuda.reset_peak_memory_stats()
            n0 = _lib.lib.mm3d_kernel_launches()
            out = f()
            torch.cuda.synchronize()
            launches[k] = _lib.lib.mm3d_kernel_launches() - n0
            peak[k] = torch.cuda.max_memory_allocated() - base
            del out
        for k in arms:
            r = {"mode": mode, "arm": k, "ms": statistics.median(ms[k]), "ms_rounds": ms[k], "launches": launches[k],
                 "peak_MiB": peak[k] / 2**20, "bytes_equal_to_eval": equal}
            results.append(r)
            print(f"{mode:7s} {k:38s} {r['ms']:7.3f} ms  (rounds {min(ms[k]):.3f}..{max(ms[k]):.3f})  "
                  f"{launches[k]:4d} launches  peak {r['peak_MiB']:8.1f} MiB  outputs byte-equal: {equal}")
    scn.set_conv_mode("fp32")
    assert _lib.lib.mm3d_take_device_error() == 0
    if a.out:
        with open(a.out, "w") as fh:
            json.dump({"info": info, "results": results}, fh, indent=1)


def _nograd(net, x):
    with torch.no_grad():
        return net(x)


if __name__ == "__main__":
    main()
