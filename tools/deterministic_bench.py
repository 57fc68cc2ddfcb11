"""Cost of the deterministic mode on the ops it covers, at benchmark size, default vs deterministic in one process.

Workload: batch-8 nuScenes-shaped scans (synth.make_batch).  One step runs, forward and backward:
  - the InputLayer (mode 4, the 3 RGB channels) and the OutputLayer of a 16-channel network output (module path);
  - the integer lift of a [8, 64, 225, 400] channels-last float32 map at one pixel per point;
  - the RGB mask, and heads3d (16 -> 10 classes) with its KL loss against random target logits.
The deterministic step rebuilds the voxel and pixel lists each time (a training step sees a new batch, so it pays
for them once per step).  Blocks of --steps steps alternate between the two settings (--rounds times each, after a
warm-up of both), timed with CUDA events; the tool prints ms/step and mm3d_kernel_launches per step for each setting
and the GPU's name and power limit read in the same run.  It also checks its own claim: two deterministic steps on
identical inputs give identical SHA-256 digests of every output and gradient.  The convolution weight gradients,
BatchNorm and the fused executor have no deterministic form yet and are not part of the step.

    python tools/deterministic_bench.py --steps 20 --rounds 5 [--json OUT]
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from mm2d3d_b200 import _lib, synth  # noqa: E402
from mm2d3d_b200 import functional as F  # noqa: E402
from mm2d3d_b200.heads import heads3d, rgb_mask  # noqa: E402
from mm2d3d_b200.lift import LiftIndices, lift2d  # noqa: E402
from mm2d3d_b200.metadata import Metadata  # noqa: E402


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        info["power_limit"] = q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        info["power_limit"] = "unknown"
    return info


class Workload:
    def __init__(self, dev):
        locs, feats = synth.make_batch("nuscenes", batch=8, seed0=0)
        self.meta = Metadata(torch.from_numpy(locs).to(dev), 4096, 1)
        n = self.meta.n_points
        g = torch.Generator(device=dev).manual_seed(0)
        self.feats = torch.from_numpy(feats).to(dev)
        self.d_out = torch.randn(n, 16, device=dev, generator=g)
        counts = np.bincount(locs[:, 3], minlength=8)
        self.lift = LiftIndices(synth.make_img_indices(counts.tolist(), seed=0), dev)
        self.fmap = torch.randn(8, 64, 225, 400, device=dev, generator=g).contiguous(memory_format=torch.channels_last)
        self.d_lift = torch.randn(n, 64, device=dev, generator=g)
        self.mask_w, self.mask_b = torch.randn(1, 3, device=dev, generator=g), torch.randn(1, device=dev, generator=g)
        self.hfeat = torch.randn(n, 16, device=dev, generator=g)
        self.hw = [torch.randn(10, 16, device=dev, generator=g) * 0.3, torch.randn(10, device=dev, generator=g),
                   torch.randn(10, 16, device=dev, generator=g) * 0.3, torch.randn(10, device=dev, generator=g)]
        self.target = torch.randn(n, 10, device=dev, generator=g)

    def step(self):
        self.meta._point_csr = None  # a new batch: the lists are built inside the step
        self.lift._pixel_lists.clear()
        x = self.feats.clone().requires_grad_(True)
        vox = F.InputLayerFn.apply(x, self.meta, 4)
        vox16 = vox.repeat(1, 6)[:, :16].detach().requires_grad_(True)  # stands in for the network's 16-channel output
        out = F.OutputLayerFn.apply(vox16, self.meta)
        fmap = self.fmap.detach().requires_grad_(True)
        lifted = lift2d(fmap, self.lift)
        ps = [self.mask_w.clone().requires_grad_(True), self.mask_b.clone().requires_grad_(True),
              self.hfeat.clone().requires_grad_(True)] + [w.clone().requires_grad_(True) for w in self.hw]
        y = rgb_mask(x, ps[0], ps[1])
        l1, l2, kl = heads3d(ps[2], *ps[3:], target=self.target)
        tot = ((out * self.d_out).sum() + (lifted * self.d_lift).sum() + (vox * 1.0).sum() + y.sum() + l1.sum()
               + l2.sum() + kl)
        grads = torch.autograd.grad(tot, [x, vox16, fmap] + ps)
        return [vox, out, lifted, y, l1, l2, kl] + list(grads)


def digest(ts):
    h = hashlib.sha256()
    for t in ts:
        h.update(t.detach().contiguous().cpu().numpy().tobytes())
    return h.hexdigest()


def timed(wl, flag, steps):
    F.DETERMINISTIC = flag
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    k0 = _lib.lib.mm3d_kernel_launches()
    start.record()
    for _ in range(steps):
        wl.step()
    end.record()
    torch.cuda.synchronize()
    return start.elapsed_time(end) / steps, (_lib.lib.mm3d_kernel_launches() - k0) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("deterministic_bench.py needs a CUDA device")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    wl = Workload(dev)
    prev = F.DETERMINISTIC
    try:
        for flag in (False, True):
            timed(wl, flag, a.warmup)
        ms = {False: [], True: []}
        launches = {}
        for _ in range(a.rounds):
            for flag in (False, True):
                t, k = timed(wl, flag, a.steps)
                ms[flag].append(t)
                launches[flag] = k
        F.DETERMINISTIC = True
        d1, d2 = digest(wl.step()), digest(wl.step())
    finally:
        F.DETERMINISTIC = prev
    _lib.raise_device_errors("deterministic_bench")
    res = dict(gpu_info())
    res.update({
        "workload": "batch-8 nuScenes-shaped scans: InputLayer(mode 4, 3 ch) + OutputLayer(16 ch) + lift "
                    "[8,64,225,400] f32 channels-last + rgb_mask + heads3d(16->10, KL), forward + backward",
        "n_points": wl.meta.n_points, "n_voxels": wl.meta.n_voxels,
        "steps_per_block": a.steps, "rounds": a.rounds,
        "default_ms_per_step": float(np.median(ms[False])), "deterministic_ms_per_step": float(np.median(ms[True])),
        "default_ms_blocks": ms[False], "deterministic_ms_blocks": ms[True],
        "default_launches_per_step": launches[False], "deterministic_launches_per_step": launches[True],
        "deterministic_digest_step1": d1, "deterministic_digest_step2": d2, "digests_equal": d1 == d2,
    })
    res["overhead"] = res["deterministic_ms_per_step"] / res["default_ms_per_step"]
    print(f"# {res['gpu']}, power limit {res['power_limit']}; {res['n_points']} points, {res['n_voxels']} voxels")
    print(f"default        {res['default_ms_per_step']:.3f} ms/step  {launches[False]:.0f} launches/step")
    print(f"deterministic  {res['deterministic_ms_per_step']:.3f} ms/step  {launches[True]:.0f} launches/step  "
          f"({res['overhead']:.2f}x)")
    print(f"two deterministic steps, SHA-256 of all outputs and gradients equal: {d1 == d2}")
    print(json.dumps(res))
    if a.json:
        with open(a.json, "w") as f:
            json.dump(res, f, indent=1)
    if d1 != d2:
        raise SystemExit("deterministic steps differ")


if __name__ == "__main__":
    main()
