"""Cost of the deterministic mode on a module-path UNetSCN training step, default vs deterministic in one process.

Workload: batch-8 nuScenes-shaped scans (synth.make_batch), UNetSCN(in_channels=3) in its reference configuration with
``net.fused = False`` (module by module: the path whose training step the mode makes bit-reproducible in the tensor-core
modes), forward + backward of a fixed upstream gradient, in each of tf32, tf32x3 and bf16.  Blocks of --steps steps
alternate between the two settings (--rounds times each, after a warm-up of both), timed with CUDA events; the tool
prints ms/step and mm3d_kernel_launches per step for each setting.  Per op, it times the weight gradient
(mm3d_conv_wgrad_ex) and the BatchNorm training forward + backward (mm3d_bnrelu_*_ex) at the network's layer shapes,
default against deterministic, alternating, on the same scans' tables.  It checks its own claim: two deterministic
steps from the same state give equal SHA-256 digests of the output, the input gradient, every parameter gradient and
the running statistics.  The GPU's name and power limit are read in the same run.

    python tools/deterministic_step_bench.py --steps 5 --rounds 3 [--json OUT]
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from mm2d3d_b200 import _lib, synth  # noqa: E402
from mm2d3d_b200 import functional as F  # noqa: E402
from mm2d3d_b200 import scn  # noqa: E402
from mm2d3d_b200._lib import check, lib, ptr  # noqa: E402
from mm2d3d_b200.metadata import Metadata  # noqa: E402
from mm2d3d_b200.unet import UNetSCN  # noqa: E402

MODES = ("tf32", "tf32x3", "bf16")


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        info["power_limit"] = q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        info["power_limit"] = "unknown"
    return info


def timed(fn, reps):
    """ms per call of fn over reps calls (CUDA events), and libmm3d launches per call."""
    torch.cuda.synchronize()
    k0 = lib.mm3d_kernel_launches()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps, (lib.mm3d_kernel_launches() - k0) / reps


def digest(ts):
    h = hashlib.sha256()
    for t in ts:
        h.update(t.detach().contiguous().cpu().numpy().tobytes())
    return h.hexdigest()


class Step:
    def __init__(self, dev):
        locs, feats = synth.make_batch("nuscenes", batch=8, seed0=0)
        self.coords, self.x = torch.from_numpy(locs).to(dev), torch.from_numpy(feats).to(dev)
        torch.manual_seed(0)
        self.net = UNetSCN(in_channels=3).to(dev)
        self.net.fused = False
        self.state = {k: v.clone() for k, v in self.net.state_dict().items()}
        self.g = torch.randn(len(locs), 16, device=dev, generator=torch.Generator(device=dev).manual_seed(1))

    def __call__(self, keep=False):
        self.net.load_state_dict(self.state)
        self.net.zero_grad(set_to_none=True)
        x = self.x.clone().requires_grad_(True)
        out = self.net([self.coords, x])
        out.backward(self.g)
        if keep:
            return [out, x.grad] + [p.grad for p in self.net.parameters()] + list(self.net.buffers())


def op_shapes(meta, m=16, levels=7):
    """(name, table, c_in, c_out) of the network's convolutions per level, and (name, rows, c) of its BatchNorms."""
    convs, bns = [], []
    s = 4096
    for lv in range(levels):
        c = m * (lv + 1)
        smc, _, _ = F.conv_tables(meta, "smc", s, plans=True)
        convs.append((f"L{lv} smc {c}->{c}", smc, c, c))
        bns.append((f"L{lv} bn {c}", smc.n_out, c))
        if lv + 1 < levels:
            down, _, _ = F.conv_tables(meta, "down", s, plans=True)
            up, _, _ = F.conv_tables(meta, "up", s // 2, plans=True)
            convs.append((f"L{lv} smc {2 * c}->{c}", smc, 2 * c, c))
            convs.append((f"L{lv} down {c}->{c + m}", down, c, c + m))
            convs.append((f"L{lv} up {c + m}->{c}", up, c + m, c))
            bns.append((f"L{lv} bn {2 * c}", smc.n_out, 2 * c))
        s //= 2
    return convs, bns


def per_op(dev, reps):
    locs, _ = synth.make_batch("nuscenes", batch=8, seed0=0)
    meta = Metadata(torch.from_numpy(locs).to(dev), 4096, 7, plans=True)
    convs, bns = op_shapes(meta)
    det = _lib.DETERMINISTIC
    rows = []
    sp = _lib.stream_ptr()
    for mode in MODES:
        mcode = _lib.MODES[mode]
        for name, t, ci, co in convs:
            x = torch.randn(t.n_in, ci, device=dev)
            g = torch.randn(t.n_out, co, device=dev)
            xo = F._tf32(x) if mode == "tf32" else F._planes(x, mode == "bf16")
            go = F._tf32(g) if mode == "tf32" else F._planes(g, mode == "bf16")
            dw = torch.empty(t.K, ci, co, device=dev)
            ws = torch.empty(max(lib.mm3d_conv_wgrad_workspace_bytes(t.n_out, ci, co, t.K, mcode, det), 1),
                             dtype=torch.uint8, device=dev)

            def call(flags):
                check(lib.mm3d_conv_wgrad_ex(ptr(xo), t.n_in, ci, ptr(go), t.n_out, co, ptr(dw), t.K, t.tbl, t.stride,
                                             t.onehot, t.plan, t.plan_cap, 0, mcode, ptr(ws), ws.numel(), sp, flags))
            res = {0: [], det: []}
            for _ in range(3):
                for flags in (0, det):
                    timed(lambda: call(flags), 2)
                    res[flags].append(timed(lambda: call(flags), reps))
            rows.append({"op": "wgrad", "mode": mode, "layer": name, "rows": t.n_out,
                         "default_ms": min(r[0] for r in res[0]), "det_ms": min(r[0] for r in res[det]),
                         "default_launches": res[0][0][1], "det_launches": res[det][0][1]})
    for name, n, c in bns:
        x, dy = torch.randn(n, c, device=dev), torch.randn(n, c, device=dev)
        gamma, beta = torch.ones(c, device=dev), torch.zeros(c, device=dev)
        rm, rv = torch.zeros(c, device=dev), torch.ones(c, device=dev)
        y, dx = torch.empty_like(x), torch.empty_like(x)
        save, dgb = torch.empty(2, c, device=dev), torch.empty(2, c, device=dev)
        ws = torch.empty(lib.mm3d_bnrelu_workspace_bytes_ex(c, det), dtype=torch.uint8, device=dev)

        def call(flags):
            check(lib.mm3d_bnrelu_fwd_ex(ptr(x), ptr(y), n, c, ptr(gamma), ptr(beta), ptr(rm), ptr(rv), ptr(save[0]),
                                         ptr(save[1]), 1e-4, 0.9, 0.0, 1, ptr(ws), ws.numel(), sp, flags))
            check(lib.mm3d_bnrelu_bwd_ex(ptr(x), ptr(dy), ptr(dx), n, c, ptr(gamma), ptr(beta), ptr(save[0]),
                                         ptr(save[1]), ptr(dgb[0]), ptr(dgb[1]), 0.0, 1, ptr(ws), ws.numel(), sp, flags))
        res = {0: [], det: []}
        for _ in range(3):
            for flags in (0, det):
                timed(lambda: call(flags), 2)
                res[flags].append(timed(lambda: call(flags), reps))
        rows.append({"op": "bn fwd+bwd", "mode": "-", "layer": name, "rows": n,
                     "default_ms": min(r[0] for r in res[0]), "det_ms": min(r[0] for r in res[det]),
                     "default_launches": res[0][0][1], "det_launches": res[det][0][1]})
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--op-reps", type=int, default=10)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("deterministic_step_bench: needs a CUDA device")
    dev = torch.device("cuda:0")
    out = {"workload": "UNetSCN(in_channels=3), net.fused=False, batch-8 nuScenes-shaped scans, training step",
           **gpu_info(), "steps": {}}
    step = Step(dev)
    prev = scn.get_conv_mode()
    try:
        for mode in MODES:
            scn.set_conv_mode(mode)
            for flag in (False, True):  # warm-up of both settings
                F.DETERMINISTIC = flag
                step()
            times = {False: [], True: []}
            launches = {}
            for _ in range(args.rounds):
                for flag in (False, True):
                    F.DETERMINISTIC = flag
                    ms, k = timed(step, args.steps)
                    times[flag].append(ms)
                    launches[flag] = k
            F.DETERMINISTIC = True
            d1, d2 = digest(step(keep=True)), digest(step(keep=True))
            out["steps"][mode] = {"default_ms_per_step": min(times[False]), "det_ms_per_step": min(times[True]),
                                  "default_ms_all_rounds": times[False], "det_ms_all_rounds": times[True],
                                  "default_launches_per_step": launches[False],
                                  "det_launches_per_step": launches[True],
                                  "det_sha256_equal": d1 == d2, "det_sha256": d1}
            print(f"{mode:7s} default {min(times[False]):8.3f} ms/step {launches[False]:6.0f} launches | "
                  f"deterministic {min(times[True]):8.3f} ms/step {launches[True]:6.0f} launches | "
                  f"ratio {min(times[True]) / min(times[False]):.3f} | sha256 equal: {d1 == d2}", flush=True)
    finally:
        F.DETERMINISTIC = None
        scn.set_conv_mode(prev)
    out["per_op"] = per_op(dev, args.op_reps)
    for r in out["per_op"]:
        print(f"{r['op']:10s} {r['mode']:7s} {r['layer']:22s} rows {r['rows']:8d}  default {r['default_ms'] * 1e3:8.1f} us "
              f"({r['default_launches']:.0f} launches)  deterministic {r['det_ms'] * 1e3:8.1f} us "
              f"({r['det_launches']:.0f} launches)  x{r['det_ms'] / r['default_ms']:.2f}")
    print(f"GPU: {out['gpu']}, power limit {out['power_limit']}")
    assert lib.mm3d_take_device_error() == 0
    if args.json:
        with open(args.json, "w") as f:
            json.dump(out, f, indent=1)
    if not all(v["det_sha256_equal"] for v in out["steps"].values()):
        raise SystemExit("deterministic steps differ")


if __name__ == "__main__":
    main()
