#!/usr/bin/env python
"""Benchmark of the hot path: UNetSCN forward+backward on synthetic nuScenes-shaped scans.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--mode fp32|tf32] [--impl ours|reference]
                    [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch (default 8 scans per GPU, BASELINE.json
configs[1]): structure build (voxel hash, 7-level pyramid, rule tables), UNetSCN forward, backward
to the point features and all parameters, and -- for N > 1 -- the flat-gradient all-reduce.
Prints ONE JSON line (rank 0).  ``--impl reference`` times the CPU restatement of the reference's
SparseConvNet path (oracle/, the dependency itself is not installable here) on the host cores.

``--dump-outputs DIR`` writes what the last timed step computed as ``DIR/<name>.npy``: the point
features ``out``, ``grad_feats`` and one ``grad.<parameter>`` per parameter.  The inputs are
seeded, so two builds run with the same arguments can be compared output for output.
``--steps K`` sets the number of timed steps of every measured loop: the headline, the end-to-end
loop, the side modes and, with ``--full-step``, the 3D-branch figures.  The kernel pass times each
launch on its own (3 repetitions); the CPU baseline of the GPU arm times 5 scans.
The benchmark writes nothing into the source tree.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "UNetSCN fwd+bwd scans/sec"
UNIT = "scans/s"
NET_KW = dict(in_channels=3, m=16, block_reps=1, residual_blocks=False, full_scale=4096, num_planes=7)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50, help="timed steps of every measured loop (see the module docstring)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    # BASELINE.json configs[1] names both arithmetic modes; the tensor-core one (tcgen05 kind::tf32, FP32
    # accumulate, parity bar 1e-2) is the headline, the FP32 SIMT parity mode (1e-4) is timed beside it
    ap.add_argument("--mode", default=os.environ.get("MM3D_BENCH_MODE", "tf32"), choices=["fp32", "tf32", "tf32x3", "bf16"])
    ap.add_argument("--no-fp32-side", action="store_true", help="skip the short FP32-mode measurement")
    ap.add_argument("--shape", default="nuscenes", choices=["nuscenes", "semantickitti"])
    ap.add_argument("--batch", type=int, default=8, help="scans per GPU per step")
    ap.add_argument("--rotate", type=int, default=4, help="distinct resident input batches cycled through")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-pipeline", dest="pipeline", action="store_false",
                    help="build each step's sparse structure inline on the compute stream instead of one step ahead")
    ap.add_argument("--no-kernel-pass", action="store_true")
    ap.add_argument("--kernel-pass-json", metavar="FILE", help="write the kernel pass's per-launch rows to FILE")
    ap.add_argument("--graph-2d", action="store_true",
                    help="--full-step: replay the dense 2D network (forward and backward, source and target pass) from CUDA graphs")
    ap.add_argument("--ab", default="", help="development: NAME=VALUE, time alternating blocks of steps with that variable set / unset")
    ap.add_argument("--full-step", action="store_true",
                    help="BASELINE configs[2]: whole MM2D3D training step (2D ResNet34-UNet stand-in on stock cuDNN + lift + "
                         "UNetSCN + heads + losses + optimiser), source and target batch, single GPU")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs and gradients of the last timed step as DIR/<name>.npy (at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.full_step):
        ap.error("--dump-outputs applies to the UNetSCN measurement (--impl ours without --full-step)")
    return args


DUMP_BYTES = 64_000_000  # file sizes included (.npy headers: < 1 kB each)


def to_host(tensors):
    """Host copies of ``{name: tensor}`` in float32 (float64 stays float64), for :func:`dump_outputs`."""
    import numpy as np

    out = {}
    for k, t in tensors.items():
        a = t.detach().cpu().numpy()
        out[k] = a if a.dtype == np.float64 else a.astype(np.float32)
    return out


def dump_outputs(path, per_point, whole):
    """Write every array as ``path/<name>.npy``.  ``per_point`` arrays share their row count; if everything
    together exceeds DUMP_BYTES they keep the same fixed, seeded sample of rows (sorted), so that two runs with the
    same arguments write the same rows.  ``whole`` arrays are written whole."""
    import numpy as np

    n = next(iter(per_point.values())).shape[0]
    row_bytes = sum(a[:1].nbytes for a in per_point.values())
    budget = DUMP_BYTES - sum(a.nbytes + 1024 for a in whole.values()) - 1024 * len(per_point)
    if n * row_bytes > budget:
        rows = np.sort(np.random.default_rng(0).choice(n, budget // row_bytes, replace=False))
        per_point = {k: a[rows] for k, a in per_point.items()}
    os.makedirs(path, exist_ok=True)
    for k, a in {**per_point, **whole}.items():
        np.save(os.path.join(path, k + ".npy"), a)


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            p = json.load(open(path))
            return {"hbm_gbs": float(p["hbm_gbs"]), "bf16_tflops": float(p.get("bf16_tflops", 0)), "source": "measured"}
        except Exception:
            pass
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "source": "fallback"}


# ------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
            t0 = time.time()
            while not self.rows and time.time() - t0 < 3.0:  # nvidia-smi needs a moment before its first line
                time.sleep(0.02)
        except Exception:
            self.proc = None

    def mark(self):
        """Samples taken from now on are 'under load' (the timed region)."""
        self.first = len(self.rows)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        first = getattr(self, "first", 0)
        rows = self.rows[first:] if len(self.rows) > first else self.rows[-1:]
        for r in rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for nme, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nme)
            except Exception:
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------ CPU baseline
def cpu_reference_scans_per_s(iters, warmup, shape):
    """The reference's CPU path restated (oracle/): SparseConvNet's CPU algorithm -- hash-map rule
    books + per-offset index_select -> matmul -> index_add_ -- incl. structure build, 1 scan/step."""
    import torch

    from mm2d3d_b200 import synth
    from mm2d3d_b200.unet import UNetSCN
    from oracle import scn_cpu

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    net = UNetSCN(backend=scn_cpu, **NET_KW)
    locs, feats = synth.make_batch(shape, batch=1, seed0=0)
    locs_t, feats_t = torch.from_numpy(locs), torch.from_numpy(feats)
    g = torch.randn(locs.shape[0], NET_KW["m"])
    times = []
    for i in range(warmup + iters):
        t0 = time.perf_counter()
        x = feats_t.clone().requires_grad_(True)
        out = net([locs_t, x])
        out.backward(g)
        dt = time.perf_counter() - t0
        for p in net.parameters():
            p.grad = None
        if i >= warmup:
            times.append(dt)
    total = sum(times)
    return {"value": len(times) / total, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{len(times)} x (1 {shape}-shaped scan, {locs.shape[0]} points, fwd+bwd incl. rulebook build), "
                      f"{warmup} warm-up, torch {torch.__version__} CPU ops, {cores} threads",
            "ms_per_scan": 1e3 * total / len(times)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    base = cpu_reference_scans_per_s(max(args.steps, 1), max(min(args.warmup, 3), 1), args.shape)
    line = {
        "impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": base["ms_per_scan"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"UNetSCN(m=16, 7 planes, full_scale=4096) fwd+bwd, {args.shape}-shaped scans; "
                               f"CPU sample: 1 scan per step", "reference": "oracle port of SparseConvNet CPU path "
                   "(sparseconvnet@dcf6a7ff is not vendored/installable: no source, no network)"},
        "cpu_baseline": {k: base[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------ kernel pass
def kernel_pass(net, locs_d, feats_d, mode, pk):
    """Time every sparse-convolution launch of one forward+backward individually (CUDA events on
    the launching stream, L2 flushed before each timed launch) through the C ABI, and report the
    roofline of the slowest one plus the time split by op family."""
    import torch

    from mm2d3d_b200 import _lib
    from mm2d3d_b200 import functional as F
    from mm2d3d_b200.scn import _ConvBase

    lib = _lib.lib
    dev = feats_d.device
    records = []

    def hook(mod, inp, out):
        x = inp[0]
        records.append((mod, x.features.detach(), x.metadata, int(x.spatial_size[0])))

    hooks = [m.register_forward_hook(hook) for m in net.modules() if isinstance(m, _ConvBase)]
    names = {m: n for n, m in net.named_modules()}
    fused, net.fused = net.fused, False  # module-by-module run so that the hooks see every layer's input
    try:
        with torch.no_grad():
            net([locs_d, feats_d])
    finally:
        net.fused = fused
    for h in hooks:
        h.remove()

    flush = torch.empty(384 << 20, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream()
    m = _lib.MODES[mode]

    def timed(fn, reps=3):
        ts = []
        for _ in range(reps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            fn()
            e1.record(stream)
            e1.synchronize()
            ts.append(e0.elapsed_time(e1))
        return sum(ts) / len(ts)

    rows = []
    for mod, x, meta, spatial in records:
        w = mod.weight.detach()
        K, c_in, c_out = w.shape[0], w.shape[2], w.shape[3]
        if mode != "fp32" and c_in % 16:
            # the product path pads odd channel counts (the 3-channel stem) to 16 in tensor-core modes
            pad = (-c_in) % 16
            x = torch.nn.functional.pad(x, (0, pad)).contiguous()
            w = torch.nn.functional.pad(w, (0, 0, 0, pad)).contiguous()
            c_in += pad
        fwd_t, bwd_t, bwd_flags = F.conv_tables(meta, mod.kind, spatial, plans=mode != "fp32")
        out = torch.empty(fwd_t.n_out, c_out, device=dev)
        dout = torch.randn(fwd_t.n_out, c_out, device=dev)
        if mode in ("tf32x3", "bf16"):  # the gathered operands carry two planes in these modes
            x, dout = F._planes(x, mode == "bf16"), F._planes(dout, mode == "bf16")
        dx = torch.empty(bwd_t.n_out, c_in, device=dev)
        dw = torch.empty_like(w)
        ws = F.scratch(max(lib.mm3d_conv_workspace_bytes(fwd_t.n_in, fwd_t.n_out, c_in, c_out, K, m),
                           lib.mm3d_conv_workspace_bytes(bwd_t.n_in, bwd_t.n_out, c_out, c_in, K, m)), dev)
        sp = _lib.stream_ptr()
        # pairs of the rule table (for flops)
        if fwd_t.onehot is None:
            lv = meta.level(spatial)
            cap = fwd_t.stride
            if mod.kind == "smc":
                t = meta._lv_view(lv, lv.o_nbr, torch.int32, 27 * cap).view(27, cap)[:, :fwd_t.n_out]
            else:
                t = meta._lv_view(lv, lv.o_child, torch.int32, 8 * cap).view(8, cap)[:, :fwd_t.n_out]
            pairs = int((t >= 0).sum())
        else:
            pairs = fwd_t.n_out

        def f_fwd():
            _lib.check(lib.mm3d_conv_fwd(x.data_ptr(), fwd_t.n_in, c_in, out.data_ptr(), fwd_t.n_out, c_out,
                                         w.data_ptr(), K, fwd_t.tbl, fwd_t.stride, fwd_t.onehot, fwd_t.plan, fwd_t.plan_cap,
                                         0, m, ws.data_ptr(), ws.numel(), sp))

        def f_dgrad():
            _lib.check(lib.mm3d_conv_fwd(dout.data_ptr(), bwd_t.n_in, c_out, dx.data_ptr(), bwd_t.n_out, c_in,
                                         w.data_ptr(), K, bwd_t.tbl, bwd_t.stride, bwd_t.onehot, bwd_t.plan, bwd_t.plan_cap,
                                         bwd_flags, m, ws.data_ptr(), ws.numel(), sp))

        def f_wgrad():
            _lib.check(lib.mm3d_conv_wgrad(x.data_ptr(), fwd_t.n_in, c_in, dout.data_ptr(), fwd_t.n_out, c_out,
                                           dw.data_ptr(), K, fwd_t.tbl, fwd_t.stride, fwd_t.onehot, fwd_t.plan,
                                           fwd_t.plan_cap, 0, m, ws.data_ptr(), ws.numel(), sp))

        tbl_bytes = 4 * K * fwd_t.n_out if fwd_t.onehot is None else 5 * fwd_t.n_out
        alg_bytes = 4 * (fwd_t.n_in * c_in + fwd_t.n_out * c_out) + 4 * K * c_in * c_out + tbl_bytes
        flops = 2 * pairs * c_in * c_out
        for direction, fn in (("fwd", f_fwd), ("dgrad", f_dgrad), ("wgrad", f_wgrad)):
            fn()  # warm
            ms = timed(fn)
            rows.append({"layer": names[mod], "kind": mod.kind, "dir": direction, "c_in": c_in, "c_out": c_out,
                         "n_in": fwd_t.n_in, "n_out": fwd_t.n_out, "pairs": pairs, "ms": ms,
                         "alg_bytes": alg_bytes, "flops": flops})
    top = max(rows, key=lambda r: r["ms"])
    ach = top["alg_bytes"] / (top["ms"] * 1e-3) / 1e9
    split = {}
    for r in rows:
        split[r["kind"] + "_" + r["dir"]] = split.get(r["kind"] + "_" + r["dir"], 0.0) + r["ms"]
    roofline = {
        "bound": "hbm", "achieved": ach, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": ach / pk["hbm_gbs"],
        "traffic": None, "peak_source": pk["source"],
        "kernel": f"conv {top['kind']} {top['dir']} {top['c_in']}->{top['c_out']} @ {top['layer']} "
                  f"({top['n_out']} rows, {top['pairs']} pairs), mode {mode}",
        "launch_ms": top["ms"], "alg_bytes_per_launch": top["alg_bytes"],
        "achieved_tflops": top["flops"] / (top["ms"] * 1e-3) / 1e12,
        "conv_ms_by_family": {k: round(v, 4) for k, v in sorted(split.items())},
        "conv_total_ms": round(sum(r["ms"] for r in rows), 4),
        "conv_total_gflop": round(sum(r["flops"] for r in rows) / 1e9, 3),
    }
    return roofline, rows


# ------------------------------------------------------------------------------------ our arm
def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if args.gpus > 1 and world == 1:
        raise SystemExit("for --gpus N > 1 launch with: python -m torch.distributed.run --nproc-per-node N bench.py --gpus N ...")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the hot path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import datetime
        # NCCL prints its version banner on stdout when the communicator is created; this script's stdout is ONE
        # JSON line, so stdout points at stderr until the communicator exists
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=180))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)

    from mm2d3d_b200 import _lib, synth
    from mm2d3d_b200 import scn as scn_mod
    from mm2d3d_b200.dp import FlatGradAllReduce
    from mm2d3d_b200.unet import UNetSCN

    scn_mod.set_conv_mode(args.mode)
    torch.manual_seed(0)
    # The network runs on a HIGH-priority stream (CUDA: lower number = more urgent; the default stream has the lowest
    # priority): forward / dgrad / BatchNorm form the step's dependent chain, and their CTAs are then dispatched ahead
    # of the weight-gradient stream's and the structure stream's whenever an SM frees up.  Measured on one box,
    # alternating processes: 2.94 against 2.98 ms per step (profiles/r2_streamk_ab.txt).  MM3D_BENCH_MAIN_PRIO=0
    # restores the default stream.
    main_prio = int(os.environ.get("MM3D_BENCH_MAIN_PRIO", "-1"))
    if main_prio:
        torch.cuda.set_stream(torch.cuda.Stream(device=dev, priority=main_prio))
    net = UNetSCN(**NET_KW).to(dev)
    flat = FlatGradAllReduce(net)
    flat.broadcast_parameters()

    # resident inputs: `rotate` distinct batches per rank (different scans on every rank)
    host, resident = [], []
    for r in range(args.rotate):
        locs, feats = synth.make_batch(args.shape, batch=args.batch, seed0=(rank * args.rotate + r) * args.batch)
        gout = np.random.default_rng(77 + r).standard_normal((locs.shape[0], NET_KW["m"]), dtype=np.float32)
        host.append((torch.from_numpy(locs).pin_memory(), torch.from_numpy(feats).pin_memory()))
        resident.append((torch.from_numpy(locs).to(dev), torch.from_numpy(feats).to(dev), torch.from_numpy(gout).to(dev)))
    n_points = [int(h[0].shape[0]) for h in host]

    # The sparse structure of step i+1 (voxel hash, rule tables, row plans: ~60 launches and the one host read-back
    # of the row counts) is built on a second stream right after step i has been enqueued -- what a prefetching data
    # loader does with UNetSCN.prepare().  Every timed step still contains exactly one structure build and one
    # forward+backward; --no-pipeline builds the structure inline, on the compute stream, as round-1 v8 did.
    prep_stream = torch.cuda.Stream(device=dev, priority=int(os.environ.get("MM3D_BENCH_PREP_PRIO", "0")))
    prepared = {}
    in_flight = []  # end-of-step events: the host stays at most one step ahead of the GPU, like a training loop
                    # that logs its loss one step late (the end-to-end loop below does exactly that)

    def prepare(i, coords=None, stream=prep_stream):
        with torch.cuda.stream(stream):
            prepared[i] = net.prepare(resident[i % args.rotate][0] if coords is None else coords)

    counter = [0]

    def step(_=None):
        i = counter[0]  # steps are numbered across all loops so that the one-step-ahead structure is always the right one
        counter[0] += 1
        locs_d, feats_d, gout = resident[i % args.rotate]
        flat.zero_()
        x = feats_d.detach().requires_grad_(True)  # d(feats) is on the path (3d_net/model.py:46-48)
        if args.pipeline:
            if i not in prepared:
                prepare(i)
            cur = prepared.pop(i)
            prepare(i + 1)  # enqueued (not waited for) before this step's own ~200 launches
            out = net([cur, x])
        else:
            out = net([locs_d, x])
        out.backward(gout)
        flat.all_reduce_mean()
        if args.pipeline:
            ev = torch.cuda.Event()
            ev.record()
            in_flight.append(ev)
            if len(in_flight) > 1:
                in_flight.pop(0).synchronize()
        return out, x

    # End to end: every step's inputs come from pinned host memory and its scalar result goes back to the host.
    # The upload of step i+1 is issued on a copy stream while step i computes (what a prefetching data loader does);
    # each step still pays for one upload and one read-back inside the timed region.
    copy_stream = torch.cuda.Stream(device=dev)
    pending = {}

    def upload(i):
        locs_h, feats_h = host[i % args.rotate]
        with torch.cuda.stream(copy_stream):
            locs_d = locs_h.to(dev, non_blocking=True)
            feats_d = feats_h.to(dev, non_blocking=True)
            # pipelined: the structure is built behind its own upload, on the copy stream
            prep = net.prepare(locs_d) if args.pipeline else None
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        pending[i] = (locs_d, feats_d, ev, prep)

    res_ring = [torch.empty((), dtype=torch.float32, pin_memory=True) for _ in range(4)]

    host_prof = {} if os.environ.get("MM3D_BENCH_HOST_PROFILE") else None

    def _tick(name, t0):
        if host_prof is not None:
            host_prof.setdefault(name, []).append(time.perf_counter() - t0)
        return time.perf_counter()

    def step_e2e(i):
        t = time.perf_counter()
        if i not in pending:
            upload(i)
        locs_d, feats_d, ev, prep = pending.pop(i)
        upload(i + 1)
        t = _tick("upload+prepare(i+1)", t)
        torch.cuda.current_stream().wait_event(ev)
        locs_d.record_stream(torch.cuda.current_stream())
        feats_d.record_stream(torch.cuda.current_stream())
        gout = resident[i % args.rotate][2]
        flat.zero_()
        x = feats_d.requires_grad_(True)
        out = net([prep if args.pipeline else locs_d, x])
        t = _tick("forward", t)
        out.backward(gout)
        t = _tick("backward", t)
        flat.all_reduce_mean()
        t = _tick("all_reduce", t)
        res = (out.detach() * gout).sum()  # the step's scalar result ...
        host_res = res_ring[i % len(res_ring)]  # pinned once: page-locking per step serialises in the driver at N > 1
        host_res.copy_(res, non_blocking=True)  # ... goes back to the host; it is waited for (and used) one step later,
        done = torch.cuda.Event()               # after the next step has been enqueued (lazy loss logging)
        done.record()
        _tick("result", t)
        return host_res, done

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for i in range(args.warmup):
        step(i)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for i in range(3):  # (every rank: steps contain a collective) keep the GPU busy until the sampler's first in-load line is due
        step(i)
    barrier()
    if rank == 0:
        sampler.mark()
    launches0 = _lib.lib.mm3d_kernel_launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps - 1):
        step(i)
    # only the last step's result is kept (for --dump-outputs): a step's output holds its whole activation arena
    last = step(args.steps - 1)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = _lib.lib.mm3d_kernel_launches() - launches0
    dumped = None
    if args.dump_outputs and rank == 0:  # copied before any further step overwrites the gradients; written later
        out, x = last
        dumped = (to_host({"out": out, "grad_feats": x.grad}),
                  to_host({"grad." + k: p.grad for k, p in net.named_parameters()}))
    del last
    # a short timed region can fall between two 50 ms samples: run on under the sampler for ~0.4 s (the same number
    # of extra steps on every rank, decided by rank 0, because steps contain a collective)
    extra = torch.tensor([0 if os.environ.get("MM3D_BENCH_NO_RUNON") else
                          max(0, int(400.0 / max(ms / args.steps, 1e-3)) - args.steps)], device=dev, dtype=torch.int64)
    if world > 1:
        dist.broadcast(extra, 0)
    for i in range(int(extra.item())):
        step(i)
        if i % 8 == 7:
            torch.cuda.synchronize()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    if dumped is not None:
        dump_outputs(args.dump_outputs, *dumped)

    if args.ab and world == 1:
        # development aid: alternate blocks of steps with an environment switch of the library set / unset (switches
        # that the library reads at every call), in ONE process on ONE box -- box-to-box variation is larger than most
        # kernel changes.  Printed on stderr; not part of the JSON line.
        name, _, val = args.ab.partition("=")
        rows = {"set": [], "unset": []}
        for rnd in range(6):
            for which in ("set", "unset"):
                if which == "set":
                    os.environ[name] = val
                else:
                    os.environ.pop(name, None)
                for i in range(3):
                    step(i)
                barrier()
                a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a0.record()
                for i in range(args.steps):
                    step(i)
                a1.record()
                barrier()
                rows[which].append(a0.elapsed_time(a1) / args.steps)
        os.environ.pop(name, None)
        for which in rows:
            v = sorted(rows[which])
            print(f"[ab] {name}={val} {which:5s}: median {v[len(v) // 2]:.3f} ms  all {' '.join(f'{x:.3f}' for x in rows[which])}", file=sys.stderr)

    # end to end: pinned host inputs -> device -> fwd+bwd (-> all-reduce) -> scalar back to the host
    # untimed lead-in: every distinct batch once (+2), so that the copy stream's allocator pool has seen all sizes and
    # no cudaMalloc (a device-wide synchronisation, slower still with N processes) falls into the timed region
    e2e_counter = [0]

    def time_e2e(steps):
        n_pre = max(min(args.warmup, 3), args.rotate + 2)
        base = e2e_counter[0]
        for i in range(base, base + n_pre):
            step_e2e(i)
        barrier()
        t0 = time.perf_counter()
        prev, acc = None, 0.0
        for i in range(base + n_pre, base + n_pre + steps):
            cur = step_e2e(i)
            if prev is not None:
                tw = time.perf_counter()
                prev[1].synchronize()
                acc += float(prev[0])
                _tick("wait(previous step)", tw)
            prev = cur
        prev[1].synchronize()
        acc += float(prev[0])
        barrier()
        dt = (time.perf_counter() - t0) * 1e3
        if host_prof:
            print(f"[rank {rank}] e2e host phases, median ms over {steps} steps: " +
                  ", ".join(f"{k} {1e3 * sorted(v)[len(v) // 2]:.3f}" for k, v in host_prof.items()), file=sys.stderr, flush=True)
            host_prof.clear()
        e2e_counter[0] = base + n_pre + steps
        pending.clear()
        if acc != acc:
            raise SystemExit("bench.py: the end-to-end loop produced NaN")
        return dt

    e2e_ms = time_e2e(args.steps)

    if world > 1:
        t = torch.tensor([ms, e2e_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_ms = float(t[0]), float(t[1])

    if rank == 0:
        pk = peaks()
        roofline, cpu = None, None
        if not args.no_kernel_pass:
            roofline, rows = kernel_pass(net, resident[0][0], resident[0][1], args.mode, pk)
            roofline["share_of_step"] = roofline["conv_total_ms"] / (ms / args.steps)
            roofline["share_note"] = ("conv_total_ms sums launches timed one by one with a cold L2; inside a step the weight-"
                                      "gradient kernels run on a second stream beside dgrad/BatchNorm and the caches are warm, "
                                      "so the sum can exceed the step time")
            if args.kernel_pass_json:
                try:
                    with open(args.kernel_pass_json, "w") as f:
                        json.dump(rows, f, indent=0)
                except OSError as e:  # a side table: the benchmark line is printed regardless
                    print(f"bench.py: could not write {args.kernel_pass_json}: {e}", file=sys.stderr)
        if world == 1 and not args.no_cpu_baseline:
            cpu = cpu_reference_scans_per_s(5, 1, args.shape)
            cpu = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")}
        # the precision-matched modes (the reference's 3D branch is FP32, SURVEY 3.3) as full measurements: same workload,
        # same loops -- device-timed value and end-to-end value.  "fp32" = SIMT FMA kernels, "tf32x3" = tensor cores with
        # three error-compensated TF32 products (both hold the 1e-4 bars)
        side = {}
        if world == 1 and args.mode == "tf32" and not args.no_fp32_side:
            notes = {"fp32": "same workload and loops in the FP32 SIMT parity mode (activations / gradients within 1e-4): the "
                             "figure to set against the reference's FP32 3D branch",
                     "tf32x3": "same workload and loops with FP32-grade arithmetic on the tensor cores: every convolution as three "
                               "error-compensated TF32 products (hi.hi + lo.hi + hi.lo), activations / gradients within 1e-4",
                     "bf16": "same workload and loops with BF16 gathered operands and weights in forward and dgrad (kind::f16, FP32 "
                             "accumulate, half the gathered bytes), TF32 weight gradients; 1e-2 per op"}
            for smode in ("fp32", "tf32x3", "bf16"):
                scn_mod.set_conv_mode(smode)
                prepared.clear()  # (row plans are built per mode)
                try:
                    n_f = args.steps
                    for i in range(3):
                        step(i)
                    barrier()
                    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    f0.record()
                    for i in range(n_f):
                        step(i)
                    f1.record()
                    barrier()
                    fms = f0.elapsed_time(f1) / n_f
                    prepared.clear()
                    fe2e = time_e2e(n_f) / n_f
                    side[smode] = {"value": args.batch / (fms * 1e-3), "unit": UNIT, "ms_per_step": fms, "steps": n_f, "warmup": 3,
                                   "dtype": {"fp32": "f32", "tf32x3": "tf32x3 (f32-grade)", "bf16": "bf16"}[smode],
                                   "e2e": {"value": args.batch / (fe2e * 1e-3), "unit": UNIT, "ms_per_step": fe2e}, "note": notes[smode]}
                finally:
                    scn_mod.set_conv_mode(args.mode)
                    prepared.clear()
        if roofline is not None:
            # DRAM traffic of the dominant kernel: from an `ncu --set full` capture (profiles/ncu_traffic.json) of the SAME
            # kernel source -- the entry records the SHA-1 of the kernel's .cu file at capture time; any other build
            # prints null rather than a stale number
            try:
                import hashlib
                tr = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
                key = roofline["kernel"].split(" @ ")[0] + f" rows {roofline['kernel'].split('(')[1].split(' rows')[0]} {args.mode}"
                ent = tr.get(key)
                srcs = (ent["src_file"], "mm2d3d_b200/csrc/tc_common.cuh", "mm2d3d_b200/csrc/plan.cuh") if ent else ()
                if ent and hashlib.sha1(b"".join(open(os.path.join(ROOT, f), "rb").read() for f in srcs)).hexdigest() == ent["src_sha1"]:
                    roofline["traffic"] = ent["dram_bytes"]
                    roofline["traffic_source"] = ent["source"]
            except Exception:
                pass
        scans = world * args.batch * args.steps
        avg_pts = sum(n_points) / len(n_points)
        line = {
            "impl": "ours", "metric": METRIC, "value": scans / (ms * 1e-3), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None,
            "dtype": {"fp32": "f32", "tf32": "tf32", "bf16": "bf16", "tf32x3": "tf32x3 (f32-grade)"}[args.mode], "data": "synthetic",
            "config": {
                "workload": f"UNetSCN(m=16, 7 planes, full_scale=4096) fwd+bwd, batch {args.batch} "
                            f"{args.shape}-shaped scans per GPU (BASELINE configs[1])",
                "scans_per_gpu": args.batch, "points_per_batch": avg_pts, "conv_mode": args.mode,
                "parallelism": f"dp{world} by scan, flat-gradient all-reduce ({flat.nbytes} B)" if world > 1 else "single GPU",
                "l2": f"{args.rotate} rotating resident input batches; one step touches >1 GB of activations/tables, "
                      "far above the 126 MB L2, so no step starts with its data cached",
                "step": "structure build + forward + backward (d_feats and all parameter grads)"
                        + (" + gradient all-reduce" if world > 1 else ""),
                "structure": "built one step ahead on a second stream (UNetSCN.prepare); one build per timed step"
                             if args.pipeline else "built inline on the compute stream",
            },
            "clocks": clocks,
            "e2e": {"value": scans / (e2e_ms * 1e-3), "unit": UNIT,
                    "h2d_bytes_per_step": int(avg_pts * (32 + 4 * NET_KW["in_channels"])), "d2h_bytes_per_step": 4,
                    "ms_per_step": e2e_ms / args.steps},
            "gpu_launches": int(launches),
        }
        if roofline is not None:
            line["roofline"] = roofline
        for smode, rec in side.items():
            line[smode + "_mode"] = rec
        if cpu is not None:
            line["cpu_baseline"] = cpu
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------ full step (configs[2])
def run_full_step(args):
    """One optimisation step of the reference's trainer (train.py:186-292): source AND target batch through the 2D and
    the 3D network (4 forwards), cross-entropy on the source, cross-modal KL on both, one backward, one optimiser step.
    The 2D network is a stock-cuDNN stand-in of the reference's Net2DSeg (tools/net2d_standin.py; channels-last, BF16
    autocast like the reference's AMP); lift, RGB mask, UNetSCN and the KL terms are this package's kernels."""
    import numpy as np
    import torch
    import torch.nn.functional as F

    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from net2d_standin import Dense2D, RGBDUNet2D

    from mm2d3d_b200 import _lib, synth
    from mm2d3d_b200 import scn as scn_mod
    from mm2d3d_b200.heads import cross_modal_kl, heads3d
    from mm2d3d_b200.lift import LiftIndices
    from mm2d3d_b200.unet import UNetSCN

    if args.gpus != 1:
        raise SystemExit("bench.py --full-step: single GPU only")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    scn_mod.set_conv_mode(args.mode)
    torch.manual_seed(0)
    C, H, W = 6, 225, 400  # nuScenes-lidarseg merged classes (config.yaml), resize [400, 225]
    net2d = RGBDUNet2D(C).to(dev).to(memory_format=torch.channels_last)
    net3d = UNetSCN(**NET_KW).to(dev)
    mask = torch.nn.Linear(3, 1).to(dev)
    head, head_aux = torch.nn.Linear(16, C).to(dev), torch.nn.Linear(16, C).to(dev)
    params = [*net2d.parameters(), *net3d.parameters(), *mask.parameters(), *head.parameters(), *head_aux.parameters()]
    opt = torch.optim.Adam(params, lr=1e-4, fused=True)

    data = {"src": [], "trg": []}
    for d, dom in enumerate(("src", "trg")):
        for r in range(args.rotate):
            seed0 = (d * args.rotate + r) * args.batch
            locs, feats = synth.make_batch(args.shape, batch=args.batch, seed0=seed0)
            counts = np.bincount(locs[:, 3], minlength=args.batch).tolist()
            idx = synth.make_img_indices(counts, H, W, seed=seed0)
            rng = np.random.default_rng(seed0)
            data[dom].append(dict(
                locs=torch.from_numpy(locs).to(dev), feats=torch.from_numpy(feats).to(dev),
                img=torch.from_numpy(rng.random((args.batch, 3, H, W), dtype=np.float32)).to(dev).contiguous(memory_format=torch.channels_last),
                depth=torch.from_numpy((rng.random((args.batch, 1, H, W), dtype=np.float32) < 0.04).astype(np.float32) * 30).to(dev),
                li=LiftIndices(idx, dev), labels=torch.from_numpy(rng.integers(0, C, locs.shape[0])).to(dev)))
    n_points = float(np.mean([b["locs"].shape[0] for dom in data for b in data[dom]]))
    ev3d = []
    # SURVEY 8(f).4: the dense 2D network (static shapes) replayed from CUDA graphs -- one graph pair (forward, backward)
    # per pass of the step, because the source and the target pass are both alive when backward starts; the lifts (a
    # different number of points every batch) stay outside
    graphed = None
    if args.graph_2d:
        b0 = data["src"][0]
        with torch.autocast("cuda", dtype=torch.bfloat16, cache_enabled=False):
            graphed = dict(zip(("src", "trg"), torch.cuda.make_graphed_callables(
                (Dense2D(net2d), Dense2D(net2d)), ((b0["img"], b0["depth"]), (b0["img"], b0["depth"])))))
    from mm2d3d_b200.lift import lift2d

    def step(i, time3d=False):
        loss = 0.0
        for dom in ("src", "trg"):
            b = data[dom][i % args.rotate]
            if graphed is not None:
                with torch.autocast("cuda", dtype=torch.bfloat16, cache_enabled=False):
                    m2d, ma2d = graphed[dom](b["img"], b["depth"])
                l2d, a2d = lift2d(m2d.float(), b["li"]), lift2d(ma2d.float(), b["li"])
            else:
                with torch.autocast("cuda", dtype=torch.bfloat16):
                    l2d, a2d, _ = net2d(b["img"], b["depth"], b["li"])
            if time3d:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
            out3d = net3d([b["locs"], b["feats"]], rgb_mask=mask)  # the RGB-mask prologue rides in the InputLayer scatter
            if time3d:
                e1.record()
                ev3d.append((e0, e1))
            # both 3D heads and the 3D side of the cross-modal loss in one pass over the [N, 16] features (SURVEY 8(f).3)
            l3d, _, xm3d = heads3d(out3d, head.weight, head.bias, head_aux.weight, head_aux.bias, l2d)
            if dom == "src":
                loss = loss + F.cross_entropy(l2d, b["labels"]) + F.cross_entropy(l3d, b["labels"])
            loss = loss + 0.1 * (xm3d + cross_modal_kl(a2d, l3d))
        loss.backward()
        opt.step()
        opt.zero_grad(set_to_none=True)
        return loss

    for i in range(max(args.warmup, 3)):
        step(i)
    torch.cuda.synchronize()
    sampler = ClockSampler(0)
    sampler.start()
    for i in range(3):
        step(i)
    torch.cuda.synchronize()
    sampler.mark()
    launches0 = _lib.lib.mm3d_kernel_launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        last = step(i)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    launches = _lib.lib.mm3d_kernel_launches() - launches0
    if not bool(torch.isfinite(last)):
        raise SystemExit("bench.py --full-step: non-finite loss")
    for i in range(max(0, int(400.0 / ms) - args.steps)):
        step(i)
    torch.cuda.synchronize()
    clocks = sampler.stop()
    # the 3D branch alone, same batches: mask + UNetSCN forward (events inside the step), and forward+backward
    for i in range(args.steps):
        step(i, time3d=True)
    torch.cuda.synchronize()
    fwd3d = sum(a.elapsed_time(b) for a, b in ev3d) / args.steps

    def only3d(i):
        for dom in ("src", "trg"):
            b = data[dom][i % args.rotate]
            x = b["feats"].detach().requires_grad_(True)
            out = net3d([b["locs"], x])
            out.backward(torch.ones_like(out))
        for p_ in net3d.parameters():
            p_.grad = None
    for i in range(3):
        only3d(i)
    torch.cuda.synchronize()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for i in range(args.steps):
        only3d(i)
    f1.record()
    torch.cuda.synchronize()
    ms3d = f0.elapsed_time(f1) / args.steps
    scans = 2 * args.batch
    line = {
        "impl": "ours", "metric": "full MM2D3D training step scans/sec (source + target)", "value": scans / (ms * 1e-3), "unit": UNIT,
        "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": {"fp32": "f32", "tf32": "tf32", "tf32x3": "tf32x3", "bf16": "bf16"}[args.mode] + " (3D) / bf16 autocast (2D)", "data": "synthetic",
        "config": {
            "workload": f"BASELINE configs[2]: full MM2D3D step -- ResNet34-UNet stand-in on {H}x{W} RGB-D (46.2 M parameters, "
                        f"stock cuDNN, channels-last, BF16 autocast{', dense part replayed from CUDA graphs' if args.graph_2d else ''}) + 2D->3D lift + RGB mask + UNetSCN(m=16, 7 planes) + 2+2 heads "
                        f"+ CE / cross-modal KL + fused Adam; batch {args.batch} source + {args.batch} target {args.shape}-shaped scans",
            "points_per_batch": n_points, "conv_mode": args.mode,
            "structure": "built inline by each 3D forward", "l2": f"{args.rotate} rotating resident batches per domain",
        },
        "clocks": clocks, "gpu_launches": int(launches),
        "branch_3d": {"forward_ms_inside_step": fwd3d, "fwd_bwd_ms_alone": ms3d, "share_of_step": ms3d / ms,
                      "note": "UNetSCN (+ mask) on the step's two batches; forward timed with events inside the full step, "
                              "forward+backward timed alone on the same batches"},
    }
    print(json.dumps(line), flush=True)


def main():
    args = parse_args()
    if os.environ.get("MM3D_ABL_SKIP"):
        # ablation builds (-DMM3D_ABLATION) skip kernel families: never a benchmark number
        raise SystemExit("bench.py: MM3D_ABL_SKIP is set -- refusing to print a benchmark line for an ablated run")
    if args.impl == "reference":
        run_reference(args)
    elif args.full_step:
        run_full_step(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
