"""bench.py --impl reference runs without a GPU (the CPU oracle port) and prints ONE JSON line with the keys the
driver reads; the product arm refuses to run without a GPU instead of falling back to anything."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "UNetSCN fwd+bwd scans/sec" and d["unit"] == "scans/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 1
    assert d["value"] > 0 and abs(d["ms_per_step"] * d["value"] - 1000.0) < 1e-3 * 1000.0  # one scan per CPU step
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["sample"] and cb["value"] == d["value"]
    e = d["e2e"]
    assert e["value"] == d["value"] and e["unit"] == d["unit"] and e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0
    assert d["vs_baseline"] is None and d["data"] == "synthetic" and "workload" in d["config"]


def test_product_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a GPU is present")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode != 0  # no CPU fallback
    assert not any(l.lstrip().startswith("{") for l in r.stdout.splitlines())


@pytest.mark.gpu
def test_product_arm_dumps_the_last_timed_step(tmp_path):
    """--dump-outputs writes the outputs and gradients of the LAST TIMED step.  With --rotate 8 --batch 1 each step
    works on one of 8 distinct seeded scans in turn; with --warmup 2 --steps 3 the last timed step is the run's 8th
    (2 warm-up, 3 lead-in steps under the clock sampler, 3 timed), so it works on scan 7.  The CPU oracle recomputes
    that step here from the same seeds and weights (a warm-up step, a step after the timed ones or a timed loop that
    ignored --steps would have worked on another scan).  A second run with the same arguments writes the same
    arrays: float32, at most 64 MB."""
    import numpy as np
    import torch

    sys.path.insert(0, ROOT)
    import bench
    from mm2d3d_b200 import synth
    from mm2d3d_b200.unet import UNetSCN
    from oracle import scn_cpu

    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--mode", "fp32", "--batch", "1", "--rotate", "8",
           "--warmup", "2", "--steps", "3", "--no-cpu-baseline", "--no-kernel-pass", "--no-fp32-side"]
    dumps = []
    for run in ("a", "b"):
        dumps.append(tmp_path / run)
        r = subprocess.run(cmd + ["--dump-outputs", str(dumps[-1])], capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        lines = [l for l in r.stdout.splitlines() if l.strip()]
        assert len(lines) == 1 and json.loads(lines[0])["steps"] == 3, lines
    names = sorted(os.listdir(dumps[0]))
    assert names == sorted(os.listdir(dumps[1]))
    assert {"out.npy", "grad_feats.npy", "grad.layer2.weight.npy"} <= set(names) and len(names) == 2 + 78  # 78 parameter tensors
    assert sum(os.path.getsize(dumps[0] / n) for n in names) <= 64_000_000
    got = {n[:-4]: np.load(dumps[0] / n) for n in names}
    for n in names:
        a, b = got[n[:-4]], np.load(dumps[1] / n)
        assert a.dtype == np.float32 and a.shape == b.shape and np.isfinite(a).all(), n
        a, b = a.astype(np.float64), b.astype(np.float64)
        if n == "out.npy":
            assert np.abs(a - b).max() <= 1e-3 * np.abs(b).max(), n
        else:  # a ReLU gate that flips between the runs moves one gradient entry by O(1)
            assert np.linalg.norm(a - b) <= 1e-2 * max(np.linalg.norm(b), 1e-30), n

    # the last timed step, recomputed by the CPU oracle: bench.py's weights (torch.manual_seed(0)), scan 7 and its
    # output gradient (seeded 77 + 7)
    torch.manual_seed(0)
    weights = UNetSCN(**bench.NET_KW).state_dict()  # built as bench.py builds it
    ref = UNetSCN(backend=scn_cpu, **bench.NET_KW)
    ref.load_state_dict(weights)
    locs, feats = synth.make_batch("nuscenes", batch=1, seed0=7)
    gout = np.random.default_rng(77 + 7).standard_normal((locs.shape[0], bench.NET_KW["m"]), dtype=np.float32)
    x = torch.from_numpy(feats).requires_grad_(True)
    out = ref([torch.from_numpy(locs), x])
    out.backward(torch.from_numpy(gout))
    want = {"out": out.detach(), "grad_feats": x.grad, **{"grad." + k: p.grad for k, p in ref.named_parameters()}}
    assert set(want) == set(got)
    for k, w in want.items():
        a, w = got[k].astype(np.float64), w.double().numpy()
        assert a.shape == w.shape, k
        if k == "out":  # the FP32 forward bar
            assert np.abs(a - w).max() <= 1e-4 * np.abs(w).max(), k
        else:  # FP32 gradients of this 60-layer BN/ReLU net are ~3e-3 (rel-L2) from FP64 on either side
            assert np.linalg.norm(a - w) <= 2e-2 * np.linalg.norm(w), k
