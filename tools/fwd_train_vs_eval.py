"""Training-mode against eval-mode forward of UNetSCN (tf32, batch of 8 nuScenes-shaped scans, structures reused),
both under torch.no_grad().  A no_grad eval forward takes the inference path (mm3d_unet_topo_infer) in the modes of
executor.INFER_MODES (bf16); in the tf32 mode timed here it runs the eval forward through UNetSCNFn, where the
inference path measured slower (tools/infer_bench.py)."""
import os, sys
sys.path.insert(0, "/root/repo")
import numpy as np, torch
from mm2d3d_b200 import scn as scn_mod, synth
from mm2d3d_b200.unet import UNetSCN
dev = torch.device("cuda", 0)
scn_mod.set_conv_mode("tf32")
torch.manual_seed(0)
net = UNetSCN(in_channels=3, m=16, block_reps=1, residual_blocks=False, full_scale=4096, num_planes=7).to(dev)
res = []
for r in range(4):
    locs, feats = synth.make_batch("nuscenes", batch=8, seed0=r * 8)
    res.append((torch.from_numpy(locs).to(dev), torch.from_numpy(feats).to(dev)))
fixed = [net.prepare(r[0]) for r in res]
torch.cuda.synchronize()
for mode in ("train", "eval", "train", "eval"):
    net.train(mode == "train")
    with torch.no_grad():
        for i in range(5):
            net([fixed[i % 4], res[i % 4][1]])
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(40):
            net([fixed[i % 4], res[i % 4][1]])
        e1.record()
        torch.cuda.synchronize()
    print(mode, "forward only, structure reused:", round(e0.elapsed_time(e1) / 40, 3), "ms")
