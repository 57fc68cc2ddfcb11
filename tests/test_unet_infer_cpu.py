"""Inference forward of the whole-network executor without a GPU: the C ABI additions, their bindings, the workspace
query against the training forward's, and the dispatch predicate."""
import ctypes as C
import os
import re

import torch

from mm2d3d_b200 import _lib
from mm2d3d_b200.executor import inference_path

NEW = ["mm3d_unet_topo_infer_bytes", "mm3d_unet_topo_infer"]
HEADER = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "mm3d.h")
TOPOLOGIES = [(reps, res) for reps in (1, 2) for res in (0, 1)]
# rows per level of a batch of 8 nuScenes-shaped scans (the order of magnitude of synth.make_batch at full_scale 4096)
ROWS = [240_000, 150_000, 70_000, 26_000, 8_500, 2_600, 800]


def _desc(rows):
    """Level descriptors with the row counts only: the size queries read nothing else."""
    W = _lib.LEVEL_DESC_WORDS
    d = (C.c_int64 * (W * len(rows)))()
    for l, n in enumerate(rows):
        d[W * l] = n
    return d


def test_new_symbols_declared_exported_bound_and_abi_still_8():
    header = open(HEADER).read()
    for name in NEW:
        assert re.search(r"MM3D_API\s+\w+\s+" + name + r"\(", header), name
        assert name in _lib.SIGNATURES and hasattr(_lib.lib, name)
    assert _lib.lib.mm3d_abi_version() == _lib.ABI_VERSION == 8


def test_infer_workspace_below_training_forward():
    """The inference workspace holds only what the forward writes: below the training forward's activations plus
    its scratch, in every mode and block topology (ratios printed)."""
    lib = _lib.lib
    for L in (7, 5):
        rows = ROWS[:L]
        desc = _desc(rows)
        n_points = 2 * rows[0]
        for name, mode in _lib.MODES.items():
            for reps, res in TOPOLOGIES:
                for in_ch, m in ((3, 16), (1, 16), (3, 32)):
                    train = (lib.mm3d_unet_topo_act_bytes(in_ch, m, L, reps, res, mode, desc, n_points)
                             + lib.mm3d_unet_topo_scratch_bytes(in_ch, m, L, reps, res, mode))
                    infer = lib.mm3d_unet_topo_infer_bytes(in_ch, m, L, reps, res, mode, desc, n_points, 0)
                    assert 0 < infer < train, (name, reps, res, in_ch, m, L, infer, train)
                    # the deterministic mode changes only the InputLayer: same workspace
                    assert lib.mm3d_unet_topo_infer_bytes(in_ch, m, L, reps, res, mode, desc, n_points,
                                                          _lib.DETERMINISTIC) == infer
                    if (in_ch, m) == (3, 16):
                        print(f"{name:7s} L={L} reps={reps} {'res' if res else 'vgg'}: inference / training forward "
                              f"workspace {infer / 2**20:8.1f} / {train / 2**20:8.1f} MiB = {infer / train:.3f}")


def test_infer_workspace_query_rejects_bad_arguments():
    lib = _lib.lib
    desc = _desc(ROWS)
    assert lib.mm3d_unet_topo_infer_bytes(3, 16, 7, 1, 0, _lib.MODE_TF32, None, 10, 0) == 0
    assert lib.mm3d_unet_topo_infer_bytes(3, 16, 7, 1, 0, _lib.MODE_TF32, desc, 10, 0x4) == 0  # unknown flag
    assert lib.mm3d_unet_topo_infer_bytes(3, 16, 7, 0, 0, _lib.MODE_TF32, desc, 10, 0) == 0  # no blocks


def test_dispatch_predicate():
    """Inference path: eval mode and autograd recording nothing (grad mode off, or no input requiring a gradient)."""
    w = torch.zeros(3, requires_grad=True)
    x = torch.zeros(3)
    assert inference_path(False, (x, None, None, w)) is False  # eval, grad mode on, a parameter requires grad
    assert inference_path(False, (x, None, None, w.detach())) is True
    assert inference_path(True, (x, None, None, w.detach())) is False  # training mode: never
    with torch.no_grad():
        assert inference_path(False, (x, None, None, w)) is True
        assert inference_path(True, (x, None, None, w)) is False
    with torch.inference_mode():
        assert inference_path(False, (x, w)) is True
    assert inference_path(False, (x.requires_grad_(True), None, None, w.detach())) is False  # features need a gradient
    mask_w = torch.zeros(1, 3, requires_grad=True)
    assert inference_path(False, (torch.zeros(3), mask_w, torch.zeros(1), w.detach())) is False  # RGB-mask weight
