"""Deterministic mode of the whole-network executor without a GPU: the C ABI additions, their bindings and the
scratch query with and without MM3D_DETERMINISTIC."""
import os
import re

from mm2d3d_b200 import _lib
from mm2d3d_b200.executor import wgrad_covered

NEW = ["mm3d_input_masked_fwd_csr", "mm3d_input_masked_bwd_ex", "mm3d_unet_topo_scratch_bytes_ex",
       "mm3d_unet_topo_forward_ex", "mm3d_unet_topo_backward_ex"]
HEADER = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "mm3d.h")
TOPOLOGIES = [(reps, res) for reps in (1, 2) for res in (0, 1)]


def test_new_symbols_declared_exported_bound_and_abi_still_8():
    header = open(HEADER).read()
    for name in NEW:
        assert re.search(r"MM3D_API\s+\w+\s+" + name + r"\(", header), name
        assert name in _lib.SIGNATURES and hasattr(_lib.lib, name)
    assert _lib.lib.mm3d_abi_version() == _lib.ABI_VERSION == 8


def test_flags_zero_scratch_query_is_the_old_one():
    lib = _lib.lib
    for mode in _lib.MODES.values():
        for reps, res in TOPOLOGIES:
            for in_ch, m, L in ((3, 16, 6), (1, 16, 7), (3, 32, 5), (3, 8, 4)):
                assert (lib.mm3d_unet_topo_scratch_bytes_ex(in_ch, m, L, reps, res, mode, 0)
                        == lib.mm3d_unet_topo_scratch_bytes(in_ch, m, L, reps, res, mode)), (mode, reps, res, m, L)


def _conv_shapes(in_ch, m, L, res):
    cin_k = (in_ch + 15) // 16 * 16
    shapes = [(cin_k, m, 27)]
    for l in range(L):
        p = m * (l + 1)
        shapes.append((p, p, 27))
        if l + 1 < L:
            q = m * (l + 2)
            shapes += [(p, q, 8), (q, p, 8), (2 * p, p, 27)] + ([(2 * p, p, 1)] if res else [])
    return shapes


def test_deterministic_scratch_query_adds_slabs_and_bn_workspace():
    lib, det = _lib.lib, _lib.DETERMINISTIC
    for mode in (_lib.MODE_TF32, _lib.MODE_TF32X3, _lib.MODE_BF16):
        for reps, res in TOPOLOGIES:
            for in_ch, m, L in ((3, 16, 6), (1, 16, 7), (3, 32, 5)):
                old = lib.mm3d_unet_topo_scratch_bytes(in_ch, m, L, reps, res, mode)
                new = lib.mm3d_unet_topo_scratch_bytes_ex(in_ch, m, L, reps, res, mode, det)
                slab = max(lib.mm3d_conv_wgrad_workspace_bytes(0, ci, co, K, mode, det)
                           for ci, co, K in _conv_shapes(in_ch, m, L, res))
                assert slab > 0
                bn = lib.mm3d_bnrelu_workspace_bytes_ex(2 * m * L, det)
                assert new >= old + slab + bn, (mode, reps, res, m, L, old, new, slab, bn)


def test_wgrad_coverage():
    for reps, res in TOPOLOGIES:
        assert not wgrad_covered(3, 16, 6, res, _lib.MODE_FP32)
        for mode in (_lib.MODE_TF32, _lib.MODE_TF32X3, _lib.MODE_BF16):
            assert wgrad_covered(3, 16, 6, res, mode)
            assert wgrad_covered(3, 32, 4, res, mode)
            assert not wgrad_covered(3, 8, 4, res, mode)  # channel counts the tcgen05 kernels do not take
