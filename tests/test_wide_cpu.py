"""Wide UNetSCN layers (up to 512 channels) without a GPU: the C queries that size them and the FP64 oracle's
conditioning at m = 32.

Layers wider than 256 channels run as slices of the shapes the kernels take (DESIGN.md section 5).  The
deterministic weight gradient then needs the slab of its largest slice: never 0 for a wide shape in a tensor-core
mode, never more than one 256 KB slab per SM plus the 256-byte table.
"""
import ctypes

import pytest

from mm2d3d_b200 import _lib
from mm2d3d_b200.executor import wgrad_covered
from tests.test_exec_fp64_cpu import conditioned_net

TC_MODES = {"tf32": _lib.MODE_TF32, "tf32x3": _lib.MODE_TF32X3, "bf16": _lib.MODE_BF16}
WIDE_SHAPES = [(384, 192, 27), (192, 384, 27), (320, 160, 27), (448, 224, 27), (512, 512, 27), (256, 288, 8),
               (288, 256, 8), (384, 192, 1)]
SMS = 148  # B200; the library's SM count without a device


def _lib_handle():
    lib = _lib.lib
    lib.mm3d_conv_wgrad_workspace_bytes.restype = ctypes.c_size_t
    lib.mm3d_conv_wgrad_workspace_bytes.argtypes = [ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                                    ctypes.c_int, ctypes.c_int]
    return lib


@pytest.mark.parametrize("mode", list(TC_MODES))
@pytest.mark.parametrize("shape", WIDE_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_deterministic_wgrad_workspace_of_wide_shapes(shape, mode):
    lib = _lib_handle()
    ci, co, k = shape
    b = lib.mm3d_conv_wgrad_workspace_bytes(0, ci, co, k, TC_MODES[mode], _lib.DETERMINISTIC)
    assert 0 < b <= 256 + SMS * 256 * 1024, (shape, mode, b)


@pytest.mark.parametrize("mode", list(TC_MODES))
@pytest.mark.parametrize("res", [0, 1])
def test_wgrad_covered_at_m32(mode, res):
    assert wgrad_covered(3, 32, 7, res, TC_MODES[mode])


def test_conditioning_opens_the_gates_at_m32():
    _, self_check = conditioned_net(1, False, m=32)
    near = self_check()
    print(f"\nm = 32 (1, VGG): {near} BatchNorm pre-activations near the kink")
