"""Deterministic weight gradient and BatchNorm without a GPU: the C ABI additions and their workspace queries."""
import torch

from mm2d3d_b200 import _lib

NEW = ["mm3d_conv_wgrad_ex", "mm3d_conv_wgrad_workspace_bytes", "mm3d_bnrelu_fwd_ex", "mm3d_bnrelu_bwd_ex",
       "mm3d_bnrelu_workspace_bytes_ex"]


def _sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count if torch.cuda.is_available() else 148


def test_new_symbols_bound_and_abi_still_8():
    for name in NEW:
        assert name in _lib.SIGNATURES and hasattr(_lib.lib, name)
    assert _lib.lib.mm3d_abi_version() == _lib.ABI_VERSION == 8


def test_flags_zero_queries_are_the_old_ones():
    lib = _lib.lib
    for mode in _lib.MODES.values():
        assert lib.mm3d_conv_wgrad_workspace_bytes(250_000, 64, 32, 27, mode, 0) == 0
    for c in (16, 96, 112, 224):
        assert lib.mm3d_bnrelu_workspace_bytes_ex(c, 0) == lib.mm3d_bnrelu_workspace_bytes(c)


def test_deterministic_wgrad_query_is_bounded_and_row_independent():
    lib, det = _lib.lib, _lib.DETERMINISTIC
    bound = _sm_count() * 256 * 1024 + 256
    for mode in (_lib.MODE_TF32, _lib.MODE_TF32X3, _lib.MODE_BF16):
        for ci, co, K in ((16, 16, 27), (32, 16, 27), (64, 32, 8), (96, 48, 27), (160, 80, 27), (192, 96, 8),
                          (256, 256, 27)):
            sizes = {lib.mm3d_conv_wgrad_workspace_bytes(n, ci, co, K, mode, det) for n in (0, 1000, 2_000_000)}
            assert len(sizes) == 1
            (b,) = sizes
            assert 256 + _sm_count() * ci * co * 4 <= b <= bound, (mode, ci, co, K, b)
        # the SIMT kernel's shapes (an unpadded 3-channel stem) have no deterministic form
        assert lib.mm3d_conv_wgrad_workspace_bytes(1000, 3, 16, 27, mode, det) == 0
    assert lib.mm3d_conv_wgrad_workspace_bytes(1000, 64, 32, 27, _lib.MODE_FP32, det) == 0


def test_deterministic_bnrelu_query_covers_a_row_per_cta():
    lib, det = _lib.lib, _lib.DETERMINISTIC
    for c in (16, 96, 224):
        b = lib.mm3d_bnrelu_workspace_bytes_ex(c, det)
        assert b >= _sm_count() * 2 * c * 8 + 2 * 2 * c * 8
