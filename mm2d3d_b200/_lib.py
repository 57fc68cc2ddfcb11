"""ctypes binding of ``libmm3d.so`` (the C ABI declared in ``include/mm3d.h``).

There is no CPU fallback: if the library has not been built (``python -m mm2d3d_b200.build``)
importing this module raises, and every op raises on a non-zero return code.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmm3d.so")

ABI_VERSION = 8


class UnetMask(C.Structure):
    """``mm3d_unet_mask`` of ``include/mm3d.h``."""
    _fields_ = [("wb", C.c_void_p), ("s", C.c_void_p), ("feats", C.c_void_p), ("d_wb", C.c_void_p),
                ("ws", C.c_void_p), ("ws_bytes", C.c_size_t)]


class UnetGroups(C.Structure):
    """``mm3d_unet_groups`` of ``include/mm3d.h``."""
    _fields_ = [("groups", C.c_int), ("bounds", C.c_void_p)]


LEVEL_DESC_WORDS = 10
BN_MAX_GROUPS = 8        # MM3D_BN_MAX_GROUPS: batch groups of one grouped call
MAX_GROUP_LEVELS = 16    # MM3D_MAX_GROUP_LEVELS

MODE_FP32, MODE_TF32, MODE_BF16, MODE_TF32X3 = 0, 1, 2, 3
MODES = {"fp32": MODE_FP32, "tf32": MODE_TF32, "bf16": MODE_BF16, "tf32x3": MODE_TF32X3}
CONV_TRANSPOSE_W, CONV_MIRROR_K = 1, 2
DETERMINISTIC = 0x100  # MM3D_DETERMINISTIC: the flags bit of the *_ex entry points
DET_CTAS = 592         # MM3D_DET_CTAS: partial slots of a deterministic reduction
STATUS_BAD_COORD = 1
STATUS_DROPPED = 2

if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} is missing: build it with `python -m mm2d3d_b200.build` "
        "(nvcc, sm_100a). mm2d3d_b200 has no CPU fallback."
    )

lib = C.CDLL(LIB_PATH)

_p, _i, _i64, _sz, _f = C.c_void_p, C.c_int, C.c_int64, C.c_size_t, C.c_float

# name: (restype, argtypes) -- mirrors include/mm3d.h one to one
SIGNATURES = {
    "mm3d_abi_version": (_i, []),
    "mm3d_last_error": (C.c_char_p, []),
    "mm3d_device_supports_tc": (_i, []),
    "mm3d_kernel_launches": (C.c_longlong, []),
    "mm3d_take_device_error": (_i, []),
    "mm3d_hash_capacity": (_i64, [_i64]),
    "mm3d_unique_workspace_bytes": (_sz, [_i64]),
    "mm3d_voxelize": (_i, [_p, _i64, _i, _p, _p, _i64, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "mm3d_coarsen": (_i, [_p, _p, _i64, _p, _p, _i64, _p, _p, _p, _p, _i64, _p, _p, _sz, _p]),
    "mm3d_build_nbr27": (_i, [_p, _p, _i64, _i, _p, _p, _i64, _p, _i64, _p]),
    "mm3d_scale_points_workspace_bytes": (_sz, [_i]),
    "mm3d_scale_points": (_i, [_p, _p, _i, _i64, _p, _f, _i, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "mm3d_voxelize_points_workspace_bytes": (_sz, [_i64, _i]),
    "mm3d_voxelize_points": (_i, [_p, _p, _i, _i64, _p, _f, _i, _p, _p, _p, _p, _p, _p, _i64, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "mm3d_input_fwd": (_i, [_p, _p, _p, _i64, _i64, _i, _i, _p, _p]),
    "mm3d_input_bwd": (_i, [_p, _p, _p, _i64, _i, _i, _p, _p]),
    "mm3d_output_fwd": (_i, [_p, _p, _i64, _i, _p, _p]),
    "mm3d_output_bwd": (_i, [_p, _p, _i64, _i64, _i, _p, _p]),
    "mm3d_conv_workspace_bytes": (_sz, [_i64, _i64, _i, _i, _i, _i]),
    "mm3d_plan_bytes": (_sz, [_i64, _i]),
    "mm3d_build_plan": (_i, [_p, _i64, _p, _p, _i64, _i, _p, _sz, _p]),
    "mm3d_build_plans": (_i, [_p, _i, _p]),
    "mm3d_conv_fwd": (_i, [_p, _i64, _i, _p, _i64, _i, _p, _i, _p, _i64, _p, _p, _i64, _i, _i, _p, _sz, _p]),
    "mm3d_round_tf32": (_i, [_p, _p, _i64, _p]),
    "mm3d_split_tf32": (_i, [_p, _p, _i64, _p]),
    "mm3d_split_bf16": (_i, [_p, _p, _i64, _p]),
    "mm3d_conv_wgrad": (_i, [_p, _i64, _i, _p, _i64, _i, _p, _i, _p, _i64, _p, _p, _i64, _i, _i, _p, _sz, _p]),
    "mm3d_conv_wgrad_workspace_bytes": (_sz, [_i64, _i, _i, _i, _i, _i]),
    "mm3d_conv_wgrad_ex": (_i, [_p, _i64, _i, _p, _i64, _i, _p, _i, _p, _i64, _p, _p, _i64, _i, _i, _p, _sz, _p, _i]),
    "mm3d_bnrelu_workspace_bytes": (_sz, [_i]),
    "mm3d_bnrelu_fwd": (_i, [_p, _p, _i64, _i, _p, _p, _p, _p, _p, _p, _f, _f, _f, _i, _p, _sz, _p]),
    "mm3d_bnrelu_bwd": (_i, [_p, _p, _p, _i64, _i, _p, _p, _p, _p, _p, _p, _f, _i, _p, _sz, _p]),
    "mm3d_bnrelu_workspace_bytes_ex": (_sz, [_i, _i]),
    "mm3d_bnrelu_fwd_ex": (_i, [_p, _p, _i64, _i, _p, _p, _p, _p, _p, _p, _f, _f, _f, _i, _p, _sz, _p, _i]),
    "mm3d_bnrelu_bwd_ex": (_i, [_p, _p, _p, _i64, _i, _p, _p, _p, _p, _p, _p, _f, _i, _p, _sz, _p, _i]),
    "mm3d_lift2d_fwd": (_i, [_p, _i, _i, _i, _i, _i, _i64, _i64, _i64, _i64, _p, _p, _i64, _p, _p]),
    "mm3d_lift2d_bwd": (_i, [_p, _i, _i, _i, _i, _i, _i64, _i64, _i64, _i64, _p, _p, _i64, _p, _p]),
    "mm3d_lift2d_bilinear_fwd": (_i, [_p, _i, _i, _i, _i, _i, _i64, _i64, _i64, _i64, _p, _p, _i64, _p, _p]),
    "mm3d_lift2d_bilinear_bwd": (_i, [_p, _i, _i, _i, _i, _i, _i64, _i64, _i64, _i64, _p, _p, _i64, _p, _p]),
    "mm3d_raster2d_workspace_bytes": (_sz, [_i, _i, _i]),
    "mm3d_raster2d": (_i, [_p, _p, _i, _i, _i, _i64, _p, _f, _p, _p, _sz, _p]),
    "mm3d_rgb_mask_fwd": (_i, [_p, _i64, _i, _p, _p, _p, _p, _p]),
    "mm3d_rgb_mask_bwd": (_i, [_p, _p, _p, _i64, _i, _p, _p, _p, _p, _p, _sz, _p]),
    "mm3d_kl_logits_fwd": (_i, [_p, _p, _i64, _i, _p, _p, _sz, _p]),
    "mm3d_kl_logits_bwd": (_i, [_p, _p, _i64, _i, _p, _p, _p]),
    "mm3d_heads3d_fwd": (_i, [_p, _i64, _i, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "mm3d_heads3d_bwd": (_i, [_p, _i64, _i, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "mm3d_unet_topo_num_params": (_i64, [_i, _i, _i]),
    "mm3d_unet_topo_act_bytes": (_sz, [_i, _i, _i, _i, _i, _i, _p, _i64]),
    "mm3d_unet_topo_bwd_bytes": (_sz, [_i, _i, _i, _i, _i, _i, _p, _i64]),
    "mm3d_unet_topo_scratch_bytes": (_sz, [_i, _i, _i, _i, _i, _i]),
    "mm3d_unet_topo_forward": (_i, [_i, _i, _i, _i, _i, _i, _i, _f, _f, _p, _i64, _p, _p, _p, _p, _p, _p, _sz, _p, _sz, _p, _p]),
    "mm3d_unet_topo_backward": (_i, [_i, _i, _i, _i, _i, _i, _i, _p, _i64, _p, _p, _p, _p, _p, _p, _p, _sz, _p, _sz, _p, _sz, _p, _p]),
    "mm3d_unet_num_params": (_i64, [_i]),
    "mm3d_unet_act_bytes": (_sz, [_i, _i, _i, _i, _p, _i64]),
    "mm3d_unet_bwd_bytes": (_sz, [_i, _i, _i, _i, _p, _i64]),
    "mm3d_unet_scratch_bytes": (_sz, [_i, _i, _i, _i]),
    "mm3d_unet_forward": (_i, [_i, _i, _i, _i, _i, _f, _f, _p, _i64, _p, _p, _p, _p, _p, _p, _sz, _p, _sz, _p, _p]),
    "mm3d_unet_backward": (_i, [_i, _i, _i, _i, _i, _p, _i64, _p, _p, _p, _p, _p, _p, _p, _sz, _p, _sz, _p, _sz, _p, _p]),
    "mm3d_input_masked_fwd": (_i, [_p, _p, _p, _i64, _i64, _i, _i, _p, _p, _p, _p]),
    "mm3d_input_masked_bwd": (_i, [_p, _p, _p, _p, _p, _i64, _i, _i, _p, _p, _p, _p, _sz, _p]),
    "mm3d_point_csr_workspace_bytes": (_sz, [_i64]),
    "mm3d_point_csr": (_i, [_p, _p, _i64, _i64, _p, _p, _p, _sz, _p]),
    "mm3d_input_fwd_csr": (_i, [_p, _p, _p, _i64, _i, _i, _p, _p]),
    "mm3d_output_bwd_csr": (_i, [_p, _p, _p, _i64, _i, _p, _p]),
    "mm3d_lift_csr_workspace_bytes": (_sz, [_i, _i, _i, _i64, _i]),
    "mm3d_lift_csr": (_i, [_p, _p, _p, _i, _i, _i, _i64, _p, _p, _p, _sz, _p]),
    "mm3d_lift2d_bwd_csr": (_i, [_p, _i, _i, _i, _i, _i, _i64, _i64, _i64, _i64, _p, _p, _p, _p]),
    "mm3d_lift2d_bilinear_bwd_csr": (_i, [_p, _i, _i, _i, _i, _i, _i64, _i64, _i64, _i64, _p, _p, _p, _p, _p]),
    "mm3d_rgb_mask_bwd_ex": (_i, [_p, _p, _p, _i64, _i, _p, _p, _p, _p, _p, _sz, _p, _i]),
    "mm3d_kl_logits_fwd_ex": (_i, [_p, _p, _i64, _i, _p, _p, _sz, _p, _i]),
    "mm3d_heads3d_fwd_ex": (_i, [_p, _i64, _i, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p, _sz, _p, _i]),
    "mm3d_heads3d_bwd_ex": (_i, [_p, _i64, _i, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _sz, _p, _i]),
    "mm3d_input_masked_fwd_csr": (_i, [_p, _p, _p, _i64, _i, _i, _p, _p, _p, _p]),
    "mm3d_input_masked_bwd_ex": (_i, [_p, _p, _p, _p, _p, _i64, _i, _i, _p, _p, _p, _p, _sz, _p, _i]),
    "mm3d_unet_topo_scratch_bytes_ex": (_sz, [_i, _i, _i, _i, _i, _i, _i]),
    "mm3d_unet_topo_forward_ex": (_i, [_i, _i, _i, _i, _i, _i, _i, _f, _f, _p, _i64, _p, _p, _p, _p, _p, _p, _p, _p, _sz, _p, _sz,
                                       _p, _p, _i]),
    "mm3d_unet_topo_backward_ex": (_i, [_i, _i, _i, _i, _i, _i, _i, _p, _i64, _p, _p, _p, _p, _p, _p, _p, _p, _p, _sz, _p, _sz,
                                        _p, _sz, _p, _p, _i]),
    "mm3d_unet_topo_infer_bytes": (_sz, [_i, _i, _i, _i, _i, _i, _p, _i64, _i]),
    "mm3d_unet_topo_infer": (_i, [_i, _i, _i, _i, _i, _i, _f, _p, _i64, _p, _p, _p, _p, _p, _p, _p, _p, _sz, _p, _p, _i]),
    "mm3d_group_bounds": (_i, [_p, _p, _i, _p, _i, _p, _p]),
    "mm3d_bnrelu_workspace_bytes_grouped": (_sz, [_i, _i, _i]),
    "mm3d_bnrelu_fwd_grouped": (_i, [_p, _p, _i64, _i, _p, _p, _p, _p, _p, _p, _f, _f, _f, _i, _p, _sz, _p, _i, _i, _p]),
    "mm3d_bnrelu_bwd_grouped": (_i, [_p, _p, _p, _i64, _i, _p, _p, _p, _p, _p, _p, _f, _i, _p, _sz, _p, _i, _i, _p]),
    "mm3d_unet_topo_act_bytes_grouped": (_sz, [_i, _i, _i, _i, _i, _i, _p, _i64, _i]),
    "mm3d_unet_topo_scratch_bytes_grouped": (_sz, [_i, _i, _i, _i, _i, _i, _i, _i]),
    "mm3d_unet_topo_forward_grouped": (_i, [_i, _i, _i, _i, _i, _i, _i, _f, _f, _p, _i64, _p, _p, _p, _p, _p, _p, _p, _p, _sz, _p,
                                            _sz, _p, _p, _i, _p]),
    "mm3d_unet_topo_backward_grouped": (_i, [_i, _i, _i, _i, _i, _i, _i, _p, _i64, _p, _p, _p, _p, _p, _p, _p, _p, _p, _sz, _p,
                                             _sz, _p, _sz, _p, _p, _i, _p]),
}

class PlanDesc(C.Structure):
    """``mm3d_plan_desc`` of include/mm3d.h."""
    _fields_ = [("tbl", _p), ("tbl_stride", _i64), ("onehot_off", _p), ("n_dev", _p), ("n_cap", _i64),
                ("n_rows_hint", _i64), ("K", _i), ("plan", _p), ("plan_bytes", _sz)]


for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)  # AttributeError here = library / header mismatch
    _fn.restype = _res
    _fn.argtypes = _args

if lib.mm3d_abi_version() != ABI_VERSION:
    raise ImportError(f"libmm3d ABI {lib.mm3d_abi_version()} != expected {ABI_VERSION}; rebuild the library")


class Mm3dError(RuntimeError):
    pass


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib.mm3d_last_error().decode("utf-8", "replace")
        raise Mm3dError(f"{what or 'libmm3d'} failed (code {rc}): {msg}")


def raise_device_errors(where: str = "") -> None:
    """Poll the sticky device-error bits (mapped host memory: no synchronisation, no CUDA call) and raise."""
    bits = lib.mm3d_take_device_error()
    if bits > 0:
        what = []
        if bits & 1:
            what.append("a kernel's internal pipeline or grid barrier timed out (results of that launch are garbage)")
        if bits & 2:
            what.append("lift2d met a pixel index outside the feature map")
        raise Mm3dError(f"{where or 'libmm3d'}: device-side error reported: " + "; ".join(what))


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


def stream_ptr():
    import torch

    return torch.cuda.current_stream().cuda_stream
