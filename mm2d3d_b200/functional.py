"""``torch.autograd.Function`` wrappers around the C ABI: PyTorch carries tensors and the autograd
graph, every arithmetic step is a ``libmm3d`` kernel launch on the current CUDA stream.

All Functions run in float32 whatever autocast says -- SparseConvNet's ops are float-only and the
reference's 3D branch therefore runs in FP32 under AMP (SURVEY.md 3.3 / A.11).  The convolution
arithmetic mode (``fp32`` SIMT parity mode, ``tf32`` / ``bf16`` tcgen05 modes) is a per-call
argument, defaulting to the module-level :data:`DEFAULT_MODE`.
"""
from __future__ import annotations

import ctypes as C
import warnings

import torch
from torch.amp import custom_bwd, custom_fwd

from . import _lib
from ._lib import MODES, check, lib, ptr

DEFAULT_MODE = "fp32"

# Deterministic mode (scn.set_deterministic): None follows torch.are_deterministic_algorithms_enabled()
DETERMINISTIC = None


def deterministic() -> bool:
    """Whether the ops called now take their deterministic (fixed summation order) forms."""
    return torch.are_deterministic_algorithms_enabled() if DETERMINISTIC is None else bool(DETERMINISTIC)


def alert_not_deterministic(what: str) -> None:
    """Called by an op that has no deterministic form yet while the mode is on: a UserWarning that its result can
    still differ between runs (Python shows it once per call site)."""
    warnings.warn(f"mm2d3d_b200: {what} has no deterministic form yet -- its result can differ in the last bits "
                  "between runs although the deterministic mode is on (see INTEGRATION.md, Deterministic mode)",
                  UserWarning, stacklevel=3)

_scratch: dict = {}


def scratch(nbytes: int, device) -> torch.Tensor:
    """Grow-only per-device scratch buffer.  Ops are stream-ordered, so consecutive ops on one
    stream can share it; do not run ops of this package concurrently on several streams."""
    key = (device.type, device.index)
    buf = _scratch.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(int(nbytes), 1 << 20), dtype=torch.uint8, device=device)
        _scratch[key] = buf
    return buf


def _f32c(t):
    return t.contiguous() if t.dtype == torch.float32 else t.float().contiguous()


def _require_cuda(t, what):
    if not t.is_cuda:
        raise RuntimeError(f"{what}: expected a CUDA tensor -- mm2d3d_b200 has no CPU path")


# ----------------------------------------------------------------------------- I/O layers
class InputLayerFn(torch.autograd.Function):
    @staticmethod
    @custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, feats, meta, mode):
        _require_cuda(feats, "InputLayer")
        feats = _f32c(feats)
        n, c = meta.n_points, feats.shape[1]
        if feats.shape[0] < n:
            raise ValueError("InputLayer: fewer feature rows than coordinates")
        out = torch.empty(meta.n_voxels, c, dtype=torch.float32, device=feats.device)
        with torch.cuda.device(feats.device):
            if deterministic():
                start, pts = meta.point_csr()
                check(lib.mm3d_input_fwd_csr(ptr(feats), ptr(start), ptr(pts), meta.n_voxels, c, mode, ptr(out),
                                             _lib.stream_ptr()), "mm3d_input_fwd_csr")
            else:
                check(lib.mm3d_input_fwd(ptr(feats), meta.p2v_ptr, meta.npts_ptr, n, meta.n_voxels, c, mode, ptr(out),
                                         _lib.stream_ptr()), "mm3d_input_fwd")
        ctx.meta, ctx.mode, ctx.rows = meta, mode, feats.shape[0]
        return out

    @staticmethod
    @custom_bwd(device_type="cuda")
    def backward(ctx, d_out):
        meta = ctx.meta
        d_out = _f32c(d_out)
        c = d_out.shape[1]
        alloc = torch.zeros if ctx.rows > meta.n_points else torch.empty
        d_feats = alloc(ctx.rows, c, dtype=torch.float32, device=d_out.device)
        with torch.cuda.device(d_out.device):
            check(lib.mm3d_input_bwd(ptr(d_out), meta.p2v_ptr, meta.npts_ptr, meta.n_points, c, ctx.mode,
                                     ptr(d_feats), _lib.stream_ptr()), "mm3d_input_bwd")
        return d_feats, None, None


class OutputLayerFn(torch.autograd.Function):
    @staticmethod
    @custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, vox, meta):
        _require_cuda(vox, "OutputLayer")
        vox = _f32c(vox)
        c = vox.shape[1]
        out = torch.empty(meta.n_points, c, dtype=torch.float32, device=vox.device)
        with torch.cuda.device(vox.device):
            check(lib.mm3d_output_fwd(ptr(vox), meta.p2v_ptr, meta.n_points, c, ptr(out), _lib.stream_ptr()),
                  "mm3d_output_fwd")
        ctx.meta, ctx.det = meta, deterministic()
        return out

    @staticmethod
    @custom_bwd(device_type="cuda")
    def backward(ctx, d_out):
        meta = ctx.meta
        d_out = _f32c(d_out)
        c = d_out.shape[1]
        d_vox = torch.empty(meta.n_voxels, c, dtype=torch.float32, device=d_out.device)
        with torch.cuda.device(d_out.device):
            if ctx.det:
                start, pts = meta.point_csr()
                check(lib.mm3d_output_bwd_csr(ptr(d_out), ptr(start), ptr(pts), meta.n_voxels, c, ptr(d_vox),
                                              _lib.stream_ptr()), "mm3d_output_bwd_csr")
            else:
                check(lib.mm3d_output_bwd(ptr(d_out), meta.p2v_ptr, meta.n_points, meta.n_voxels, c, ptr(d_vox),
                                          _lib.stream_ptr()), "mm3d_output_bwd")
        return d_vox, None


# ----------------------------------------------------------------------------- convolutions
class _Table:
    """Rule table of one convolution direction, in C-ABI terms."""
    __slots__ = ("tbl", "stride", "onehot", "n_in", "n_out", "K", "plan", "plan_cap")

    def __init__(self, tbl, stride, onehot, n_in, n_out, K, plan=(None, 0)):
        self.tbl, self.stride, self.onehot, self.n_in, self.n_out, self.K = tbl, stride, onehot, n_in, n_out, K
        self.plan, self.plan_cap = plan


def conv_tables(meta, kind: str, spatial_in: int, plans: bool = False):
    """(forward table, dgrad table, dgrad flags) of a layer applied at ``spatial_in``; with ``plans`` the
    tables carry their row plans (tensor-core modes).

    smc : out rows = in rows, table = 3^3 neighbours; dgrad = same table, W^T with mirrored offsets.
    down: out rows = coarse, table = children [8];   dgrad = one-hot (parent, off) over fine rows, W^T.
    up  : out rows = fine, one-hot (parent, off);     dgrad = children table over coarse rows, W^T.
    """
    if kind == "smc":
        lv = meta.nbr(spatial_in)
        t = _Table(lv.ptr(lv.o_nbr), lv.tstride, None, lv.n, lv.n, 27,
                   meta.plan("smc", spatial_in) if plans else (None, 0))
        return t, t, _lib.CONV_TRANSPOSE_W | _lib.CONV_MIRROR_K
    if kind == "down":
        s_fine = int(spatial_in)
    elif kind == "up":
        s_fine = int(spatial_in) * 2
    else:
        raise ValueError(kind)
    fine, coarse = meta.down(s_fine)
    child = _Table(fine.ptr(fine.o_child), fine.tstride, None, fine.n, coarse.n, 8,
                   meta.plan("down", s_fine) if plans else (None, 0))
    onehot = _Table(fine.ptr(fine.o_parent), 0, fine.ptr(fine.o_off), coarse.n, fine.n, 8,
                    meta.plan("up", s_fine) if plans else (None, 0))
    return (child, onehot, _lib.CONV_TRANSPOSE_W) if kind == "down" else (onehot, child, _lib.CONV_TRANSPOSE_W)


def _tf32(t: torch.Tensor, inplace: bool = False) -> torch.Tensor:
    """RNA-round a contiguous float32 tensor to TF32 (operands of the tensor-core convolutions: the MMA itself would
    truncate).  The whole-network executor's producers store rounded values themselves; this is the module path."""
    out = t if inplace else torch.empty_like(t)
    if t.numel():
        with torch.cuda.device(t.device):
            check(lib.mm3d_round_tf32(ptr(t), ptr(out), t.numel(), _lib.stream_ptr()), "mm3d_round_tf32")
    return out


def _planes(t: torch.Tensor, bf16: bool = False) -> torch.Tensor:
    """[2, n, c]: hi = tf32(t) and lo = tf32(t - hi), the operand planes of the error-compensated "tf32x3" mode.
    ``bf16``: the planes of the "bf16" mode instead -- tf32(t) as float32, then bf16(t) (n * c bfloat16 values at the
    start of the second plane)."""
    t = t.contiguous()
    out = torch.empty((2,) + tuple(t.shape), dtype=torch.float32, device=t.device)
    if t.numel():
        with torch.cuda.device(t.device):
            if bf16:
                check(lib.mm3d_split_bf16(ptr(t), ptr(out), t.numel(), _lib.stream_ptr()), "mm3d_split_bf16")
            else:
                check(lib.mm3d_split_tf32(ptr(t), ptr(out), t.numel(), _lib.stream_ptr()), "mm3d_split_tf32")
    return out


class TableConvFn(torch.autograd.Function):
    @staticmethod
    @custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, x, weight, meta, kind, spatial_in, mode):
        _require_cuda(x, "convolution")
        x, w = _f32c(x), _f32c(weight)
        K, c_in, c_out = w.shape[0], w.shape[-2], w.shape[-1]
        m = MODES[mode]
        if m in (_lib.MODE_TF32X3, _lib.MODE_BF16) and c_out % 16:
            m = _lib.MODE_FP32  # (dgrad / wgrad of such a layer have no tensor-core path; no layer of the network is one)
        fwd_t, bwd_t, bwd_flags = conv_tables(meta, kind, spatial_in, plans=m != _lib.MODE_FP32)
        if x.shape[0] != fwd_t.n_in or x.shape[1] != c_in or K != fwd_t.K:
            raise ValueError(f"{kind} convolution: input {tuple(x.shape)} / weight {tuple(w.shape)} do not match "
                             f"the active set ({fwd_t.n_in} rows, {fwd_t.K} offsets)")
        # tensor-core modes gather rows in 64-byte pieces: pad an odd channel count (the 3-channel
        # stem) with zero channels instead of using the SIMT kernels
        pad = 0
        if m != _lib.MODE_FP32:
            pad = (-c_in) % 16
        if pad:
            x = torch.nn.functional.pad(x, (0, pad))
            w = torch.nn.functional.pad(w, (0, 0, 0, pad))
            c_in += pad
        ctx.pad = pad
        if m in (_lib.MODE_TF32X3, _lib.MODE_BF16):
            x = _planes(x, m == _lib.MODE_BF16)  # two planes (saved: wgrad reads the same operand)
        elif m != _lib.MODE_FP32:
            x = _tf32(x, inplace=bool(pad))  # (the saved x is the rounded one: wgrad reads the same operand)
        out = torch.empty(fwd_t.n_out, c_out, dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):
            wsb = lib.mm3d_conv_workspace_bytes(fwd_t.n_in, fwd_t.n_out, c_in, c_out, K, m)
            ws = scratch(wsb, x.device)
            check(lib.mm3d_conv_fwd(ptr(x), fwd_t.n_in, c_in, ptr(out), fwd_t.n_out, c_out, ptr(w), K, fwd_t.tbl,
                                    fwd_t.stride, fwd_t.onehot, fwd_t.plan, fwd_t.plan_cap, 0, m, ptr(ws), ws.numel(),
                                    _lib.stream_ptr()), "mm3d_conv_fwd")
        ctx.save_for_backward(x, w)
        ctx.meta, ctx.tables, ctx.mode, ctx.wshape = meta, (fwd_t, bwd_t, bwd_flags), m, weight.shape
        ctx.det = deterministic()
        return out

    @staticmethod
    @custom_bwd(device_type="cuda")
    def backward(ctx, d_out):
        x, w = ctx.saved_tensors
        fwd_t, bwd_t, bwd_flags = ctx.tables
        d_out = _f32c(d_out)
        K, c_in, c_out = w.shape[0], w.shape[-2], w.shape[-1]
        m = ctx.mode
        if m in (_lib.MODE_TF32X3, _lib.MODE_BF16):
            d_out = _planes(d_out, m == _lib.MODE_BF16)
        elif m != _lib.MODE_FP32:
            d_out = _tf32(d_out)
        d_x = d_w = None
        with torch.cuda.device(x.device):
            stream = _lib.stream_ptr()
            wsb = lib.mm3d_conv_workspace_bytes(bwd_t.n_in, bwd_t.n_out, c_out, c_in, K, m)
            ws = scratch(wsb, x.device)
            if ctx.needs_input_grad[0]:
                d_x = torch.empty(bwd_t.n_out, c_in, dtype=torch.float32, device=x.device)
                check(lib.mm3d_conv_fwd(ptr(d_out), bwd_t.n_in, c_out, ptr(d_x), bwd_t.n_out, c_in, ptr(w), K,
                                        bwd_t.tbl, bwd_t.stride, bwd_t.onehot, bwd_t.plan, bwd_t.plan_cap, bwd_flags, m,
                                        ptr(ws), ws.numel(), stream), "mm3d_conv_fwd(dgrad)")
            if ctx.needs_input_grad[1]:
                d_w = torch.empty(w.shape, dtype=torch.float32, device=x.device)
                # deterministic form: per-CTA slabs summed in CTA order (0 bytes = none: the fp32 mode's SIMT kernel)
                det_wsb = (lib.mm3d_conv_wgrad_workspace_bytes(fwd_t.n_out, c_in, c_out, K, m, _lib.DETERMINISTIC)
                           if ctx.det else 0)
                if ctx.det and not det_wsb:
                    alert_not_deterministic("the sparse-convolution weight gradient in the fp32 mode")
                if det_wsb:
                    ws = scratch(max(wsb, det_wsb), x.device)
                    check(lib.mm3d_conv_wgrad_ex(ptr(x), fwd_t.n_in, c_in, ptr(d_out), fwd_t.n_out, c_out, ptr(d_w), K,
                                                 fwd_t.tbl, fwd_t.stride, fwd_t.onehot, fwd_t.plan, fwd_t.plan_cap, 0, m,
                                                 ptr(ws), ws.numel(), stream, _lib.DETERMINISTIC), "mm3d_conv_wgrad_ex")
                else:
                    check(lib.mm3d_conv_wgrad(ptr(x), fwd_t.n_in, c_in, ptr(d_out), fwd_t.n_out, c_out, ptr(d_w), K,
                                              fwd_t.tbl, fwd_t.stride, fwd_t.onehot, fwd_t.plan, fwd_t.plan_cap, 0, m, ptr(ws),
                                              ws.numel(), stream), "mm3d_conv_wgrad")
        if ctx.pad:
            d_x = d_x[:, :c_in - ctx.pad] if d_x is not None else None
            d_w = d_w[..., :c_in - ctx.pad, :] if d_w is not None else None
        return d_x, d_w, None, None, None, None


# ----------------------------------------------------------------------------- BN + ReLU
class BatchNormReLUFn(torch.autograd.Function):
    @staticmethod
    @custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, x, gamma, beta, running_mean, running_var, eps, momentum, leakiness, training, bounds=None):
        """``bounds``: the row boundaries of batch groups (``Metadata.group_bounds``), each normalised with its own
        statistics in training mode (``mm3d_bnrelu_fwd_grouped``); ``None`` = one group."""
        _require_cuda(x, "BatchNormReLU")
        x = _f32c(x)
        n, c = x.shape
        y = torch.empty_like(x)
        grouped = bounds is not None and len(bounds) > 2 and training
        G = len(bounds) - 1 if grouped else 1
        save = torch.empty(2, G, c, dtype=torch.float32, device=x.device)
        # deterministic: every reduction over rows (the training forward's statistics, and every backward: d_gamma /
        # d_beta are row sums in eval mode too) in its fixed-order form
        det = deterministic()
        with torch.cuda.device(x.device):
            if grouped:
                flags = _lib.DETERMINISTIC if det else 0
                b = (C.c_int64 * (G + 1))(*bounds)
                ws = scratch(lib.mm3d_bnrelu_workspace_bytes_grouped(c, G, flags), x.device)
                check(lib.mm3d_bnrelu_fwd_grouped(ptr(x), ptr(y), n, c, ptr(gamma), ptr(beta), ptr(running_mean),
                                                  ptr(running_var), ptr(save[0]), ptr(save[1]), eps, momentum, leakiness, 1,
                                                  ptr(ws), ws.numel(), _lib.stream_ptr(), flags, G, b),
                      "mm3d_bnrelu_fwd_grouped")
            elif det and training:
                ws = scratch(lib.mm3d_bnrelu_workspace_bytes_ex(c, _lib.DETERMINISTIC), x.device)
                check(lib.mm3d_bnrelu_fwd_ex(ptr(x), ptr(y), n, c, ptr(gamma), ptr(beta), ptr(running_mean),
                                             ptr(running_var), ptr(save[0]), ptr(save[1]), eps, momentum, leakiness, 1,
                                             ptr(ws), ws.numel(), _lib.stream_ptr(), _lib.DETERMINISTIC), "mm3d_bnrelu_fwd_ex")
            else:
                wsb = lib.mm3d_bnrelu_workspace_bytes(c)
                ws = scratch(wsb, x.device)
                check(lib.mm3d_bnrelu_fwd(ptr(x), ptr(y), n, c, ptr(gamma), ptr(beta), ptr(running_mean), ptr(running_var),
                                          ptr(save[0]), ptr(save[1]), eps, momentum, leakiness, int(training), ptr(ws),
                                          ws.numel(), _lib.stream_ptr()), "mm3d_bnrelu_fwd")
        ctx.save_for_backward(x, gamma, beta, save)
        ctx.leak, ctx.training, ctx.det = leakiness, bool(training), det
        ctx.bounds = tuple(bounds) if grouped else None
        return y

    @staticmethod
    @custom_bwd(device_type="cuda")
    def backward(ctx, dy):
        x, gamma, beta, save = ctx.saved_tensors
        dy = _f32c(dy)
        n, c = x.shape
        dx = torch.empty_like(x)
        dgb = torch.empty(2, c, dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):
            if ctx.bounds is not None:
                G = len(ctx.bounds) - 1
                flags = _lib.DETERMINISTIC if ctx.det else 0
                b = (C.c_int64 * (G + 1))(*ctx.bounds)
                ws = scratch(lib.mm3d_bnrelu_workspace_bytes_grouped(c, G, flags), x.device)
                check(lib.mm3d_bnrelu_bwd_grouped(ptr(x), ptr(dy), ptr(dx), n, c, ptr(gamma), ptr(beta), ptr(save[0]),
                                                  ptr(save[1]), ptr(dgb[0]), ptr(dgb[1]), ctx.leak, int(ctx.training),
                                                  ptr(ws), ws.numel(), _lib.stream_ptr(), flags, G, b),
                      "mm3d_bnrelu_bwd_grouped")
            elif ctx.det:
                ws = scratch(lib.mm3d_bnrelu_workspace_bytes_ex(c, _lib.DETERMINISTIC), x.device)
                check(lib.mm3d_bnrelu_bwd_ex(ptr(x), ptr(dy), ptr(dx), n, c, ptr(gamma), ptr(beta), ptr(save[0]),
                                             ptr(save[1]), ptr(dgb[0]), ptr(dgb[1]), ctx.leak, int(ctx.training), ptr(ws),
                                             ws.numel(), _lib.stream_ptr(), _lib.DETERMINISTIC), "mm3d_bnrelu_bwd_ex")
            else:
                wsb = lib.mm3d_bnrelu_workspace_bytes(c)
                ws = scratch(wsb, x.device)
                check(lib.mm3d_bnrelu_bwd(ptr(x), ptr(dy), ptr(dx), n, c, ptr(gamma), ptr(beta), ptr(save[0]), ptr(save[1]),
                                          ptr(dgb[0]), ptr(dgb[1]), ctx.leak, int(ctx.training), ptr(ws), ws.numel(),
                                          _lib.stream_ptr()), "mm3d_bnrelu_bwd")
        return dx, dgb[0], dgb[1], None, None, None, None, None, None, None


# ----------------------------------------------------------------------------- 2D -> 3D lift
_LIFT_DTYPES = {torch.float32: 0, torch.float16: 1, torch.bfloat16: 2}


def lift_csr(idx, uv, offsets, B, H, W):
    """(pix_start int32 [B H W + 1], pix_ent int32 [n or 4 n]): the lift's entries grouped by pixel in ascending
    order (``mm3d_lift_csr``), on the current stream.  ``idx`` int64 [n, 2] or, for the bilinear lift, ``uv``."""
    t = idx if idx is not None else uv
    n = int(t.shape[0])
    bil = uv is not None
    start = torch.empty(B * H * W + 1, dtype=torch.int32, device=t.device)
    ent = torch.empty(max((4 if bil else 1) * n, 1), dtype=torch.int32, device=t.device)
    with torch.cuda.device(t.device):
        ws = torch.empty(lib.mm3d_lift_csr_workspace_bytes(B, H, W, n, int(bil)), dtype=torch.uint8, device=t.device)
        check(lib.mm3d_lift_csr(ptr(idx), ptr(uv), ptr(offsets), B, H, W, n, ptr(start), ptr(ent), ptr(ws), ws.numel(),
                                _lib.stream_ptr()), "mm3d_lift_csr")
    return start, ent


def _dense_map(t):
    """The map as it is when its memory is dense in NCHW or channels-last (NHWC) order, else a contiguous copy."""
    if t.is_contiguous() or t.is_contiguous(memory_format=torch.channels_last):
        return t
    return t.contiguous()


class Lift2DFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, fmap, idx, offsets, lists=None):
        """``lists``: an object whose ``pixel_lists(B, H, W)`` caches the pixel lists of ``idx`` (LiftIndices)."""
        _require_cuda(fmap, "lift2d")
        if fmap.dtype not in _LIFT_DTYPES:
            raise TypeError(f"lift2d: unsupported dtype {fmap.dtype}")
        fmap = _dense_map(fmap)  # channels-last maps (cuDNN's layout for the 2D network) are gathered in place
        B, C, H, W = fmap.shape
        n = idx.shape[0]
        out = torch.empty(n, C, dtype=fmap.dtype, device=fmap.device)
        with torch.cuda.device(fmap.device):
            check(lib.mm3d_lift2d_fwd(ptr(fmap), _LIFT_DTYPES[fmap.dtype], B, C, H, W, *fmap.stride(), ptr(idx), ptr(offsets), n,
                                      ptr(out), _lib.stream_ptr()), "mm3d_lift2d_fwd")
        ctx.save_for_backward(idx, offsets)
        ctx.shape = (B, C, H, W)
        ctx.channels_last = not fmap.is_contiguous()
        ctx.lists, ctx.det = lists, deterministic()
        return out

    @staticmethod
    def backward(ctx, d_out):
        idx, offsets = ctx.saved_tensors
        B, C, H, W = ctx.shape
        d_out = d_out.contiguous()
        # the gradient has the map's memory format: the scatter-add then touches one contiguous piece per point
        d_fmap = torch.empty(B, C, H, W, dtype=d_out.dtype, device=d_out.device,
                             memory_format=torch.channels_last if ctx.channels_last else torch.contiguous_format).zero_()
        with torch.cuda.device(d_out.device):
            if ctx.det:
                start, ent = (ctx.lists.pixel_lists(B, H, W) if ctx.lists is not None
                              else lift_csr(idx, None, offsets, B, H, W))
                check(lib.mm3d_lift2d_bwd_csr(ptr(d_out), _LIFT_DTYPES[d_out.dtype], B, C, H, W, *d_fmap.stride(), ptr(start),
                                              ptr(ent), ptr(d_fmap), _lib.stream_ptr()), "mm3d_lift2d_bwd_csr")
            else:
                check(lib.mm3d_lift2d_bwd(ptr(d_out), _LIFT_DTYPES[d_out.dtype], B, C, H, W, *d_fmap.stride(), ptr(idx),
                                          ptr(offsets), idx.shape[0], ptr(d_fmap), _lib.stream_ptr()), "mm3d_lift2d_bwd")
        return d_fmap, None, None, None


class Lift2DBilinearFn(torch.autograd.Function):
    """Bilinear lift (an extension of the reference's integer gather): ``uv`` float32 ``[N, 2]`` = (row, col)."""

    @staticmethod
    def forward(ctx, fmap, uv, offsets):
        _require_cuda(fmap, "lift2d_bilinear")
        if fmap.dtype not in _LIFT_DTYPES:
            raise TypeError(f"lift2d_bilinear: unsupported dtype {fmap.dtype}")
        fmap = _dense_map(fmap)
        B, C, H, W = fmap.shape
        n = uv.shape[0]
        out = torch.empty(n, C, dtype=fmap.dtype, device=fmap.device)
        with torch.cuda.device(fmap.device):
            check(lib.mm3d_lift2d_bilinear_fwd(ptr(fmap), _LIFT_DTYPES[fmap.dtype], B, C, H, W, *fmap.stride(), ptr(uv),
                                               ptr(offsets), n, ptr(out), _lib.stream_ptr()), "mm3d_lift2d_bilinear_fwd")
        ctx.save_for_backward(uv, offsets)
        ctx.shape = (B, C, H, W)
        ctx.channels_last = not fmap.is_contiguous()
        ctx.det = deterministic()
        return out

    @staticmethod
    def backward(ctx, d_out):
        uv, offsets = ctx.saved_tensors
        B, C, H, W = ctx.shape
        d_out = d_out.contiguous()
        d_fmap = torch.empty(B, C, H, W, dtype=d_out.dtype, device=d_out.device,
                             memory_format=torch.channels_last if ctx.channels_last else torch.contiguous_format).zero_()
        with torch.cuda.device(d_out.device):
            if ctx.det:  # (point, tap) lists of this call's coordinates
                start, ent = lift_csr(None, uv, offsets, B, H, W)
                check(lib.mm3d_lift2d_bilinear_bwd_csr(ptr(d_out), _LIFT_DTYPES[d_out.dtype], B, C, H, W, *d_fmap.stride(),
                                                       ptr(uv), ptr(start), ptr(ent), ptr(d_fmap), _lib.stream_ptr()),
                      "mm3d_lift2d_bilinear_bwd_csr")
            else:
                check(lib.mm3d_lift2d_bilinear_bwd(ptr(d_out), _LIFT_DTYPES[d_out.dtype], B, C, H, W, *d_fmap.stride(),
                                                   ptr(uv), ptr(offsets), uv.shape[0], ptr(d_fmap), _lib.stream_ptr()),
                      "mm3d_lift2d_bilinear_bwd")
        return d_fmap, None, None
