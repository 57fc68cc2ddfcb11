"""Point-wise prologue and loss around the 3D network (SURVEY.md 8(f).3), each one kernel per direction.

* :func:`rgb_mask` -- ``Net3DSeg.forward``'s ``feats *= sigmoid(linear_rgb_mask(feats))``
  (``3d_net/model.py:46-48``); takes the ``nn.Linear(C, 1)`` parameters as they are.
* :func:`cross_modal_kl` -- one term of ``TrainModel.cross_modal_loss`` (``train.py:157-184``):
  ``F.kl_div(F.log_softmax(pred, 1), F.softmax(target.detach(), 1), reduction="none").sum(1).mean()``.
* :func:`heads3d` -- the two ``Linear(16, classes)`` heads of ``Net3DSeg`` (``3d_net/model.py:38,49`` and
  ``L2G_classifier_3D.linear_point`` ``:73,85``) and the 3D side of the cross-modal loss in one pass over the features.
"""
from __future__ import annotations

import torch

from . import _lib
from ._lib import check, lib, ptr
from .functional import deterministic


def _det_flags():
    """(flags, partial slots of a reduction's workspace) of the deterministic mode as it is now"""
    return (_lib.DETERMINISTIC, _lib.DET_CTAS) if deterministic() else (0, 1)


def _f32c(t):
    return t.detach().to(torch.float32).contiguous()


class _RgbMaskFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, feats, weight, bias):
        if not feats.is_cuda:
            raise RuntimeError("rgb_mask: CUDA tensors expected (there is no CPU path)")
        x, w, b = _f32c(feats), _f32c(weight).reshape(-1), _f32c(bias).reshape(-1)
        n, c = x.shape
        if w.numel() != c or b.numel() != 1:
            raise ValueError("rgb_mask: weight must be [1, C] and bias [1] (nn.Linear(C, 1))")
        y = torch.empty_like(x)
        s = torch.empty(n, dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):
            check(lib.mm3d_rgb_mask_fwd(ptr(x), n, c, ptr(w), ptr(b), ptr(y), ptr(s), _lib.stream_ptr()), "mm3d_rgb_mask_fwd")
        ctx.save_for_backward(x, s, w)
        ctx.shapes = (weight.shape, bias.shape)
        ctx.det = _det_flags()
        return y

    @staticmethod
    def backward(ctx, dy):
        x, s, w = ctx.saved_tensors
        dy = _f32c(dy)
        n, c = x.shape
        dx = torch.empty_like(x) if ctx.needs_input_grad[0] else None
        dwb = torch.empty(c + 1, dtype=torch.float32, device=x.device)
        flags, slots = ctx.det
        ws = torch.empty((c + 1) * slots, dtype=torch.float64, device=x.device)
        with torch.cuda.device(x.device):
            check(lib.mm3d_rgb_mask_bwd_ex(ptr(x), ptr(s), ptr(dy), n, c, ptr(w), ptr(dx), ptr(dwb), dwb.data_ptr() + 4 * c,
                                           ptr(ws), ws.numel() * 8, _lib.stream_ptr(), flags), "mm3d_rgb_mask_bwd")
        return dx, dwb[:c].reshape(ctx.shapes[0]), dwb[c:].reshape(ctx.shapes[1])


def rgb_mask(feats: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor) -> torch.Tensor:
    """``feats * sigmoid(feats @ weight.T + bias)``; feats ``[N, C]`` (C <= 8), ``weight [1, C]``, ``bias [1]``."""
    return _RgbMaskFn.apply(feats, weight, bias)


class _KlFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pred, target):
        if not pred.is_cuda:
            raise RuntimeError("cross_modal_kl: CUDA tensors expected (there is no CPU path)")
        p, t = _f32c(pred), _f32c(target)
        if p.shape != t.shape or p.dim() != 2 or p.shape[0] == 0:
            raise ValueError("cross_modal_kl: two non-empty [N, C] logit tensors expected")
        n, C = p.shape
        loss = torch.empty((), dtype=torch.float32, device=p.device)
        flags, slots = _det_flags()
        ws = torch.empty(slots, dtype=torch.float64, device=p.device)
        with torch.cuda.device(p.device):
            check(lib.mm3d_kl_logits_fwd_ex(ptr(p), ptr(t), n, C, ptr(loss), ptr(ws), ws.numel() * 8, _lib.stream_ptr(), flags),
                  "mm3d_kl_logits_fwd")
        ctx.save_for_backward(p, t)
        return loss

    @staticmethod
    def backward(ctx, dloss):
        p, t = ctx.saved_tensors
        n, C = p.shape
        d = _f32c(dloss).reshape(1)
        dpred = torch.empty_like(p)
        with torch.cuda.device(p.device):
            check(lib.mm3d_kl_logits_bwd(ptr(p), ptr(t), n, C, ptr(d), ptr(dpred), _lib.stream_ptr()), "mm3d_kl_logits_bwd")
        return dpred, None


def cross_modal_kl(pred: torch.Tensor, target: torch.Tensor) -> torch.Tensor:
    """Mean over rows of ``KL(softmax(target) || softmax(pred))``; ``target`` is treated as detached."""
    return _KlFn.apply(pred, target)


class _Heads3DFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, feat, w1, b1, w2, b2, target):
        if not feat.is_cuda:
            raise RuntimeError("heads3d: CUDA tensors expected (there is no CPU path)")
        x, w1c, b1c, w2c, b2c = _f32c(feat), _f32c(w1), _f32c(b1), _f32c(w2), _f32c(b2)
        n, f = x.shape
        C = w1c.shape[0]
        if w1c.shape != (C, f) or w2c.shape != (C, f) or b1c.shape != (C,) or b2c.shape != (C,):
            raise ValueError("heads3d: weights must be [C, f] and biases [C] (two nn.Linear(f, C))")
        t = _f32c(target) if target is not None else None
        if t is not None and t.shape != (n, C):
            raise ValueError("heads3d: target must be [N, C] logits")
        l1 = torch.empty(n, C, dtype=torch.float32, device=x.device)
        l2 = torch.empty(n, C, dtype=torch.float32, device=x.device)
        loss = torch.zeros((), dtype=torch.float32, device=x.device)
        flags, slots = ctx.det = _det_flags()
        ws = torch.empty(slots, dtype=torch.float64, device=x.device)
        with torch.cuda.device(x.device):
            check(lib.mm3d_heads3d_fwd_ex(ptr(x), n, f, C, ptr(w1c), ptr(b1c), ptr(w2c), ptr(b2c),
                                          ptr(t) if t is not None else None, ptr(l1), ptr(l2),
                                          ptr(loss) if t is not None and n else None, ptr(ws), ws.numel() * 8,
                                          _lib.stream_ptr(), flags), "mm3d_heads3d_fwd")
        ctx.save_for_backward(x, w1c, w2c, b2c, *([t] if t is not None else []))
        ctx.has_target = t is not None
        return l1, l2, loss

    @staticmethod
    def backward(ctx, d1, d2, dloss):
        saved = ctx.saved_tensors
        x, w1, w2, b2 = saved[:4]
        t = saved[4] if ctx.has_target else None
        n, f = x.shape
        C = w1.shape[0]
        d1 = _f32c(d1) if d1 is not None else None
        d2 = _f32c(d2) if d2 is not None else None
        dl = _f32c(dloss).reshape(1) if (dloss is not None and t is not None) else None
        dx = torch.empty_like(x) if ctx.needs_input_grad[0] else None
        dw1, db1 = torch.empty_like(w1), torch.empty(C, dtype=torch.float32, device=x.device)
        dw2, db2 = torch.empty_like(w2), torch.empty(C, dtype=torch.float32, device=x.device)
        flags, slots = ctx.det
        ws = torch.empty((2 * C * f + 2 * C) * slots, dtype=torch.float64, device=x.device)
        with torch.cuda.device(x.device):
            check(lib.mm3d_heads3d_bwd_ex(ptr(x), n, f, C, ptr(w1), ptr(w2), ptr(b2), ptr(t) if t is not None else None,
                                          ptr(d1) if d1 is not None else None, ptr(d2) if d2 is not None else None,
                                          ptr(dl) if dl is not None else None, ptr(dx) if dx is not None else None,
                                          ptr(dw1), ptr(db1), ptr(dw2), ptr(db2), ptr(ws), ws.numel() * 8, _lib.stream_ptr(),
                                          flags), "mm3d_heads3d_bwd")
        return dx, dw1, db1, dw2, db2, None


def heads3d(feat, w1, b1, w2, b2, target=None):
    """``(feat @ w1.T + b1, feat @ w2.T + b2, mean KL(softmax(target) || softmax(second logits)))`` in one pass over
    ``feat`` ``[N, f]`` (f a multiple of 4, <= 32; C <= 20 classes).  ``w*``/``b*`` are the parameters of two
    ``nn.Linear(f, C)``; ``target`` ``[N, C]`` logits is treated as detached; without it the loss is 0."""
    return _Heads3DFn.apply(feat, w1, b1, w2, b2, target)
