"""``sparseconvnet``-shaped module surface backed by ``libmm3d`` (CUDA, sm_100a).

Drop-in for the names the reference uses (``3d_net/scn_unet.py:38-52,56-81,113-117``): same
constructor argument order, same parameter / buffer names and shapes (SURVEY.md 8(b), Appendix
B), same ``SparseConvNetTensor`` fields.  ``sys.modules["sparseconvnet"] = mm2d3d_b200.scn`` is
enough for the reference's ``scn_unet.py`` to run on it unchanged (see INTEGRATION.md).

Only what SparseConvNet itself restricts to CUDA-float is supported: dimension 3, float32
features, filter 3 (submanifold) and 2/2 (strided), ``groups == 1``.  Anything else raises.
"""
from __future__ import annotations

import math

import torch
import torch.nn as nn

from .. import _lib  # noqa: F401  (raises ImportError when libmm3d.so has not been built)
from .. import functional as F
from ..metadata import Metadata

__all__ = [
    "SparseConvNetTensor", "Sequential", "ConcatTable", "JoinTable", "AddTable", "Identity", "InputLayer",
    "OutputLayer", "SubmanifoldConvolution", "Convolution", "Deconvolution", "BatchNormReLU",
    "BatchNormLeakyReLU", "NetworkInNetwork", "set_conv_mode", "get_conv_mode", "set_deterministic", "get_deterministic",
]


def set_conv_mode(mode: str) -> None:
    """Arithmetic of the sparse convolutions: "fp32" (SIMT FMA, the parity mode), "tf32" (tcgen05, 1e-2), "tf32x3"
    (tcgen05 with three error-compensated TF32 products: FP32-grade results, 1e-4) or "bf16" (tcgen05 kind::f16 on
    BF16 copies of the gathered operands and weights in forward, dgrad and -- up to 128 input channels -- the weight
    gradient, FP32 accumulate: 1e-2 per op)."""
    if mode not in _lib.MODES:
        raise ValueError(f"unknown mode {mode!r}; expected one of {sorted(_lib.MODES)}")
    F.DEFAULT_MODE = mode


def get_conv_mode() -> str:
    return F.DEFAULT_MODE


def set_deterministic(flag) -> None:
    """Deterministic mode: ``True`` makes the ops below sum in a fixed order, so that they return the same bits on
    every run and in every process (same device model, build, inputs and settings); ``False`` keeps the default
    kernels, whose floating-point atomics may land in any order; ``None`` (the default) follows
    ``torch.use_deterministic_algorithms`` (what Lightning's ``Trainer(deterministic=True)`` sets).  The setting is
    read when an op runs forward, and its backward keeps that choice.

    Covered: the InputLayer forward and OutputLayer backward of the module path, the lift backward (``lift2d``,
    ``lift2d_bilinear``), ``rgb_mask``, ``cross_modal_kl`` and ``heads3d``.  Not yet covered: the convolution weight
    gradients, the BatchNorm statistics and the whole-network executor (``UNetSCN``'s fused path); while the mode is
    on, these issue a ``UserWarning`` when they run."""
    if flag is not None and not isinstance(flag, bool):
        raise TypeError(f"set_deterministic: True, False or None expected, got {flag!r}")
    F.DETERMINISTIC = flag


def get_deterministic() -> bool:
    """Whether the deterministic mode is on now (the setting of :func:`set_deterministic`, resolved)."""
    return F.deterministic()


class SparseConvNetTensor:
    def __init__(self, features=None, metadata=None, spatial_size=None):
        self.features = features
        self.metadata = metadata
        self.spatial_size = spatial_size

    def cuda(self):
        self.features = self.features.cuda()
        return self

    def __repr__(self):
        return f"SparseConvNetTensor(features={tuple(self.features.shape)}, spatial_size={self.spatial_size.tolist()})"


def _spatial(sz, dimension):
    if isinstance(sz, int):
        return torch.LongTensor([sz] * dimension)
    return torch.as_tensor(sz, dtype=torch.long)


def _ss(x: SparseConvNetTensor) -> int:
    s = x.spatial_size
    if int(s.min()) != int(s.max()):
        raise NotImplementedError("only cubic spatial sizes are supported")
    return int(s[0])


# ------------------------------------------------------------------------------- containers
class Sequential(nn.Sequential):
    def add(self, module):
        self._modules[str(len(self._modules))] = module
        return self

    def forward(self, x):
        for m in self._modules.values():
            x = m(x)
        return x


class ConcatTable(nn.Sequential):
    def add(self, module):
        self._modules[str(len(self._modules))] = module
        return self

    def forward(self, x):
        return [m(x) for m in self._modules.values()]


class Identity(nn.Module):
    def forward(self, x):
        return x


class JoinTable(nn.Module):
    def forward(self, xs):
        return SparseConvNetTensor(torch.cat([x.features for x in xs], 1), xs[0].metadata, xs[0].spatial_size)


class AddTable(nn.Module):
    def forward(self, xs):
        out = xs[0].features
        for x in xs[1:]:
            out = out + x.features
        return SparseConvNetTensor(out, xs[0].metadata, xs[0].spatial_size)


# ------------------------------------------------------------------------------- I/O layers
class InputLayer(nn.Module):
    """``forward([coords int64 [N,4] (x,y,z,batch), features [N,C]])`` -> SparseConvNetTensor.
    mode 4 = mean over duplicate coordinates, 3 = sum.  ``prebuild_levels`` > 1 makes this layer
    build that many levels of the stride-2 pyramid (and their 3^3 tables) in the same pass, so a
    whole U-Net forward costs one host synchronisation."""

    def __init__(self, dimension, spatial_size, mode=3):
        super().__init__()
        if dimension != 3:
            raise NotImplementedError("InputLayer: dimension 3 only")
        if mode not in (3, 4):
            raise NotImplementedError("InputLayer: modes 3 (sum) and 4 (mean) only")
        self.dimension = dimension
        self.spatial_size = _spatial(spatial_size, dimension)
        self.mode = mode
        self.prebuild_levels = 1

    def forward(self, x):
        coords, feats = x[0], x[1]
        if not feats.is_cuda:
            raise RuntimeError("InputLayer: features must be a CUDA tensor -- mm2d3d_b200 has no CPU path")
        if coords.device != feats.device:
            coords = coords.to(feats.device, non_blocking=True)
        meta = Metadata(coords, int(self.spatial_size[0]), self.prebuild_levels, plans=F.DEFAULT_MODE != "fp32")
        return SparseConvNetTensor(F.InputLayerFn.apply(feats, meta, self.mode), meta, self.spatial_size)


class OutputLayer(nn.Module):
    def __init__(self, dimension):
        super().__init__()
        self.dimension = dimension

    def forward(self, x):
        return F.OutputLayerFn.apply(x.features, x.metadata)


# ------------------------------------------------------------------------------- convolutions
class _ConvBase(nn.Module):
    kind = ""

    def __init__(self, dimension, nIn, nOut, filter_volume, bias, groups):
        super().__init__()
        if dimension != 3 or groups != 1:
            raise NotImplementedError("dimension 3 and groups == 1 only")
        self.dimension, self.nIn, self.nOut = dimension, nIn, nOut
        self.filter_volume = filter_volume
        std = math.sqrt(2.0 / (nIn * filter_volume))
        self.weight = nn.Parameter(torch.empty(filter_volume, groups, nIn, nOut).normal_(0, std))
        if bias:
            self.bias = nn.Parameter(torch.zeros(nOut))
        self.mode = None  # None -> functional.DEFAULT_MODE at call time

    def _apply_conv(self, x, spatial_in):
        y = F.TableConvFn.apply(x.features, self.weight, x.metadata, self.kind, spatial_in,
                                self.mode or F.DEFAULT_MODE)
        if hasattr(self, "bias"):
            y = y + self.bias
        return y


class SubmanifoldConvolution(_ConvBase):
    kind = "smc"

    def __init__(self, dimension, nIn, nOut, filter_size, bias, groups=1):
        if filter_size != 3:
            raise NotImplementedError("SubmanifoldConvolution: filter_size 3 only")
        super().__init__(dimension, nIn, nOut, 27, bias, groups)

    def forward(self, x):
        return SparseConvNetTensor(self._apply_conv(x, _ss(x)), x.metadata, x.spatial_size)


class Convolution(_ConvBase):
    kind = "down"

    def __init__(self, dimension, nIn, nOut, filter_size, filter_stride, bias, groups=1):
        if filter_size != 2 or filter_stride != 2:
            raise NotImplementedError("Convolution: filter_size 2 / filter_stride 2 only")
        super().__init__(dimension, nIn, nOut, 8, bias, groups)

    def forward(self, x):
        return SparseConvNetTensor(self._apply_conv(x, _ss(x)), x.metadata, (x.spatial_size - 2) // 2 + 1)


class Deconvolution(_ConvBase):
    kind = "up"

    def __init__(self, dimension, nIn, nOut, filter_size, filter_stride, bias, groups=1):
        if filter_size != 2 or filter_stride != 2:
            raise NotImplementedError("Deconvolution: filter_size 2 / filter_stride 2 only")
        super().__init__(dimension, nIn, nOut, 8, bias, groups)

    def forward(self, x):
        return SparseConvNetTensor(self._apply_conv(x, _ss(x)), x.metadata, (x.spatial_size - 1) * 2 + 2)


# ------------------------------------------------------------------------------- normalisation
class BatchNormLeakyReLU(nn.Module):
    def __init__(self, nPlanes, eps=1e-4, momentum=0.9, leakiness=0.333):
        super().__init__()
        self.nPlanes, self.eps, self.momentum, self.leakiness = nPlanes, eps, momentum, leakiness
        self.weight = nn.Parameter(torch.ones(nPlanes))
        self.bias = nn.Parameter(torch.zeros(nPlanes))
        self.register_buffer("running_mean", torch.zeros(nPlanes))
        self.register_buffer("running_var", torch.ones(nPlanes))

    def forward(self, x):
        # a structure of several batch groups (UNetSCN.forward_groups): each group normalised with its own statistics
        meta = x.metadata
        bounds = meta.group_bounds(_ss(x)) if self.training and getattr(meta, "groups", 1) > 1 else None
        y = F.BatchNormReLUFn.apply(x.features, self.weight, self.bias, self.running_mean, self.running_var,
                                    float(self.eps), float(self.momentum), float(self.leakiness), self.training, bounds)
        return SparseConvNetTensor(y, x.metadata, x.spatial_size)

    def extra_repr(self):
        return f"{self.nPlanes}, eps={self.eps}, momentum={self.momentum}, leakiness={self.leakiness}"


class BatchNormReLU(BatchNormLeakyReLU):
    def __init__(self, nPlanes, eps=1e-4, momentum=0.9):
        super().__init__(nPlanes, eps, momentum, leakiness=0.0)


class NetworkInNetwork(nn.Module):
    """1x1 convolution (``features @ W``) -- only on the residual-block path, a library GEMM."""

    def __init__(self, nIn, nOut, bias):
        super().__init__()
        self.weight = nn.Parameter(torch.empty(nIn, nOut).normal_(0, math.sqrt(2.0 / nIn)))
        if bias:
            self.bias = nn.Parameter(torch.zeros(nOut))

    def forward(self, x):
        y = x.features @ self.weight
        if hasattr(self, "bias"):
            y = y + self.bias
        return SparseConvNetTensor(y, x.metadata, x.spatial_size)
