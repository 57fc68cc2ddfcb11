"""``UNetSCN`` -- the 3D backbone of MM2D3D, on this package's ``scn`` modules.

Drop-in for ``3d_net/scn_unet.py:90-126`` of the reference: same constructor arguments
(``config.yaml:22-28``), same attributes (``in_channels``, ``out_channels``), same
``forward([coords, feats]) -> [N, m]`` and the same module tree, so parameter names and shapes
match a SparseConvNet checkpoint (SURVEY.md Appendix B):

    layer1 InputLayer(3, full_scale, mode=4)      layer4 BatchNormReLU(m)
    layer2 SubmanifoldConvolution(in, m, 3)       layer5 OutputLayer
    layer3 U-Net: per level  [BN-ReLU -> SMC]*reps, then (unless deepest)
           ConcatTable{Identity | BN-ReLU -> Conv 2/2 -> deeper level -> BN-ReLU -> Deconv 2/2}
           -> JoinTable -> [BN-ReLU -> SMC]*reps with the first one taking 2p planes

The topology is described once as data (``level_plan``) and then materialised with whatever
``scn``-shaped backend is passed in; tests pass the CPU oracle's module set to get the
reference network, the default is the CUDA implementation in ``mm2d3d_b200.scn``.
"""
from __future__ import annotations

import torch
import torch.nn as nn

DIMENSION = 3


def level_plan(planes, reps):
    """Yield, shallow to deep, ``(p, p_next | None)`` with the (in, out) plane pairs of the
    pre- and post-join blocks of each level (``scn_unet.py:55-84``)."""
    plan = []
    for lvl, p in enumerate(planes):
        deeper = planes[lvl + 1] if lvl + 1 < len(planes) else None
        pre = [(p, p)] * reps
        post = [(2 * p if r == 0 else p, p) for r in range(reps)] if deeper is not None else []
        plan.append({"planes": p, "deeper": deeper, "pre": pre, "post": post})
    return plan


def _append_block(scn, seq, a, b, residual, leakiness):
    """One VGG (``scn_unet.py:48-53``) or pre-activation ResNet (``:36-47``) block."""
    body = scn.Sequential()
    body.add(scn.BatchNormLeakyReLU(a, leakiness=leakiness))
    body.add(scn.SubmanifoldConvolution(DIMENSION, a, b, 3, False))
    if not residual:
        seq.add(body)
        return
    body.add(scn.BatchNormLeakyReLU(b, leakiness=leakiness))
    body.add(scn.SubmanifoldConvolution(DIMENSION, b, b, 3, False))
    shortcut = scn.Identity() if a == b else scn.NetworkInNetwork(a, b, False)
    seq.add(scn.ConcatTable().add(shortcut).add(body))
    seq.add(scn.AddTable())


def build_unet(scn, reps, planes, residual_blocks=False, downsample=(2, 2), leakiness=0):
    """Materialise the U-Net bottom-up (deepest level first) so no recursion is needed."""
    plan = level_plan(list(planes), reps)
    inner = None
    for lvl in reversed(plan):
        seq = scn.Sequential()
        for a, b in lvl["pre"]:
            _append_block(scn, seq, a, b, residual_blocks, leakiness)
        if lvl["deeper"] is not None:
            p, q = lvl["planes"], lvl["deeper"]
            branch = scn.Sequential()
            branch.add(scn.BatchNormLeakyReLU(p, leakiness=leakiness))
            branch.add(scn.Convolution(DIMENSION, p, q, downsample[0], downsample[1], False))
            branch.add(inner)
            branch.add(scn.BatchNormLeakyReLU(q, leakiness=leakiness))
            branch.add(scn.Deconvolution(DIMENSION, q, p, downsample[0], downsample[1], False))
            seq.add(scn.ConcatTable().add(scn.Identity()).add(branch))
            seq.add(scn.JoinTable())
            for a, b in lvl["post"]:
                _append_block(scn, seq, a, b, residual_blocks, leakiness)
        inner = seq
    return inner


class UNetSCN(nn.Module):
    def __init__(self, in_channels=1, m=16, block_reps=1, residual_blocks=False,
                 full_scale=4096, num_planes=7, backend=None):
        super().__init__()
        if backend is None:
            from . import scn as backend  # CUDA implementation; raises if the library is missing
        scn = backend
        self._native = scn.__name__ == "mm2d3d_b200.scn"
        self._num_planes, self._block_reps, self._residual = num_planes, block_reps, residual_blocks
        self.fused = True  # set False to run module by module (same kernels, ~110 autograd nodes)
        self.in_channels = in_channels
        self.out_channels = m
        self.full_scale = full_scale
        planes = [(i + 1) * m for i in range(num_planes)]
        self.layer1 = scn.InputLayer(DIMENSION, full_scale, mode=4)
        if hasattr(self.layer1, "prebuild_levels"):
            # build the whole num_planes-level pyramid in the InputLayer pass: one host sync per forward
            self.layer1.prebuild_levels = num_planes
        self.layer2 = scn.SubmanifoldConvolution(DIMENSION, in_channels, m, 3, False)
        self.layer3 = build_unet(scn, block_reps, planes, residual_blocks)
        self.layer4 = scn.BatchNormReLU(m)
        self.layer5 = scn.OutputLayer(DIMENSION)

    def prepare(self, coords, wait=False):
        """Enqueue the sparse-structure build of a batch ahead of time on the current stream (see
        ``executor.PreparedScans``); ``forward([prepared, feats])`` then skips the structure build."""
        from . import executor
        if not (self.fused and self._native and executor.fusable(self)):
            raise RuntimeError("UNetSCN.prepare needs the fused executor (native backend, fused=True)")
        return executor.prepare(self, coords, wait)

    def prepare_points(self, points, sample_offsets, rot, transl_u, scale, wait=False):
        """:meth:`prepare` from raw float points ``[N, 3]`` (metres, samples concatenated): the reference's
        ``augment_and_scale_3d`` + integer cast + receptive-field filter (``lib/utils/augmentation_3d.py:83-158``,
        ``nuscenes_dataloader.py:312-327``) evaluated inside the voxel-hash insert -- the int64 ``[N, 4]`` coordinate
        tensor of the collate never exists (SURVEY 8(f).1).  See ``executor.prepare_points``."""
        from . import executor
        if not (self.fused and self._native and executor.fusable(self)):
            raise RuntimeError("UNetSCN.prepare_points needs the fused executor (native backend, fused=True)")
        return executor.prepare_points(self, points, sample_offsets, rot, transl_u, scale, wait)

    def prepare_groups(self, coords, wait=False):
        """:meth:`prepare` for :meth:`forward_groups`: one structure build for several batch groups (a list of
        coordinate tensors, each group's batch column starting from 0), enqueued on the current stream."""
        from . import executor
        self._check_groups(coords)
        if len(coords) == 1:
            return self.prepare(coords[0], wait)
        if not (self.fused and self._native and executor.fusable(self)):
            raise RuntimeError("UNetSCN.prepare_groups needs the fused executor (native backend, fused=True)")
        return executor.prepare_groups(self, coords, wait)

    def forward_groups(self, coords, feats, rgb_mask=None):
        """Several batches through one structure build, one forward and one backward: ``coords`` a list of
        ``[N_g, 4]`` coordinate tensors (each group's batch column starting from 0) or what :meth:`prepare_groups`
        returned, ``feats`` the list of the groups' ``[N_g, C]`` features.  Returns the list of the groups' ``[N_g, m]``
        outputs (views of one tensor).  The result is that of ``[self([coords[g], feats[g]]) for g in groups]`` run in
        that order: in training mode every BatchNorm normalises each group with the group's own batch statistics and
        updates the running statistics once per group, in group order; feature gradients are per group, parameter
        (and RGB-mask) gradients the sums over the groups, in one flat gradient tensor.  In eval mode the groups change
        nothing: coordinate lists then run as plain calls, a prepared structure as one eval forward over it.  At most
        8 groups (``MM3D_BN_MAX_GROUPS``); the two-domain step of MM2D3D needs 2.  A prepared structure takes the
        same path as coordinates: the executor when it takes the network, else module by module."""
        from . import executor
        feats = list(feats) if isinstance(feats, (list, tuple)) else feats
        if not isinstance(feats, list):
            raise ValueError("UNetSCN.forward_groups: feats must be a list of the groups' feature tensors")
        if isinstance(coords, executor.PreparedScans):
            if coords.sizes is None:  # (prepare_groups of one group: the plain path)
                if len(feats) != 1:
                    raise ValueError(f"UNetSCN.forward_groups: 1 coordinate group but {len(feats)} feature groups")
                return [self([coords, feats[0]], rgb_mask)]
        else:
            self._check_groups(coords)
            if len(coords) != len(feats):
                raise ValueError(f"UNetSCN.forward_groups: {len(coords)} coordinate groups but {len(feats)} feature "
                                 "groups")
            if len(coords) == 1:  # one group is a plain call
                return [self([coords[0], feats[0]], rgb_mask)]
            if not self.training:
                # eval mode normalises with the running statistics: the groups change nothing, and plain calls give
                # each group the bits of its own call (a shared structure tiles the convolutions' rows differently)
                out = torch.cat([self([c, x], rgb_mask) for c, x in zip(coords, feats)])
                return list(out.split([int(c.shape[0]) for c in coords]))
        if not self._native:
            raise RuntimeError("UNetSCN.forward_groups needs the native backend")
        rgb_mask = self._mask_pair(rgb_mask)
        meta, sizes = executor.group_structure(self, coords, feats)
        if self.fused and executor.fusable(self) and (rgb_mask is None or self.in_channels == 3):
            return executor.run_groups(self, meta, sizes, feats, rgb_mask)
        # module by module over the groups' structure: every BatchNorm finds the groups in the metadata
        from . import functional as F
        from .scn import SparseConvNetTensor
        x = torch.cat(feats)
        if rgb_mask is not None:
            from .heads import rgb_mask as _mask
            x = _mask(x, rgb_mask[0], rgb_mask[1])
        y = SparseConvNetTensor(F.InputLayerFn.apply(x, meta, self.layer1.mode), meta, self.layer1.spatial_size)
        for layer in (self.layer2, self.layer3, self.layer4, self.layer5):
            y = layer(y)
        return list(y.split(sizes))

    @staticmethod
    def _check_groups(coords):
        from ._lib import BN_MAX_GROUPS
        if not isinstance(coords, (list, tuple)) or not coords:
            raise ValueError("UNetSCN.forward_groups: a non-empty list of the groups' coordinate tensors expected")
        if len(coords) > BN_MAX_GROUPS:
            raise ValueError(f"UNetSCN.forward_groups: {len(coords)} groups; at most {BN_MAX_GROUPS} are supported")

    @staticmethod
    def _mask_pair(rgb_mask):
        if rgb_mask is not None and not isinstance(rgb_mask, (tuple, list)):
            return (rgb_mask.weight, rgb_mask.bias)
        return rgb_mask

    def forward(self, x, rgb_mask=None):
        """``x = [coords, feats]`` as in the reference.  ``rgb_mask``: an ``nn.Linear(in_channels, 1)`` (or its
        ``(weight, bias)``) -- the prologue of ``Net3DSeg.forward`` (``3d_net/model.py:46-48``,
        ``feats *= sigmoid(linear_rgb_mask(feats))``): the executor folds it into the InputLayer scatter, so that
        ``net_3d(data_batch["x"], rgb_mask=self.linear_rgb_mask)`` replaces the three lines and the call."""
        if rgb_mask is not None and not isinstance(rgb_mask, (tuple, list)):
            rgb_mask = (rgb_mask.weight, rgb_mask.bias)
        if self.fused and self._native:
            from . import executor
            if executor.fusable(self) and (rgb_mask is None or self.in_channels == 3):
                # whole forward (and backward) as one native call each: csrc/unet_exec.cu
                return executor.run(self, x[0], x[1], rgb_mask)
        if rgb_mask is not None:  # module-by-module path (or the oracle backend): the prologue as its own op
            if self._native:
                from .heads import rgb_mask as _mask
                x = [x[0], _mask(x[1], rgb_mask[0], rgb_mask[1])]
            else:
                x = [x[0], x[1] * torch.sigmoid(torch.nn.functional.linear(x[1], rgb_mask[0], rgb_mask[1]))]
        for layer in (self.layer1, self.layer2, self.layer3, self.layer4, self.layer5):
            x = layer(x)
        return x
