"""2D->3D feature lift: sample the 2D network's ``[B, C, H, W]`` map at the pixel every LiDAR
point projects to.

Replaces the per-sample advanced-indexing loop of the reference
(``2d_net/model.py:131-137`` and ``:163-173``)::

    for i in range(B): out.append(fmap.permute(0, 2, 3, 1)[i][img_indices[i][:, 0], img_indices[i][:, 1]])
    out = torch.cat(out, 0)

with one gather kernel over all samples (forward) and one scatter-add kernel (backward,
duplicates accumulate like ``index_put_(accumulate=True)``).  Indices are integer pixels
(row, col) -- the reference never interpolates.  ``LiftIndices`` uploads the per-sample numpy
index arrays ONCE per batch; the reference converts and uploads them at every use.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib  # noqa: F401  (raises when the library is missing)
from .functional import Lift2DBilinearFn, Lift2DFn, lift_csr


class LiftIndices:
    """Device-resident concatenation of the reference's ``img_indices`` list."""

    def __init__(self, img_indices, device):
        counts = [int(len(ix)) for ix in img_indices]
        offs = np.zeros(len(counts) + 1, dtype=np.int64)
        np.cumsum(counts, out=offs[1:])
        if counts and offs[-1] > 0:
            cat = np.concatenate([np.asarray(ix, dtype=np.int64).reshape(-1, 2) for ix in img_indices], 0)
        else:
            cat = np.zeros((0, 2), dtype=np.int64)
        self.counts = counts
        # host-side bounds of the indices, so that lift2d can refuse an out-of-image index synchronously like the
        # reference's advanced indexing does (IndexError), without reading anything back from the device
        self.lo = (int(cat[:, 0].min()), int(cat[:, 1].min())) if len(cat) else (0, 0)
        self.hi = (int(cat[:, 0].max()), int(cat[:, 1].max())) if len(cat) else (-1, -1)
        self.idx = torch.from_numpy(np.ascontiguousarray(cat)).to(device, non_blocking=True)
        self.offsets = torch.from_numpy(offs).to(device, non_blocking=True)
        self._pixel_lists = {}

    def pixel_lists(self, B, H, W):
        """The points grouped by pixel of a [B, ., H, W] map (deterministic lift backward), built on first use."""
        key = (int(B), int(H), int(W))
        if key not in self._pixel_lists:
            self._pixel_lists[key] = lift_csr(self.idx, None, self.offsets, *key)
        return self._pixel_lists[key]

    @property
    def n(self):
        return int(self.idx.shape[0])


def lift2d(fmap: torch.Tensor, img_indices) -> torch.Tensor:
    """``[B, C, H, W]`` map + per-sample (row, col) indices -> ``[sum N_i, C]`` (same dtype)."""
    if not isinstance(img_indices, LiftIndices):
        img_indices = LiftIndices(img_indices, fmap.device)
    if len(img_indices.counts) != fmap.shape[0]:
        raise ValueError("lift2d: one index array per sample expected")
    H, W = int(fmap.shape[2]), int(fmap.shape[3])
    if img_indices.lo[0] < -H or img_indices.hi[0] >= H or img_indices.lo[1] < -W or img_indices.hi[1] >= W:
        raise IndexError(f"lift2d: pixel index out of range for a {H}x{W} map "
                         f"(rows {img_indices.lo[0]}..{img_indices.hi[0]}, columns {img_indices.lo[1]}..{img_indices.hi[1]})")
    return Lift2DFn.apply(fmap, img_indices.idx, img_indices.offsets, img_indices)


def lift2d_bilinear(fmap: torch.Tensor, pixel_coords) -> torch.Tensor:
    """Bilinear variant of :func:`lift2d` -- an extension: the reference only gathers at integer pixels.

    ``pixel_coords``: one float array ``[N_i, 2]`` of (row, col) per sample, in pixel units with pixel centres at the
    integers (the un-floored projection of the LiDAR points).  Returns ``[sum N_i, C]``: the blend of the four
    neighbouring pixels, a neighbour outside the map contributing zero -- ``F.grid_sample(fmap[i:i+1], grid,
    mode="bilinear", padding_mode="zeros", align_corners=True)`` on the normalised coordinates.  At integer coordinates
    inside the map it equals :func:`lift2d`.  Differentiable with respect to the map."""
    counts = [int(len(c)) for c in pixel_coords]
    if len(counts) != fmap.shape[0]:
        raise ValueError("lift2d_bilinear: one coordinate array per sample expected")
    offs = np.zeros(len(counts) + 1, dtype=np.int64)
    np.cumsum(counts, out=offs[1:])
    if offs[-1] > 0:
        cat = np.concatenate([np.asarray(c, dtype=np.float32).reshape(-1, 2) for c in pixel_coords], 0)
    else:
        cat = np.zeros((0, 2), dtype=np.float32)
    uv = torch.from_numpy(np.ascontiguousarray(cat)).to(fmap.device, non_blocking=True)
    offsets = torch.from_numpy(offs).to(fmap.device, non_blocking=True)
    return Lift2DBilinearFn.apply(fmap, uv, offsets)


def rasterize_points(img_indices, values, height: int, width: int, fill: float = 0.0) -> torch.Tensor:
    """Per-point values -> ``[B, H, W]`` float32 maps pre-filled with ``fill``.

    The loaders' sparse depth map and 2D label map (``lib/dataset/nuscenes_dataloader.py:275-278`` and
    ``:287-292``)::

        depth = np.zeros((H, W));             depth[idx[:, 0], idx[:, 1]] = pts_cam_coord[:, 2]
        seg_labels_2d = np.ones((H, W)) * -100;  seg_labels_2d[idx[:, 0], idx[:, 1]] = seg_label

    Where several points fall on one pixel the last one wins, as numpy's indexed assignment does.
    ``values``: float32 CUDA tensor ``[sum N_i]`` in the order of the concatenated index arrays.
    """
    if not values.is_cuda:
        raise RuntimeError("rasterize_points: CUDA tensor expected (there is no CPU path)")
    if not isinstance(img_indices, LiftIndices):
        img_indices = LiftIndices(img_indices, values.device)
    B = len(img_indices.counts)
    vals = values.detach().to(torch.float32).contiguous().reshape(-1)
    if vals.numel() != img_indices.n:
        raise ValueError("rasterize_points: one value per point expected")
    out = torch.empty((B, int(height), int(width)), dtype=torch.float32, device=values.device)
    ws_bytes = _lib.lib.mm3d_raster2d_workspace_bytes(B, int(height), int(width))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=values.device)
    _lib.check(_lib.lib.mm3d_raster2d(_lib.ptr(img_indices.idx), _lib.ptr(img_indices.offsets), B, int(height), int(width),
                                      img_indices.n, _lib.ptr(vals), float(fill), _lib.ptr(out), _lib.ptr(ws), ws_bytes,
                                      _lib.stream_ptr()), "mm3d_raster2d")
    return out
