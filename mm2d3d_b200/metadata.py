"""Per-forward sparse structure on the GPU -- the counterpart of SparseConvNet's ``Metadata``.

One ``Metadata`` is created by ``InputLayer`` and shared by every layer of that forward
(SURVEY.md A.1, a12).  It owns, per spatial size ("level"): the voxel keys in row order, the
voxel hash, the 3^3 neighbour table and the stride-2 tables (parent / offset / child).  All of
it is built by ``libmm3d`` kernels on the current stream; the only host synchronisation is one
read of the per-level row counts after a build (SparseConvNet builds all of this on the CPU and
re-uploads rule lists at every layer call).

Buffers are carved from one ``uint8`` tensor per build and handed to the C ABI as raw pointers;
tensor views are only materialised for inspection (tests, debugging).
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib
from ._lib import check, lib

_ALIGN = 256


def _al(x):
    return (x + _ALIGN - 1) // _ALIGN * _ALIGN


class Level:
    """Structure of one spatial size.  ``cap`` = row capacity the buffers were sized for,
    ``n`` = actual row count (host int, known after the build's sync)."""

    __slots__ = ("spatial", "cap", "tstride", "n", "buf", "base", "o_keys", "o_hkeys", "o_hvals", "hcap",
                 "o_nbr", "o_parent", "o_off", "o_child", "has_nbr", "has_down", "count_slot", "plans")

    def ptr(self, off):
        return self.base + off


class Metadata:
    MAX_LEVELS = 16

    _side = {}  # per-device side stream for the neighbour tables

    def __init__(self, coords: torch.Tensor, spatial_size: int, prebuild_levels: int = 1, plans: bool = False,
                 defer_sync: bool = False, points=None, batch_start=None):
        """``defer_sync``: enqueue the build and an asynchronous read-back of the row counts, but do not wait for
        them; :meth:`finish` (called by every accessor that needs a row count) does.  Lets a caller enqueue a build
        on a side stream and keep launching other work.

        ``points`` (with ``coords=None``): build level 0 from raw float points with ``mm3d_voxelize_points`` -- a
        dict of device tensors ``points [N,3] f32, offsets [B+1] i64, rot [B,9] f32, u [B,3] f64 or None, keep [N] u8,
        min_value [B,3] f32, offset [B,3] f64`` and the float ``scale`` (see ``augment.voxelize_points``).  If the
        batch holds a point outside the receptive field :attr:`dropped` is set once the counts are known and the
        structure must not be used.

        ``batch_start`` (see :func:`group_coords`): the coordinates are several batch groups one after the other, group
        k's scans with batch indices ``[batch_start[k], batch_start[k + 1])`` (device int64 ``[G + 1]``).  Every level
        of the pre-built pyramid then also gets its group row boundaries (:meth:`group_bounds`), computed on the device
        and read back with the row counts."""
        self.dropped = False
        self.groups = 1 if batch_start is None else int(batch_start.numel()) - 1
        self._group_bounds = None
        self._points = points  # (keeps the build's input tensors alive)
        if points is not None:
            if coords is not None:
                raise ValueError("Metadata: pass coords or points, not both")
            self.device = points["points"].device
            self.n_points = int(points["points"].shape[0])
        else:
            if not isinstance(coords, torch.Tensor):
                raise TypeError("Metadata: coords must be a tensor [N, 4] = (x, y, z, batch)")
            if coords.dim() != 2 or coords.shape[1] != 4:
                raise ValueError("coords must be [N, 4] = (x, y, z, batch)")
            if not coords.is_cuda:
                coords = coords.cuda(non_blocking=True)
            coords = coords.to(torch.int64).contiguous()
            self.device = coords.device
            self.n_points = int(coords.shape[0])
        self._pending = None
        self._point_csr = None
        self.spatial_size0 = int(spatial_size)
        self.levels: dict[int, Level] = {}
        self._order: list[Level] = []
        n = self.n_points
        L = max(1, min(int(prebuild_levels), self.MAX_LEVELS))
        # spatial sizes halve while they stay even and > 1
        sizes = [self.spatial_size0]
        while len(sizes) < L and sizes[-1] % 2 == 0 and sizes[-1] > 1:
            sizes.append(sizes[-1] // 2)
        L = len(sizes)

        with torch.cuda.device(self.device):
            stream = _lib.stream_ptr()
            # row counts, status word, then (groups) each level's group boundaries
            n_bounds = self.MAX_LEVELS * (self.groups + 1) if batch_start is not None else 0
            self._counts = torch.zeros(self.MAX_LEVELS + 1 + n_bounds, dtype=torch.int32, device=self.device)
            if points is not None:
                B = int(points["offsets"].numel()) - 1
                ws_bytes = lib.mm3d_voxelize_points_workspace_bytes(n, B)
            else:
                ws_bytes = lib.mm3d_unique_workspace_bytes(n)
            head = _al(4 * n) * 2 + _al(ws_bytes)
            per_level, lay = self._level_layout(n)
            self._buf = torch.empty(head + per_level * L, dtype=torch.uint8, device=self.device)
            base = self._buf.data_ptr()
            self._o_p2v, self._o_npts, o_ws = 0, _al(4 * n), 2 * _al(4 * n)
            self._ws = (base + o_ws, ws_bytes)
            for i, s in enumerate(sizes):
                lv = self._make_level(s, n, self._buf, head + per_level * i, lay, count_slot=i)
                self.levels[s] = lv
                self._order.append(lv)
            l0 = self._order[0]
            cp = self._counts.data_ptr()
            if points is not None:
                q = points
                check(lib.mm3d_voxelize_points(q["points"].data_ptr(), q["offsets"].data_ptr(), B, n, q["rot"].data_ptr(),
                                               float(q["scale"]), self.spatial_size0,
                                               None if q["u"] is None else q["u"].data_ptr(), q["keep"].data_ptr(),
                                               q["min_value"].data_ptr(), q["offset"].data_ptr(), l0.ptr(l0.o_hkeys),
                                               l0.ptr(l0.o_hvals), l0.hcap, base + self._o_p2v, l0.ptr(l0.o_keys),
                                               base + self._o_npts, cp, cp + 4 * self.MAX_LEVELS, self._ws[0],
                                               self._ws[1], stream), "mm3d_voxelize_points")
            else:
                check(lib.mm3d_voxelize(coords.data_ptr(), n, self.spatial_size0, l0.ptr(l0.o_hkeys), l0.ptr(l0.o_hvals),
                                        l0.hcap, base + self._o_p2v, l0.ptr(l0.o_keys), base + self._o_npts,
                                        cp, cp + 4 * self.MAX_LEVELS, self._ws[0], self._ws[1], stream), "mm3d_voxelize")
            # The level chain (coarsen l -> l+1) is a sequence of small latency-bound kernels; the 3^3 table of a
            # level only needs that level's hash, so it runs beside the chain on a second stream.
            main = torch.cuda.current_stream()
            side = self._side.get(self.device.index)
            if side is None:
                side = self._side[self.device.index] = torch.cuda.Stream(device=self.device)
            ready = torch.cuda.Event()
            ready.record(main)
            side.wait_event(ready)
            self._build_nbr(l0, side.cuda_stream)
            for i in range(1, L):
                self._build_down(self._order[i - 1], self._order[i], stream)
                ready = torch.cuda.Event()
                ready.record(main)
                side.wait_event(ready)
                self._build_nbr(self._order[i], side.cuda_stream)
            done = torch.cuda.Event()
            done.record(side)
            main.wait_event(done)
            if plans:
                # row plans of every table, before the host learns the row counts (launch sized by capacity)
                # heaviest tables first (3^3: 27 offsets per row): the launch is ~1.6 waves of one-per-SM CTAs and the
                # hardware hands out CTAs in index order, so the second wave should be the light ones
                specs = [("smc", s) for s in sizes] + [("down", s) for s in sizes[:-1]] + [("up", s) for s in sizes[:-1]]
                self.build_plans(specs)
            if batch_start is not None:
                self._batch_start = batch_start  # (kept alive until the launch is done)
                keys = (C.c_void_p * L)(*[lv.ptr(lv.o_keys) for lv in self._order])
                check(lib.mm3d_group_bounds(keys, cp, L, batch_start.data_ptr(), self.groups,
                                            cp + 4 * (self.MAX_LEVELS + 1), stream), "mm3d_group_bounds")
            if defer_sync:
                host = torch.empty(self._counts.numel(), dtype=torch.int32, pin_memory=True)
                host.copy_(self._counts, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record()
                self._pending = (host, ev)
            else:
                self._sync_counts()

    # ------------------------------------------------------------------ construction helpers
    @staticmethod
    def _level_layout(cap):
        hcap = lib.mm3d_hash_capacity(cap)
        o = {}
        off = 0
        ts = (cap + 3) // 4 * 4  # table plane stride: multiple of 4 rows so 16-byte copies stay aligned
        for name, nbytes in (("keys", 8 * cap), ("hkeys", 8 * hcap), ("hvals", 4 * hcap), ("nbr", 108 * ts),
                             ("parent", 4 * cap), ("off", cap), ("child", 32 * ts)):
            o[name] = off
            off += _al(nbytes)
        o["hcap"] = hcap
        o["tstride"] = ts
        return off, o

    @staticmethod
    def _make_level(spatial, cap, buf, base_off, lay, count_slot):
        lv = Level()
        lv.spatial, lv.cap, lv.n, lv.tstride = spatial, cap, None, lay["tstride"]
        lv.buf, lv.base = buf, buf.data_ptr() + base_off
        lv.o_keys, lv.o_hkeys, lv.o_hvals, lv.hcap = lay["keys"], lay["hkeys"], lay["hvals"], lay["hcap"]
        lv.o_nbr, lv.o_parent, lv.o_off, lv.o_child = lay["nbr"], lay["parent"], lay["off"], lay["child"]
        lv.has_nbr = lv.has_down = False
        lv.count_slot = count_slot
        lv.plans = {}
        return lv

    def _count_ptr(self, lv):
        return self._counts.data_ptr() + 4 * lv.count_slot

    def _build_nbr(self, lv, stream):
        check(lib.mm3d_build_nbr27(lv.ptr(lv.o_keys), self._count_ptr(lv), lv.cap, lv.spatial, lv.ptr(lv.o_hkeys),
                                   lv.ptr(lv.o_hvals), lv.hcap, lv.ptr(lv.o_nbr), lv.tstride, stream), "mm3d_build_nbr27")
        lv.has_nbr = True

    def _build_down(self, fine, coarse, stream):
        # parent/off/child of the 2/2 convolution live with the FINE level; keys/hash with the coarse one
        check(lib.mm3d_coarsen(fine.ptr(fine.o_keys), self._count_ptr(fine), fine.cap, coarse.ptr(coarse.o_hkeys),
                               coarse.ptr(coarse.o_hvals), coarse.hcap, fine.ptr(fine.o_parent), fine.ptr(fine.o_off),
                               coarse.ptr(coarse.o_keys), fine.ptr(fine.o_child), fine.tstride, self._count_ptr(coarse),
                               self._ws[0], self._ws[1], stream), "mm3d_coarsen")
        fine.has_down = True

    def finish(self):
        """Wait for a deferred build's row counts (no-op otherwise)."""
        if self._pending is not None:
            host, ev = self._pending
            self._pending = None
            ev.synchronize()
            self._sync_counts(host)
        return self

    def _sync_counts(self, host=None):
        if host is None:
            host = self._counts.cpu()  # the one host synchronisation of a build
        if int(host[self.MAX_LEVELS]) & _lib.STATUS_BAD_COORD:
            raise ValueError("InputLayer: coordinates must lie in [0, spatial_size) and batch index in [0, 32768)")
        if int(host[self.MAX_LEVELS]) & _lib.STATUS_DROPPED:
            self.dropped = True  # (a point outside the receptive field: the owner rebuilds from the kept points)
        for lv in self._order:
            if lv.n is None:
                lv.n = int(host[lv.count_slot])
        if self.groups > 1 or host.numel() > self.MAX_LEVELS + 1:
            g1 = self.groups + 1
            b = host[self.MAX_LEVELS + 1:].view(self.MAX_LEVELS, g1)
            self._group_bounds = [tuple(int(v) for v in b[lv.count_slot]) for lv in self._order]

    def group_bounds(self, spatial_size=None):
        """Group row boundaries (a structure built from :func:`group_coords`): per pre-built level, shallow to deep, a
        tuple of ``groups + 1`` row indices -- group k = rows ``[b[k], b[k + 1])``; with ``spatial_size`` that level's
        tuple only.  ``None`` for an ungrouped structure."""
        self.finish()
        if self._group_bounds is None:
            return None
        if spatial_size is None:
            return self._group_bounds
        lv = self.levels[int(spatial_size)]
        if lv.count_slot >= len(self._group_bounds):
            raise ValueError(f"no group boundaries for spatial size {spatial_size} (not a pre-built level)")
        return self._group_bounds[lv.count_slot]

    def record_stream(self, stream):
        """Tell the caching allocator that ``stream`` uses this structure's buffers (needed when the structure
        was built on another stream than the one the network runs on, see ``UNetSCN.prepare``)."""
        seen = set()
        bufs = [self._buf, self._counts] + [lv.buf for lv in self._order]
        bufs += [pl[0] for lv in self._order for pl in lv.plans.values()]
        bufs += list(self._point_csr or ())
        for b in bufs:
            key = b.untyped_storage().data_ptr()
            if key not in seen:
                seen.add(key)
                b.record_stream(stream)

    def point_csr(self):
        """(vox_start int32 [n_voxels + 1], vox_pts int32 [n_points]): the points of every voxel in ascending point
        index, for the deterministic InputLayer forward and OutputLayer backward.  Built on the current stream at
        first use and kept.  Called before a deferred build's row counts are known (``UNetSCN.prepare`` with the
        deterministic mode on), it does not wait for them: the lists are built over the point count, a bound on the
        voxel count (the build zeroes the per-voxel counts that far, so the voxels past the real ones are empty and
        ``vox_start`` is longer than ``n_voxels + 1``, with the same first ``n_voxels + 1`` entries)."""
        if self._point_csr is None:
            n = self.n_points
            nv = n if self._pending is not None else self.n_voxels
            start = torch.empty(nv + 1, dtype=torch.int32, device=self.device)
            pts = torch.empty(max(n, 1), dtype=torch.int32, device=self.device)
            with torch.cuda.device(self.device):
                ws = torch.empty(lib.mm3d_point_csr_workspace_bytes(nv), dtype=torch.uint8, device=self.device)
                check(lib.mm3d_point_csr(self.p2v_ptr, self.npts_ptr, n, nv, start.data_ptr(), pts.data_ptr(),
                                         ws.data_ptr(), ws.numel(), _lib.stream_ptr()), "mm3d_point_csr")
            self._point_csr = (start, pts)
        return self._point_csr

    # ------------------------------------------------------------------ lookups used by the layers
    def level(self, spatial_size: int) -> Level:
        self.finish()
        return self.levels[int(spatial_size)]

    def nbr(self, spatial_size: int) -> Level:
        self.finish()
        lv = self.levels[int(spatial_size)]
        if not lv.has_nbr:
            with torch.cuda.device(self.device):
                self._build_nbr(lv, _lib.stream_ptr())
        return lv

    def down(self, spatial_size: int):
        """(fine level, coarse level) of the 2/2 convolution from ``spatial_size``; built lazily
        (one extra host sync) when it was not part of the pre-built pyramid."""
        self.finish()
        s = int(spatial_size)
        fine = self.levels[s]
        if not fine.has_down:
            if s % 2 or s < 2:
                raise ValueError(f"cannot apply a 2/2 convolution at spatial size {s}")
            if len(self._order) >= self.MAX_LEVELS:
                raise ValueError("too many levels")
            with torch.cuda.device(self.device):
                # capacity of the fine level, not its row count: mm3d_coarsen sizes the coarse hash for n_fine_cap rows
                # (the pre-built pyramid does the same: every level has the capacity of the point count)
                cap = fine.cap
                per_level, lay = self._level_layout(cap)
                buf = torch.empty(per_level, dtype=torch.uint8, device=self.device)
                coarse = self._make_level(s // 2, cap, buf, 0, lay, count_slot=len(self._order))
                self.levels[s // 2] = coarse
                self._order.append(coarse)
                self._build_down(fine, coarse, _lib.stream_ptr())
                self._sync_counts()
        return fine, self.levels[s // 2]

    def _plan_level(self, kind, spatial_size):
        return self.nbr(spatial_size) if kind == "smc" else self.down(spatial_size)[0]

    def build_plans(self, specs):
        """Build the row plans (``csrc/plan.cuh``) of several rule tables in ONE launch on the current stream
        (no host synchronisation).  ``specs``: iterable of ``(kind, spatial_size)`` with ``kind`` ``"smc"`` =
        3^3 table of the level, ``"down"`` = child table of the 2/2 convolution FROM ``spatial_size`` (rows =
        coarse voxels), ``"up"`` = its (parent, offset) table (rows = fine voxels).  Already built plans are
        skipped.  The tensor-core modes need them."""
        todo = []
        for kind, s in specs:
            lv = self._plan_level(kind, s)
            if kind not in lv.plans and (kind, int(s)) not in [(k, int(z)) for k, z, _ in todo]:
                todo.append((kind, s, lv))
        if not todo:
            return
        with torch.cuda.device(self.device):
            sizes = []
            for kind, s, lv in todo:
                K = 27 if kind == "smc" else 8
                sizes.append(_al(lib.mm3d_plan_bytes(lv.cap, K)))
            buf = torch.empty(sum(sizes), dtype=torch.uint8, device=self.device)
            descs = (_lib.PlanDesc * len(todo))()
            off = 0
            for d, (kind, s, lv), nbytes in zip(descs, todo, sizes):
                if kind == "smc":
                    d.tbl, d.tbl_stride, d.onehot_off, cnt_lv = lv.ptr(lv.o_nbr), lv.tstride, None, lv
                elif kind == "down":
                    d.tbl, d.tbl_stride, d.onehot_off = lv.ptr(lv.o_child), lv.tstride, None
                    cnt_lv = self.levels[int(s) // 2]
                elif kind == "up":
                    d.tbl, d.tbl_stride, d.onehot_off, cnt_lv = lv.ptr(lv.o_parent), 0, lv.ptr(lv.o_off), lv
                else:
                    raise ValueError(kind)
                d.n_dev, d.n_cap, d.n_rows_hint = self._count_ptr(cnt_lv), lv.cap, (cnt_lv.n or 0)  # 0: size by capacity
                d.K = 27 if kind == "smc" else 8
                d.plan, d.plan_bytes = buf.data_ptr() + off, nbytes
                lv.plans[kind] = (buf[off:off + nbytes], lv.cap)
                off += nbytes
            check(lib.mm3d_build_plans(descs, len(todo), _lib.stream_ptr()), "mm3d_build_plans")

    def plan(self, kind: str, spatial_size: int):
        """(device pointer, capacity) of one row plan, built on first use (see :meth:`build_plans`)."""
        lv = self._plan_level(kind, spatial_size)
        if kind not in lv.plans:
            self.build_plans([(kind, spatial_size)])
        buf, cap = lv.plans[kind]
        return buf.data_ptr(), cap

    def plan_tensors(self, kind: str, spatial_size: int):
        """(perm int32 [T*128], tile_mask int32 [T], table int32 [K, T*128], tile order int32 [T]) views of a
        plan (tests)."""
        self.plan(kind, spatial_size)
        lv = self.levels[int(spatial_size)]
        buf, cap = lv.plans[kind]
        K = 27 if kind == "smc" else 8
        T = (cap + 127) // 128
        al = lambda x: (x + 255) // 256 * 256
        o_mask = al(T * 128 * 4)
        o_order = o_mask + al(T * 4)
        o_tbl = o_order + al(T * 4) + 256
        perm = buf[:T * 128 * 4].view(torch.int32)
        mask = buf[o_mask:o_mask + T * 4].view(torch.int32)
        tbl = buf[o_tbl:o_tbl + K * T * 128 * 4].view(torch.int32).view(K, T * 128)
        order = buf[o_order:o_order + T * 4].view(torch.int32)
        return perm, mask, tbl, order

    # ------------------------------------------------------------------ inspection (tests)
    @property
    def p2v_ptr(self):
        return self._buf.data_ptr() + self._o_p2v

    @property
    def npts_ptr(self):
        return self._buf.data_ptr() + self._o_npts

    @property
    def n_voxels(self):
        self.finish()
        return self._order[0].n

    def _view(self, buf, byte_off, dtype, numel):
        esz = torch.empty(0, dtype=dtype).element_size()
        start = (byte_off) // 1
        return buf[start:start + numel * esz].view(dtype)

    def p2v(self) -> torch.Tensor:
        return self._view(self._buf, self._o_p2v, torch.int32, self.n_points)

    def npts(self) -> torch.Tensor:
        return self._view(self._buf, self._o_npts, torch.int32, self.n_voxels)

    def _lv_view(self, lv, off, dtype, numel):
        return self._view(lv.buf, lv.base - lv.buf.data_ptr() + off, dtype, numel)

    def coords_at(self, spatial_size) -> torch.Tensor:
        """int64 [n, 4] (x, y, z, batch) of the level's rows, decoded from the keys."""
        lv = self.level(spatial_size)
        k = self._lv_view(lv, lv.o_keys, torch.int64, lv.n)
        return torch.stack([(k >> 32) & 0xFFFF, (k >> 16) & 0xFFFF, k & 0xFFFF, k >> 48], 1)

    def nbr_table(self, spatial_size) -> torch.Tensor:
        """int32 [n, 27] (row-major copy of the offset-major device table)."""
        lv = self.nbr(spatial_size)
        t = self._lv_view(lv, lv.o_nbr, torch.int32, 27 * lv.tstride).view(27, lv.tstride)
        return t[:, :lv.n].t().contiguous()

    def down_tables(self, spatial_size):
        """(parent int32 [n_fine], off uint8 [n_fine], child int32 [n_coarse, 8])."""
        fine, coarse = self.down(spatial_size)
        parent = self._lv_view(fine, fine.o_parent, torch.int32, fine.n)
        off = self._lv_view(fine, fine.o_off, torch.uint8, fine.n)
        child = self._lv_view(fine, fine.o_child, torch.int32, 8 * fine.tstride).view(8, fine.tstride)
        return parent, off, child[:, :coarse.n].t().contiguous()


def group_coords(coords_list, device=None):
    """Concatenate the coordinates of several batch groups into one structure's input, keeping the groups apart:
    group k's batch column (each group's starting from 0) is offset by the scans of the groups before it.  The offsets
    are computed on the device (no host synchronisation).  Returns ``(coords [sum N_k, 4] int64, batch_start int64
    [G + 1])`` for ``Metadata(..., batch_start=...)``."""
    if not isinstance(coords_list, (list, tuple)) or not coords_list:
        raise ValueError("group_coords: a non-empty list of [N, 4] coordinate tensors expected")
    if len(coords_list) > _lib.BN_MAX_GROUPS:
        raise ValueError(f"group_coords: {len(coords_list)} groups; at most {_lib.BN_MAX_GROUPS} are supported")
    cs = []
    for c in coords_list:
        if not isinstance(c, torch.Tensor) or c.dim() != 2 or c.shape[1] != 4:
            raise ValueError("group_coords: every group's coordinates must be a tensor [N, 4] = (x, y, z, batch)")
        if device is not None and c.device != torch.device(device):
            c = c.to(device, non_blocking=True)
        cs.append(c.to(torch.int64))
    dev = cs[0].device
    if any(c.device != dev for c in cs):
        raise ValueError("group_coords: the groups' coordinates are on different devices")
    # scans per group = its largest batch index + 1 (0 for an empty group), summed up on the device
    counts = [c[:, 3].max().reshape(1) + 1 if c.shape[0] else torch.zeros(1, dtype=torch.int64, device=dev) for c in cs]
    batch_start = torch.cat([torch.zeros(1, dtype=torch.int64, device=dev), torch.cat(counts).cumsum(0)])
    out = torch.cat(cs)
    row = cs[0].shape[0]
    for k in range(1, len(cs)):  # (device scalars: no host synchronisation)
        out[row:row + cs[k].shape[0], 3] += batch_start[k]
        row += cs[k].shape[0]
    return out, batch_start
