"""Fused execution of ``UNetSCN``: the whole forward (and the whole backward) is ONE call into
``libmm3d`` (``csrc/unet_exec.cu``) instead of ~110 Python autograd nodes (about twice that with
``block_reps=2``).

``UNetSCN.forward`` uses this path for every block topology of the constructor (any ``block_reps``,
VGG or residual blocks) with InputLayer mode 4 (``config/config.yaml:22-28``); what the executor does
not implement (per-layer conv modes, conv or NetworkInNetwork bias, leaky ReLU) runs module by module.
Results are the same kernels in the same order, so parity is unchanged; the one exception is the
residual blocks' NetworkInNetwork, which the module path runs as an FP32 torch matmul and the executor
as this library's K = 1 rule-table convolution in the network's convolution mode.

Deterministic mode (``scn.set_deterministic``, or ``torch.use_deterministic_algorithms``), read at the forward and
kept by its backward: the executor then sums the InputLayer and OutputLayer over the voxels' point lists, runs every
BatchNorm and the masked InputLayer's mask gradient in their fixed-order forms and every weight gradient through the
fixed-order tcgen05 form, so a training step in the ``tf32``, ``tf32x3`` and ``bf16`` modes is the same bits on every
run.  The ``fp32`` mode's weight gradients (the SIMT kernel) have no such form: there the step warns.

Inference (validation, test, deployment): in the bf16 mode (``INFER_MODES``), a network in eval mode whose forward
autograd would not record -- grad mode off, or no input of the call (features, RGB-mask weight and bias, parameters)
requiring a gradient -- runs ``mm3d_unet_topo_infer`` instead: every BatchNorm+ReLU in the epilogue of the convolution that produces its input, no
JoinTable copies, a workspace of only what the forward writes, no autograd node.  The output is the same bits as the
eval forward through ``UNetSCNFn`` (which ``net(x).detach()`` with grad mode on still runs).

Grouped BatchNorm statistics (``UNetSCN.forward_groups`` / ``prepare_groups``, :func:`run_groups`): several batches
through one structure (``metadata.group_coords``), one forward and one backward; in training mode the executor's
``mm3d_unet_topo_*_grouped`` calls normalise each group's rows with the group's own statistics, level by level.
"""
from __future__ import annotations

import ctypes as C
import functools

import torch

from . import _lib
from . import functional as F
from ._lib import check, lib
from .metadata import Metadata, group_coords


def collect_slots(net):
    """Parameters and BN buffers of ``net`` in the executor's slot order, which is module-tree order: per
    BatchNorm ``weight, bias, running_mean, running_var``, per convolution or NetworkInNetwork ``weight``.
    For the reference configuration: stem.w | per level: pre_bn pre.w [dn_bn dn.w <deeper> up_bn up.w post_bn
    post.w] | head_bn.

    The module walk is cached as (parameter or buffer dict of the module, name) pairs and the slots are read through
    them on every call, so a parameter or buffer replaced by a new object (``conv.weight = nn.Parameter(...)``,
    ``bn.running_mean = torch.zeros(...)``, ``load_state_dict(..., assign=True)``, buffers moved by ``.to()``) is the
    one the executor reads and writes the gradient of."""
    from . import scn
    refs = getattr(net, "_exec_slot_refs", None)
    # (host time per call, measured on an x86 CPU: the walk ~70 us for the reference configuration; reading its 130
    # slots through the refs ~5 us, the 331 of block_reps = 2 with residual blocks ~11 us)
    if refs is None:
        refs = []
        for mod in net.modules():
            if isinstance(mod, scn.BatchNormLeakyReLU):
                refs += [(mod._parameters, "weight"), (mod._parameters, "bias"), (mod._buffers, "running_mean"),
                         (mod._buffers, "running_var")]
            elif isinstance(mod, (scn._ConvBase, scn.NetworkInNetwork)):
                refs.append((mod._parameters, "weight"))
        net._exec_slot_refs = refs
    return [d[k] for d, k in refs]


def topology(net):
    """``(block_reps, residual)`` of a ``UNetSCN``: the block topology argument of the ``mm3d_unet_topo_*`` calls."""
    return int(getattr(net, "_block_reps", 1)), int(bool(getattr(net, "_residual", False)))


def fusable(net) -> bool:
    """Whether ``net`` has the shape the executor implements.  The module walk costs ~0.35 ms, so the answer is
    cached on the network together with what it depends on (per-layer conv modes, leakiness, InputLayer mode)."""
    from . import scn
    mods = getattr(net, "_exec_mods", None)
    if mods is None:
        mods = net._exec_mods = [m for m in net.modules()
                                 if isinstance(m, (scn._ConvBase, scn.NetworkInNetwork, scn.BatchNormLeakyReLU))]
    key = (net.layer1.mode if isinstance(net.layer1, scn.InputLayer) else None,
           tuple((m.mode, hasattr(m, "bias")) if isinstance(m, scn._ConvBase)
                 else hasattr(m, "bias") if isinstance(m, scn.NetworkInNetwork) else m.leakiness for m in mods))
    cached = getattr(net, "_exec_fusable", None)
    if cached is not None and cached[0] == key:
        return cached[1]
    ok = _fusable(net)
    net._exec_fusable = (key, ok)
    return ok


def _fusable(net) -> bool:
    from . import scn
    if not isinstance(net.layer1, scn.InputLayer) or net.layer1.mode != 4:
        return False
    if int(getattr(net, "_block_reps", 1)) < 1:
        return False
    for mod in net.modules():
        if isinstance(mod, scn._ConvBase) and (mod.mode is not None or hasattr(mod, "bias")):
            return False
        if isinstance(mod, scn.NetworkInNetwork) and hasattr(mod, "bias"):
            return False
        if isinstance(mod, scn.BatchNormLeakyReLU) and mod.leakiness != 0:
            return False
    return True


@functools.lru_cache(maxsize=None)
def wgrad_covered(in_ch: int, m: int, L: int, residual: int, mode: int) -> bool:
    """Whether every weight gradient of this network shape has a deterministic form (the tcgen05 kernel takes it):
    never in the fp32 mode; in the tensor-core modes for the usual widths (multiples of 16).  The executor runs the
    default kernel for a shape without one, so the caller warns."""
    if mode == _lib.MODE_FP32:
        return False
    cin_k = (in_ch + 15) // 16 * 16  # the stem input as the kernels see it (padded)
    shapes = {(cin_k, m, 27)}
    for l in range(L):
        p = m * (l + 1)
        shapes.add((p, p, 27))
        if l + 1 < L:
            q = m * (l + 2)
            shapes |= {(p, q, 8), (q, p, 8), (2 * p, p, 27)}
            if residual:
                shapes.add((2 * p, p, 1))  # NetworkInNetwork of the first post block
    return all(lib.mm3d_conv_wgrad_workspace_bytes(0, ci, co, K, mode, _lib.DETERMINISTIC) > 0 for ci, co, K in shapes)


def _level_desc(meta: Metadata, num_planes: int, spatial0: int, plans: bool):
    W = _lib.LEVEL_DESC_WORDS
    desc = (C.c_int64 * (W * num_planes))()
    if plans:  # every table of the forward in one launch
        specs, s = [], spatial0
        for l in range(num_planes):
            specs.append(("smc", s))
            if l + 1 < num_planes:
                specs += [("down", s), ("up", s)]
            s //= 2
        meta.build_plans(specs)
    s = spatial0
    for l in range(num_planes):
        lv = meta.nbr(s)
        desc[W * l + 0] = lv.n
        desc[W * l + 1] = lv.ptr(lv.o_nbr)
        desc[W * l + 2] = lv.tstride
        if plans:
            desc[W * l + 6], desc[W * l + 9] = meta.plan("smc", s)
        if l + 1 < num_planes:
            fine, _ = meta.down(s)
            desc[W * l + 3] = fine.ptr(fine.o_parent)
            desc[W * l + 4] = fine.ptr(fine.o_off)
            desc[W * l + 5] = fine.ptr(fine.o_child)
            if plans:
                desc[W * l + 7] = meta.plan("down", s)[0]
                desc[W * l + 8] = meta.plan("up", s)[0]
        s //= 2
    return desc


def _unet_groups(meta: Metadata, num_planes: int):
    """(``mm3d_unet_groups``, its bounds array) of a grouped structure's first ``num_planes`` levels."""
    G = meta.groups
    flat = [b for lv in meta.group_bounds()[:num_planes] for b in lv]
    if len(flat) != num_planes * (G + 1):
        raise ValueError("UNetSCN: the grouped structure has fewer levels than the network")
    bounds = (C.c_int64 * len(flat))(*flat)
    return _lib.UnetGroups(G, C.addressof(bounds)), bounds


class UNetSCNFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, feats, meta, cfg, mask_w, mask_b, *slots):
        in_ch, m, L, mode, training, eps, momentum, spatial0, reps, res = cfg
        det = F.deterministic()
        if det and not wgrad_covered(in_ch, m, L, res, mode):
            F.alert_not_deterministic("the sparse-convolution weight gradient in the fp32 mode" if mode == _lib.MODE_FP32
                                      else f"the sparse-convolution weight gradient with m = {m} (channel counts that "
                                           "are not multiples of 16)")
        flags = _lib.DETERMINISTIC if det else 0
        feats = feats.float().contiguous()
        dev = feats.device
        # optional RGB mask of Net3DSeg.forward (3d_net/model.py:46-48), folded into the InputLayer scatter
        masked = mask_w is not None
        wb = _mask_wb(in_ch, mask_w, mask_b) if masked else None  # (checked before anything is allocated)
        n_points = meta.n_points
        desc = _level_desc(meta, L, spatial0, plans=mode != _lib.MODE_FP32)
        # a structure of several batch groups (UNetSCN.forward_groups), training mode: every BatchNorm per group
        groups = _unet_groups(meta, L) if training and meta.groups > 1 else None
        G = meta.groups if groups is not None else 1
        with torch.cuda.device(dev):
            # sticky device-error words (mapped host memory): whatever a kernel of an earlier call raised surfaces
            # here -- no synchronisation, a few nanoseconds
            _lib.raise_device_errors("UNetSCN.forward")
            if groups is None:
                act_bytes = lib.mm3d_unet_topo_act_bytes(in_ch, m, L, reps, res, mode, desc, n_points)
                scr = F.scratch(lib.mm3d_unet_topo_scratch_bytes_ex(in_ch, m, L, reps, res, mode, flags), dev)
            else:
                act_bytes = lib.mm3d_unet_topo_act_bytes_grouped(in_ch, m, L, reps, res, mode, desc, n_points, G)
                scr = F.scratch(lib.mm3d_unet_topo_scratch_bytes_grouped(in_ch, m, L, reps, res, mode, flags, G), dev)
            act = torch.empty(act_bytes, dtype=torch.uint8, device=dev)
            out = torch.empty(n_points, m, dtype=torch.float32, device=dev)
            vox_start, vox_pts = meta.point_csr() if det else (None, None)
            params = (C.c_void_p * len(slots))(*[t.data_ptr() for t in slots])
            mask, gate = None, None
            if masked:
                gate = torch.empty(max(n_points, 1), dtype=torch.float32, device=dev)
                mask = C.byref(_lib.UnetMask(wb.data_ptr(), gate.data_ptr(), None, None, None, 0))
            if groups is not None:
                check(lib.mm3d_unet_topo_forward_grouped(in_ch, m, L, reps, res, mode, int(training), eps, momentum, desc,
                                                         n_points, meta.p2v_ptr, meta.npts_ptr, _lib.ptr(vox_start),
                                                         _lib.ptr(vox_pts), feats.data_ptr(), out.data_ptr(), params,
                                                         act.data_ptr(), act_bytes, scr.data_ptr(), scr.numel(), mask,
                                                         _lib.stream_ptr(), flags, C.byref(groups[0])),
                      "mm3d_unet_topo_forward_grouped")
            elif det:
                check(lib.mm3d_unet_topo_forward_ex(in_ch, m, L, reps, res, mode, int(training), eps, momentum, desc, n_points,
                                                    meta.p2v_ptr, meta.npts_ptr, vox_start.data_ptr(), vox_pts.data_ptr(),
                                                    feats.data_ptr(), out.data_ptr(), params, act.data_ptr(), act_bytes,
                                                    scr.data_ptr(), scr.numel(), mask, _lib.stream_ptr(), flags),
                      "mm3d_unet_topo_forward_ex")
            else:
                check(lib.mm3d_unet_topo_forward(in_ch, m, L, reps, res, mode, int(training), eps, momentum, desc, n_points,
                                                 meta.p2v_ptr, meta.npts_ptr, feats.data_ptr(), out.data_ptr(), params,
                                                 act.data_ptr(), act_bytes, scr.data_ptr(), scr.numel(), mask,
                                                 _lib.stream_ptr()), "mm3d_unet_topo_forward")
        ctx.meta, ctx.cfg, ctx.desc, ctx.act, ctx.slots = meta, cfg, desc, act, slots
        ctx.flags = flags  # the backward keeps the forward's choice
        ctx.groups = groups
        ctx.feats_shape = feats.shape
        ctx.mask = (feats, wb, gate, mask_w.shape, mask_b.shape) if masked else None
        return out

    @staticmethod
    def backward(ctx, d_out):
        in_ch, m, L, mode, training, eps, momentum, spatial0, reps, res = ctx.cfg
        meta, slots, desc, act = ctx.meta, ctx.slots, ctx.desc, ctx.act
        d_out = d_out.float().contiguous()
        dev = d_out.device
        n_points = meta.n_points
        need_feats = ctx.needs_input_grad[0]
        flags = ctx.flags
        with torch.cuda.device(dev):
            _lib.raise_device_errors("UNetSCN.backward")
            # one flat buffer for every parameter gradient; the returned grads are views into it
            live = [t for t in slots if t.requires_grad]
            flat = torch.empty(sum(t.numel() for t in live), dtype=torch.float32, device=dev)
            # all views in one native call (what DDP's buckets use) instead of ~130 slice + view calls
            views = iter(torch._utils._unflatten_dense_tensors(flat, live)) if live else iter(())
            gptrs, grads = [], []
            for t in slots:
                if t.requires_grad:
                    g = next(views)
                    gptrs.append(g.data_ptr())
                    grads.append(g)
                else:
                    gptrs.append(None)
                    grads.append(None)
            d_feats = torch.empty(ctx.feats_shape, dtype=torch.float32, device=dev) if need_feats else None
            if need_feats and ctx.feats_shape[0] > n_points:
                d_feats.zero_()
            tmp_bytes = lib.mm3d_unet_topo_bwd_bytes(in_ch, m, L, reps, res, mode, desc, n_points)
            tmp = torch.empty(tmp_bytes, dtype=torch.uint8, device=dev)
            groups = ctx.groups
            if groups is None:
                scr = F.scratch(lib.mm3d_unet_topo_scratch_bytes_ex(in_ch, m, L, reps, res, mode, flags), dev)
            else:
                scr = F.scratch(lib.mm3d_unet_topo_scratch_bytes_grouped(in_ch, m, L, reps, res, mode, flags,
                                                                         groups[0].groups), dev)
            params = (C.c_void_p * len(slots))(*[t.data_ptr() for t in slots])
            gp = (C.c_void_p * len(slots))(*gptrs)
            mask, d_mw, d_mb = None, None, None
            if ctx.mask is not None:
                feats, wb, gate, w_shape, b_shape = ctx.mask
                d_wb = torch.empty(in_ch + 1, dtype=torch.float32, device=dev)
                # (deterministic: one row of partial sums per CTA)
                mws = torch.empty((in_ch + 1) * (_lib.DET_CTAS if flags else 1), dtype=torch.float64, device=dev)
                mask = C.byref(_lib.UnetMask(wb.data_ptr(), gate.data_ptr(), feats.data_ptr(), d_wb.data_ptr(), mws.data_ptr(),
                                             mws.numel() * 8))
                d_mw, d_mb = d_wb[:in_ch].reshape(w_shape), d_wb[in_ch:].reshape(b_shape)
            d_feats_ptr = d_feats.data_ptr() if need_feats else None
            if groups is not None:
                vox_start, vox_pts = meta.point_csr() if flags else (None, None)
                check(lib.mm3d_unet_topo_backward_grouped(in_ch, m, L, reps, res, mode, int(training), desc, n_points,
                                                          meta.p2v_ptr, meta.npts_ptr, _lib.ptr(vox_start),
                                                          _lib.ptr(vox_pts), d_out.data_ptr(), d_feats_ptr, params, gp,
                                                          act.data_ptr(), act.numel(), tmp.data_ptr(), tmp_bytes,
                                                          scr.data_ptr(), scr.numel(), mask, _lib.stream_ptr(), flags,
                                                          C.byref(groups[0])), "mm3d_unet_topo_backward_grouped")
            elif flags:
                vox_start, vox_pts = meta.point_csr()
                check(lib.mm3d_unet_topo_backward_ex(in_ch, m, L, reps, res, mode, int(training), desc, n_points, meta.p2v_ptr,
                                                     meta.npts_ptr, vox_start.data_ptr(), vox_pts.data_ptr(), d_out.data_ptr(),
                                                     d_feats_ptr, params, gp, act.data_ptr(), act.numel(), tmp.data_ptr(),
                                                     tmp_bytes, scr.data_ptr(), scr.numel(), mask, _lib.stream_ptr(), flags),
                      "mm3d_unet_topo_backward_ex")
            else:
                check(lib.mm3d_unet_topo_backward(in_ch, m, L, reps, res, mode, int(training), desc, n_points, meta.p2v_ptr,
                                                  meta.npts_ptr, d_out.data_ptr(), d_feats_ptr, params, gp, act.data_ptr(),
                                                  act.numel(), tmp.data_ptr(), tmp_bytes, scr.data_ptr(), scr.numel(), mask,
                                                  _lib.stream_ptr()), "mm3d_unet_topo_backward")
        return (d_feats, None, None, d_mw, d_mb, *grads)


class PreparedScans:
    """Sparse structure of one batch (voxels, rule tables, row plans), built ahead of the forward that uses it --
    typically on a side stream while the previous step still computes, the way a prefetching data loader prepares
    the next batch.  Pass it to ``UNetSCN.forward`` in place of the coordinate tensor."""

    __slots__ = ("meta", "event", "stream", "mode", "spatial0", "levels", "points", "sizes")

    def __init__(self, meta, mode, spatial0, levels, points=None, sizes=None):
        self.meta, self.mode, self.spatial0, self.levels = meta, mode, spatial0, levels
        self.points = points  # augment.PointStructure when the batch was prepared from raw float points
        self.sizes = sizes  # prepare_groups: the groups' point counts (None: one batch)
        self.stream = torch.cuda.current_stream(meta.device)
        self.event = torch.cuda.Event()
        self.event.record(self.stream)

    def kept(self):
        """Prepared from points (``UNetSCN.prepare_points``): ``None`` when every point lies inside the receptive
        field, else the bool ``[N]`` mask of the points the reference's loader keeps -- features and labels passed
        to the forward must be filtered with it.  Waits for the build's row counts (the build's one host sync)."""
        if self.points is None:
            return None
        meta, keep = self.points.resolve()
        if meta is not self.meta:  # rebuilt from the kept points, on the stream current at the time of this call
            self.meta = meta
            self.stream = torch.cuda.current_stream(meta.device)
            self.event = torch.cuda.Event()
            self.event.record(self.stream)
        return keep

    @property
    def min_value(self):
        return self.points.min_value

    @property
    def offset(self):
        return self.points.offset

    @property
    def n_points(self):
        return self.meta.n_points


def prepare(net, coords, wait=False):
    """Enqueue the structure build for ``coords`` ([N, 4] int64: x, y, z, batch) on the CURRENT stream and return a
    :class:`PreparedScans`.  Nothing blocks here unless ``wait``: the one host synchronisation of a build (reading
    the row counts) is deferred to the forward that uses the structure, by which time a build enqueued one step
    ahead has long finished."""
    if not isinstance(coords, torch.Tensor) or not coords.is_cuda:
        raise RuntimeError("UNetSCN.prepare: coordinates must be a CUDA tensor -- mm2d3d_b200 has no CPU path")
    spatial0 = int(net.layer1.spatial_size[0])
    L = net._num_planes
    with torch.cuda.device(coords.device):
        meta = Metadata(coords, spatial0, L, plans=F.DEFAULT_MODE != "fp32", defer_sync=not wait)
        if F.deterministic():  # the voxels' point lists too, one step ahead like the rest of the structure
            meta.point_csr()
        return PreparedScans(meta, F.DEFAULT_MODE, spatial0, L)


def prepare_groups(net, coords_list, wait=False):
    """:func:`prepare` for several batch groups (``UNetSCN.forward_groups``): one structure build of the groups one
    after the other, their row boundaries at every level computed on the device and read back with the row counts."""
    if not isinstance(coords_list, (list, tuple)) or not all(isinstance(c, torch.Tensor) and c.is_cuda for c in coords_list):
        raise RuntimeError("UNetSCN.prepare_groups: a list of CUDA coordinate tensors expected -- mm2d3d_b200 has no "
                           "CPU path")
    spatial0 = int(net.layer1.spatial_size[0])
    L = net._num_planes
    with torch.cuda.device(coords_list[0].device):
        coords, batch_start = group_coords(coords_list)
        meta = Metadata(coords, spatial0, L, plans=F.DEFAULT_MODE != "fp32", defer_sync=not wait, batch_start=batch_start)
        if F.deterministic():
            meta.point_csr()
        return PreparedScans(meta, F.DEFAULT_MODE, spatial0, L, sizes=[int(c.shape[0]) for c in coords_list])


def prepare_points(net, points, sample_offsets, rot, transl_u, scale, wait=False):
    """:func:`prepare` from raw float points: the reference's ``augment_and_scale_3d`` + cast + filter fused into the
    voxel-hash insert (``augment.voxelize_points``).  ``rot`` / ``transl_u`` are the host-side random draws
    (``augment.draw_augmentation``).  The returned handle's :meth:`PreparedScans.kept` tells which points survive
    (``None`` = all), ``.min_value`` / ``.offset`` are what ``augment_and_scale_3d`` returns beside the coordinates."""
    from .augment import voxelize_points
    spatial0 = int(net.layer1.spatial_size[0])
    L = net._num_planes
    ps = voxelize_points(points, sample_offsets, rot, transl_u, scale, spatial0, L, plans=F.DEFAULT_MODE != "fp32",
                         defer_sync=not wait)
    with torch.cuda.device(ps.meta.device):
        if F.deterministic():  # (a structure rebuilt from the kept points builds its lists at the forward)
            ps.meta.point_csr()
        prep = PreparedScans(ps.meta, F.DEFAULT_MODE, spatial0, L, points=ps)
    if wait:
        prep.kept()
    return prep


# Convolution modes that take the inference path: those where it measured faster than the eval forward through
# UNetSCNFn on a batch of 8 nuScenes-shaped scans (tools/infer_bench.py, profiles/r4_infer_bench.txt, B200).  In the
# fp32, tf32 and tf32x3 modes the BatchNorm arithmetic and the extra row stores in the convolution epilogues cost more
# than the passes they remove, so there the eval forward stays on UNetSCNFn.
INFER_MODES = frozenset({_lib.MODE_BF16})


def inference_path(training: bool, inputs) -> bool:
    """Whether a forward takes the inference path: the network is in eval mode and autograd would record nothing --
    grad mode is off, or none of ``inputs`` (the call's tensors; ``None`` entries ignored) requires a gradient."""
    if training:
        return False
    if not torch.is_grad_enabled():
        return True
    return not any(t is not None and t.requires_grad for t in inputs)


def _mask_wb(in_ch, mask_w, mask_b):
    """The RGB mask of Net3DSeg.forward (3d_net/model.py:46-48) as the executor takes it: [weight | bias], FP32."""
    if mask_w.numel() != in_ch or mask_b is None or mask_b.numel() != 1:
        raise ValueError("UNetSCN: rgb_mask must be the weight [1, C] and bias [1] of an nn.Linear(C, 1)")
    return torch.cat([mask_w.detach().reshape(-1), mask_b.detach().reshape(-1)]).float().contiguous()


def infer(feats, meta, cfg, mask_w, mask_b, slots):
    """The inference forward (``mm3d_unet_topo_infer``): plain tensors in, a plain ``[n_points, m]`` tensor out, nothing
    kept.  ``cfg`` as for :class:`UNetSCNFn` (its training flag and momentum unused)."""
    in_ch, m, L, mode, _, eps, _, spatial0, reps, res = cfg
    flags = _lib.DETERMINISTIC if F.deterministic() else 0
    feats = feats.detach().float().contiguous()
    dev = feats.device
    wb = _mask_wb(in_ch, mask_w, mask_b) if mask_w is not None else None
    n_points = meta.n_points
    desc = _level_desc(meta, L, spatial0, plans=mode != _lib.MODE_FP32)
    with torch.cuda.device(dev):
        _lib.raise_device_errors("UNetSCN.forward")
        ws_bytes = lib.mm3d_unet_topo_infer_bytes(in_ch, m, L, reps, res, mode, desc, n_points, flags)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        out = torch.empty(n_points, m, dtype=torch.float32, device=dev)
        vox_start, vox_pts = meta.point_csr() if flags else (None, None)
        params = (C.c_void_p * len(slots))(*[t.data_ptr() for t in slots])
        mask = None
        if wb is not None:
            gate = torch.empty(max(n_points, 1), dtype=torch.float32, device=dev)
            mask = C.byref(_lib.UnetMask(wb.data_ptr(), gate.data_ptr(), None, None, None, 0))
        check(lib.mm3d_unet_topo_infer(in_ch, m, L, reps, res, mode, eps, desc, n_points, meta.p2v_ptr, meta.npts_ptr,
                                       _lib.ptr(vox_start), _lib.ptr(vox_pts), feats.data_ptr(), out.data_ptr(), params,
                                       ws.data_ptr(), ws_bytes, mask, _lib.stream_ptr(), flags), "mm3d_unet_topo_infer")
    return out


def _resolve(net, coords, feats):
    """The structure of a forward: a prepared one (waited for on this stream) or one built now from ``coords``."""
    spatial0 = int(net.layer1.spatial_size[0])
    L = net._num_planes
    if isinstance(coords, PreparedScans):
        prep = coords
        if (prep.mode, prep.spatial0, prep.levels) != (F.DEFAULT_MODE, spatial0, L) or prep.meta.device != feats.device:
            raise ValueError("UNetSCN: the prepared structure was built for another network, device or convolution mode")
        prep.kept()  # (prepared from points: settles which structure is used)
        meta = prep.meta.finish()
        cur = torch.cuda.current_stream(feats.device)
        if cur != prep.stream:
            cur.wait_event(prep.event)
            meta.record_stream(cur)
    else:
        if coords.device != feats.device:
            coords = coords.to(feats.device, non_blocking=True)
        meta = Metadata(coords, spatial0, L, plans=F.DEFAULT_MODE != "fp32")
    return meta


def run(net, coords, feats, rgb_mask=None):
    if not feats.is_cuda:
        raise RuntimeError("UNetSCN: features must be a CUDA tensor -- mm2d3d_b200 has no CPU path")
    if isinstance(coords, PreparedScans) and coords.sizes is not None:
        raise ValueError("UNetSCN: a structure from prepare_groups goes to forward_groups")
    return _run(net, _resolve(net, coords, feats), feats, rgb_mask)


def group_structure(net, coords, feats):
    """(structure, the groups' point counts) of ``UNetSCN.forward_groups``: a structure from :func:`prepare_groups`
    (waited for on this stream), or one built now from the list of the groups' coordinate tensors."""
    if isinstance(coords, PreparedScans):
        if coords.sizes is None:
            raise ValueError("UNetSCN.forward_groups: the prepared structure is not grouped (use prepare_groups)")
        check_group_feats(coords.sizes, feats)
        return _resolve(net, coords, feats[0]), coords.sizes
    sizes = [int(c.shape[0]) for c in coords]
    check_group_feats(sizes, feats)
    with torch.cuda.device(feats[0].device):
        c, batch_start = group_coords(coords, feats[0].device)
        meta = Metadata(c, int(net.layer1.spatial_size[0]), net._num_planes, plans=F.DEFAULT_MODE != "fp32",
                        batch_start=batch_start)
    return meta, sizes


def run_groups(net, meta, sizes, feats, rgb_mask=None):
    """``UNetSCN.forward_groups`` on the executor: one forward over the groups' structure (training mode: every
    BatchNorm per group), the output split back into the groups (views of one tensor)."""
    return list(_run(net, meta, torch.cat(list(feats)), rgb_mask).split(sizes))


def check_group_feats(sizes, feats):
    if len(feats) != len(sizes):
        raise ValueError(f"UNetSCN.forward_groups: {len(sizes)} coordinate groups but {len(feats)} feature groups")
    for k, (n, f) in enumerate(zip(sizes, feats)):
        if not isinstance(f, torch.Tensor) or not f.is_cuda:
            raise RuntimeError("UNetSCN: features must be a CUDA tensor -- mm2d3d_b200 has no CPU path")
        if f.dim() != 2 or f.shape[0] != n:
            raise ValueError(f"UNetSCN.forward_groups: group {k} has {n} points but features of shape {tuple(f.shape)}")


def _run(net, meta, feats, rgb_mask):
    spatial0 = int(net.layer1.spatial_size[0])
    L = net._num_planes
    if feats.shape[0] < meta.n_points:
        raise ValueError(f"UNetSCN: {feats.shape[0]} feature rows for {meta.n_points} points")
    bn0 = net.layer4
    cfg = (net.in_channels, net.out_channels, L, _lib.MODES[F.DEFAULT_MODE], bool(net.training), float(bn0.eps),
           float(bn0.momentum), spatial0, *topology(net))
    mask_w, mask_b = rgb_mask if rgb_mask is not None else (None, None)
    slots = collect_slots(net)
    if cfg[3] in INFER_MODES and inference_path(net.training, (feats, mask_w, mask_b, *slots)):
        return infer(feats, meta, cfg, mask_w, mask_b, slots)
    with torch.autocast("cuda", enabled=False):
        return UNetSCNFn.apply(feats, meta, cfg, mask_w, mask_b, *slots)
