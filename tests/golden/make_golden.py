"""Generates the committed golden fixtures.  Run in the BUILD container (needs /root/reference for
the lift fixture):  ``python tests/golden/make_golden.py``.

* ``lift_ref.npz``    -- produced by the REFERENCE ITSELF: its ``L2G_classifier_2D``
  (``2d_net/model.py:145-180``) is imported and run on CPU; we record the map it lifts from
  (``seg_logit_avg_2d``), the per-sample pixel indices and what it returns (``seg_logit_avg``),
  plus the gradient torch autograd gives for the map.  This pins the lift oracle and kernel.
* ``unet_small.npz``  -- produced by the CPU ORACLE (SparseConvNet is not available; see
  oracle/__init__.py): a small UNetSCN (m=4, 4 planes, full_scale 64) forward + backward with
  seeded weights on a seeded 2-sample cloud: inputs, parameters, output, all gradients.
* ``structure_small.npz`` -- oracle voxel ids / level coords / rule tables for a seeded cloud.
* ``augment_ref.npz`` -- produced by the REFERENCE ITSELF: ``augment_and_scale_3d``
  (``lib/utils/augmentation_3d.py``) + the loader's integer cast and range filter.
* ``heads3d_ref.npz`` -- the two 3D heads by the REFERENCE's ``Net3DSeg.forward`` with its real heads (backbone replaced by a
  16-channel pass-through), 3D cross-modal term by the torch lines of ``train.py:174-182``.
* ``heads_ref.npz`` -- RGB mask by the REFERENCE's ``Net3DSeg.forward`` (``3d_net/model.py:44-58``, backbone replaced by
  a pass-through), cross-modal KL term by the torch lines of ``train.py:157-184``.
* ``unetscn_tree.json`` -- the SPEC of the reference's ``UNetSCN(in_channels=3)`` module tree (``3d_net/scn_unet.py:8-126``)
  as state_dict keys in order with their shapes, spelled out from SURVEY.md Appendix B without ``mm2d3d_b200``.  It is
  not produced by running the reference; where the reference is at hand, its own tree is what to store here.
"""
import importlib.util
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import scn_cpu  # noqa: E402
from oracle import scn_oracle as O  # noqa: E402
from mm2d3d_b200.unet import UNetSCN  # noqa: E402

REF_2D = "/root/reference/experiments_USA_SING/rgbd_rgbxyz_sigmoid_for_rgb/2d_net/model.py"


def lift_from_reference():
    # import only the class definitions of the reference file (its package-relative import of
    # .backbones is not needed for L2G_classifier_2D)
    src = open(REF_2D).read().replace("from .backbones import Backbone", "Backbone = None")
    mod = type(sys)("ref_2d_model")
    exec(compile(src, REF_2D, "exec"), mod.__dict__)
    torch.manual_seed(7)
    rng = np.random.default_rng(7)
    B, C_in, H, W, classes = 3, 8, 23, 40, 6
    head = mod.L2G_classifier_2D(C_in, classes).double()
    feat = torch.randn(B, C_in, H, W, dtype=torch.float64)
    counts = [57, 0, 131]
    img_indices = []
    for i, n in enumerate(counts):
        r = rng.integers(0, H, n)
        c = rng.integers(0, W, n)
        if i == 2:  # duplicate-heavy sample
            r, c = r % 4, c % 4
        img_indices.append(np.stack([r, c], 1).astype(np.int64))
    preds = head(feat, img_indices)
    fmap = preds["seg_logit_avg_2d"].detach().clone().requires_grad_(True)
    # re-run the reference's lift lines on the recorded map to get the autograd gradient
    lifted = []
    for i in range(B):
        lifted.append(fmap.permute(0, 2, 3, 1)[i][img_indices[i][:, 0], img_indices[i][:, 1]])
    lifted = torch.cat(lifted, 0)
    assert torch.equal(lifted.detach(), preds["seg_logit_avg"].detach())
    g = torch.randn_like(lifted)
    (d_fmap,) = torch.autograd.grad(lifted, fmap, g)
    np.savez_compressed(
        os.path.join(HERE, "lift_ref.npz"), fmap=fmap.detach().numpy(), lifted=preds["seg_logit_avg"].detach().numpy(),
        idx=np.concatenate(img_indices, 0), counts=np.asarray(counts), grad_out=g.numpy(), grad_fmap=d_fmap.numpy())


def small_cloud(seed, n=220, b=2, span=28, origin=5):
    rng = np.random.default_rng(seed)
    # surface-like: points near two planes so that 3^3 neighbourhoods are populated
    pts = []
    for s in range(b):
        u = rng.integers(0, span, (n, 2))
        z = (u[:, 0] // 3 + rng.integers(0, 2, n)) % span
        c = np.stack([u[:, 0], u[:, 1], z], 1) + origin
        pts.append(np.concatenate([c, np.full((n, 1), s)], 1))
    coords = np.concatenate(pts, 0).astype(np.int64)
    feats = rng.random((coords.shape[0], 3), dtype=np.float32)
    return coords, feats


def unet_small():
    torch.manual_seed(11)
    coords, feats = small_cloud(11)
    net = UNetSCN(in_channels=3, m=4, num_planes=4, full_scale=64, backend=scn_cpu).double()
    # non-trivial BN affine parameters
    for name, p in net.named_parameters():
        if p.dim() == 1:
            with torch.no_grad():
                p.add_(0.1 * torch.randn_like(p))
    x = torch.from_numpy(feats).double().requires_grad_(True)
    out = net([torch.from_numpy(coords), x])
    g = torch.randn_like(out)
    params = dict(net.named_parameters())
    grads = torch.autograd.grad(out, [x] + list(params.values()), g)
    blob = {"coords": coords, "feats": feats, "out": out.detach().numpy(), "grad_out": g.numpy(),
            "grad_feats": grads[0].numpy()}
    for (name, p), gr in zip(params.items(), grads[1:]):
        blob["param:" + name] = p.detach().numpy()
        blob["grad:" + name] = gr.numpy()
    for name, b in net.named_buffers():
        blob["buffer_after:" + name] = b.detach().numpy()
    np.savez_compressed(os.path.join(HERE, "unet_small.npz"), **blob)


def structure_small():
    coords, _ = small_cloud(23, n=400, b=3, span=40, origin=100)
    meta = O.Metadata(coords, 4096)
    blob = {"coords": coords, "p2v": meta.p2v, "npts": meta.npts}
    s = 4096
    for lvl in range(4):
        blob[f"coords_l{lvl}"] = meta.coords_at(s)
        blob[f"nbr_l{lvl}"] = meta.nbr(s)
        if lvl < 3:
            parent, off, nc = meta.down(s)
            blob[f"parent_l{lvl}"], blob[f"off_l{lvl}"] = parent, off
            blob[f"child_l{lvl}"] = O.child_table(parent, off, nc)
        s //= 2
    np.savez_compressed(os.path.join(HERE, "structure_small.npz"), **blob)


def augment_from_reference():
    """``augment_ref.npz`` -- produced by the REFERENCE ITSELF: ``augment_and_scale_3d``
    (``lib/utils/augmentation_3d.py:83-158``) is imported and run with a seeded ``numpy.random`` on three synthetic
    sweeps with different settings, followed by the data loader's ``astype(int64)`` + range filter
    (``nuscenes_dataloader.py:323-327``).  The random draws are replayed with ``mm2d3d_b200.augment.draw_augmentation``
    on the same seed (asserted equal to what the reference returned)."""
    from mm2d3d_b200 import synth
    from mm2d3d_b200.augment import draw_augmentation
    spec = importlib.util.spec_from_file_location("ref_aug", "/root/reference/lib/utils/augmentation_3d.py")
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    settings = [
        dict(),                                                                  # validation: no augmentation
        dict(noisy_rot=0.1, flip_x=0.5, rot_z=6.2831, transl=True),              # nuScenes training settings
        dict(noisy_rot=0.1, flip_y=0.5, rot_y=6.2831, transl=True),              # camera-coordinate variant
    ]
    scale, full_scale = 20, 4096
    pts, offs, rots, us, coords, keeps, mins, offsets = [], [0], [], [], [], [], [], []
    for i, kw in enumerate(settings):
        p = synth.raycast_points("nuscenes", seed=40 + i)[::3].copy()
        np.random.seed(100 + i)
        c, min_value, offset, rot = ref.augment_and_scale_3d(p, scale, full_scale, **kw)
        np.random.seed(100 + i)
        rot2, u = draw_augmentation(**kw)
        assert np.array_equal(rot, rot2) and rot.dtype == np.float32
        ci = c.astype(np.int64)
        idxs = (ci.min(1) >= 0) * (ci.max(1) < full_scale)
        pts.append(p); offs.append(offs[-1] + p.shape[0]); rots.append(rot)
        us.append(u if u is not None else np.zeros(3)); coords.append(ci); keeps.append(idxs)
        mins.append(min_value.astype(np.float32)); offsets.append(np.asarray(offset, dtype=np.float64))
    # the same sweeps through a receptive field they do not fit into (no translation): exercises the range filter
    small = 1500
    coords_s, keep_s = [], []
    for i, kw in enumerate(settings):
        kw = dict(kw, transl=False)
        np.random.seed(100 + i)
        c, _, _, rot = ref.augment_and_scale_3d(pts[i], scale, small, **kw)
        assert np.array_equal(rot, rots[i])
        ci = c.astype(np.int64)
        coords_s.append(ci)
        keep_s.append((ci.min(1) >= 0) * (ci.max(1) < small))
    np.savez_compressed(os.path.join(HERE, "augment_ref.npz"), points=np.concatenate(pts), offsets=np.array(offs),
                        small_full_scale=small, coords_small=np.concatenate(coords_s), keep_small=np.concatenate(keep_s),
                        rot=np.stack(rots), u=np.stack(us), transl=np.array([bool(s.get("transl")) for s in settings]),
                        coords=np.concatenate(coords), keep=np.concatenate(keeps), min_value=np.stack(mins),
                        offset=np.stack(offsets), scale=scale, full_scale=full_scale)


REF_3D_DIR = "/root/reference/experiments_USA_SING/rgbd_rgbxyz_sigmoid_for_rgb/3d_net"


def heads_from_reference():
    """``heads_ref.npz``: the RGB mask computed by the reference's own ``Net3DSeg.forward`` (CPU; its sparse backbone is
    replaced by a pass-through that returns the -- already masked -- point features, and the heads by 16-channel-free
    stand-ins), with autograd gradients; and the cross-modal KL term computed by the torch lines of
    ``train.py:157-184``."""
    import torch.nn as nn
    src = open(os.path.join(REF_3D_DIR, "model.py")).read().replace("from .scn_unet import UNetSCN", "UNetSCN = None")
    mod = type(sys)("ref_3d_model")
    exec(compile(src, os.path.join(REF_3D_DIR, "model.py"), "exec"), mod.__dict__)

    class PassThrough(nn.Module):  # stands in for UNetSCN: hands the (masked) features on
        out_channels = 3

        def forward(self, x):
            return x[1]

    mod.UNetSCN = lambda **kw: PassThrough()
    mod.L2G_classifier_3D = lambda c, k: nn.Identity()
    torch.manual_seed(11)
    net = mod.Net3DSeg(num_classes=6, dual_head=True, backbone_3d_kwargs={})
    rng = np.random.default_rng(11)
    feats = torch.from_numpy(rng.random((2000, 3), dtype=np.float32))
    w = net.linear_rgb_mask.weight.detach().clone()
    b = net.linear_rgb_mask.bias.detach().clone()
    x_in = feats.clone()
    _, masked, _ = net({"x": [torch.zeros(2000, 4, dtype=torch.int64), x_in]})   # model.py:44-58
    g = torch.from_numpy(rng.standard_normal((2000, 3)).astype(np.float32))
    net.zero_grad()
    x_leaf = feats.clone().requires_grad_(True)
    m = torch.sigmoid(net.linear_rgb_mask(x_leaf))
    (x_leaf * m).backward(g)                                                      # same ops, out of place, for dx
    # cross-modal loss (train.py:157-184)
    import torch.nn.functional as F
    pred = torch.from_numpy((3 * rng.standard_normal((1500, 6))).astype(np.float32)).requires_grad_(True)
    target = torch.from_numpy((3 * rng.standard_normal((1500, 6))).astype(np.float32))
    loss = F.kl_div(F.log_softmax(pred, dim=1), F.softmax(target.detach(), dim=1), reduction="none").sum(1).mean()
    loss.backward()
    np.savez_compressed(os.path.join(HERE, "heads_ref.npz"), feats=feats.numpy(), w=w.numpy(), b=b.numpy(),
                        masked=masked.detach().numpy(), g=g.numpy(), dx=x_leaf.grad.numpy(),
                        dw=net.linear_rgb_mask.weight.grad.numpy(), db=net.linear_rgb_mask.bias.grad.numpy(),
                        pred=pred.detach().numpy(), target=target.numpy(), loss=loss.detach().numpy(),
                        dpred=pred.grad.numpy())


def heads3d_from_reference():
    """``heads3d_ref.npz``: ``seg_logit`` and ``seg_logit_point`` computed by the reference's own ``Net3DSeg.forward``
    (``3d_net/model.py:44-58``, real ``linear`` and ``L2G_classifier_3D`` heads; its sparse backbone replaced by a
    pass-through that hands on a recorded 16-channel feature tensor), the 3D term of the cross-modal loss by the torch
    lines of ``train.py:174-182``, and the autograd gradients of  sum(seg_logit * g1) + sum(seg_logit_point * g2) +
    lam * loss_3d  with respect to the features and the four head parameters."""
    import torch.nn as nn
    import torch.nn.functional as F
    src = open(os.path.join(REF_3D_DIR, "model.py")).read().replace("from .scn_unet import UNetSCN", "UNetSCN = None")
    mod = type(sys)("ref_3d_model_heads")
    exec(compile(src, os.path.join(REF_3D_DIR, "model.py"), "exec"), mod.__dict__)
    rng = np.random.default_rng(23)
    n, classes = 1777, 6
    feat = torch.from_numpy(rng.standard_normal((n, 16)).astype(np.float32)).requires_grad_(True)

    class PassThrough(nn.Module):  # stands in for UNetSCN: hands on the recorded backbone output
        out_channels = 16

        def forward(self, x):
            return feat

    mod.UNetSCN = lambda **kw: PassThrough()
    torch.manual_seed(23)
    net = mod.Net3DSeg(num_classes=classes, dual_head=True, backbone_3d_kwargs={})
    preds, out_feat, out_aux = net({"x": [torch.zeros(n, 4, dtype=torch.int64), torch.rand(n, 3)]})   # model.py:44-58
    l1, l2 = preds["seg_logit"], out_aux["seg_logit_point"]
    target = torch.from_numpy((2 * rng.standard_normal((n, classes))).astype(np.float32))           # 2D logits
    loss = F.kl_div(F.log_softmax(l2, dim=1), F.softmax(target.detach(), dim=1), reduction="none").sum(1).mean()
    g1 = torch.from_numpy(rng.standard_normal((n, classes)).astype(np.float32))
    g2 = torch.from_numpy(rng.standard_normal((n, classes)).astype(np.float32))
    lam = 0.7
    ((l1 * g1).sum() + (l2 * g2).sum() + lam * loss).backward()
    np.savez_compressed(
        os.path.join(HERE, "heads3d_ref.npz"), feat=feat.detach().numpy(), target=target.numpy(), g1=g1.numpy(), g2=g2.numpy(),
        lam=np.float32(lam), w1=net.linear.weight.detach().numpy(), b1=net.linear.bias.detach().numpy(),
        w2=net.aux.linear_point.weight.detach().numpy(), b2=net.aux.linear_point.bias.detach().numpy(),
        logit1=l1.detach().numpy(), logit2=l2.detach().numpy(), loss=loss.detach().numpy(), d_feat=feat.grad.numpy(),
        d_w1=net.linear.weight.grad.numpy(), d_b1=net.linear.bias.grad.numpy(),
        d_w2=net.aux.linear_point.weight.grad.numpy(), d_b2=net.aux.linear_point.bias.grad.numpy())


def unetscn_tree(in_channels=3, m=16, num_planes=7):
    """``unetscn_tree.json``: SURVEY.md Appendix B's recursion -- level l at ``prefix`` with p = m(l+1) planes holds
    BN-ReLU ``.0.0`` and SMC ``.0.1``; every level but the deepest adds BN-ReLU ``.1.1.0``, Conv 2/2 ``.1.1.1``, the
    next level ``.1.1.2``, BN-ReLU ``.1.1.3``, Deconv 2/2 ``.1.1.4``, then BN-ReLU ``.3.0`` and SMC ``.3.1`` on 2p."""
    tree = []

    def bn(prefix, c):
        tree.extend([f"{prefix}.{k}", [c]] for k in ("weight", "bias", "running_mean", "running_var"))

    def level(prefix, lvl):
        p = m * (lvl + 1)
        bn(f"{prefix}.0.0", p)
        tree.append([f"{prefix}.0.1.weight", [27, 1, p, p]])
        if lvl + 1 < num_planes:
            q = m * (lvl + 2)
            bn(f"{prefix}.1.1.0", p)
            tree.append([f"{prefix}.1.1.1.weight", [8, 1, p, q]])
            level(f"{prefix}.1.1.2", lvl + 1)
            bn(f"{prefix}.1.1.3", q)
            tree.append([f"{prefix}.1.1.4.weight", [8, 1, q, p]])
            bn(f"{prefix}.3.0", 2 * p)
            tree.append([f"{prefix}.3.1.weight", [27, 1, 2 * p, p]])

    tree.append(["layer2.weight", [27, 1, in_channels, m]])
    level("layer3", 0)
    bn("layer4", m)
    with open(os.path.join(HERE, "unetscn_tree.json"), "w") as f:
        json.dump({"in_channels": in_channels, "m": m, "num_planes": num_planes, "state_dict": tree}, f, indent=0)
        f.write("\n")


if __name__ == "__main__":
    only = sys.argv[1] if len(sys.argv) > 1 else None  # e.g. `make_golden.py augment` regenerates one fixture
    if only in (None, "lift"):
        lift_from_reference()
    if only in (None, "unet"):
        unet_small()
    if only in (None, "structure"):
        structure_small()
    if only in (None, "augment"):
        augment_from_reference()
    if only in (None, "heads"):
        heads_from_reference()
    if only in (None, "heads3d"):
        heads3d_from_reference()
    if only in (None, "tree"):
        unetscn_tree()
    for f in sorted(os.listdir(HERE)):
        if f.endswith((".npz", ".json")):
            print(f, os.path.getsize(os.path.join(HERE, f)))
