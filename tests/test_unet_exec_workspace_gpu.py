"""The whole-network executor's backward-workspace query is the exact need, and the backward checks it before it
issues anything: one byte short fails with MM3D_ERR_WORKSPACE and launches no kernel, the queried size runs."""
import pytest
import torch

from mm2d3d_b200 import synth
from tests.test_gpu_parity import DEV, _no_device_error

pytestmark = pytest.mark.gpu

MM3D_ERR_WORKSPACE = 3
TMP_BYTES = 18  # position of tmp_bytes among mm3d_unet_topo_backward's arguments


class _ShortTmp:
    """The executor's library handle with mm3d_unet_topo_backward told `short` bytes less backward workspace than
    the executor queried and allocated (the buffer itself stays full size, so a missing check could not write out of
    bounds); records the return code and the kernels the call launched."""

    def __init__(self, lib, short):
        self._lib, self.short = lib, short
        self.rc = self.launches = None

    def __getattr__(self, name):
        return getattr(self._lib, name)

    def mm3d_unet_topo_backward(self, *args):
        args = list(args)
        args[TMP_BYTES] -= self.short
        n0 = self._lib.mm3d_kernel_launches()
        self.rc = self._lib.mm3d_unet_topo_backward(*args)
        self.launches = self._lib.mm3d_kernel_launches() - n0
        return self.rc


@pytest.mark.parametrize("mode", ["tf32", "tf32x3"])
@pytest.mark.parametrize("reps,res", [(1, False), (2, True)], ids=["reps1-vgg", "reps2-res"])
def test_backward_workspace_query_is_exact(monkeypatch, reps, res, mode):
    import mm2d3d_b200.scn as scn
    from mm2d3d_b200 import _lib, executor
    from mm2d3d_b200.unet import UNetSCN
    torch.manual_seed(3)
    locs, feats = synth.make_batch("nuscenes", batch=1, seed0=11)
    locs[:, :3] //= 8  # a small scan
    coords, feats = torch.from_numpy(locs).to(DEV), torch.from_numpy(feats).to(DEV)
    net = UNetSCN(in_channels=3, block_reps=reps, residual_blocks=res).to(DEV)
    g = torch.randn(coords.shape[0], 16, device=DEV)
    scn.set_conv_mode(mode)
    try:
        for short in (1, 0):
            x = feats.clone().requires_grad_(True)
            out = net([coords, x])
            shim = _ShortTmp(_lib.lib, short)
            with monkeypatch.context() as mp:
                mp.setattr(executor, "lib", shim)
                if short:
                    with pytest.raises(_lib.Mm3dError, match="backward workspace too small"):
                        torch.autograd.grad(out, [x], g)
                else:
                    torch.autograd.grad(out, [x], g)
            torch.cuda.synchronize()
            if short:
                assert shim.rc == MM3D_ERR_WORKSPACE and shim.launches == 0, (shim.rc, shim.launches)
            else:
                assert shim.rc == 0 and shim.launches > 0, (shim.rc, shim.launches)
    finally:
        scn.set_conv_mode("fp32")
    _no_device_error()
