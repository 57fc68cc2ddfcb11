"""Host side of the whole-network executor for every UNetSCN block topology (no GPU needed): the parameter slot walk,
its agreement with the library's slot count, and which networks the executor takes."""
import pytest
import torch

from mm2d3d_b200 import _lib, executor
from mm2d3d_b200.unet import UNetSCN


def _reference_walk(net):
    """The hand-written slot walk of the reference configuration (block_reps = 1, VGG blocks):
    stem.w | per level: pre_bn pre.w [dn_bn dn.w <deeper> up_bn up.w post_bn post.w] | head_bn."""

    def bn(mod):
        return [mod.weight, mod.bias, mod.running_mean, mod.running_var]

    def level(seq):
        mods = list(seq._modules.values())
        out = bn(mods[0][0]) + [mods[0][1].weight]
        if len(mods) > 1:
            branch = list(mods[1][1]._modules.values())  # ConcatTable[Identity, Sequential[BN, Conv, U, BN, Deconv]]
            out += bn(branch[0]) + [branch[1].weight]
            out += level(branch[2])
            out += bn(branch[3]) + [branch[4].weight]
            out += bn(mods[3][0]) + [mods[3][1].weight]
        return out

    return [net.layer2.weight] + level(net.layer3) + bn(net.layer4)


@pytest.mark.parametrize("num_planes", [1, 2, 7])
def test_generic_slot_walk_equals_reference_walk(num_planes):
    net = UNetSCN(in_channels=3, m=16, num_planes=num_planes)
    slots, ref = executor.collect_slots(net), _reference_walk(net)
    assert len(slots) == len(ref) == _lib.lib.mm3d_unet_num_params(num_planes)
    assert all(a is b for a, b in zip(slots, ref))


@pytest.mark.parametrize("residual", [False, True])
@pytest.mark.parametrize("reps", [1, 2, 3])
@pytest.mark.parametrize("num_planes", [1, 2, 4, 7])
def test_slot_count_matches_library_and_network_is_fusable(num_planes, reps, residual):
    from mm2d3d_b200 import scn
    net = UNetSCN(in_channels=3, m=16, block_reps=reps, residual_blocks=residual, num_planes=num_planes)
    slots = executor.collect_slots(net)
    assert len(slots) == _lib.lib.mm3d_unet_topo_num_params(num_planes, reps, int(residual))
    assert executor.fusable(net)
    assert executor.topology(net) == (reps, int(residual))
    # every parameter exactly once, in module-tree (= parameters()) order; the running statistics in between
    params = [s for s in slots if isinstance(s, torch.nn.Parameter)]
    assert len(params) == len(list(net.parameters())) and all(a is b for a, b in zip(params, net.parameters()))
    nins = [m for m in net.modules() if isinstance(m, scn.NetworkInNetwork)]
    assert len(nins) == (num_planes - 1 if residual else 0)  # the first post block of every level but the deepest
    assert _lib.lib.mm3d_unet_topo_scratch_bytes(3, 16, num_planes, reps, int(residual), _lib.MODE_TF32) > 0


def test_reference_entry_points_are_the_reference_topology():
    for L in (1, 4, 7):
        assert _lib.lib.mm3d_unet_num_params(L) == _lib.lib.mm3d_unet_topo_num_params(L, 1, 0)
        for mode in _lib.MODES.values():
            assert _lib.lib.mm3d_unet_scratch_bytes(3, 16, L, mode) == _lib.lib.mm3d_unet_topo_scratch_bytes(3, 16, L, 1, 0, mode)
    assert _lib.lib.mm3d_unet_topo_num_params(7, 0, 0) < 0  # no such topology


def test_executor_rejects_what_it_does_not_implement():
    from mm2d3d_b200 import scn
    net = UNetSCN(in_channels=3, m=16, residual_blocks=True, num_planes=3)
    assert executor.fusable(net)
    nin = next(m for m in net.modules() if isinstance(m, scn.NetworkInNetwork))
    nin.bias = torch.nn.Parameter(torch.zeros(nin.weight.shape[1]))
    assert not executor.fusable(net)
    net = UNetSCN(in_channels=3, m=16, block_reps=2, num_planes=3)
    next(m for m in net.modules() if isinstance(m, scn.BatchNormLeakyReLU)).leakiness = 0.1
    assert not executor.fusable(net)
