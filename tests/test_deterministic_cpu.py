"""Deterministic mode without a GPU: the switch, the ABI and the group-by statement the GPU tests compare against."""
import numpy as np
import torch

from mm2d3d_b200 import _lib, scn


def groupby_reference(keys, n_keys):
    """(start [n_keys + 1], entries) of the group-by-key lists: the entries with key k (key < 0 = none) in ascending
    entry index -- a stable argsort of the keys."""
    keys = np.asarray(keys, dtype=np.int64)
    valid = np.nonzero(keys >= 0)[0]
    order = valid[np.argsort(keys[valid], kind="stable")]
    start = np.zeros(n_keys + 1, dtype=np.int64)
    np.cumsum(np.bincount(keys[valid], minlength=n_keys), out=start[1:])
    return start, order


def test_switch_follows_torch_flag_and_overrides():
    prev_torch = torch.are_deterministic_algorithms_enabled()
    prev = scn.get_deterministic()
    try:
        scn.set_deterministic(None)
        torch.use_deterministic_algorithms(True, warn_only=True)
        assert scn.get_deterministic() is True
        torch.use_deterministic_algorithms(False)
        assert scn.get_deterministic() is False
        scn.set_deterministic(True)
        assert scn.get_deterministic() is True
        torch.use_deterministic_algorithms(True, warn_only=True)
        scn.set_deterministic(False)
        assert scn.get_deterministic() is False
    finally:
        torch.use_deterministic_algorithms(prev_torch)
        scn.set_deterministic(None)
    assert scn.get_deterministic() == prev_torch == prev


def test_switch_rejects_other_values():
    import pytest
    with pytest.raises(TypeError):
        scn.set_deterministic(1)
    assert scn.get_deterministic() is torch.are_deterministic_algorithms_enabled()


def test_abi_version_8():
    assert _lib.ABI_VERSION == 8 == _lib.lib.mm3d_abi_version()
    assert _lib.DETERMINISTIC == 0x100


def test_deterministic_workspace_queries():
    lib = _lib.lib
    assert lib.mm3d_point_csr_workspace_bytes(0) > 0
    assert lib.mm3d_point_csr_workspace_bytes(100_000) >= 2 * 4 * 100_000
    i = lib.mm3d_lift_csr_workspace_bytes(8, 225, 400, 30_000, 0)
    b = lib.mm3d_lift_csr_workspace_bytes(8, 225, 400, 30_000, 1)
    assert b > i >= 2 * 4 * 8 * 225 * 400


def test_groupby_reference():
    keys = np.array([3, -1, 0, 3, 1, 0, 3, -1, 1])
    start, ent = groupby_reference(keys, 5)
    assert start.tolist() == [0, 2, 4, 4, 7, 7]
    assert ent.tolist() == [2, 5, 4, 8, 0, 3, 6]
    for k in range(5):
        seg = ent[start[k]:start[k + 1]]
        assert (keys[seg] == k).all() and (np.diff(seg) > 0).all()
