"""Host side of serving the branched policy, on CPU: the centre-crop table and the argument checks of the C ABI's branched
serving entry points (they reject before any CUDA call, so fake device addresses are enough)."""
import ctypes as C

import numpy as np
import pytest


def test_center_crop_table_is_augment_tables_identity_row():
    from carla_imitation_learning_b200.data import augment_table, center_crop_table
    t = center_crop_table(6, (288, 320), mean=0.5, std=0.25)
    assert t.dtype == np.float32 and t.shape == augment_table(0, 6, (288, 320)).shape
    assert np.array_equal(t, np.tile(np.array([16, 32, 1, 1, 1, 0.5, 4, 0], np.float32), (6, 1)))
    assert np.array_equal(center_crop_table(2, (256, 256))[:, :2], np.zeros((2, 2), np.float32))
    assert np.array_equal(center_crop_table(1, (257, 259))[0, :2], np.array([0, 1], np.float32))   # odd margins round down
    with pytest.raises(ValueError):
        center_crop_table(1, (255, 300))


def _fake(batch, hbatch, arena=0x10000):
    from carla_imitation_learning_b200 import _lib
    c = _lib.BcCtx()
    c.obs_size, c.n_actions, c.batch = 4, 3, batch
    c.params, c.act[1], c.act[3] = 0x20000, 0x30000, 0x40000
    h = _lib.BcBranched()
    h.n_branches, h.n_out, h.batch = 4, 3, hbatch
    h.command, h.params, h.out = 0x50000, arena, 0x60000
    return c, h


@pytest.mark.parametrize("tail", [0, 1])
def test_branched_serving_arguments_are_rejected_before_any_launch(tail):
    from carla_imitation_learning_b200 import _lib
    _lib.build()
    lib = _lib.lib()
    for (batch, hbatch, arena), words in (((8, 7, 0x10000), "batch"), ((8, 8, 0x10004), "16 B"),
                                          ((65, 65, 0x10000), "64" if tail else None)):
        if words is None:
            continue
        c, h = _fake(batch, hbatch, arena)
        rc = lib.bc_forward_branched_act(C.byref(c), C.byref(h), None, tail, None)
        assert rc == -1, (batch, hbatch, arena)
        assert words in lib.bc_last_error_string().decode()
    c, h = _fake(65, 65)
    assert lib.bc_policy_tail_branched(C.byref(c), C.byref(h), None, None) == -1
    assert "batch" in lib.bc_last_error_string().decode()
    c, h = _fake(8, 8, 0x10004)
    assert lib.bc_policy_tail_branched(C.byref(c), C.byref(h), None, None) == -1
    c, h = _fake(8, 8)
    h.n_branches = 17
    assert lib.bc_policy_tail_branched(C.byref(c), C.byref(h), None, None) == -1
