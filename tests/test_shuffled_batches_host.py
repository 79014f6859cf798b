"""Host side of shuffled minibatches, on CPU: valid_starts on episode layouts, the per-epoch permutation and its rank shards
(ShuffledFrames' order is a host numpy PCG64 permutation, so it is checked without a device), the datamodule keys, and the
argument checks of bc_stage_gather (they reject before any CUDA call, so fake device addresses are enough)."""
import types

import numpy as np
import pytest


def test_valid_starts_on_episode_layouts():
    from carla_imitation_learning_b200.data import valid_starts
    assert valid_starts([10]).tolist() == list(range(6))
    assert valid_starts([5, 5]).tolist() == [0, 5]
    assert valid_starts([4, 6, 0, 3, 7]).tolist() == [4, 5, 13, 14, 15]        # 4, 0 and 3 frames hold no sample
    assert valid_starts([]).size == 0 and valid_starts([2, 4]).size == 0
    assert valid_starts([9, 8], frame_skip=2).tolist() == list(range(7)) + list(range(9, 15))
    rng = np.random.default_rng(0)
    for _ in range(20):
        lengths = rng.integers(0, 40, size=rng.integers(1, 12))
        got = valid_starts(lengths)
        # brute force: window [i, i+4) and label frame i+4 inside one episode
        ep = np.repeat(np.arange(len(lengths)), lengths)
        want = [i for i in range(len(ep) - 4) if ep[i] == ep[i + 4]]
        assert got.dtype == np.int64 and got.tolist() == want
    with pytest.raises(ValueError, match="non-negative"):
        valid_starts([3, -1])


def _shuffled(n_samples, batch, seed=0, starts=None, rank=0, world=1):
    """A ShuffledFrames' order methods without a device: they read only starts, seed, rank, world and batch_size."""
    from carla_imitation_learning_b200.data import ShuffledFrames
    sf = ShuffledFrames.__new__(ShuffledFrames)
    sf.starts = np.arange(n_samples, dtype=np.int64) if starts is None else np.asarray(starts, np.int64)
    sf.seed, sf.rank, sf.world, sf.batch_size, sf.epoch = seed, rank, world, batch, 0
    return sf


@pytest.mark.parametrize("n", [1, 7, 256, 1001])
def test_each_epoch_covers_every_start_once_and_is_deterministic(n):
    sf = _shuffled(n, 64, seed=3)
    perms = [sf.permutation(e) for e in range(4)]
    for p in perms:
        assert sorted(p.tolist()) == list(range(n))
    assert all(np.array_equal(sf.permutation(e), perms[e]) for e in range(4))
    assert np.array_equal(_shuffled(n, 64, seed=3).permutation(2), perms[2])
    if n > 6:
        assert not np.array_equal(perms[0], perms[1]) and not np.array_equal(perms[1], perms[2])
        assert not np.array_equal(_shuffled(n, 64, seed=4).permutation(0), perms[0])
    # the epoch seeds numpy PCG64(seed + epoch): reproducible anywhere
    assert np.array_equal(perms[1], np.random.Generator(np.random.PCG64(4)).permutation(n))


def test_permutation_draws_from_the_given_starts():
    from carla_imitation_learning_b200.data import valid_starts
    starts = valid_starts([30, 3, 50, 12])
    sf = _shuffled(0, 16, seed=9, starts=starts)
    for e in range(3):
        p = sf.permutation(e)
        assert sorted(p.tolist()) == starts.tolist()


@pytest.mark.parametrize("world", [1, 2, 3, 8])
@pytest.mark.parametrize("n", [5, 64, 1000])
def test_rank_shards_are_disjoint_and_cover_the_epoch(world, n):
    B = 16
    shards = [_shuffled(n, B, seed=1, rank=r, world=world) for r in range(world)]
    for e in range(3):
        parts = [s.shard(e) for s in shards]
        joined = np.concatenate(parts)
        assert len(joined) == n and sorted(joined.tolist()) == list(range(n))
        assert max(len(p) for p in parts) - min(len(p) for p in parts) <= 1
        assert np.array_equal(joined[np.argsort(np.concatenate([np.arange(r, n, world) for r in range(world)]))],
                              shards[0].permutation(e))
    for s in shards:
        assert len(s) == (len(s.shard(0)) + B - 1) // B     # batches per epoch; the last one may be short


def test_datamodule_shuffle_keys_parse():
    from carla_imitation_learning_b200.config import compose
    from carla_imitation_learning_b200.data import _datamodule_key
    hp = compose("config", overrides=["model=imitation"])
    assert hp.datamodule.shuffle is False and hp.datamodule.shuffle_seed == 0
    assert _datamodule_key(hp, "shuffle", None) is False and _datamodule_key(hp, "shuffle_seed", None) == 0
    hp.datamodule["shuffle"], hp.datamodule["shuffle_seed"] = True, 7
    assert _datamodule_key(hp, "shuffle", False) is True and _datamodule_key(hp, "shuffle_seed", 0) == 7
    assert _datamodule_key({"shuffle": True}, "shuffle", False) is True                 # flat hparams, as the modules pass
    assert _datamodule_key({"BATCH_SIZE": 8}, "shuffle", False) is False


def test_stage_gather_arguments_are_rejected_before_any_launch():
    from carla_imitation_learning_b200 import _lib
    _lib.build()
    lib = _lib.lib()
    good_store = dict(frames=0x10000, n_frames=100, cams=1, src_h=256, src_w=256, labels=0x20000, commands=None,
                      targets=None, n_out=0)
    good = dict(index=0x30000, batch=8, table=None, out=0x40000, dt=_lib.BC_BF16_TP, y=0x50000, command=None, target=None,
                err=0x60000)
    cases = [(dict(frames=None), {}, "null"), ({}, dict(index=None), "null"), ({}, dict(out=None), "null"),
             ({}, dict(err=None), "null"), ({}, dict(batch=0), "batch"), (dict(cams=2), {}, "cams"),
             (dict(n_frames=4), {}, "n_frames"), (dict(src_h=255), dict(table=0x70000), "smaller"),
             (dict(src_w=200), dict(table=0x70000), "smaller"), (dict(src_h=288, src_w=320), {}, "crop table"),
             ({}, dict(out=0x40008), "16 B"), ({}, dict(table=0x70004), "16 B"), ({}, dict(dt=_lib.BC_BF16), "BC_F32 or BC_BF16_TP"),
             ({}, dict(index=0x30004), "8 B"), (dict(frames=0x10001), {}, "4 B"),
             (dict(targets=0x80000, n_out=0), dict(target=0x90000), "n_out"),
             (dict(cams=3), dict(batch=200000), "32-bit")]
    for s_change, a_change, words in cases:
        s, a = {**good_store, **s_change}, {**good, **a_change}
        st = _lib.BcFrameStore(s["frames"], s["n_frames"], s["cams"], s["src_h"], s["src_w"], s["labels"], s["commands"],
                               s["targets"], s["n_out"])
        rc = lib.bc_stage_gather(st, a["index"], a["batch"], a["table"], a["out"], a["dt"], a["y"], a["command"],
                                 a["target"], a["err"], None)
        assert rc == -1, (s_change, a_change)
        assert words in lib.bc_last_error_string().decode(), (s_change, a_change, lib.bc_last_error_string())
    assert lib.bc_stage_gather(None, 0x30000, 8, None, 0x40000, _lib.BC_F32, None, None, None, 0x60000, None) == -1


def test_step_gather_rejects_bad_inputs_before_any_launch():
    """TrainStep.step_gather's checks run before the engine is touched: a fake step whose engine raises on any use."""
    import torch
    from carla_imitation_learning_b200.trainer import TrainStep

    class _NoLaunch:
        obs_size, device, conv_mode = 4, torch.device("cpu"), 0

        def ensure_packed(self):
            raise AssertionError("step_gather reached the launch path")

    st = TrainStep.__new__(TrainStep)
    st.eng, st.batch, st.bf16 = _NoLaunch(), 4, False
    store = types.SimpleNamespace(struct=object(), device=torch.device("cpu"), cams=1, src_hw=(256, 256), labels=object())
    idx = torch.zeros(4, dtype=torch.int64)
    bad = [(dict(store=types.SimpleNamespace(device=torch.device("cpu"))), "FrameStore"),
           (dict(store=types.SimpleNamespace(**{**store.__dict__, "cams": 3})), "camera"),
           (dict(store=types.SimpleNamespace(**{**store.__dict__, "src_hw": (288, 320)})), "stages"),
           (dict(store=types.SimpleNamespace(**{**store.__dict__, "labels": None})), "labels"),
           (dict(index=torch.zeros(5, dtype=torch.int64)), "index"), (dict(index=idx.int()), "index"),
           (dict(index=torch.zeros((4, 2), dtype=torch.int64)[:, 0]), "index"), (dict(index=idx.numpy()), "index")]
    for change, words in bad:
        a = dict(store=store, index=idx)
        a.update(change)
        with pytest.raises(ValueError, match=words):
            st.step_gather(a["store"], a["index"])


def test_gather_graph_key_names_every_field_of_the_store():
    """A captured step_gather graph holds the whole bc_frame_store by value: two stores over the same frames that differ in
    any field (labels, commands, targets, size) must not share a graph."""
    import types
    from carla_imitation_learning_b200 import _lib
    from carla_imitation_learning_b200.trainer import _GatherInput
    base = dict(frames=0x10000, n_frames=100, cams=1, src_h=256, src_w=256, labels=0x20000, commands=None, targets=None, n_out=0)
    idx = types.SimpleNamespace(data_ptr=lambda: 0x30000)
    tab = types.SimpleNamespace(data_ptr=lambda: 0x40000)

    def key(table=None, **change):
        f = {**base, **change}
        st = _lib.BcFrameStore(f["frames"], f["n_frames"], f["cams"], f["src_h"], f["src_w"], f["labels"], f["commands"],
                               f["targets"], f["n_out"])
        return _GatherInput.gather_key(types.SimpleNamespace(struct=st), idx, table)

    k0 = key()
    assert key() == k0
    for change in (dict(labels=0x20100), dict(labels=None), dict(commands=0x50000), dict(targets=0x60000, n_out=3),
                   dict(n_frames=99), dict(cams=3), dict(src_h=288, src_w=320), dict(frames=0x10100)):
        assert key(**change) != k0, change
    assert key(table=tab) != k0
