"""Host side of closed-loop serving with per-agent frame histories, on CPU: the ring model against a brute-force per-agent
frame stack, the argument checks of bc_stage_history (they reject before any CUDA call, so fake device addresses are
enough), and RolloutActStep's input checks (they reject before anything is staged or launched)."""
import collections
import ctypes as C
import types

import numpy as np
import pytest
import torch

from tests.rollout_model import RingModel


@pytest.mark.parametrize("cams", [1, 3])
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_ring_model_equals_a_per_agent_frame_stack(cams, seed):
    rng = np.random.default_rng(seed)
    n, ticks = 7, 40
    model = RingModel(n, cams)
    stacks = [collections.deque(maxlen=4) for _ in range(n)]
    for t in range(ticks):
        reset_all = t == 0 or (t == 23)
        reset = rng.random(n) < 0.15
        ids = t * n + np.arange(n)
        s = model.tick(ids, reset, reset_all)
        assert s == t % 4
        win = model.window(s)
        for a in range(n):
            if reset_all or reset[a]:
                stacks[a].extend([ids[a]] * 4)
            else:
                stacks[a].append(ids[a])
            assert list(win[a]) == list(stacks[a]), (t, a)
            # channel cams * f + k of the window is plane (s + 1 + f) * cams + k of the agent's ring: frame f, camera k
            planes = model.window_planes(s, a)
            for f in range(4):
                for k in range(cams):
                    p = planes[cams * f + k]
                    assert p == model.plane(a, s + 1 + f, k)
                    assert model.slots[a, (p // cams) % 8] == stacks[a][f]


def test_stage_history_arguments_are_rejected_before_any_launch():
    from carla_imitation_learning_b200 import _lib
    _lib.build()
    lib = _lib.lib()
    good = dict(rgb=0x10000, n=4, cams=1, hs=256, ws=256, table=None, reset=0x20000, all=0, ring=0x30000, slot=0,
                dt=_lib.BC_BF16_TP)
    cases = [(dict(n=0), "n_agents"), (dict(cams=2), "cams"), (dict(slot=4), "slot"), (dict(slot=-1), "slot"),
             (dict(hs=255, table=0x40000), "smaller"), (dict(ws=200, table=0x40000), "smaller"),
             (dict(hs=288, ws=320), "crop table"), (dict(ring=0x30008), "16 B"), (dict(table=0x40004), "16 B"),
             (dict(dt=_lib.BC_BF16), "BC_F32 or BC_BF16_TP"), (dict(ring=None), "null"), (dict(rgb=0x10001), "4 B"),
             (dict(n=200000, cams=3), "32-bit")]
    for change, words in cases:
        a = {**good, **change}
        rc = lib.bc_stage_history(a["rgb"], a["n"], a["cams"], a["hs"], a["ws"], a["table"], a["reset"], a["all"],
                                  a["ring"], a["slot"], a["dt"], None)
        assert rc == -1, change
        assert words in lib.bc_last_error_string().decode(), (change, lib.bc_last_error_string())


class _NoLaunchEngine:
    """The engine surface RolloutActStep touches at construction, on the CPU; any path that would launch raises."""

    def __init__(self, obs_size):
        self.obs_size, self.n_actions, self.conv_mode, self.device = obs_size, 9, 0, torch.device("cpu")
        self.tail_batch = 8

    def alloc(self, batch, x, y, backward):
        return types.SimpleNamespace(batch=batch, x=x, logits=torch.empty(batch, self.n_actions))

    def ensure_packed(self):
        raise AssertionError("RolloutActStep reached the launch path")

    ctx = ensure_packed


def _fake_net(obs_size, branched):
    eng = _NoLaunchEngine(obs_size)
    net = types.SimpleNamespace(engine=lambda: eng, n_actions=9)
    if branched:
        net._barena = types.SimpleNamespace(is_cuda=True, device=torch.device("cpu"))
        net.tail_batch, net.branch_loss = 8, "ce"
    return net


def _step(obs_size=4, branched=False, n=3, src_hw=None):
    from carla_imitation_learning_b200.trainer import RolloutActStep
    return RolloutActStep(_fake_net(obs_size, branched), n, src_hw=src_hw)


def test_branched_rollout_refuses_stacked_cameras():
    with pytest.raises(ValueError, match="obs_size must be 4"):
        _step(12, True)


def test_rollout_refuses_bad_construction():
    with pytest.raises(ValueError, match="at least 1"):
        _step(n=0)
    with pytest.raises(ValueError, match="smaller"):
        _step(src_hw=(255, 320))


def _good(n, cams, hw=(256, 256), table=False):
    fr = torch.zeros((n * cams, *hw, 3), dtype=torch.uint8)
    return fr, torch.zeros(n, dtype=torch.bool), (torch.zeros((n * cams, 8)) if table else None)


@pytest.mark.parametrize("obs_size", [4, 12])
def test_rollout_rejects_bad_inputs_before_any_launch(obs_size):
    n, cams = 3, obs_size // 4
    st = _step(obs_size, n=n)
    fr, reset, _ = _good(n, cams)
    bad = [
        (dict(frames=fr[:-1]), "frames"),
        (dict(frames=torch.zeros((n * cams, 256, 256, 3), dtype=torch.int16)), "frames"),
        (dict(frames=torch.zeros((n * cams, 256, 257, 3), dtype=torch.uint8)), "frames"),
        (dict(frames=torch.zeros((n * cams, 3, 256, 256), dtype=torch.uint8).permute(0, 2, 3, 1)), "frames"),
        (dict(frames=fr.numpy()), "frames"),
        (dict(reset=torch.zeros(n + 1, dtype=torch.bool)), "reset"),
        (dict(reset=torch.zeros(n, dtype=torch.int64)), "reset"),
        (dict(reset=torch.zeros((n, 1), dtype=torch.uint8)), "reset"),
        (dict(reset=None), "reset"),
        (dict(table=torch.zeros((n * cams, 8))), "table must be None"),
        (dict(command=torch.zeros(n, dtype=torch.int64)), "takes no command"),
    ]
    for change, words in bad:
        a = dict(frames=fr, reset=reset, table=None, command=None, **{})
        a.update(change)
        with pytest.raises(ValueError, match=words):
            st.act(a["frames"], a["reset"], a["table"], a["command"])
    assert st._tick == 0 and not st._seen


def test_rollout_rejects_bad_table_and_command_before_any_launch():
    n = 3
    st = _step(4, True, n=n, src_hw=(288, 320))
    fr, reset, table = _good(n, 1, (288, 320), table=True)
    cmd = torch.zeros(n, dtype=torch.int64)
    bad = [
        (dict(table=None), "table"),
        (dict(table=table[:-1]), "table"),
        (dict(table=table.double()), "table"),
        (dict(table=torch.zeros((n, 16))[:, ::2]), "table"),
        (dict(frames=torch.zeros((n, 256, 256, 3), dtype=torch.uint8)), "frames"),
        (dict(command=None), "command"),
        (dict(command=cmd.int()), "command"),
        (dict(command=torch.zeros(n + 1, dtype=torch.int64)), "command"),
        (dict(command=torch.zeros((n, 2), dtype=torch.int64)[:, 0]), "command"),
    ]
    for change, words in bad:
        a = dict(frames=fr, reset=reset, table=table, command=cmd)
        a.update(change)
        with pytest.raises(ValueError, match=words):
            st.act(a["frames"], a["reset"], a["table"], a["command"])
    assert st._tick == 0 and not st._seen
