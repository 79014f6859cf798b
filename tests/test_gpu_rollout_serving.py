"""Closed-loop serving of N independent agents (trainer.RolloutActStep, bc_stage_history) against explicit references.

* The history ring, tick by tick, against the host model of tests/rollout_model.py: every live plane bitwise equal to the
  existing staging kernel's output (bc_stage_gray / bc_stage_gray_tp / bc_stage_augment) for the frame the model assigns it,
  every other plane and the guard planes around the ring still holding their sentinel.
* RolloutActStep's outputs on every tick bitwise equal to the same forward (same path, same kernels) on windows stacked
  explicitly from the host model: conv1 then reads identical bytes in the same non-sliding mode.
* On three ticks, every stage bounded against f64 on the windows the host model gives (the bound of tests/test_gpu_serving.py),
  so a model and a device that agree with each other but are both wrong still fail.
* Captured graphs against an eager run, the centre crop from 288x320 frames, and new weights in the middle of an episode.
Every output is filled with NaN and the actions with -1 before each tick, so an element the kernels failed to write fails.
"""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from tests.rollout_model import RingModel
from tests.test_gpu_batch_edges import _check_forward, _cpu64, _planes_from_tp
from tests.test_gpu_serving import _check_action, _check_conv12, _check_tail

pytestmark = pytest.mark.gpu

NAN = float("nan")
TICKS = 12
SRC_HW = (288, 320)
SENTINEL = {"tp": 0x7FC3, "f32": 0x7FC00123}           # NaN bit patterns no staging kernel writes


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (no CPU fallback exists to run instead)")
    torch.set_num_threads(os.cpu_count() or 1)
    return torch.device("cuda", 0)


def _lib():
    from carla_imitation_learning_b200 import _lib as L
    return L


def _stream():
    from carla_imitation_learning_b200.engine import _stream_ptr
    return _stream_ptr()


def _schedule(N, seed, ticks=TICKS):
    """(reset (N,) bool, reset_all) per tick: every agent at tick 0, single agents mid-run (tick 5), on two consecutive ticks
    (6 and 7) and on the tick the slot wraps (8), reset_all at tick 10, and seeded random resets elsewhere."""
    rng = np.random.default_rng(seed)
    out = []
    for t in range(ticks):
        r = rng.random(N) < 0.1
        if t == 0:
            r[:] = True
        for tt, a in ((5, 1), (6, 2), (7, 2), (8, 3)):
            if t == tt:
                r[a % N] = True
        out.append((r, t == 10))
    return out


def _net(mode, kind, obs=4, seed=7):
    if kind == "single":
        from src.architectures.nets import ConvNet1
        torch.manual_seed(seed)
        return ConvNet1({"obs_size": obs, "n_actions": 9, "precision": mode}).cuda()
    from src.architectures.branched import ConvNet1Branched
    torch.manual_seed(seed)
    return ConvNet1Branched({"obs_size": 4, "n_actions": 3 if kind == "l1" else 9, "n_branches": 4, "branch_loss": kind,
                             "precision": mode}).cuda()


class _Feed:
    """The frames of every tick (seeded, generated on the device) and the planes the EXISTING staging kernels make of them."""

    def __init__(self, dev, rows, tp, src_hw=None, table="none", seed=0):
        self.dev, self.rows, self.tp, self.src_hw, self.table, self.seed = dev, rows, tp, src_hw, table, seed
        self.hw = src_hw or (256, 256)

    def frames(self, t):
        g = torch.Generator(device=self.dev).manual_seed(1000 * self.seed + t)
        return torch.randint(0, 256, (self.rows, *self.hw, 3), generator=g, dtype=torch.uint8, device=self.dev)

    def table_of(self, t):
        from carla_imitation_learning_b200.data import augment_table, center_crop_table
        if self.table == "none":
            return None
        rows = (augment_table(77 * self.seed + t, self.rows, self.hw) if self.table == "augment"
                else center_crop_table(self.rows, self.hw, mean=0.25, std=0.5))
        return torch.from_numpy(rows).to(self.dev)

    def reference(self, fr, table):
        """(rows, TP) bf16 or (rows, 256, 256) f32: bc_stage_gray_tp / bc_stage_gray(BC_F32) / bc_stage_augment."""
        from carla_imitation_learning_b200 import stage_augmented, stage_gray
        if table is not None:
            r = stage_augmented(fr, table, layout="tp" if self.tp else "plain")
            return r.tp if self.tp else r
        if not self.tp:
            return stage_gray(fr)
        L = _lib()
        out = torch.empty((fr.shape[0], L.TP_PLANE_ELEMS), dtype=torch.bfloat16, device=self.dev)
        L.check(L.lib().bc_stage_gray_tp(fr.data_ptr(), out.data_ptr(), None, fr.shape[0], _stream()), "bc_stage_gray_tp")
        return out


def _bits(t):
    return t.view(torch.int16) if t.dtype == torch.bfloat16 else t.view(torch.int32)


def _gather(refs, ids, rows_of, shape_like, fill=None):
    """Planes picked from the per-tick reference planes: out[i] = refs[ids[i]][rows_of[i]] for ids[i] >= 0, else `fill`."""
    out = torch.empty((len(ids), *shape_like.shape[1:]), dtype=shape_like.dtype, device=shape_like.device)
    if fill is not None:
        _bits(out).fill_(fill)
    ids, rows_of = np.asarray(ids), np.asarray(rows_of)
    for u in np.unique(ids[ids >= 0]):
        sel = np.nonzero(ids == u)[0]
        src = refs[int(u)].index_select(0, torch.from_numpy(rows_of[sel]).to(shape_like.device))
        out.index_copy_(0, torch.from_numpy(sel).to(shape_like.device), src)
    return out


# ------------------------------------------------------------------------------- 1. the ring, plane by plane
def _ring_case(dev, N, cams, layout, table, ticks, seed):
    L = _lib()
    tp = layout == "tp"
    feed = _Feed(dev, N * cams, tp, SRC_HW if table != "none" else None, table, seed)
    R, G = N * 8 * cams, 3                                   # ring planes, guard planes on each side
    shape = (R + 2 * G, L.TP_PLANE_ELEMS) if tp else (R + 2 * G, 256, 256)
    buf = torch.empty(shape, dtype=torch.bfloat16 if tp else torch.float32, device=dev)
    _bits(buf).fill_(SENTINEL[layout])
    ring = buf[G:G + R]
    model = RingModel(N, cams)
    refs = {}
    reset_dev = torch.zeros(N, dtype=torch.uint8, device=dev)
    for t, (reset, reset_all) in enumerate(_schedule(N, seed, ticks)):
        fr, tab = feed.frames(t), feed.table_of(t)
        refs[t] = feed.reference(fr, tab)
        reset_dev.copy_(torch.from_numpy(reset.astype(np.uint8)))
        s = model.tick(np.full(N, t), reset, reset_all)
        L.check(L.lib().bc_stage_history(fr.data_ptr(), N, cams, feed.hw[0], feed.hw[1],
                                         None if tab is None else tab.data_ptr(), reset_dev.data_ptr(), int(reset_all),
                                         ring.data_ptr(), s, L.BC_BF16_TP if tp else L.BC_F32, _stream()), "bc_stage_history")
        # the expected ring: plane (a*8 + j)*cams + k holds frame row a*cams + k of the tick the model assigns to slot j
        a, j, k = np.meshgrid(np.arange(N), np.arange(8), np.arange(cams), indexing="ij")
        ids = model.slots[a, j].reshape(-1)
        exp = _gather(refs, ids, (a * cams + k).reshape(-1), buf, fill=SENTINEL[layout])
        torch.cuda.synchronize()
        guards_ok = bool((_bits(buf[:G]) == SENTINEL[layout]).all()) and bool((_bits(buf[G + R:]) == SENTINEL[layout]).all())
        if not (guards_ok and torch.equal(_bits(ring), _bits(exp))):
            bad = (_bits(ring) != _bits(exp)).flatten(1).any(1).nonzero().flatten().tolist()
            pytest.fail(f"{layout} cams={cams} table={table} N={N} tick {t} (slot {s}): guards intact {guards_ok}, "
                        f"{len(bad)} ring planes differ from the model, first {bad[:8]} "
                        f"(agent, slot, camera) {[(p // (8 * cams), (p // cams) % 8, p % cams) for p in bad[:8]]}")
        for u in [u for u in refs if u not in set(model.slots.reshape(-1).tolist())]:
            del refs[u]


@pytest.mark.parametrize("table", ["none", "augment"])
@pytest.mark.parametrize("layout", ["f32", "tp"])
@pytest.mark.parametrize("cams", [1, 3])
def test_ring_holds_what_the_staging_kernels_write(dev, cams, layout, table):
    """12 ticks (three rotations of the 4 tick slots), 5 agents: resets of every agent, of single agents, on consecutive ticks
    and on the tick the slot wraps, and reset_all. Without a table the planes are bc_stage_gray(BC_F32) / bc_stage_gray_tp's,
    with one (288x320 sources, random crop and jitter per frame) bc_stage_augment's, bit for bit."""
    _ring_case(dev, 5, cams, layout, table, TICKS, seed=11 + cams)


def test_ring_addresses_past_32_bits(dev):
    """4096 agents x 3 cameras x 8 slots of Toeplitz-ready planes = 8.5e9 bf16 elements (17 GB): the offsets of the last
    agents do not fit in 32 bits."""
    _ring_case(dev, 4096, 3, "tp", "none", 6, seed=5)
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------- 2. windows equal explicit stacks
def _stacked_forward(net, step, model, s, refs, command):
    """The forward RolloutActStep ran, on the path it chose, on windows stacked explicitly from the host model: (N, obs)
    planes with strides (obs, 1) planes. Returns (out or logits, actions or None) on fresh, poisoned buffers."""
    from carla_imitation_learning_b200 import StagedBatch
    L = _lib()
    eng, N, cams = step.eng, step.batch, step.cams
    obs = 4 * cams
    win = model.window(s)                                                 # (N, 4) ticks, oldest first
    a, f, k = np.meshgrid(np.arange(N), np.arange(4), np.arange(cams), indexing="ij")   # channel = cams * f + k
    like = next(iter(refs.values()))
    stacked = _gather(refs, win[a, f].reshape(-1), (a * cams + k).reshape(-1), like)
    if step.bf16:
        bufs = eng.alloc(N, StagedBatch(stacked, None, obs, cams), None, False)
        bufs.x_tp_strides = (obs * L.TP_PLANE_ELEMS, L.TP_PLANE_ELEMS)
    else:
        bufs = eng.alloc(N, stacked.view(N, obs, 256, 256), None, False)
    if step.branched:
        out = torch.full((N, net.n_actions), NAN, device=eng.device)
        actions = torch.full((N,), -1, dtype=torch.int64, device=eng.device) if net.branch_loss == "ce" else None
        net._serve(bufs, out, actions, command, step.tail)
    else:
        bufs.logits.fill_(NAN)
        out, actions = bufs.logits, torch.full((N,), -1, dtype=torch.int64, device=eng.device)
        c = eng.ctx(bufs)
        L.check(eng.lib.bc_forward_act(C.byref(c), actions.data_ptr(), int(step.tail), _stream()), "bc_forward_act")
    return out, actions, stacked


def _rollout(dev, net, N, seed, src_hw=None, on_tick=None, ticks=TICKS, step=None):
    """Run `ticks` ticks through a RolloutActStep (graph=True: persistent input buffers rewritten in place, so ticks 0-3 run
    eagerly, 4-7 capture and 8-11 replay) and compare every tick with the explicitly stacked forward, bitwise."""
    from carla_imitation_learning_b200.trainer import RolloutActStep
    step = step or RolloutActStep(net, N, src_hw=src_hw)
    cams = step.cams
    feed = _Feed(dev, N * cams, step.bf16, src_hw, "none" if src_hw is None else "center", seed)
    frames = torch.empty((N * cams, *feed.hw, 3), dtype=torch.uint8, device=dev)
    reset_dev = torch.zeros(N, dtype=torch.bool, device=dev)
    command = torch.zeros(N, dtype=torch.int64, device=dev) if step.branched else None
    table = feed.table_of(0)
    model, refs = RingModel(N, cams), {}
    for t, (reset, reset_all) in enumerate(_schedule(N, seed, ticks)):
        if t == 10:
            step.reset_all()
        frames.copy_(feed.frames(t))
        refs[t] = feed.reference(frames, table)
        reset_dev.copy_(torch.from_numpy(reset))
        if command is not None:
            command.copy_((torch.arange(N, device=dev) + t) % net.n_branches)      # alternating, rewritten every tick
        s = model.tick(np.full(N, t), reset, reset_all or t == 0)
        step.out.fill_(NAN)
        if step.actions is not None:
            step.actions.fill_(-1)
        out, actions = step.act(frames, reset_dev, table, command)
        ref_out, ref_actions, stacked = _stacked_forward(net, step, model, s, refs, command)
        torch.cuda.synchronize()
        tag = f"{'bf16' if step.bf16 else 'fp32'} N={N} obs={4 * cams} tick {t} slot {s}"
        assert torch.equal(out, ref_out), f"{tag}: outputs differ from the explicitly stacked windows"
        assert (actions is None) == (ref_actions is None)
        if actions is not None:
            assert torch.equal(actions, ref_actions), f"{tag}: actions differ"
        if on_tick is not None:
            on_tick(t, s, step, stacked)
        for u in [u for u in refs if u not in set(model.slots.reshape(-1).tolist())]:
            del refs[u]
    step.check()
    return step


@pytest.mark.parametrize("kind", ["single", "l1", "ce"])
@pytest.mark.parametrize("N", [1, 2, 7, 8, 9, 64, 65, 300])
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_windows_equal_explicit_stacks(dev, mode, N, kind):
    _rollout(dev, _net(mode, kind), N, seed=N)


@pytest.mark.parametrize("N", [1, 8, 33])
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_stacked_camera_windows_equal_explicit_stacks(dev, mode, N):
    """obs_size 12: three cameras per agent, channel = 3 * frame + camera."""
    step = _rollout(dev, _net(mode, "single", obs=12), N, seed=50 + N)
    assert step.cams == 3


def test_4096_agents_equal_explicit_stacks(dev):
    _rollout(dev, _net("bf16", "single"), 4096, seed=4096, ticks=6)
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------- 3. anchored to f64
@pytest.mark.parametrize("N", [7, 9])
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_rollout_is_exact_on_the_model_windows(dev, mode, N):
    """On ticks 3, 8 and 11 every stage is bounded against f64 on the host model's windows (conv1 on the planes the existing
    staging kernel makes of the frames the model assigns): the tail (N = 7) or the layer chain (N = 9)."""
    net = _net(mode, "single")
    P = {k: _cpu64(v) for k, v in net.state_dict().items()}
    checked = []

    def on_tick(t, s, step, stacked):
        if t not in (3, 8, 11):
            return
        planes = (_planes_from_tp(stacked).double() if step.bf16 else _cpu64(stacked)).reshape(N, 4, 256, 256)
        tag = f"rollout {mode} N={N} tick {t}"
        print(f"\n{tag}")
        # the rollout's own buffers (the stacked forward wrote buffers of its own)
        if step.tail:
            _check_conv12(tag, step.bufs, P, planes, N, step.bf16)
            _check_tail(tag, step.bufs, P, N, 9, step.actions)
        else:
            _check_forward(tag, step.bufs, P, planes, N, 9, step.bf16)
            _check_action(tag, step.actions, step.bufs.logits)
        checked.append(t)

    step = _rollout(dev, net, N, seed=300 + N, on_tick=on_tick)
    assert step.tail == (N <= 8) and checked == [3, 8, 11]


# ------------------------------------------------------------------------------- 4. graphs
@pytest.mark.parametrize("kind", ["single", "ce"])
@pytest.mark.parametrize("N", [8, 65])
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_captured_ticks_equal_eager_ticks(dev, mode, N, kind):
    """16 ticks over two input slots that alternate: every (input slot, tick slot) graph runs eagerly, is captured and is
    replayed twice. reset and command are rewritten in place between replays. Bitwise equal to graph=False on the same
    sequence."""
    from carla_imitation_learning_b200.trainer import RolloutActStep
    net = _net(mode, kind, seed=21)
    steps = [RolloutActStep(net, N), RolloutActStep(net, N, graph=False)]
    slots = [dict(frames=torch.empty((N, 256, 256, 3), dtype=torch.uint8, device=dev),
                  reset=torch.zeros(N, dtype=torch.uint8, device=dev),
                  command=torch.zeros(N, dtype=torch.int64, device=dev) if kind != "single" else None) for _ in range(2)]
    feed = _Feed(dev, N, mode == "bf16", seed=N)
    sched = _schedule(N, 40 + N, 16)
    for t in range(16):
        sl = slots[t % 2]
        sl["frames"].copy_(feed.frames(t))
        sl["reset"].copy_(torch.from_numpy(sched[t][0].astype(np.uint8)))
        if sl["command"] is not None:
            sl["command"].copy_(torch.from_numpy((np.arange(N) * 7 + 3 * t) % 4))
        got = []
        for st in steps:
            st.out.fill_(NAN)
            st.actions.fill_(-1)
            out, actions = st.act(sl["frames"], sl["reset"], None, sl["command"])
            got.append((out.clone(), actions.clone()))
        torch.cuda.synchronize()
        assert torch.equal(got[0][0], got[1][0]) and torch.equal(got[0][1], got[1][1]), (mode, N, kind, t)
    assert len(steps[0]._graphs) == 4 and not steps[1]._graphs
    for st in steps:
        st.check()


# ------------------------------------------------------------------------------- 5. centre crop
@pytest.mark.parametrize("kind", ["single", "l1"])
@pytest.mark.parametrize("N", [8, 65])
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_center_crop_serving_equals_stacked_augmented_planes(dev, mode, N, kind):
    """288x320 frames through data.center_crop_table (the configs[2] policy's serving input): the reference windows are
    stacked from stage_augmented's planes."""
    _rollout(dev, _net(mode, kind, seed=9), N, seed=600 + N, src_hw=SRC_HW)


# ------------------------------------------------------------------------------- 6. new weights mid-episode
@pytest.mark.parametrize("kind", ["single", "l1"])
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_new_weights_mid_episode(dev, mode, kind):
    """load_state_dict between ticks 8 and 9 (ticks 8-11 replay captured graphs): tick 9 onwards uses the new weights (bf16:
    re-packed operand images) on the history staged before the load, bitwise equal to a net built with those weights that
    saw the same frames; tick 8 still ran the old weights."""
    from carla_imitation_learning_b200.trainer import RolloutActStep
    N = 9
    net, other = _net(mode, kind, seed=1), _net(mode, kind, seed=2)
    outs = {"reloaded": {}, "built": {}}

    def recorder(name, load):
        def on_tick(t, s, st, stacked):
            outs[name][t] = st.out.clone()
            if load and t == 8:
                net.load_state_dict(other.state_dict())
        return on_tick

    _rollout(dev, net, N, seed=77, on_tick=recorder("reloaded", True), step=RolloutActStep(net, N))
    _rollout(dev, other, N, seed=77, on_tick=recorder("built", False), step=RolloutActStep(other, N))
    assert not torch.equal(outs["reloaded"][8], outs["built"][8])
    for t in (9, 10, 11):
        assert torch.equal(outs["reloaded"][t], outs["built"][t]), f"tick {t} after the reload differs"
