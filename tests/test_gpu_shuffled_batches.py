"""Shuffled minibatches from a device-resident frame store (bc_stage_gather, data.FrameStore / ShuffledFrames,
TrainStep.step_gather, BranchedTrainStep.step_gather): every gathered plane bitwise what the existing staging kernels write
for the explicitly gathered frames, the side data of frame i+4, invalid indices, a store larger than 2^32 bytes, and the
training steps and the module path bitwise equal to the same engine on explicitly staged batches (and to the f64 oracle on
sequential_samples(...)[index] within the usual tolerances)."""
import os

import numpy as np
import pytest
import torch

from oracle import bc_oracle as O

pytestmark = pytest.mark.gpu

TP = 86688
REL_F32, REL_BF16 = 1e-5, 2e-2


def _dev():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (no CPU fallback exists to run instead)")
    return torch.device("cuda", 0)


def _rel(got, ref):
    got, ref = got.detach().double().cpu(), ref.detach().double().cpu()
    return float((got - ref).abs().max() / ref.abs().max().clamp_min(1e-30))


def _store(n_frames, cams=1, hw=(256, 256), seed=0, n_actions=9, G=4, n_out=3):
    from carla_imitation_learning_b200.data import FrameStore
    g = torch.Generator().manual_seed(seed)
    frames = torch.randint(0, 256, (n_frames * cams, hw[0], hw[1], 3), generator=g, dtype=torch.uint8)
    labels = torch.randint(0, n_actions, (n_frames,), generator=g)
    commands = torch.randint(0, G, (n_frames,), generator=g)
    targets = torch.rand((n_frames, n_out), generator=g) * 2 - 1
    return FrameStore(frames.to(_dev()), labels, commands, targets, cams=cams)


def _rows(store, index):
    """Store rows of the explicitly gathered window frames, plane order b*4*cams + cams*j + k."""
    c = store.cams
    return torch.tensor([(int(i) + j) * c + k for i in index for j in range(4) for k in range(c)], dtype=torch.int64,
                        device=store.device)


def _indices(n_frames, B, seed):
    """B sample ids with 0, n_frames - 5 and repeated ones among them."""
    rng = np.random.default_rng(seed)
    idx = rng.integers(0, n_frames - 4, size=B)
    idx[0] = 0
    if B > 1:
        idx[-1] = n_frames - 5
    if B > 4:
        idx[2] = idx[3] = idx[1]
    return idx


def _explicit(store, index, layout, table_rows=None):
    """The same batch staged the existing way: the window frames gathered by a torch index op, then bc_stage_gray(_tp) or
    bc_stage_augment with each sample's table row repeated over its 4 frames."""
    from carla_imitation_learning_b200 import _lib
    from carla_imitation_learning_b200.engine import _stream_ptr, stage_augmented, stage_gray
    fr = store.frames.index_select(0, _rows(store, index)).contiguous()
    n, c = fr.shape[0], store.cams
    if table_rows is not None:
        rep = table_rows.view(len(index), 1, c, 8).expand(len(index), 4, c, 8).reshape(n, 8).contiguous()
        out = stage_augmented(fr, rep, layout="tp" if layout == "tp" else "plain")
        return out.tp if layout == "tp" else out.view(len(index), 4 * c, 256, 256)
    if layout == "tp":
        tp = torch.empty((n, TP), dtype=torch.bfloat16, device=fr.device)
        _lib.check(_lib.lib().bc_stage_gray_tp(fr.data_ptr(), tp.data_ptr(), None, n, _stream_ptr()), "bc_stage_gray_tp")
        return tp
    return stage_gray(fr).view(len(index), 4 * c, 256, 256)


def _guarded_out(layout, B, cams, guard=3):
    """Output buffer with `guard` planes of a fill pattern on both sides; returns (whole buffer, the destination)."""
    from carla_imitation_learning_b200.engine import StagedBatch
    dev, n = _dev(), B * 4 * cams
    if layout == "tp":
        whole = torch.full((n + 2 * guard, TP), 7.0, dtype=torch.bfloat16, device=dev)
        return whole, StagedBatch(whole[guard:guard + n], None, 4 * cams, 4 * cams)
    whole = torch.full((n + 2 * guard, 256, 256), -3.0, dtype=torch.float32, device=dev)
    return whole, whole[guard:guard + n].view(B, 4 * cams, 256, 256)


def _bits(t):
    t = t.tp if hasattr(t, "tp") else t
    return t.contiguous().view(torch.int16 if t.dtype == torch.bfloat16 else torch.int32)


# ------------------------------------------------------------------------------------------------ staging, bitwise
@pytest.mark.parametrize("cams", [1, 3])
@pytest.mark.parametrize("layout", ["plain", "tp"])
@pytest.mark.parametrize("aug", [False, True])
def test_gathered_planes_are_bitwise_the_existing_staging(cams, layout, aug):
    from carla_imitation_learning_b200.data import augment_table
    from carla_imitation_learning_b200.engine import stage_gather
    hw = (288, 320) if aug else (256, 256)
    store = _store(40, cams, hw, seed=cams)
    guard = 3
    for B in (1, 7, 256, 300):
        index = _indices(store.n_frames, B, B)
        idx = torch.from_numpy(index).to(store.device)
        table = torch.from_numpy(augment_table(B, B * cams, hw)).to(store.device) if aug else None
        whole, out = _guarded_out(layout, B, cams, guard)
        got = stage_gather(store, idx, layout, out=out, table=table)
        assert got is out
        ref = _explicit(store, index, layout, table)
        torch.cuda.synchronize()
        assert torch.equal(_bits(got), _bits(ref)), (B, cams, layout, aug)
        fill = 7.0 if layout == "tp" else -3.0
        assert bool((whole[:guard] == fill).all()) and bool((whole[-guard:] == fill).all()), "a guard plane was written"
    store.check()


def test_side_data_is_that_of_frame_i_plus_4():
    from carla_imitation_learning_b200.engine import stage_gather
    store = _store(60, 1, seed=5)
    B = 37
    index = _indices(store.n_frames, B, 1)
    idx = torch.from_numpy(index).to(store.device)
    y = torch.full((B,), -9, dtype=torch.int64, device=store.device)
    cmd, tgt = torch.full_like(y, -9), torch.full((B, 3), 5.0, device=store.device)
    stage_gather(store, idx, "tp", y=y, command=cmd, target=tgt)
    i4 = idx + 4
    assert torch.equal(y, store.labels[i4]) and torch.equal(cmd, store.commands[i4]) and torch.equal(tgt, store.targets[i4])
    store.check()


def test_invalid_indices_raise_flag_5_and_zero_only_their_samples():
    from carla_imitation_learning_b200.engine import stage_gather
    for layout in ("plain", "tp"):
        store = _store(30, 1, seed=2)
        n = store.n_frames
        index = np.array([3, -1, 0, n - 4, 7, 2 ** 40, n - 5], dtype=np.int64)
        bad = np.array([False, True, False, True, False, True, False])
        B = len(index)
        idx = torch.from_numpy(index).to(store.device)
        y, cmd = torch.full((B,), -9, dtype=torch.int64, device=store.device), torch.full((B,), -9, dtype=torch.int64, device=store.device)
        tgt = torch.full((B, 3), 5.0, device=store.device)
        got = stage_gather(store, idx, layout, y=y, command=cmd, target=tgt)
        with pytest.raises(RuntimeError, match="sample index"):
            store.check()
        store.check()                                        # the flag was cleared
        planes = _bits(got).view(B, 4, -1)
        ok = np.flatnonzero(~bad)
        ref = _explicit(store, index[ok], layout)
        assert torch.equal(planes[torch.from_numpy(ok)], _bits(ref).view(len(ok), 4, -1))
        assert not bool(planes[torch.from_numpy(np.flatnonzero(bad))].any())
        okd = torch.from_numpy(ok).to(store.device)
        badd = torch.from_numpy(np.flatnonzero(bad)).to(store.device)
        assert torch.equal(y[okd], store.labels[idx[okd] + 4]) and not bool(y[badd].any())
        assert torch.equal(cmd[okd], store.commands[idx[okd] + 4]) and not bool(cmd[badd].any())
        assert torch.equal(tgt[okd], store.targets[idx[okd] + 4]) and not bool(tgt[badd].any())
        del store


def test_store_larger_than_4_gib_with_indices_near_its_end():
    """22,000 frames of 256x256 RGB = 4.33e9 bytes: sample offsets past 2^32 bytes."""
    from carla_imitation_learning_b200.data import FrameStore
    from carla_imitation_learning_b200.engine import stage_gather
    dev = _dev()
    n = 22000
    frames = torch.empty((n, 256, 256, 3), dtype=torch.uint8, device=dev)
    g = torch.Generator(device=dev).manual_seed(7)
    for lo in range(0, n, 2000):
        frames[lo:lo + 2000] = torch.randint(0, 256, (min(2000, n - lo), 256, 256, 3), generator=g, dtype=torch.uint8, device=dev)
    labels = torch.arange(n, dtype=torch.int64, device=dev) % 9
    store = FrameStore(frames, labels)
    assert store.frames.data_ptr() == frames.data_ptr() and frames.numel() > 2 ** 32
    index = np.array([n - 5, n - 6, 0, 21900, 2 ** 32 // (256 * 256 * 3) - 2, n - 5], dtype=np.int64)
    idx = torch.from_numpy(index).to(dev)
    for layout in ("plain", "tp"):
        y = torch.empty(len(index), dtype=torch.int64, device=dev)
        got = stage_gather(store, idx, layout, y=y)
        ref = _explicit(store, index, layout)
        assert torch.equal(_bits(got), _bits(ref)), layout
        assert torch.equal(y, labels[idx + 4])
    store.check()


def test_invalid_index_does_not_mask_an_earlier_error_code():
    from carla_imitation_learning_b200.engine import stage_gather
    store = _store(30, 1, seed=4)
    store.err_flag.fill_(3)
    stage_gather(store, torch.tensor([-1, 2], dtype=torch.int64, device=store.device), "tp")
    assert int(store.err_flag.item()) == 3
    store.err_flag.zero_()


# ------------------------------------------------------------------------------------------------ single-head training
def _net(obs=4, precision="bf16", seed=12345):
    from src.architectures.nets import ConvNet1
    torch.manual_seed(seed)
    return ConvNet1({"obs_size": obs, "n_actions": 9, "precision": precision}).to(_dev())


def _explicit_step(ts, store, index):
    """The same training step on the explicitly gathered and staged batch: the existing staging kernels write the step's
    gather buffer, the labels come from a torch index, then the step's own enqueue runs eagerly."""
    ts.eng.ensure_packed()
    ts._point(True)
    x = ts._gather_x()
    ref = _explicit(store, index, "tp" if ts.bf16 else "plain")
    (x.tp if ts.bf16 else x).copy_(ref)
    ts.bufs.y = store.labels[torch.from_numpy(np.asarray(index) + 4).to(store.device)].contiguous()
    ts._train()
    return ts.bufs.loss


@pytest.mark.parametrize("obs,precision", [(4, "bf16"), (4, "fp32"), (12, "bf16")])
def test_step_gather_graph_replays_equal_the_explicit_path_bitwise(obs, precision):
    """Graph-replayed step_gather over two rotating index slots, one slot rewritten in place between replays, against the
    same engine driven eagerly on the explicitly gathered and staged batches: losses, parameters and Adam moments bitwise;
    a captured run equals an eager (graph=False) run too."""
    from carla_imitation_learning_b200 import FusedAdam
    from carla_imitation_learning_b200.trainer import TrainStep
    B, steps = 256 if precision == "bf16" else 32, 7
    store = _store(600, obs // 4, seed=obs)
    rng = np.random.default_rng(0)
    plan = [rng.integers(0, store.n_frames - 4, size=B) for _ in range(steps)]
    runs = {}
    for mode in ("graph", "eager", "explicit"):
        net = _net(obs, precision)
        opt = FusedAdam(list(net.parameters()), lr=1e-3)
        ts = TrainStep(net, opt, B, graph=(mode == "graph"))
        slots = [torch.zeros(B, dtype=torch.int64, device=store.device) for _ in range(2)]
        losses = []
        for s in range(steps):
            if mode == "explicit":
                losses.append(_explicit_step(ts, store, plan[s]).clone())
            else:
                slots[s % 2].copy_(torch.from_numpy(plan[s]))        # rewritten in place: the graph follows the contents
                losses.append(ts.step_gather(store, slots[s % 2]).clone())
        torch.cuda.synchronize()
        ts.check()
        if mode == "graph":
            assert len(ts._graphs) == 2
        runs[mode] = (torch.stack(losses).cpu(), net._arena.detach().clone(), [t.clone() for t in opt._bind()[1:3]])
    for mode in ("eager", "explicit"):
        assert torch.equal(runs["graph"][0], runs[mode][0]), (mode, runs["graph"][0], runs[mode][0])
        assert torch.equal(runs["graph"][1], runs[mode][1]), mode
        for a, b in zip(runs["graph"][2], runs[mode][2]):
            assert torch.equal(a, b), mode


def test_step_gather_then_step_keeps_the_sequential_path():
    """step() after step_gather() trains on the sequential window again (the step's buffers are re-pointed): alternating
    step_gather and step equals alternating the explicit gathered path and step, bitwise."""
    from carla_imitation_learning_b200 import FusedAdam
    from carla_imitation_learning_b200.trainer import TrainStep
    B = 64
    store = _store(300, 1, seed=9)
    idx = torch.from_numpy(_indices(store.n_frames, B, 4)).to(store.device)
    frames = store.frames[:B + 4].contiguous()
    labels = store.labels[4:B + 4].contiguous()
    out = []
    for explicit in (False, True):
        net = _net()
        opt = FusedAdam(list(net.parameters()), lr=1e-3)
        ts = TrainStep(net, opt, B, graph=False)
        for _ in range(2):
            if explicit:
                _explicit_step(ts, store, idx.cpu().numpy())
            else:
                ts.step_gather(store, idx)
            ts.step(frames, labels)
        torch.cuda.synchronize()
        out.append(net._arena.detach().clone())
    assert torch.equal(out[0], out[1])


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_step_gather_gradients_match_the_oracle_on_the_indexed_samples(precision):
    """One step_gather: loss and all 14 gradients against the f64 oracle on sequential_samples(frames, labels)[index],
    given the device's pool routing (and, in bf16 mode, its ReLU masks): rel 1e-5 (fp32), 2e-2 (bf16)."""
    from carla_imitation_learning_b200 import FusedAdam
    from carla_imitation_learning_b200.data import FrameStore
    from carla_imitation_learning_b200.trainer import TrainStep
    dev = _dev()
    B = 16
    frames, labels = O.synth_frames(3, 80)
    store = FrameStore(frames, labels)
    index = _indices(store.n_frames, B, 11)
    net = _net(4, precision)
    P = {k: v.detach().cpu().clone() for k, v in net.state_dict().items()}
    ts = TrainStep(net, FusedAdam(list(net.parameters()), lr=1e-3), B, graph=False)
    loss = float(ts.step_gather(store, torch.from_numpy(index).to(dev)))
    torch.cuda.synchronize()
    ts.check()
    bufs, eng = ts.bufs, ts.eng
    got = {k: eng.grads[p._bc_offset:p._bc_offset + p.numel()].view(p.shape).cpu() for k, p in net.named_parameters()}
    x, y = O.sequential_samples(frames, labels)
    xb, yb = torch.from_numpy(x[index]), torch.from_numpy(y[index])
    assert torch.equal(bufs.y.cpu(), yb)
    amax = [a.cpu().long() for a in bufs.amax]
    relu = ({"pooled": [a.cpu() > 0 for a in bufs.act], "fc": [bufs.hid1.cpu() > 0, bufs.hid2.cpu() > 0]}
            if precision == "bf16" else None)
    torch.set_num_threads(os.cpu_count() or 1)
    ref_loss, _lg, ref, _ = O.explicit_backward(P, xb, yb, dtype=torch.float64, argmax_override=amax, relu_override=relu)
    tol = REL_BF16 if precision == "bf16" else REL_F32
    assert abs(loss - float(ref_loss)) <= tol * float(ref_loss), (loss, float(ref_loss))
    worst = {k: _rel(got[k], ref[k]) for k in O.PARAM_ORDER}
    assert max(worst.values()) <= tol, worst


def test_step_gather_graphs_follow_the_store_not_only_its_frames():
    """Two stores over the SAME device frames with different labels: after the first store's graph is captured and
    replayed, a step on the second store trains on the second store's labels (its own graph), equal to the explicit path."""
    from carla_imitation_learning_b200 import FusedAdam
    from carla_imitation_learning_b200.data import FrameStore
    from carla_imitation_learning_b200.trainer import TrainStep
    B = 64
    base = _store(200, 1, seed=12)
    other = (base.labels + 1) % 9
    a, b = FrameStore(base.frames, base.labels), FrameStore(base.frames, other)
    assert a.frames.data_ptr() == b.frames.data_ptr()
    index = _indices(base.n_frames, B, 6)
    idx = torch.from_numpy(index).to(base.device)
    arenas = []
    for explicit in (False, True):
        net = _net()
        ts = TrainStep(net, FusedAdam(list(net.parameters()), lr=1e-3), B, graph=not explicit)
        losses = []
        for store in (a, a, a, b, b, b, a):
            if explicit:
                losses.append(_explicit_step(ts, store, index).clone())
            else:
                losses.append(ts.step_gather(store, idx).clone())
                assert torch.equal(ts.bufs.y, store.labels[idx + 4])
        torch.cuda.synchronize()
        if not explicit:
            assert len(ts._graphs) == 2
        arenas.append((torch.stack(losses).cpu(), net._arena.detach().clone()))
    assert torch.equal(arenas[0][0], arenas[1][0]) and torch.equal(arenas[0][1], arenas[1][1])


def test_branched_step_gather_graphs_follow_the_store_targets():
    from carla_imitation_learning_b200.data import FrameStore
    from carla_imitation_learning_b200.trainer import BranchedTrainStep
    from src.architectures.branched import ConvNet1Branched
    B = 32
    base = _store(120, 1, seed=13)
    a = FrameStore(base.frames, commands=base.commands, targets=base.targets)
    b = FrameStore(base.frames, commands=base.commands, targets=-base.targets)
    idx = torch.from_numpy(_indices(base.n_frames, B, 2)).to(base.device)
    torch.manual_seed(12345)
    net = ConvNet1Branched({"obs_size": 4, "n_actions": 3, "n_branches": 4, "branch_loss": "l1", "precision": "bf16"}).to(_dev())
    st = BranchedTrainStep(net, net.configure_optimizer(lr=1e-3), B)
    for store in (a, a, a, b, b):
        st.step_gather(store, idx)
        torch.cuda.synchronize()
        assert torch.equal(st._gside[1], store.targets[idx + 4])
    assert len(st._graphs) == 2


# ------------------------------------------------------------------------------------------------ branched training
@pytest.mark.parametrize("kind,aug", [("ce", False), ("l1", True), ("l1", False), ("ce", True)])
def test_branched_step_gather_equals_the_explicit_path_bitwise(kind, aug):
    from carla_imitation_learning_b200.data import augment_table
    from carla_imitation_learning_b200.trainer import BranchedTrainStep
    from src.architectures.branched import ConvNet1Branched
    B, steps, G, n_out = 64, 4, 4, (9 if kind == "ce" else 3)
    hw = (288, 320) if aug else None
    store = _store(300, 1, hw or (256, 256), seed=21, n_actions=n_out, G=G, n_out=n_out)
    dev = store.device
    rng = np.random.default_rng(1)
    plan = [rng.integers(0, store.n_frames - 4, size=B) for _ in range(steps)]
    tables = [torch.from_numpy(augment_table(50 + s, B, hw)).to(dev) if aug else None for s in range(steps)]
    runs = []
    for explicit in (False, True):
        torch.manual_seed(12345)
        net = ConvNet1Branched({"obs_size": 4, "n_actions": n_out, "n_branches": G, "branch_loss": kind,
                                "precision": "bf16"}).to(dev)
        opt = net.configure_optimizer(lr=1e-3)
        st = BranchedTrainStep(net, opt, B, src_hw=hw, graph=not explicit)
        slots = [torch.zeros(B, dtype=torch.int64, device=dev) for _ in range(2)]
        tslots = [torch.zeros((B, 8), device=dev) for _ in range(2)] if aug else [None, None]
        losses = []
        for s in range(steps):
            if explicit:
                st.eng.ensure_packed()
                st._point(True)
                st._gather_x().tp.copy_(_explicit(store, plan[s], "tp", tables[s]))
                i4 = torch.from_numpy(plan[s] + 4).to(dev)
                target = store.labels[i4] if kind == "ce" else store.targets[i4].contiguous()
                st.opt.prepare()
                st._train(store.commands[i4].contiguous(), target.contiguous())
                losses.append(st.hb["loss"].clone())
            else:
                slots[s % 2].copy_(torch.from_numpy(plan[s]))
                if aug:
                    tslots[s % 2].copy_(tables[s])
                losses.append(st.step_gather(store, slots[s % 2], tslots[s % 2]).clone())
        torch.cuda.synchronize()
        st.check()
        runs.append((torch.stack(losses).cpu(), net._arena.detach().clone(), net._barena.detach().clone()))
    for a, b in zip(runs[0], runs[1]):
        assert torch.equal(a, b), kind


# ------------------------------------------------------------------------------------------------ module path
@pytest.mark.parametrize("branched", [False, True])
def test_trainer_fit_over_shuffled_frames_equals_a_manual_loop(branched):
    """Trainer.fit with a ShuffledFrames train loader (cuda_graph: true for Imitation) runs an epoch and equals a manual
    loop over the same permutation's batches staged explicitly -- parameters bitwise."""
    from carla_imitation_learning_b200.data import FrameStore, ShuffledFrames
    from carla_imitation_learning_b200.trainer import Trainer
    from src.architectures.branched import ConvNet1Branched
    from src.architectures.nets import ConvNet1
    from src.models.imitation import Imitation
    from src.models.imitation_branched import ImitationBranched
    dev = _dev()
    B, n = 32, 150
    src = _store(n, 1, seed=33, n_actions=3, n_out=3)
    results = []
    for manual in (False, True):
        torch.manual_seed(12345)
        if branched:
            hp = {"obs_size": 4, "n_actions": 3, "n_branches": 4, "branch_loss": "l1", "precision": "bf16"}
            net = ConvNet1Branched(hp).to(dev)
            store = FrameStore(src.frames, commands=src.commands, targets=src.targets)
            model = ImitationBranched(hp, net, {})
        else:
            hp = {"obs_size": 4, "n_actions": 9, "precision": "bf16", "cuda_graph": True}
            net = ConvNet1(hp).to(dev)
            store = FrameStore(src.frames, src.labels)
            model = Imitation(hp, net, {})
        loader = ShuffledFrames(store, B, seed=5, layout="tp")
        if not manual:
            model.data_loader = {"train_dataloader": loader}
            Trainer(max_epochs=1).fit(model)
            assert loader.epoch == 1
        else:
            from carla_imitation_learning_b200.engine import StagedBatch
            opt = model.configure_optimizers()[0][0]
            order = loader.shard(0)
            for k in range(len(loader)):
                index = order[k * B:(k + 1) * B]
                x = StagedBatch(_explicit(store, index, "tp"), None, 4, 4)
                i4 = torch.from_numpy(index + 4).to(dev)
                batch = ((x, src.commands[i4].contiguous(), src.targets[i4].contiguous()) if branched
                         else (x, src.labels[i4].contiguous()))
                loss = model.training_step(batch, k)
                opt.zero_grad()
                loss.backward()
                opt.step()
        torch.cuda.synchronize()
        results.append([p.detach().clone() for p in net.parameters()])
    for a, b in zip(*results):
        assert torch.equal(a, b)


def test_shuffled_frames_batches_and_datamodule():
    """ShuffledFrames yields the permutation's samples (short last batch included) with their labels; the datamodule's
    `shuffle: true` makes the train split a ShuffledFrames and leaves validation sequential."""
    from carla_imitation_learning_b200.data import (FrameStore, SequentialFrames, ShuffledFrames,
                                                    sequential_train_val_test_iterator, synthetic_sequence)
    full = _store(100, 1, seed=8)
    store = FrameStore(full.frames, full.labels)             # no commands: (x, y) batches
    B = 28                                                   # 96 samples: 3 full batches and a short one of 12
    sf = ShuffledFrames(store, B, seed=2, layout="plain")
    order = sf.shard(0)
    seen = []
    for k, (x, y) in enumerate(sf):
        index = order[k * B:(k + 1) * B]
        assert x.shape == (len(index), 4, 256, 256)
        assert torch.equal(x, _explicit(store, index, "plain"))
        assert torch.equal(y, store.labels[torch.from_numpy(index + 4).to(store.device)])
        seen.extend(index.tolist())
    assert sorted(seen) == list(range(store.n_samples)) and len(order) % B != 0
    dls = sequential_train_val_test_iterator({"BATCH_SIZE": 16, "frame_skip": 4, "n_actions": 9, "precision": "bf16",
                                              "shuffle": True, "shuffle_seed": 3})
    assert isinstance(dls["train_dataloader"], ShuffledFrames) and dls["train_dataloader"].seed == 3
    assert isinstance(dls["val_dataloader"], SequentialFrames)
    frames, labels = synthetic_sequence(0, 8 * 16 + 4)
    assert np.array_equal(dls["train_dataloader"].store.frames.cpu().numpy(), frames)
