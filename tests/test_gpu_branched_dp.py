"""EXTENSION -- NO REFERENCE PARITY. Data-parallel training of the command-conditioned branched policy: the two-arena peer
exchange (bc_adam_step_exchange_arenas, parallel.BranchedPeerExchange) inside BranchedTrainStep's CUDA graph and behind
MultiArenaAdam.step on the module path.

On a world of one rank the exchange reads one term and scales it by 1: both arenas' parameters, both moments and every loss
equal the one-GPU step bit for bit. On two GPUs (skipped below that) the replicas stay bitwise identical and equal the
single-process step on the global batch within rounding."""
import json
import os
import socket

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

SRC_HW = (288, 320)
KINDS = (("ce", 9), ("l1", 3), ("mse", 3))


def _free_port() -> int:
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _net(kind, n_out, precision, dev, G=4):
    from src.architectures.branched import ConvNet1Branched
    torch.manual_seed(12345)
    return ConvNet1Branched({"obs_size": 4, "n_actions": n_out, "n_branches": G, "branch_loss": kind,
                             "precision": precision}).to(dev)


def _state(opt):
    """Both arenas' parameters and Adam moments (copies)."""
    return [t.detach().clone() for c in opt.children_ for t in (c._bound[0], c._bound[1], c._bound[2])]


def _global_data(seed, steps, Bg, n_out, kind, hw, G=4, world=2):
    """Per step: frames (Bg+4, H, W, 3) u8, frame table (Bg+4, 8) or None, commands and targets of the global batch. The
    commands of shard r are drawn from [r, r + G - world + 1): on two ranks branch 0 is absent from rank 1's samples and
    branch G-1 from rank 0's."""
    from carla_imitation_learning_b200.data import augment_table
    gen = torch.Generator().manual_seed(seed)
    h, w = hw or (256, 256)
    per = Bg // world
    out = []
    for s in range(steps):
        frames = torch.randint(0, 256, (Bg + 4, h, w, 3), generator=gen, dtype=torch.uint8)
        table = None if hw is None else torch.from_numpy(augment_table(seed + s, Bg + 4, hw))
        command = torch.cat([torch.randint(r, r + G - world + 1, (per,), generator=gen) for r in range(world)])
        target = torch.randint(0, n_out, (Bg,), generator=gen) if kind == "ce" else torch.rand((Bg, n_out), generator=gen) * 2 - 1
        out.append((frames, table, command, target))
    return out


def _store(seed, n_frames, n_out, hw, G=4):
    from carla_imitation_learning_b200.data import FrameStore
    g = torch.Generator().manual_seed(seed)
    h, w = hw or (256, 256)
    frames = torch.randint(0, 256, (n_frames, h, w, 3), generator=g, dtype=torch.uint8)
    labels = torch.randint(0, n_out, (n_frames,), generator=g)
    commands = torch.randint(0, G, (n_frames,), generator=g)
    targets = torch.rand((n_frames, n_out), generator=g) * 2 - 1
    return FrameStore(frames, labels, commands, targets)


def _run_step(net, opt, B, hw, data, lo, hi, group=None, exchange=None):
    """BranchedTrainStep.step over `data`, this rank's shard [lo, hi) of each global batch, rotating over two device slots
    (per slot: eager, capture + replay, replays). Returns the losses."""
    from carla_imitation_learning_b200.trainer import BranchedTrainStep
    dev = net._barena.device
    st = BranchedTrainStep(net, opt, B, src_hw=hw, group=group, exchange=exchange)
    f0, t0, c0, y0 = data[0]
    slots = [[torch.empty_like(f0[:B + 4], device=dev), None if t0 is None else torch.empty_like(t0[:B + 4], device=dev),
              torch.empty_like(c0[:B], device=dev), torch.empty_like(y0[:B], device=dev)] for _ in range(2)]
    losses = []
    for s, (f, t, c, y) in enumerate(data):
        sl = slots[s & 1]
        sl[0].copy_(f[lo:hi + 4])
        if t is not None:
            sl[1].copy_(t[lo:hi + 4])
        sl[2].copy_(c[lo:hi])
        sl[3].copy_(y[lo:hi])
        losses.append(st.step(*sl).clone())
    torch.cuda.synchronize()
    st.check()
    return torch.stack(losses)


def _run_gather(net, opt, B, hw, store, plan, tables, rank, world, group=None, exchange=None):
    """BranchedTrainStep.step_gather over the global index `plan[s]`, this rank's shard index[rank::world]."""
    from carla_imitation_learning_b200.trainer import BranchedTrainStep
    dev = store.device
    st = BranchedTrainStep(net, opt, B, src_hw=hw, group=group, exchange=exchange)
    idx = [torch.zeros(B, dtype=torch.int64, device=dev) for _ in range(2)]
    tab = [torch.zeros((B, 8), device=dev) for _ in range(2)] if hw else [None, None]
    losses = []
    for s in range(len(plan)):
        idx[s & 1].copy_(torch.from_numpy(plan[s][rank::world]))
        if hw:
            tab[s & 1].copy_(tables[s][rank::world])
        losses.append(st.step_gather(store, idx[s & 1], tab[s & 1]).clone())
    torch.cuda.synchronize()
    st.check()
    return torch.stack(losses)


def _module_batches(data, lo, hi, precision, dev):
    from carla_imitation_learning_b200 import sliding_window, stage_gray, stage_frames
    out = []
    for f, _t, c, y in data:
        fr = f[lo:hi + 4].to(dev)
        x = stage_frames(fr) if precision == "bf16" else sliding_window(stage_gray(fr))
        out.append((x, c[lo:hi].to(dev), y[lo:hi].to(dev)))
    return out


def _module_loop(model, opt, batches):
    for i, b in enumerate(batches):
        loss = model.training_step(b, i)
        opt.zero_grad()
        loss.backward()
        opt.step()
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------- world of one: bitwise
def _world1_worker(_proc, out_path, port):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    dist.init_process_group("nccl", rank=0, world_size=1, device_id=dev)
    try:
        from src.models.imitation_branched import ImitationBranched
        from carla_imitation_learning_b200.data import augment_table
        from carla_imitation_learning_b200.parallel import BranchedPeerExchange
        B, steps = 8, 8
        rng = np.random.default_rng(3)
        res = {}
        for precision in ("fp32", "bf16"):
            for kind, n_out in KINDS:
                for aug in (False, True):
                    hw = SRC_HW if aug else None
                    data = _global_data(7, steps, B, n_out, kind, hw, world=1)
                    store = _store(11, 200, n_out, hw)
                    plan = [rng.integers(0, store.n_frames - 4, size=B) for _ in range(steps)]
                    tables = [torch.from_numpy(augment_table(90 + s, B, hw)).to(dev) if aug else None for s in range(steps)]
                    for path in ("step", "gather"):
                        runs = []
                        for exchange in ("peer", None):
                            net = _net(kind, n_out, precision, dev)
                            opt = net.configure_optimizer(lr=1e-3)
                            if path == "step":
                                losses = _run_step(net, opt, B, hw, data, 0, B, exchange=exchange)
                            else:
                                losses = _run_gather(net, opt, B, hw, store, plan, tables, 0, 1, exchange=exchange)
                            runs.append([losses] + _state(opt))
                        key = f"{precision}/{kind}/{'aug' if aug else 'plain'}/{path}"
                        res[key] = all(torch.equal(a, b) for a, b in zip(*runs)) and bool(torch.isfinite(runs[0][0]).all())
        for precision in ("fp32", "bf16"):                 # module path: training_step -> backward -> MultiArenaAdam.step
            data = _global_data(5, 4, B, 3, "l1", None, world=1)
            runs = []
            for dp in (True, False):
                hp = {"obs_size": 4, "n_actions": 3, "n_branches": 4, "branch_loss": "l1", "precision": precision}
                net = _net("l1", 3, precision, dev)
                model = ImitationBranched(dict(hp), net, {})
                opt = model.configure_optimizers()[0][0]
                if dp:
                    BranchedPeerExchange(net, opt)
                _module_loop(model, opt, _module_batches(data, 0, B, precision, dev) * 2)
                net.engine().check_device_errors()
                if dp:
                    net.engine().peer.check()
                runs.append(_state(opt))
            res[f"module/{precision}"] = all(torch.equal(a, b) for a, b in zip(*runs))
        with open(out_path, "w") as fh:
            json.dump(res, fh)
    finally:
        dist.destroy_process_group()


def test_world_of_one_exchange_equals_the_one_gpu_step_bitwise(tmp_path):
    """BranchedTrainStep(exchange='peer') on a one-rank NCCL group -- trunk and branch gradients written straight into the
    double-buffered peer halves, one two-arena exchange launch inside the graph -- == today's one-GPU BranchedTrainStep:
    both arenas' parameters and moments and all 8 losses (6 of them graph replays), bit for bit, for CE / L1 / MSE, fp32
    and bf16, with and without augmentation, through step() and step_gather(); and the module path
    (MultiArenaAdam.step -> BranchedPeerExchange) == the module path without it."""
    import torch.multiprocessing as mp
    out = str(tmp_path / "w1.json")
    mp.spawn(_world1_worker, args=(out, _free_port()), nprocs=1, join=True)
    with open(out) as fh:
        res = json.load(fh)
    assert len(res) == 2 * 3 * 2 * 2 + 2
    assert all(res.values()), [k for k, v in res.items() if not v]


# ------------------------------------------------------------------------------- two ranks
def _two_rank_worker(rank, world, port, out_dir):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        from carla_imitation_learning_b200.data import augment_table
        from carla_imitation_learning_b200.trainer import Trainer, replicas_identical
        from src.models.imitation_branched import ImitationBranched
        solo = [dist.new_group([r]) for r in range(world)][rank]     # the single-process reference, run on every rank
        Bl, steps = 8, 6
        Bg = Bl * world
        lo, hi = rank * Bl, (rank + 1) * Bl
        rng = np.random.default_rng(4)
        res = {}
        for precision in ("fp32", "bf16"):
            tol = 5e-5 if precision == "fp32" else 4e-3
            for kind, n_out in KINDS:
                data = _global_data(17, steps, Bg, n_out, kind, SRC_HW, world=world)
                store = _store(19, 200, n_out, SRC_HW)
                plan = [rng.integers(0, store.n_frames - 4, size=Bg) for _ in range(steps)]
                tables = [torch.from_numpy(augment_table(70 + s, Bg, SRC_HW)).to(dev) for s in range(steps)]
                for path in ("step", "gather"):
                    states = []
                    for dp in (True, False):
                        net = _net(kind, n_out, precision, dev)
                        opt = net.configure_optimizer(lr=1e-3)
                        if path == "step":
                            _run_step(net, opt, Bl if dp else Bg, SRC_HW, data, lo if dp else 0, hi if dp else Bg,
                                      group=None if dp else solo)
                        else:
                            _run_gather(net, opt, Bl if dp else Bg, SRC_HW, store, plan, tables, rank if dp else 0,
                                        world if dp else 1, group=None if dp else solo)
                        if dp:
                            same = replicas_identical(net._arena) and replicas_identical(net._barena)
                        states.append((net._arena.detach().clone(), net._barena.detach().clone()))
                    err = max(float((a - b).abs().max()) for a, b in zip(*states))
                    res[f"{precision}/{kind}/{path}"] = bool(same) and err <= tol
            # module path: Trainer.fit(ImitationBranched) on each rank's shard == the manual module loop on the global batch
            data = _global_data(23, 4, Bg, 3, "l1", None, world=world)
            hp = {"obs_size": 4, "n_actions": 3, "n_branches": 4, "branch_loss": "l1", "precision": precision}
            net = _net("l1", 3, precision, dev)
            model = ImitationBranched(dict(hp), net, {"train_dataloader": _module_batches(data, lo, hi, precision, dev)})
            Trainer(max_epochs=2, ddp_exchange="peer").fit(model)
            torch.cuda.synchronize()
            same = replicas_identical(net._arena) and replicas_identical(net._barena)
            ref_net = _net("l1", 3, precision, dev)
            ref_model = ImitationBranched(dict(hp), ref_net, {})
            ref_opt = ref_model.configure_optimizers()[0][0]
            _module_loop(ref_model, ref_opt, _module_batches(data, 0, Bg, precision, dev) * 2)
            err = max(float((net._arena - ref_net._arena).abs().max()), float((net._barena - ref_net._barena).abs().max()))
            res[f"module/{precision}"] = bool(same) and err <= tol
        with open(os.path.join(out_dir, f"r{rank}.json"), "w") as fh:
            json.dump(res, fh)
    finally:
        dist.destroy_process_group()


def test_two_rank_exchange_keeps_replicas_identical_and_equals_the_global_batch(tmp_path):
    """2 GPUs (skipped on a 1-GPU box): after 6 graph-step replays both arenas are bitwise identical across ranks and equal
    the single-process step on the concatenated global batch (<= 5e-5 fp32, <= 4e-3 bf16), for CE / L1 / MSE, with the
    commands mixed so that a branch is present on one rank and absent on the other; the same for step_gather on the index
    sharded [rank::world] and for Trainer.fit(ImitationBranched) over each rank's shard."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs (tools/branched_dp_bench.py is the torchrun version)")
    import torch.multiprocessing as mp
    mp.spawn(_two_rank_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    for r in range(2):
        with open(tmp_path / f"r{r}.json") as fh:
            res = json.load(fh)
        assert len(res) == 2 * 3 * 2 + 2
        assert all(res.values()), (r, [k for k, v in res.items() if not v])
