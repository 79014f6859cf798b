"""Data-parallel training of the command-conditioned branched policy (BASELINE configs[2]: bf16, B = 256 per rank, G = 4
branches, L1 on 3 outputs, crop + colour jitter from 288x320 sources) on 1, 2, 4 or 8 GPUs, one process per GPU. One JSON
line from rank 0; with --out DIR also DIR/bench_branched_dp.json.

    python -m torch.distributed.run --nproc_per_node N tools/branched_dp_bench.py [--steps 300] [--out DIR]
    python tools/branched_dp_bench.py                       # one process = a world of one rank

Every rank runs the same thing; rank 0 reports.

1. step / step_gather: BranchedTrainStep with the two-arena peer exchange inside its CUDA graph (exchange='peer', also at
   world 1), p50 / p90 of per-replay CUDA events over --steps replays after warm-up. step() rotates over 4 device slots of
   260 frames of 288x320x3 u8 (72 MB each, 288 MB in all: more than the 126 MB L2); step_gather() draws 256 random
   samples per step from a FrameStore of --frames 288x320 frames (2.2 GB at 8000, far more than L2), index buffers
   rotating over 4 slots.
2. one_gpu: step() and step_gather() of today's one-GPU BranchedTrainStep (no exchange) on every rank at once, timed in
   the same process: the reference of the weak-scaling efficiency = one_gpu p50 / data-parallel p50 (B per rank fixed).
3. exchange_ab: the exchange alone, one launch per step of each form, alternated block by block in the same process:
   A = one bc_adam_step_exchange_arenas launch over [trunk | branch], B = two back-to-back bc_adam_step_exchange launches,
   the trunk on one PeerGrads and the branch arena on a second one (built here from the existing ABI only). Each is
   captured as a graph of --ab-launches exchanges and timed by CUDA events around whole replays.
4. replicas_identical on both arenas of the step() run, checked before the line is printed, with the card name and
   power limit read in the same run."""
from __future__ import annotations

import argparse
import json
import os
import sys
from types import SimpleNamespace

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from tools.branched_step_bench import branched_net, device_meta, slot_inputs  # noqa: E402

NSLOT = 4
B, G, N_OUT, KIND, SRC_HW = 256, 4, 3, "l1", (288, 320)


def _events(run, steps):
    """p50 / p90 of CUDA events around each of `steps` calls, and the mean over the whole window."""
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0.record()
    for i, (a, b) in enumerate(ev):
        a.record()
        run(i)
        b.record()
    w1.record()
    torch.cuda.synchronize()
    per = np.array([a.elapsed_time(b) for a, b in ev])
    return {"ms_p50": round(float(np.percentile(per, 50)), 4), "ms_p90": round(float(np.percentile(per, 90)), 4),
            "ms_mean_window": round(w0.elapsed_time(w1) / steps, 4), "replays": steps}


def _step_run(dev, exchange, steps, warmup, group=None):
    from carla_imitation_learning_b200.trainer import BranchedTrainStep
    net = branched_net(dev, G, N_OUT, KIND, "bf16")
    st = BranchedTrainStep(net, net.configure_optimizer(lr=1e-3), B, src_hw=SRC_HW, exchange=exchange, group=group)
    slots = [slot_inputs(dev, B, G, N_OUT, KIND, SRC_HW, 100 + 10 * dist.get_rank() + s) for s in range(NSLOT)]
    for i in range(max(warmup, 3 * NSLOT)):                  # per slot: eager, capture, replays
        st.step(*slots[i % NSLOT])
    torch.cuda.synchronize()
    res = _events(lambda i: st.step(*slots[i % NSLOT]), steps)
    st.check()
    res["final_loss"] = float(st.hb["loss"])
    return res, net, st


def _gather_run(dev, store, steps, warmup, exchange, group=None):
    from carla_imitation_learning_b200.data import augment_table
    from carla_imitation_learning_b200.trainer import BranchedTrainStep
    net = branched_net(dev, G, N_OUT, KIND, "bf16")
    st = BranchedTrainStep(net, net.configure_optimizer(lr=1e-3), B, src_hw=SRC_HW, exchange=exchange, group=group)
    g = torch.Generator(device=dev).manual_seed(7 + dist.get_rank())
    idx = [torch.randint(0, store.n_frames - 4, (B,), generator=g, device=dev) for _ in range(NSLOT)]
    tab = [torch.from_numpy(augment_table(300 + 10 * dist.get_rank() + s, B, SRC_HW)).to(dev) for s in range(NSLOT)]
    for i in range(max(warmup, 3 * NSLOT)):
        st.step_gather(store, idx[i % NSLOT], tab[i % NSLOT])
    torch.cuda.synchronize()
    res = _events(lambda i: st.step_gather(store, idx[i % NSLOT], tab[i % NSLOT]), steps)
    st.check()
    return res


def _exchange_ab(dev, rounds, block, launches):
    """A: one two-arena launch; B: two single-arena launches on two PeerGrads. Graphs of `launches` exchanges each."""
    from carla_imitation_learning_b200.parallel import BranchedPeerExchange, PeerGrads
    net_a = branched_net(dev, G, N_OUT, KIND, "bf16")
    opt_a = net_a.configure_optimizer(lr=1e-3)
    xa = BranchedPeerExchange(net_a, opt_a)
    net_b = branched_net(dev, G, N_OUT, KIND, "bf16")
    opt_b = net_b.configure_optimizer(lr=1e-3)
    trunk_opt, branch_opt = opt_b.children_
    peer_t = PeerGrads(net_b.engine())
    peer_b = PeerGrads(SimpleNamespace(arena=net_b._barena, device=dev, obs_size=4, n_actions=N_OUT))
    for c, p in ((trunk_opt, peer_t), (branch_opt, peer_b)):
        c.set_grad_scale(1.0 / p.world)
    opt_b.prepare()
    net_a.engine().ensure_packed()
    net_b.engine().ensure_packed()

    def a_once():
        xa.exchange()

    def b_once():
        trunk_opt.step_exchange(peer_t)
        branch_opt.step_exchange(peer_b)

    graphs = {}
    for name, once in (("one_two_arena_launch", a_once), ("two_single_arena_launches", b_once)):
        once()                                                   # eager warm-up
        torch.cuda.synchronize()
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            for _ in range(launches):
                once()
        graphs[name] = gr
    for gr in graphs.values():
        gr.replay()
    torch.cuda.synchronize()
    per = {k: [] for k in graphs}
    for _ in range(rounds):
        for k, gr in graphs.items():
            dist.barrier()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(block):
                gr.replay()
            e1.record()
            torch.cuda.synchronize()
            per[k].append(1000.0 * e0.elapsed_time(e1) / (block * launches))
    for p in (xa.peer, peer_t, peer_b):
        p.check()
    out = {k: {"us_per_exchange_median": round(float(np.median(v)), 3), "us_per_exchange_min": round(float(min(v)), 3)}
           for k, v in per.items()}
    out.update(rounds=rounds, replays_per_block=block, exchanges_per_replay=launches,
               trunk_floats=int(net_a._arena.numel()), branch_floats=int(net_a._barena.numel()))
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=300, help="timed graph replays per step variant")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--frames", type=int, default=8000, help="frames of the step_gather store (288x320x3 u8 each)")
    ap.add_argument("--ab-rounds", type=int, default=8)
    ap.add_argument("--ab-block", type=int, default=20, help="graph replays per form and round")
    ap.add_argument("--ab-launches", type=int, default=20, help="exchanges captured in one graph")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("branched_dp_bench: no CUDA device (this measures the B200 path; there is no CPU fallback)")
    for k, v in (("MASTER_ADDR", "127.0.0.1"), ("MASTER_PORT", "29541"), ("RANK", "0"), ("WORLD_SIZE", "1"), ("LOCAL_RANK", "0")):
        os.environ.setdefault(k, v)
    local = int(os.environ["LOCAL_RANK"])
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    try:
        from carla_imitation_learning_b200 import _lib
        from carla_imitation_learning_b200.data import FrameStore
        from carla_imitation_learning_b200.trainer import replicas_identical
        _lib.build()
        world, rank = dist.get_world_size(), dist.get_rank()
        res = {"workload": "branched_train_step_data_parallel", "config": "BASELINE configs[2]", "world": world,
               "batch_per_rank": B, "global_batch": B * world, "n_branches": G, "n_out": N_OUT, "loss": KIND,
               "precision": "bf16", "augment_src_hw": list(SRC_HW), **device_meta(dev)}
        solo = [dist.new_group([r]) for r in range(world)][rank]   # a group of this rank alone: the one-GPU step
        one, _net1, _st1 = _step_run(dev, None, args.steps, args.warmup, group=solo)
        dist.barrier()
        step, net, _st = _step_run(dev, "peer", args.steps, args.warmup)
        same = bool(replicas_identical(net._arena) and replicas_identical(net._barena))
        g = torch.Generator(device=dev).manual_seed(1000 + rank)
        store = FrameStore(torch.randint(0, 256, (args.frames, *SRC_HW, 3), generator=g, dtype=torch.uint8, device=dev),
                           commands=torch.randint(0, G, (args.frames,), generator=g, device=dev),
                           targets=torch.rand((args.frames, N_OUT), generator=g, device=dev) * 2 - 1)
        one_gather = _gather_run(dev, store, args.steps, args.warmup, None, group=solo)
        dist.barrier()
        gather = _gather_run(dev, store, args.steps, args.warmup, "peer")
        dist.barrier()
        ab = _exchange_ab(dev, args.ab_rounds, args.ab_block, args.ab_launches)
        if not same:
            raise SystemExit("branched_dp_bench: the replicas differ after the timed steps")
        for r, ref in ((step, one), (gather, one_gather)):
            r["global_samples_per_s"] = round(B * world / (r["ms_mean_window"] / 1000.0), 1)
            r["weak_scaling_efficiency_p50"] = round(ref["ms_p50"] / r["ms_p50"], 4)
        for r in (one, one_gather):
            r["samples_per_s"] = round(B / (r["ms_mean_window"] / 1000.0), 1)
        res.update(replicas_identical=same, one_gpu={"step": one, "step_gather": one_gather}, step=step, step_gather=gather,
                   exchange_ab=ab,
                   inputs={"step": f"{NSLOT} rotating device slots of {B + 4} frames 288x320x3 u8 "
                                   f"({NSLOT * (B + 4) * 288 * 320 * 3 / 1e6:.0f} MB: larger than the 126 MB L2)",
                           "step_gather": f"FrameStore of {args.frames} frames 288x320x3 u8 "
                                          f"({args.frames * 288 * 320 * 3 / 1e9:.1f} GB), {NSLOT} rotating index slots"},
                   value=step["global_samples_per_s"], unit="samples/s")
        if rank == 0:
            line = json.dumps(res)
            print(line)
            if args.out:
                os.makedirs(args.out, exist_ok=True)
                with open(os.path.join(args.out, "bench_branched_dp.json"), "w") as f:
                    f.write(line + "\n")
    finally:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
