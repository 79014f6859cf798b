"""What shuffled minibatches cost on one GPU: bc_stage_gather against the other graphable way to stage the same batch, and the
bf16 training steps on shuffled against sequential batches. One JSON line; with --out DIR also DIR/shuffled_step_bench.json.

    python tools/shuffled_step_bench.py [--replays 400] [--block 40] [--frames 20000] [--out DIR]

Every part times CUDA-graph replays with a pair of CUDA events around each replay; variants that are compared run in the same
process, alternated block by block (--block replays of one, then of the other, ...), and report p50 / p90 over --replays
replays each. Inputs rotate over NSLOT device slots (index buffers for the gathered variants, frame buffers for the
sequential ones), one graph per slot.

1. gather: bc_stage_gather alone, B = 256, obs 4, Toeplitz-ready bf16 planes, from a store of --frames 256x256 frames (>= 20 K:
   3.9 GB, far more than the 126 MB L2), random indices. GB/s against the bytes the batch must move: 4B source frames read
   (4B x 196,608 B) + 4B TP planes written (4B x 173,376 B).
2. index_copy_then_stage: the same batch through existing kernels -- torch index_select of the 4B window frames into a u8
   scratch buffer, then bc_stage_gray_tp on it.
3. step: TrainStep.step (sequential: 260 consecutive frames staged per step) against TrainStep.step_gather (256 shuffled
   samples), bf16, B = 256; and breakdown_us: every launch of the step timed on its own (bench.py's method) on both inputs.
4. branched: the configs[2] step (BranchedTrainStep: bf16, B = 256, 4 branches, L1 on 3 outputs, crop + colour jitter from
   288x320 sources), step against step_gather (table rows per sample) from a store of --frames 288x320 frames."""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from tools.branched_step_bench import device_meta  # noqa: E402

NSLOT = 4
B = 256
FRAME_BYTES = 256 * 256 * 3
TP_BYTES = 86688 * 2


def _random_frames(dev, n, hw, seed):
    out = torch.empty((n, hw[0], hw[1], 3), dtype=torch.uint8, device=dev)
    g = torch.Generator(device=dev).manual_seed(seed)
    for lo in range(0, n, 2000):
        hi = min(n, lo + 2000)
        out[lo:hi] = torch.randint(0, 256, (hi - lo, hw[0], hw[1], 3), generator=g, dtype=torch.uint8, device=dev)
    return out


def _capture(fn):
    fn()                                   # eager pass: allocations and first-launch work outside the capture
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    return g


def _alternate(variants: dict, replays: int, block: int) -> dict:
    """variants: name -> list of NSLOT graphs. Per-replay event times (ms), alternated in blocks; p50 / p90 per variant."""
    times = {k: [] for k in variants}
    for gs in variants.values():                               # warm every graph
        for g in gs:
            g.replay()
    torch.cuda.synchronize()
    i = 0
    while min(len(t) for t in times.values()) < replays:
        for name, gs in variants.items():
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(block + 1)]
            ev[0].record()
            for r in range(block):
                gs[(i + r) % len(gs)].replay()
                ev[r + 1].record()
            torch.cuda.synchronize()
            times[name].extend(ev[r].elapsed_time(ev[r + 1]) for r in range(block))
        i += block
    return {k: {"p50_ms": float(np.percentile(v, 50)), "p90_ms": float(np.percentile(v, 90)), "n": len(v)}
            for k, v in times.items()}


def bench_staging(dev, store, replays, block):
    from carla_imitation_learning_b200 import _lib
    from carla_imitation_learning_b200.engine import StagedBatch, _stream_ptr, stage_gather
    rng = np.random.default_rng(0)
    idx = [torch.from_numpy(rng.integers(0, store.n_samples, size=B)).to(dev) for _ in range(NSLOT)]
    rows = [(i[:, None] + torch.arange(4, device=dev)[None, :]).reshape(-1).contiguous() for i in idx]
    out = StagedBatch(torch.empty((4 * B, 86688), dtype=torch.bfloat16, device=dev), None, 4, 4)
    scratch = torch.empty((4 * B, 256, 256, 3), dtype=torch.uint8, device=dev)
    tp2 = torch.empty((4 * B, 86688), dtype=torch.bfloat16, device=dev)

    def copy_then_stage(r):
        torch.index_select(store.frames, 0, r, out=scratch)
        _lib.check(_lib.lib().bc_stage_gray_tp(scratch.data_ptr(), tp2.data_ptr(), None, 4 * B, _stream_ptr()), "bc_stage_gray_tp")
    variants = {"gather": [_capture(lambda i=i: stage_gather(store, i, "tp", out=out)) for i in idx],
                "index_copy_then_stage": [_capture(lambda r=r: copy_then_stage(r)) for r in rows]}
    res = _alternate(variants, replays, block)
    torch.cuda.synchronize()
    assert torch.equal(out.tp.view(torch.int16), tp2.view(torch.int16))       # last slot of each: the same planes
    need = 4 * B * (FRAME_BYTES + TP_BYTES)
    for k, v in res.items():
        v["bytes_moved_min"] = need
        v["gb_per_s_p50"] = need / (v["p50_ms"] * 1e-3) / 1e9
    res["index_copy_then_stage"]["bytes_moved_actual"] = need + 2 * 4 * B * FRAME_BYTES     # + the scratch write and re-read
    return res


def bench_steps(dev, store, replays, block):
    from carla_imitation_learning_b200 import FusedAdam
    from carla_imitation_learning_b200.trainer import TrainStep
    from src.architectures.nets import ConvNet1
    torch.manual_seed(12345)
    net = ConvNet1({"obs_size": 4, "n_actions": 9, "precision": "bf16"}).to(dev)
    ts = TrainStep(net, FusedAdam(list(net.parameters()), lr=1e-3), B)
    rng = np.random.default_rng(1)
    lo = [int(v) for v in rng.integers(0, store.n_frames - (B + 4), size=NSLOT)]
    seq = [(store.frames[s:s + B + 4].contiguous(), store.labels[s + 4:s + 4 + B].contiguous()) for s in lo]
    idx = [torch.from_numpy(rng.integers(0, store.n_samples, size=B)).to(dev) for _ in range(NSLOT)]
    for _ in range(2):                                         # eager pass, capture: every slot of both kinds
        for f, y in seq:
            ts.step(f, y)
        for i in idx:
            ts.step_gather(store, i)
    torch.cuda.synchronize()
    variants = {"sequential_step": [ts._graphs[(f.data_ptr(), y.data_ptr())] for f, y in seq],
                "shuffled_step_gather": [ts._graphs[ts.gather_key(store, i)] for i in idx]}
    res = _alternate(variants, replays, block)
    torch.cuda.synchronize()
    ts.check()
    res["breakdown_us"] = breakdown(ts, store, seq, idx)
    return res


def _event_us(fn, reps=20, warm=3):
    for _ in range(warm):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps * 1e3


def breakdown(ts, store, seq, idx, rounds=5):
    """Every launch of the step timed on its own (bench.py's breakdown_us: CUDA events around 20 back-to-back launches), on
    the sequential input (sliding window: conv1 shares each plane between 4 samples, weight gradient conv1_wgrad3) and on the
    materialised one (stage_gather: 4 planes per sample, the non-window conv1 kernels). The two inputs alternate round by
    round; the median over `rounds` is reported. Staging rotates over the NSLOT input slots, as in the timed step."""
    import ctypes as C
    from carla_imitation_learning_b200 import _lib
    from carla_imitation_learning_b200.engine import _stream_ptr, stage_gather
    eng, L = ts.eng, ts.eng.lib
    rot = [0]

    def stage_seq():
        rot[0] = (rot[0] + 1) % NSLOT
        ts._stage(seq[rot[0]][0])

    def stage_gathered():
        rot[0] = (rot[0] + 1) % NSLOT
        stage_gather(store, idx[rot[0]], "tp", out=ts._gather_x(), y=ts._gy, err_flag=eng.err_flag)

    times = {"sequential": {}, "shuffled": {}}
    for _ in range(rounds):
        for kind, stage in (("sequential", stage_seq), ("shuffled", stage_gathered)):
            ts._point(kind == "shuffled")
            ts.bufs.y = seq[0][1] if kind == "sequential" else ts._gy
            stage()
            c = eng.ctx(ts.bufs)
            cref, s = C.byref(c), _stream_ptr()
            ops = [("stage", stage)]
            ops += [(f"conv{l + 1}_fwd", (lambda l=l: _lib.check(L.bc_conv_relu_pool_fwd(cref, l, s)))) for l in range(4)]
            ops.append(("head_fwd_ce_bwd", lambda: _lib.check(L.bc_head(cref, 3, s))))
            for l in (3, 2, 1):
                ops.append((f"conv{l + 1}_wgrad", (lambda l=l: _lib.check(L.bc_conv_bwd_wgrad(cref, l, s)))))
                ops.append((f"conv{l + 1}_dgrad", (lambda l=l: _lib.check(L.bc_conv_bwd_dgrad(cref, l, s)))))
            ops.append(("conv1_wgrad", lambda: _lib.check(L.bc_conv_bwd_wgrad(cref, 0, s))))
            ops.append(("reduce_partials", lambda: _lib.check(L.bc_reduce_partials(cref, 1, s))))
            for name, fn in ops:
                times[kind].setdefault(name, []).append(_event_us(fn))
    ts._point(False)
    eng.check_device_errors()
    out = {k: {n: round(float(np.median(v)), 1) for n, v in t.items()} for k, t in times.items()}
    for k in out:
        out[k]["sum"] = round(sum(out[k].values()), 1)
    return out


def bench_branched(dev, n_frames, replays, block):
    from carla_imitation_learning_b200.data import FrameStore, augment_table
    from carla_imitation_learning_b200.trainer import BranchedTrainStep
    from src.architectures.branched import ConvNet1Branched
    hw = (288, 320)
    torch.manual_seed(12345)
    net = ConvNet1Branched({"obs_size": 4, "n_actions": 3, "n_branches": 4, "branch_loss": "l1", "precision": "bf16"}).to(dev)
    st = BranchedTrainStep(net, net.configure_optimizer(lr=1e-3), B, src_hw=hw)
    g = torch.Generator(device=dev).manual_seed(3)
    store = FrameStore(_random_frames(dev, n_frames, hw, 5), commands=torch.randint(0, 4, (n_frames,), generator=g, device=dev),
                       targets=torch.rand((n_frames, 3), generator=g, device=dev) * 2 - 1)
    rng = np.random.default_rng(2)
    lo = [int(v) for v in rng.integers(0, n_frames - (B + 4), size=NSLOT)]
    seq = [(store.frames[s:s + B + 4].contiguous(), torch.from_numpy(augment_table(10 + k, B + 4, hw)).to(dev),
            store.commands[s + 4:s + 4 + B].contiguous(), store.targets[s + 4:s + 4 + B].contiguous()) for k, s in enumerate(lo)]
    idx = [torch.from_numpy(rng.integers(0, store.n_samples, size=B)).to(dev) for _ in range(NSLOT)]
    tab = [torch.from_numpy(augment_table(20 + k, B, hw)).to(dev) for k in range(NSLOT)]
    for _ in range(2):
        for a in seq:
            st.step(*a)
        for i, t in zip(idx, tab):
            st.step_gather(store, i, t)
    torch.cuda.synchronize()
    variants = {"sequential_step": [st._graphs[(f.data_ptr(), t.data_ptr(), c.data_ptr(), y.data_ptr())] for f, t, c, y in seq],
                "shuffled_step_gather": [st._graphs[st.gather_key(store, i, t)]
                                         for i, t in zip(idx, tab)]}
    res = _alternate(variants, replays, block)
    torch.cuda.synchronize()
    st.check()
    return res


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--replays", type=int, default=400)
    ap.add_argument("--block", type=int, default=40)
    ap.add_argument("--frames", type=int, default=20000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("shuffled_step_bench measures on a CUDA device; there is nothing to measure without one")
    import __graft_entry__
    __graft_entry__.build()
    from carla_imitation_learning_b200.data import FrameStore
    dev = torch.device("cuda", 0)
    res = {"meta": {**device_meta(dev), "batch": B, "store_frames": a.frames, "replays": a.replays, "block": a.block}}
    store = FrameStore(_random_frames(dev, a.frames, (256, 256), 1),
                       torch.randint(0, 9, (a.frames,), generator=torch.Generator(device=dev).manual_seed(2), device=dev))
    res["meta"]["store_bytes"] = store.frames.numel()
    res["staging"] = bench_staging(dev, store, a.replays, a.block)
    res["step_bf16"] = bench_steps(dev, store, a.replays, a.block)
    del store
    torch.cuda.empty_cache()
    res["branched_configs2"] = bench_branched(dev, a.frames, a.replays, a.block)
    line = json.dumps(res)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "shuffled_step_bench.json"), "w") as f:
            f.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
