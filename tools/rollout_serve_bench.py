"""Closed-loop serving of N independent agents (BASELINE configs[4]), per-tick latency, printed as one JSON line.

    python tools/rollout_serve_bench.py [--replays 300] [--out DIR] [--agents 1,2,4,...]

* Workloads: ConvNet1 single head (obs 4, n_actions 9, 256x256 frames) and the configs[2] policy (ConvNet1Branched, G = 4,
  L1, n_out 3, 288x320 frames through data.center_crop_table), each in bf16 and fp32; N = 1 .. 4096 agents.
* (a) trainer.RolloutActStep: one new frame per agent per tick, staged into each agent's on-device history
  (bc_stage_history), the windows read in place. One CUDA graph per (input buffer, tick slot).
* (b) what an N-agent caller can build from the existing entry points as one graph: it keeps each agent's last 4 frames and
  stages all 4N of them per tick (bc_stage_gray_tp / bc_stage_gray / bc_stage_augment) into (4N) planes read with strides
  (4, 1) planes, then bc_forward_act / bc_forward_branched_act. Same path choice (tail up to tail_batch) as (a).
* At N = 1 also BranchedActStep, the single-stream step (5 frames staged per tick, sliding window).
* Each replay is timed by its own pair of CUDA events; p50 / p99 over >= 300 replays per path, (a) and (b) alternated in
  blocks of 50 in the same process. Input buffers rotate; there are enough of them that each path's frames exceed the
  126 MB L2 (the history ring of (a) is state, not input, and stays where the hardware keeps it).
* The card's name and power limit are read in the same process.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import math
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from tools.branched_step_bench import device_meta  # noqa: E402

AGENTS = (1, 2, 4, 8, 16, 64, 256, 1024, 4096)
SRC_HW = (288, 320)
L2_BYTES = 126e6
BLOCK = 50


def make_net(kind, precision):
    torch.manual_seed(12345)
    if kind == "single":
        from src.architectures.nets import ConvNet1
        return ConvNet1({"obs_size": 4, "n_actions": 9, "precision": precision}).cuda()
    from src.architectures.branched import ConvNet1Branched
    return ConvNet1Branched({"obs_size": 4, "n_actions": 3, "n_branches": 4, "branch_loss": "l1",
                             "precision": precision}).cuda()


def n_inputs(frame_bytes, multiple):
    """Input buffers to rotate over: their frames together exceed 1.5x the L2; a multiple of `multiple`."""
    k = max(multiple, math.ceil(1.5 * L2_BYTES / frame_bytes))
    return -(-k // multiple) * multiple


class StackedStep:
    """Path (b): stage the 4 frames of each of the N windows with the existing kernels, serve with strides (4, 1) planes."""

    def __init__(self, net, N, src_hw):
        from carla_imitation_learning_b200 import StagedBatch, _lib
        self.net, self.N, self.src_hw, self.eng = net, N, src_hw, net.engine()
        self.lib, self.L = self.eng.lib, _lib
        self.branched = hasattr(net, "_barena")
        self.tail = N <= (net.tail_batch if self.branched else self.eng.tail_batch)
        dev = self.eng.device
        self.bf16 = bool(self.eng.conv_mode)
        E = _lib.TP_PLANE_ELEMS
        if self.bf16:
            self.planes = torch.empty((4 * N, E), dtype=torch.bfloat16, device=dev)
            self.bufs = self.eng.alloc(N, StagedBatch(self.planes, None, 4), None, False)
            self.bufs.x_tp_strides = (4 * E, E)
        else:
            self.planes = torch.empty((4 * N, 256, 256), dtype=torch.float32, device=dev)
            self.bufs = self.eng.alloc(N, self.planes.view(N, 4, 256, 256), None, False)
        self.out = torch.empty((N, net.n_actions), dtype=torch.float32, device=dev) if self.branched else self.bufs.logits
        self.actions = None if self.branched else torch.empty(N, dtype=torch.int64, device=dev)
        self._seen, self._graphs = set(), {}

    def _enqueue(self, frames, table, command):
        from carla_imitation_learning_b200.engine import _stream_ptr
        L, s, n = self.L, _stream_ptr(), 4 * self.N
        code = L.BC_BF16_TP if self.bf16 else L.BC_F32
        if table is not None:
            L.check(self.lib.bc_stage_augment(frames.data_ptr(), n, frames.shape[1], frames.shape[2], table.data_ptr(),
                                              self.planes.data_ptr(), code, s), "bc_stage_augment")
        elif self.bf16:
            L.check(self.lib.bc_stage_gray_tp(frames.data_ptr(), self.planes.data_ptr(), None, n, s), "bc_stage_gray_tp")
        else:
            L.check(self.lib.bc_stage_gray(frames.data_ptr(), self.planes.data_ptr(), n * 65536, code, s), "bc_stage_gray")
        if self.branched:
            self.net._serve(self.bufs, self.out, None, command, self.tail)
        else:
            c = self.eng.ctx(self.bufs)
            L.check(self.lib.bc_forward_act(C.byref(c), self.actions.data_ptr(), int(self.tail), s), "bc_forward_act")

    def act(self, frames, table, command):
        key = (frames.data_ptr(), None if table is None else table.data_ptr(), None if command is None else command.data_ptr())
        g = self._graphs.get(key)
        if g is None and key in self._seen:
            g = self._graphs[key] = torch.cuda.CUDAGraph()
            with torch.no_grad(), torch.cuda.graph(g):
                self._enqueue(frames, table, command)
        if g is not None:
            g.replay()
        else:
            self._seen.add(key)
            with torch.no_grad():
                self._enqueue(frames, table, command)

    def check(self):
        self.eng.check_device_errors()


def _frames(dev, gen, n, hw):
    return torch.randint(0, 256, (n, *hw, 3), generator=gen, dtype=torch.uint8, device=dev)


def _timed(call, i0, n, ev):
    for i in range(i0, i0 + n):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        call(i)
        b.record()
        ev.append((a, b))


def _stats(ev, N):
    t = np.array([a.elapsed_time(b) for a, b in ev]) * 1000.0
    p50 = float(np.percentile(t, 50))
    return {"p50_us": round(p50, 2), "p99_us": round(float(np.percentile(t, 99)), 2), "replays": len(ev),
            "agent_frames_per_s_p50": round(N / p50 * 1e6)}


def bench_point(net, kind, N, replays, dev, seed):
    from carla_imitation_learning_b200.data import center_crop_table
    from carla_imitation_learning_b200.trainer import RolloutActStep
    src_hw = SRC_HW if kind == "l1" else None
    hw = src_hw or (256, 256)
    fb = hw[0] * hw[1] * 3
    gen = torch.Generator(device=dev).manual_seed(seed)
    command = torch.randint(0, 4, (N,), generator=gen, device=dev) if kind == "l1" else None
    # (a): N frames per tick; input i at tick i, tick slot i % 4 -> one graph per input (inputs are a multiple of 4)
    ka = n_inputs(N * fb, 4)
    ins_a = [_frames(dev, gen, N, hw) for _ in range(ka)]
    reset = torch.zeros(N, dtype=torch.uint8, device=dev)
    table_a = None if src_hw is None else torch.from_numpy(center_crop_table(N, src_hw)).to(dev)
    step_a = RolloutActStep(net, N, src_hw=src_hw)
    # (b): the 4N frames of the N windows per tick
    kb = n_inputs(4 * N * fb, 1)
    ins_b = [_frames(dev, gen, 4 * N, hw) for _ in range(kb)]
    table_b = None if src_hw is None else torch.from_numpy(center_crop_table(4 * N, src_hw)).to(dev)
    step_b = StackedStep(net, N, src_hw)
    call_a = lambda i: step_a.act(ins_a[i % ka], reset, table_a, command)
    call_b = lambda i: step_b.act(ins_b[i % kb], table_b, command)
    for i in range(2 * ka + 8):                     # every (input, slot) key: eager pass, capture, then replays
        call_a(i)
    for i in range(2 * kb + 8):
        call_b(i)
    torch.cuda.synchronize()
    ev_a, ev_b, done = [], [], 0
    while done < replays:                          # alternate the two paths in blocks
        _timed(call_a, 2 * ka + 8 + done, BLOCK, ev_a)
        _timed(call_b, 2 * kb + 8 + done, BLOCK, ev_b)
        done += BLOCK
    torch.cuda.synchronize()
    step_a.check()
    step_b.check()
    assert len(step_a._graphs) == ka, (len(step_a._graphs), ka)
    tail = step_a.tail
    rows = [{"path": "rollout", "inputs": ka, "frames_staged_per_tick": N, "tail": tail, **_stats(ev_a, N)},
            {"path": "stacked", "inputs": kb, "frames_staged_per_tick": 4 * N, "tail": tail, **_stats(ev_b, N)}]
    return rows


def bench_single_stream(net, replays, dev, seed):
    """BranchedActStep at batch 1: 5 frames per tick (its sliding window), centre crop from 288x320."""
    from carla_imitation_learning_b200.data import center_crop_table
    from carla_imitation_learning_b200.trainer import BranchedActStep
    gen = torch.Generator(device=dev).manual_seed(seed)
    k = n_inputs(5 * SRC_HW[0] * SRC_HW[1] * 3, 1)
    ins = [_frames(dev, gen, 5, SRC_HW) for _ in range(k)]
    table = torch.from_numpy(center_crop_table(5, SRC_HW)).to(dev)
    command = torch.zeros(1, dtype=torch.int64, device=dev)
    step = BranchedActStep(net, 1, src_hw=SRC_HW)
    call = lambda i: step.act(ins[i % k], table, command)
    for i in range(2 * k + 8):
        call(i)
    torch.cuda.synchronize()
    ev = []
    _timed(call, 2 * k + 8, replays, ev)
    torch.cuda.synchronize()
    step.check()
    return {"path": "branched_act_step_single_stream", "inputs": k, "frames_staged_per_tick": 5, **_stats(ev, 1)}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--replays", type=int, default=300, help="timed replays per path and point (>= 300)")
    ap.add_argument("--agents", default=",".join(map(str, AGENTS)))
    ap.add_argument("--out", default=None, help="directory for bench_rollout_serve.json")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("rollout_serve_bench: no CUDA device (this measures the B200 path; there is no CPU fallback)")
    from carla_imitation_learning_b200 import _lib
    _lib.build()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    replays = -(-max(args.replays, 300) // BLOCK) * BLOCK
    agents = [int(v) for v in args.agents.split(",")]
    res = {"workload": "rollout_serve", "config": "BASELINE configs[4]: N independent agents per tick", **device_meta(dev),
           "timing": "per-replay CUDA events around one tick (one graph replay: staging + forward), p50 / p99",
           "nets": {"single": "ConvNet1 obs 4, n_actions 9, 256x256 frames",
                    "l1": "ConvNet1Branched G=4, L1, n_out 3, 288x320 frames through center_crop_table (configs[2])"}}
    rows = []
    for kind in ("single", "l1"):
        for precision in ("bf16", "fp32"):
            net = make_net(kind, precision)
            for N in agents:
                for r in bench_point(net, kind, N, replays, dev, 1000 + N):
                    rows.append({"net": kind, "precision": precision, "agents": N, **r})
                    print(json.dumps(rows[-1]), file=sys.stderr, flush=True)
                torch.cuda.empty_cache()
            if kind == "l1" and 1 in agents:
                rows.append({"net": kind, "precision": precision, "agents": 1, **bench_single_stream(net, replays, dev, 7)})
                print(json.dumps(rows[-1]), file=sys.stderr, flush=True)
            del net
            torch.cuda.empty_cache()
    res["rows"] = rows
    res["rollout_over_stacked_p50"] = {
        f"{r['net']}/{r['precision']}/{r['agents']}": round(r["p50_us"] / s["p50_us"], 3)
        for r in rows if r["path"] == "rollout"
        for s in rows if s["path"] == "stacked" and (s["net"], s["precision"], s["agents"]) == (r["net"], r["precision"], r["agents"])}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bench_rollout_serve.json"), "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
