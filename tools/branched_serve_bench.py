"""Serving latency of the command-conditioned branched policy (the closed-loop rollout of BASELINE configs[4] with the
configs[2] policy), printed as one JSON line.

    python tools/branched_serve_bench.py [--replays 300] [--out DIR]

* Workload: ConvNet1Branched, G = 4 branches, L1, n_out = 3, bf16, frames of 288x320 staged through a centre-crop table
  (data.center_crop_table); one CE row (G = 4, n_out = 9) covers the greedy-action path. trainer.BranchedActStep, one
  CUDA graph per batch and input slot.
* Sweep B = 1 .. 4096. Each replay is timed by its own pair of CUDA events: p50 / p99 over >= 200 replays. Every input
  slot has its own random commands. Slots rotate; from B = 256 there are enough of them that the frames exceed the 126 MB
  L2. Up to B = 64 both paths are timed (the one-launch tail and the layer path), which locates the crossover.
* Before: the eager net.forward(x, command) + torch.argmax at B = 1, 8 and 256 (staging included, as the captured step has it).
* The card's name and power limit are read in the same process.
"""
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

SRC_HW = (288, 320)
BATCHES = (1, 2, 4, 8, 16, 32, 64, 256, 1024, 4096)
L2_BYTES = 126e6


def make_net(dev, n_out, kind):
    from src.architectures.branched import ConvNet1Branched
    torch.manual_seed(12345)
    return ConvNet1Branched({"obs_size": 4, "n_actions": n_out, "n_branches": 4, "branch_loss": kind,
                             "precision": "bf16"}).to(dev)


def n_slots(B):
    """Input slots to rotate over: at least 3, and from B = 256 enough that their frames do not fit in L2."""
    per = (B + 4) * SRC_HW[0] * SRC_HW[1] * 3
    return max(3, int(np.ceil(1.5 * L2_BYTES / per))) if B >= 256 else 3


def slots_for(dev, B, seed):
    from carla_imitation_learning_b200.data import center_crop_table
    g = torch.Generator(device=dev).manual_seed(seed)
    table = torch.from_numpy(center_crop_table(B + 4, SRC_HW)).to(dev)
    return [(torch.randint(0, 256, (B + 4, *SRC_HW, 3), generator=g, dtype=torch.uint8, device=dev), table,
             torch.randint(0, 4, (B,), generator=g, device=dev)) for _ in range(n_slots(B))]


def time_step(step, slots, replays, warmup):
    for i in range(max(warmup, 2 * len(slots))):          # every slot: eager pass, capture, then warm replays
        step.act(*slots[i % len(slots)])
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(replays)]
    for i, (a, b) in enumerate(ev):
        a.record()
        step.act(*slots[i % len(slots)])
        b.record()
    torch.cuda.synchronize()
    step.check()
    t = np.array([a.elapsed_time(b) for a, b in ev]) * 1000.0
    return {"p50_us": round(float(np.percentile(t, 50)), 2), "p99_us": round(float(np.percentile(t, 99)), 2),
            "replays": replays, "slots": len(slots)}


def time_eager(net, slots, replays, warmup):
    """The eager path an agent had before: stage (crop table) + net.forward(x, command) + torch.argmax."""
    from carla_imitation_learning_b200 import stage_augmented

    def once(f, t, c):
        x = stage_augmented(f, t, layout="tp")
        return torch.argmax(net(x, c), 1)
    for i in range(warmup):
        once(*slots[i % len(slots)])
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(replays)]
    for i, (a, b) in enumerate(ev):
        a.record()
        once(*slots[i % len(slots)])
        b.record()
    torch.cuda.synchronize()
    t = np.array([a.elapsed_time(b) for a, b in ev]) * 1000.0
    return {"p50_us": round(float(np.percentile(t, 50)), 2), "p99_us": round(float(np.percentile(t, 99)), 2), "replays": replays}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--replays", type=int, default=300, help="timed replays per point (>= 200)")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", default=None, help="directory for bench_branched_serve.json")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("branched_serve_bench: no CUDA device (this measures the B200 path; there is no CPU fallback)")
    from carla_imitation_learning_b200 import _lib
    from carla_imitation_learning_b200.trainer import BranchedActStep
    _lib.build()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    replays = max(args.replays, 200)
    res = {"workload": "branched_serve", "config": "BASELINE configs[2] policy served as configs[4]", **device_meta(dev),
           "precision": "bf16", "n_branches": 4, "src_hw": list(SRC_HW), "staging": "stage_augmented with center_crop_table",
           "timing": "per-replay CUDA events around BranchedActStep.act (one graph replay: staging + forward)"}
    rows = []
    for kind, n_out in (("l1", 3), ("ce", 9)):
        net = make_net(dev, n_out, kind)
        for B in (BATCHES if kind == "l1" else (1, 8, 256)):
            slots = slots_for(dev, B, 1000 + B)
            paths = (True, False) if B <= _lib.POLICY_TAIL_MAX_BATCH else (False,)
            for tail in paths:
                step = BranchedActStep(net, B, src_hw=SRC_HW)
                step.tail = tail
                r = time_step(step, slots, replays, args.warmup)
                rows.append({"loss": kind, "n_out": n_out, "batch": B, "path": "tail" if tail else "layers", **r})
                print(json.dumps(rows[-1]), file=sys.stderr)
                del step
            del slots
            torch.cuda.empty_cache()
    res["sweep"] = rows
    eager = []
    net = make_net(dev, 3, "l1")
    for B in (1, 8, 256):
        slots = slots_for(dev, B, 2000 + B)
        eager.append({"batch": B, **time_eager(net, slots, replays, args.warmup)})
    res["eager_forward_argmax"] = eager
    cross = {}
    for B in BATCHES:
        t = [r for r in rows if r["loss"] == "l1" and r["batch"] == B]
        if len(t) == 2:
            cross[B] = min(t, key=lambda r: r["p50_us"])["path"]
    res["faster_path_by_batch"] = cross
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bench_branched_serve.json"), "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
