"""Timing of the command-conditioned branched policy's training step (BASELINE configs[2]: the CNN BC policy on one B200,
bf16, batch 256, fused augment + encoder + branched heads), printed as one JSON line.

    python tools/branched_step_bench.py [--steps 200] [--warmup 20] [--out DIR]
    python tools/branched_step_bench.py --only-kernel            # bc_head_branched mode 3 alone
    python tools/branched_step_bench.py --dump-outputs DIR       # the head's results on seeded inputs, as .npy files

* main: trainer.BranchedTrainStep at B = 256, bf16, G = 4 branches, n_out = 3, L1 loss, augmentation (crop + colour jitter
  + normalise in the staging kernel) from 288x320 sources. Inputs rotate over 4 device slots of 260 frames (72 MB of
  frames each, 288 MB in all: more than the 126 MB L2). Per-step CUDA events over >= 200 graph replays -> p50 / p90.
* comparisons, timed in the same process and alternated block by block: the single-head CE TrainStep (no augmentation),
  BranchedTrainStep with G = 1, CE, n_out = 9 (no augmentation: the branched head against head_kernel), and the eager module
  path of the main workload (net.loss -> zero_grad -> backward -> MultiArenaAdam.step, staging included).
* kernel: bc_head_branched mode 3 (head forward + loss + backward + the partial reduction) alone, B = 256, G = 4, L1.

The kernel part and --dump-outputs use only ConvNet1Branched and bc_head_branched, which older checkouts have too, so a
copy of this script measures / dumps an older build the same way (--only-kernel skips the step parts)."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

NSLOT = 4


def device_meta(dev) -> dict:
    """Device name and power limit, from read-only queries."""
    meta = {"device": torch.cuda.get_device_name(dev), "power_limit_w": None, "sm_max_mhz": None}
    try:
        r = subprocess.run(["nvidia-smi", f"--id={dev.index}", "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30)
        if r.returncode == 0:
            p, c = [v.strip() for v in r.stdout.strip().split(",")[:2]]
            meta["power_limit_w"], meta["sm_max_mhz"] = float(p), float(c)
    except (OSError, ValueError, subprocess.SubprocessError):
        pass
    return meta


def _gen(dev, seed):
    return torch.Generator(device=dev).manual_seed(seed)


def branched_net(dev, G, n_out, kind, precision):
    from src.architectures.branched import ConvNet1Branched
    torch.manual_seed(12345)
    return ConvNet1Branched({"obs_size": 4, "n_actions": n_out, "n_branches": G, "branch_loss": kind,
                             "precision": precision}).to(dev)


def slot_inputs(dev, B, G, n_out, kind, src_hw, seed):
    """Seeded device inputs of one slot: frames (B+4, Hs, Ws, 3) u8, table or None, command, target."""
    from carla_imitation_learning_b200.data import augment_table
    g = _gen(dev, seed)
    hw = src_hw or (256, 256)
    frames = torch.randint(0, 256, (B + 4, hw[0], hw[1], 3), generator=g, dtype=torch.uint8, device=dev)
    table = None if src_hw is None else torch.from_numpy(augment_table(seed, B + 4, src_hw)).to(dev)
    command = torch.randint(0, G, (B,), generator=g, device=dev)
    target = (torch.randint(0, n_out, (B,), generator=g, device=dev) if kind == "ce"
              else torch.rand((B, n_out), generator=g, device=dev) * 2 - 1)
    return frames, table, command, target


# ------------------------------------------------------------------------------------------------ the head alone
def head_fixture(dev, B, G, n_out, kind, precision, seed):
    """A net with features from its trunk on seeded frames, the head's buffers and seeded commands / targets."""
    from carla_imitation_learning_b200 import sliding_window, stage_frames, stage_gray
    net = branched_net(dev, G, n_out, kind, precision)
    frames, _t, command, target = slot_inputs(dev, B, G, n_out, kind, None, seed)
    x = stage_frames(frames) if precision == "bf16" else sliding_window(stage_gray(frames))
    bufs = net._trunk_forward(net.engine().check_input(x), True)
    hb = net._bbufs(B)
    bufs.ghead.zero_()
    torch.cuda.synchronize()
    return net, bufs, hb, command, target


def time_head_kernel(dev, iters=2000, warmup=100):
    B, G, n_out, kind = 256, 4, 3, "l1"
    net, bufs, hb, command, target = head_fixture(dev, B, G, n_out, kind, "bf16", 7)
    for _ in range(warmup):
        net._head(bufs, hb, command, target, 3)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        net._head(bufs, hb, command, target, 3)
    e1.record()
    torch.cuda.synchronize()
    net.engine().check_device_errors()
    return {"what": "bc_head_branched mode 3 (head kernel + partial reduction), back-to-back launches",
            "batch": B, "n_branches": G, "n_out": n_out, "loss": kind, "iters": iters,
            "us_per_call": round(1000.0 * e0.elapsed_time(e1) / iters, 3)}


DUMP_CASES = (   # (name, B, G, n_out, kind, precision)
    ("b256_g4_l1_bf16", 256, 4, 3, "l1", "bf16"),
    ("b256_g4_ce_fp32", 256, 4, 9, "ce", "fp32"),
    ("b1000_g16_mse_fp32", 1000, 16, 3, "mse", "fp32"),
    ("b3000_g3_l1_bf16", 3000, 3, 3, "l1", "bf16"),
    ("b7_g1_ce_fp32", 7, 1, 9, "ce", "fp32"),
)


def dump_outputs(dev, out_dir):
    """mode 1 then mode 2 (the module path's two launches) and mode 3, on seeded inputs: out, dout, loss, gfeat and the
    branch gradients of each, as float32 .npy files (two builds run on the same inputs compare file for file)."""
    os.makedirs(out_dir, exist_ok=True)
    names = []
    for name, B, G, n_out, kind, prec in DUMP_CASES:
        net, bufs, hb, command, target = head_fixture(dev, B, G, n_out, kind, prec, 11)
        for mode_name, modes in (("m12", (1, 2)), ("m3", (3,))):
            for m in modes:
                net._head(bufs, hb, command, target if m & 1 else None, m)
            torch.cuda.synchronize()
            for key, t in (("out", hb["out"]), ("dout", hb["dout"]), ("loss", hb["loss"]), ("gfeat", bufs.ghead),
                           ("grads", hb["grads"])):
                fn = f"{name}_{mode_name}_{key}.npy"
                np.save(os.path.join(out_dir, fn), t.detach().float().cpu().numpy())
                names.append(fn)
        net._head(bufs, hb, command, None, 0)
        torch.cuda.synchronize()
        fn = f"{name}_m0_out.npy"
        np.save(os.path.join(out_dir, fn), hb["out"].detach().float().cpu().numpy())
        names.append(fn)
        net.engine().check_device_errors()
    return names


# ------------------------------------------------------------------------------------------------ steps
class Variant:
    def __init__(self, name, run, slots):
        self.name, self.run, self.slots, self.i = name, run, slots, 0

    def step(self):
        self.run(*self.slots[self.i % len(self.slots)])
        self.i += 1


def make_variants(dev):
    from carla_imitation_learning_b200 import FusedAdam, stage_augmented
    from carla_imitation_learning_b200.trainer import BranchedTrainStep, TrainStep
    from src.architectures.nets import ConvNet1
    B = 256
    v = {}
    # configs[2]: G = 4, n_out = 3, L1, augmentation from 288x320 sources
    net = branched_net(dev, 4, 3, "l1", "bf16")
    opt = net.configure_optimizer(lr=1e-3)
    st = BranchedTrainStep(net, opt, B, src_hw=(288, 320))
    aug_slots = [slot_inputs(dev, B, 4, 3, "l1", (288, 320), 100 + s) for s in range(NSLOT)]
    v["branched_g4_l1_aug"] = Variant("branched_g4_l1_aug", st.step, aug_slots)
    v["branched_g4_l1_aug"].owner = st
    # single-head CE TrainStep (what bench.py times), no augmentation
    torch.manual_seed(12345)
    net1 = ConvNet1({"obs_size": 4, "n_actions": 9, "precision": "bf16"}).to(dev)
    ts = TrainStep(net1, FusedAdam(list(net1.parameters()), lr=1e-3), B)
    ce_slots = [slot_inputs(dev, B, 1, 9, "ce", None, 200 + s) for s in range(NSLOT)]
    v["single_head_ce"] = Variant("single_head_ce", lambda f, t, c, y: ts.step(f, y), ce_slots)
    # G = 1, CE, n_out = 9, no augmentation: the branched head in place of head_kernel
    net_g1 = branched_net(dev, 1, 9, "ce", "bf16")
    st1 = BranchedTrainStep(net_g1, net_g1.configure_optimizer(lr=1e-3), B)
    v["branched_g1_ce"] = Variant("branched_g1_ce", st1.step, ce_slots)
    # the eager module path of the main workload, staging included
    net_e = branched_net(dev, 4, 3, "l1", "bf16")
    opt_e = net_e.configure_optimizer(lr=1e-3)

    def eager(f, t, c, y):
        x = stage_augmented(f, t, layout="tp")
        loss = net_e.loss(x, c, y)
        opt_e.zero_grad()
        loss.backward()
        opt_e.step()
    v["eager_module_g4_l1_aug"] = Variant("eager_module_g4_l1_aug", eager, aug_slots)
    return v, net


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=200, help="timed graph replays of the main workload (>= 200)")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5, help="alternated rounds of the comparisons")
    ap.add_argument("--block", type=int, default=40, help="steps per variant and round")
    ap.add_argument("--out", default=None, help="directory for bench_branched_step.json")
    ap.add_argument("--only-kernel", action="store_true", help="time bc_head_branched alone (runs on older checkouts too)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR", help="write the head's results on seeded inputs and exit")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("branched_step_bench: no CUDA device (this measures the B200 path; there is no CPU fallback)")
    from carla_imitation_learning_b200 import _lib
    _lib.build()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    if args.dump_outputs:
        names = dump_outputs(dev, args.dump_outputs)
        print(json.dumps({"dumped": len(names), "dir": args.dump_outputs}))
        return
    res = {"workload": "branched_train_step", "config": "BASELINE configs[2]", **device_meta(dev)}
    res["kernel"] = time_head_kernel(dev)
    if not args.only_kernel:
        B = 256
        v, net = make_variants(dev)
        main_v = v["branched_g4_l1_aug"]
        for var in v.values():                       # every slot: one eager pass, one capture, then warm replays
            for _ in range(max(args.warmup, 2 * NSLOT)):
                var.step()
        torch.cuda.synchronize()
        steps = max(args.steps, 200)
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0.record()
        for a, b in ev:
            a.record()
            main_v.step()
            b.record()
        w1.record()
        torch.cuda.synchronize()
        main_v.owner.check()
        per = np.array([a.elapsed_time(b) for a, b in ev])
        window_ms = w0.elapsed_time(w1)
        res["main"] = {
            "what": "BranchedTrainStep graph replay: augmenting staging + conv1..4 + branched heads (L1) + trunk backward "
                    "+ Adam on both arenas", "batch": B, "n_branches": 4, "n_out": 3, "loss": "l1", "precision": "bf16",
            "augment_src_hw": [288, 320], "steps": steps,
            "ms_per_step_p50": round(float(np.percentile(per, 50)), 4), "ms_per_step_p90": round(float(np.percentile(per, 90)), 4),
            "ms_per_step_mean_window": round(window_ms / steps, 4),
            "frames_per_s": round(B * steps / (window_ms / 1000.0), 1),
            "inputs": f"{NSLOT} rotating device slots of {B + 4} frames 288x320x3 u8 "
                      f"({(B + 4) * 288 * 320 * 3 / 1e6:.1f} MB each, {NSLOT * (B + 4) * 288 * 320 * 3 / 1e6:.0f} MB in all: larger than the 126 MB L2)",
            "final_loss": float(main_v.owner.hb["loss"]),
        }
        # alternated comparisons: each round times every variant over one block of steps
        blocks = {k: [] for k in v}
        for _ in range(args.rounds):
            for k, var in v.items():
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0 = time.perf_counter()
                e0.record()
                for _ in range(args.block):
                    var.step()
                e1.record()
                torch.cuda.synchronize()
                blocks[k].append((e0.elapsed_time(e1) / args.block, 1000.0 * (time.perf_counter() - t0) / args.block))
        res["compare"] = {"rounds": args.rounds, "steps_per_block": args.block, "batch": B, "variants": {
            k: {"ms_per_step_median": round(float(np.median([d for d, _ in bl])), 4),
                "ms_per_step_min": round(float(min(d for d, _ in bl)), 4),
                "host_ms_per_step_median": round(float(np.median([h for _, h in bl])), 4)} for k, bl in blocks.items()}}
        res["compare"]["notes"] = {
            "single_head_ce": "trainer.TrainStep, ConvNet1 single head + CE (n_out 9), plain staging",
            "branched_g1_ce": "BranchedTrainStep, G = 1, CE, n_out 9, plain staging",
            "branched_g4_l1_aug": "the main workload",
            "eager_module_g4_l1_aug": "stage_augmented + net.loss + zero_grad + backward + MultiArenaAdam.step, no graph"}
        res["value"] = res["main"]["frames_per_s"]
        res["unit"] = "frames/s"
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bench_branched_step.json"), "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
