"""bench.py -- BC train frames/s on N B200s (BASELINE.json metric), with roofline and CPU baseline.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl b200|reference] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...          (N > 1)

One "step" = one optimisation step of the BC policy on `batch` frames per GPU:
stage (u8 RGB -> gray planes) -> conv1..4 (+ReLU+pool) -> head + CE -> backward -> [allreduce] -> Adam.
`value` = frames/s with the u8 frames already resident in HBM; `e2e` = the same step driven
from pinned HOST buffers (H2D of the frames and labels, D2H of the loss, every step).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "bc_train_frames_per_sec"
UNIT = "frames/s"
FLOPS_FWD = (44255232, 14745600, 5308416, 589824)          # SURVEY 8(d), per frame, conv1..4
FLOPS_TRAIN = 150505152
FRAME_BYTES = 256 * 256 * 3
# dram__bytes_read.sum + dram__bytes_write.sum per launch at B=256 from the `ncu --set full` captures under profiles/
TRAFFIC = {"conv1_fwd": 45933056,      # dram read + write per launch, profiles/r2P_ncu_full_raw.csv (44.81 MB + 1.12 MB)
           "conv1_wgrad": 54615552}    # same capture: 54.38 MB read (44.9 MB of planes, 1.21x) + 0.24 MB written


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def window(self, t0, t1):
        """Keep only samples taken inside [t0, t1] (host clock around the timed region)."""
        inside = [r for (t, r) in self.rows if t0 <= t <= t1 + 0.15]
        self.rows = [(0, r) for r in (inside if inside else [r for (_t, r) in self.rows][-3:])]

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        rows = [r for (_t, r) in self.rows]
        sm = sorted(float(r[0]) for r in rows if r and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def bind_to_gpu_numa_node(index: int):
    """Run this rank (and first-touch its pinned buffers) on the CPUs of the NUMA node its GPU hangs off. With 8 ranks
    uploading 51 MB per step each, host pages on the wrong socket halve the H2D rate. Best effort: returns the node or None."""
    try:
        bus = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=10).stdout.strip().lower()
        if bus.startswith("00000000:"):
            bus = bus[4:]                                     # sysfs uses a 4-digit PCI domain
        with open(f"/sys/bus/pci/devices/{bus}/numa_node") as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = set()
            for part in f.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if allowed:
            os.sched_setaffinity(0, allowed)
            return node
    except Exception:
        pass
    return None


def synth_host_frames(seed: int, n: int):
    """Uniform-noise CARLA-shaped u8 RGB frames + uniform labels (worst case for caches; SURVEY 8d)."""
    import numpy as np
    rng = np.random.Generator(np.random.PCG64(seed))
    return rng.integers(0, 256, size=(n, 256, 256, 3), dtype=np.uint8), rng.integers(0, 9, size=n, dtype=np.int64)


# ----------------------------------------------------------------------------------------------
REF_ROOT = "/root/reference"


def _cpu_trainer(B):
    """(step callable, kind, description): the reference's own CPU training loop for one batch. In the build container the
    UNMODIFIED reference classes are imported from /root/reference through the two import stubs in oracle/_stubs (`kind`
    "reference"); on the GPU box /root/reference does not exist and the oracle port runs (`kind` "port")."""
    import torch
    from oracle import bc_oracle as O
    frames, labels = synth_host_frames(0, B + 4)
    x, y = O.sequential_samples(frames, labels)
    x, y = torch.from_numpy(x), torch.from_numpy(y)
    if os.path.isdir(os.path.join(REF_ROOT, "src")) and not os.environ.get("BC_BENCH_FORCE_PORT"):
        try:
            sys.path[:0] = [os.path.join(ROOT, "oracle", "_stubs"), REF_ROOT]
            saved = {k: sys.modules.pop(k) for k in list(sys.modules) if k == "src" or k.startswith("src.")}
            from src.architectures.nets import ConvNet1 as RefNet       # /root/reference/src/architectures/nets.py:6
            from src.models.imitation import Imitation as RefImitation  # /root/reference/src/models/imitation.py:27
            torch.manual_seed(12345)
            hp = {"obs_size": 4, "n_actions": 9}
            model = RefImitation(hp, RefNet(hp), {})
            opt = model.configure_optimizers()[0][0]

            def step():
                loss = model.training_step((x, y), 0)
                opt.zero_grad()
                loss.backward()
                opt.step()
                return float(loss)
            return step, "reference", f"unmodified reference Imitation/ConvNet1 from {REF_ROOT} (torch {torch.__version__} CPU f32)"
        except Exception as e:  # pragma: no cover - falls through to the port
            sys.stderr.write(f"reference import failed ({e!r}); timing the oracle port instead\n")
        finally:
            for k in [k for k in sys.modules if k == "src" or k.startswith("src.")]:
                del sys.modules[k]
            sys.modules.update(saved)
            sys.path[:] = [p_ for p_ in sys.path if p_ not in (os.path.join(ROOT, "oracle", "_stubs"), REF_ROOT)]
    tr = O.OracleTrainer(O.init_params(12345))
    return (lambda: tr.step(x, y)), "port", f"oracle port of the reference loop (torch {torch.__version__} CPU f32)"


def run_reference(args):
    """The reference's own CPU path on the box's host cores, all threads, on the b200 arm's workload (batch `--batch`)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    B = args.batch
    step, kind, what = _cpu_trainer(B)
    warm = min(args.warmup, 3)
    for _ in range(warm):
        step()
    # bounded: the whole arm ends within a few minutes whatever --steps says
    n, t0 = 0, time.perf_counter()
    while n < args.steps and time.perf_counter() - t0 < 150.0:
        step()
        n += 1
    dt = time.perf_counter() - t0
    fps = B * n / dt
    sample = f"{what}, {cores} threads, {n} full steps of the {B}-frame batch, {1e3 * dt / n:.1f} ms/step"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus, "steps": n,
        "warmup": warm, "ms_per_step": 1e3 * dt / n, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD.format(B=B), "cpu_batch": B},
        "cpu_baseline": {"value": fps, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}), flush=True)


def cpu_baseline(B):
    import torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    step, kind, what = _cpu_trainer(B)
    for _ in range(2):
        step()
    n, t0 = 0, time.perf_counter()
    while n < 200 and time.perf_counter() - t0 < 12.0:
        step()
        n += 1
    dt = time.perf_counter() - t0
    return {"value": B * n / dt, "unit": UNIT, "cores": cores, "kind": kind,
            "sample": f"{what}, {cores} threads, {n} steps of the full {B}-frame batch in {dt:.1f} s, {1e3 * dt / n:.1f} ms/step"}


WORKLOAD = ("ConvNet1 BC train step (BASELINE configs[1]), obs 4x256x256, 9 actions, batch {B}/GPU, "
            "u8 RGB frames staged on the device, sliding 4-frame window")


def dump_outputs(out_dir, eng, bufs):
    """What the last timed step handed its caller, as float32 .npy files: the loss, the logits of its batch, and the
    parameters after its Adam update and the gradients of the step, both flattened in the module's parameter order.
    With the peer exchange the gradients are this rank's, from the half of the double-buffered arena the last step wrote."""
    import numpy as np
    import torch
    peer = eng.peer
    if peer is not None:
        half = peer.host_epoch & 1           # peer.current() is the half the NEXT step writes
        grads = peer.buf[half * peer.n:(half + 1) * peer.n]
    else:
        grads = eng.grads
    arrays = {"loss": bufs.loss.reshape(1), "logits": bufs.logits,
              "params": torch.cat([eng.arena[o:o + n] for o, n in zip(eng.offsets, eng.sizes)]),
              "grads": torch.cat([grads[o:o + n] for o, n in zip(eng.offsets, eng.sizes)])}
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t.detach().float().cpu().numpy())


def _event_ms(fn, reps=10, warm=3):
    import torch
    for _ in range(warm):
        fn()
    k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    k0.record()
    for _ in range(reps):
        fn()
    k1.record()
    torch.cuda.synchronize()
    return k0.elapsed_time(k1) / reps


# ----------------------------------------------------------------------------------------------
def run_b200(args):
    import ctypes as C
    import numpy as np
    import torch
    import torch.distributed as dist
    from carla_imitation_learning_b200 import FusedAdam, _lib
    from carla_imitation_learning_b200.data import SequentialFrames
    from carla_imitation_learning_b200.trainer import TrainStep, arena_checksum, replicas_identical
    from src.architectures.nets import ConvNet1
    from src.models.imitation import Imitation

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world == 1 and args.gpus > 1:
        raise SystemExit("launch N>1 with torch.distributed.run (see module docstring)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_numa_node(local)      # pinned host buffers are first-touched on the GPU's own NUMA node (e2e H2D path)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    _lib.build()
    B = args.batch
    hp = {"obs_size": 4, "n_actions": 9, "precision": ("bf16" if args.mode == "bf16" else "fp32")}
    torch.manual_seed(12345)
    net = ConvNet1(hp).to(dev)
    eng = net.engine()
    opt = FusedAdam(list(net.parameters()), lr=1e-3)
    ts = TrainStep(net, opt, B, exchange=args.dp, overlap=bool(args.overlap), graph=not args.no_graph, dp_overlap=bool(args.dp_overlap))

    # ---- data: NBUF distinct frame windows per rank (rotated so inputs are never L2-resident) ----
    NBUF = args.nbuf
    host_frames, host_labels, dev_frames, dev_labels = [], [], [], []
    for i in range(NBUF):
        f, l = synth_host_frames(1000 * rank + i, B + 4)
        hf = torch.from_numpy(f).pin_memory()
        hl = torch.from_numpy(l[4:4 + B].copy()).pin_memory()
        host_frames.append(hf); host_labels.append(hl)
        dev_frames.append(hf.to(dev)); dev_labels.append(hl.to(dev))

    def step(i):
        ts.step(dev_frames[i % NBUF], dev_labels[i % NBUF])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for i in range(max(args.warmup, 3, 2 * NBUF)):      # every input slot: one eager pass, one capture
        step(i)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_host0 = time.time()
    e0.record()
    for i in range(args.steps):
        step(i)
    e1.record()
    barrier()
    t_host1 = time.time()
    ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        # taken here, before the passes below rewrite the loss, logits and gradient buffers
        dump_outputs(args.dump_outputs, eng, ts.bufs)
    clocks = None
    if rank == 0:
        time.sleep(0.25)       # let the 100 ms sampler emit the rows that cover the end of the region
        sampler.window(t_host0, t_host1)
        clocks = sampler.stop()
    loss_dev = float(ts.bufs.loss)
    ts.check()

    # ---- e2e: host buffers in, loss out, every step -------------------------------------------
    # Default (`--e2e-api module`): through the reference-facing module contract -- the pinned-host loader
    # (data.SequentialFrames: H2D + staging on a side stream, step i+1's upload under step i's compute) feeds
    # Imitation.training_step -> zero_grad -> loss.backward() -> FusedAdam.step (train.py:125-129's loop), and the loss is read
    # on the host every step. `--e2e-api engine`: the same from two pinned slots straight into TrainStep.
    loss_host = torch.zeros((), dtype=torch.float32).pin_memory()
    e2e_api = args.e2e_api
    if e2e_api == "module":
        hp_m = dict(hp, cuda_graph=not args.no_graph, overlap_backward=bool(args.overlap))
        torch.manual_seed(12345)
        net_m = ConvNet1(hp_m).to(dev)
        model = Imitation(hp_m, net_m, {})
        opt_m = model.configure_optimizers()[0][0]
        if world > 1:
            from carla_imitation_learning_b200.parallel import ModuleExchange
            ModuleExchange(net_m.engine(), opt_m)
        seq = np.concatenate([host_frames[i].numpy()[: (B if i < NBUF - 1 else B + 4)] for i in range(NBUF)])     # NBUF*B + 4 frames
        lab = np.concatenate([np.zeros(4, np.int64)] + [host_labels[i].numpy() for i in range(NBUF)])
        loader = SequentialFrames(seq, lab, batch_size=B, device=dev, dtype=torch.float32, layout=("tp" if args.mode == "bf16" else "plain"))

        it = loader.cycle()       # endless: the next pass's first batch is uploaded under the current pass's last one

        def e2e_step(i):
            x, y = next(it)
            loss = model.training_step((x, y), i)
            opt_m.zero_grad()
            loss.backward()
            opt_m.step()
            loss_host.copy_(loss.detach(), non_blocking=True)
            torch.cuda.current_stream().synchronize()
            return float(loss_host)
    else:
        slots = [(torch.empty_like(dev_frames[0]), torch.empty_like(dev_labels[0])) for _ in range(2)]
        copy_stream = torch.cuda.Stream(dev)
        up_done = [torch.cuda.Event(), torch.cuda.Event()]

        def upload(i):
            fr, lb = slots[i & 1]
            with torch.cuda.stream(copy_stream):
                fr.copy_(host_frames[i % NBUF], non_blocking=True)
                lb.copy_(host_labels[i % NBUF], non_blocking=True)
                up_done[i & 1].record(copy_stream)

        def e2e_step(i):
            upload(i + 1)                                         # next step's inputs, overlapping this step's compute
            torch.cuda.current_stream().wait_event(up_done[i & 1])
            ts.step(*slots[i & 1])
            loss_host.copy_(ts.bufs.loss, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            return float(loss_host)
        upload(0)
    for i in range(max(6, 2 * NBUF + 2) if e2e_api == "module" else 6):
        e2e_step(i)
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    e2e_loss = 0.0
    for i in range(100, 100 + args.steps):
        e2e_loss = e2e_step(i)
    f1.record()
    barrier()
    ms_e2e = f0.elapsed_time(f1)
    if e2e_api == "module":
        net_m.engine().check_device_errors()
        if getattr(net_m.engine(), "peer", None) is not None:
            net_m.engine().peer.check()
        same_m = replicas_identical(net_m._arena)
    else:
        same_m = None

    # ---- the module path with device-resident inputs (the drop-in contract without the PCIe ceiling) --------------------
    module_dev = None
    if e2e_api == "module" and not args.no_module:
        from carla_imitation_learning_b200 import StagedBatch, stage_frames, stage_gray, sliding_window
        stg = [StagedBatch(torch.empty((B + 4, _lib.TP_PLANE_ELEMS), dtype=torch.bfloat16, device=dev), None, 4) for _ in range(2)] if args.mode == "bf16" \
            else [torch.empty((B + 4, 256, 256), dtype=torch.float32, device=dev) for _ in range(2)]

        def module_step(i):
            fr, lb = dev_frames[i % NBUF], dev_labels[i % NBUF]
            k = i & 1                      # two staging slots, like the loader's
            if args.mode == "bf16":
                x = stage_frames(fr, out=stg[k])
            else:
                x = sliding_window(stage_gray(fr, out=stg[k]))
            loss = model.training_step((x, lb), i)
            opt_m.zero_grad()
            loss.backward()
            opt_m.step()
        for i in range(max(6, 2 * NBUF + 2)):
            module_step(i)
        barrier()
        m0, m1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        m0.record()
        for i in range(args.steps):
            module_step(i)
        m1.record()
        barrier()
        module_dev = m0.elapsed_time(m1)
        net_m.engine().check_device_errors()

    # ---- per-kernel times, measured live with CUDA events on the launching stream (no profiler) -------
    bufs = ts.bufs
    c = eng.ctx(bufs)
    cref = C.byref(c)
    s = torch.cuda.current_stream().cuda_stream
    L = eng.lib
    # the staging kernel streams: its input rotates over the NBUF frame buffers (NBUF x 51 MB > L2), like in the timed loop --
    # on ONE buffer the frames stay L2-resident and the kernel looks faster than it is in the step
    rot = [0]
    def stage_rot():
        rot[0] = (rot[0] + 1) % NBUF
        ts._stage(dev_frames[rot[0]])
    ops = [("stage_gray", stage_rot)]
    ops += [(f"conv{l + 1}_fwd", (lambda l=l: _lib.check(L.bc_conv_relu_pool_fwd(cref, l, s)))) for l in range(4)]
    ops.append(("head_fwd_ce_bwd", lambda: _lib.check(L.bc_head(cref, 3, s))))
    for l in (3, 2, 1):
        ops.append((f"conv{l + 1}_wgrad", (lambda l=l: _lib.check(L.bc_conv_bwd_wgrad(cref, l, s)))))
        ops.append((f"conv{l + 1}_dgrad", (lambda l=l: _lib.check(L.bc_conv_bwd_dgrad(cref, l, s)))))
    ops.append(("conv1_wgrad", lambda: _lib.check(L.bc_conv_bwd_wgrad(cref, 0, s))))
    if world == 1:
        ops.append(("reduce_partials", lambda: _lib.check(L.bc_reduce_partials(cref, 1, s))))
    breakdown = {name: round(_event_ms(fn) * 1e3, 1) for name, fn in ops}
    if world == 1:
        # Adam (+ the bf16 operand refresh) on a scratch copy of the optimiser state: timing it must not train
        sp, sm, sv = eng.arena.clone(), torch.zeros_like(eng.arena), torch.zeros_like(eng.arena)
        sst = opt._bind()[3].clone()
        wp = eng.packed_ptr()
        scratch_pack = torch.empty_like(eng.w_packed) if wp else None
        breakdown["adam_tick_step" + ("_pack" if wp else "")] = round(_event_ms(lambda: _lib.check(L.bc_adam_tick_step(
            sp.data_ptr(), eng.grads.data_ptr(), sm.data_ptr(), sv.data_ptr(), sst.data_ptr(), sp.numel(),
            scratch_pack.data_ptr() if wp else None, 4, 9, s))) * 1e3, 1)
    if world > 1 and args.dp == "peer":
        # the fused exchange + Adam launch, timed live on every rank at once (it really exchanges: all ranks run the same 13 launches,
        # on the gradients of the last step -- the replicas stay identical, which the check below verifies after it)
        def xchg():
            c2 = eng.ctx(bufs)
            _lib.check(L.bc_reduce_partials(C.byref(c2), 1, s))
            ts.dp.exchange()
        ts.dp._bufs = bufs
        dist.barrier()
        breakdown["reduce_then_adam_exchange"] = round(_event_ms(xchg) * 1e3, 1)
        ts.check()
    eng.check_device_errors()
    stage_ms = breakdown["stage_gray"] * 1e-3
    # algorithmic bytes of the staging kernel: u8 RGB in; gray planes out (bf16 mode: Toeplitz-ready bf16 planes)
    stage_bytes = (B + 4) * (FRAME_BYTES + (2 * _lib.TP_PLANE_ELEMS if args.mode == "bf16" else 65536 * 4))

    if not (loss_dev == loss_dev and 0.0 < loss_dev < 20.0) or not (e2e_loss == e2e_loss and 0.0 < e2e_loss < 20.0):
        raise RuntimeError(f"training diverged or produced a non-finite loss ({loss_dev}, e2e {e2e_loss}): the timed run is invalid")
    same = replicas_identical(eng.arena)
    if not same or same_m is False:
        raise RuntimeError("data-parallel replicas DIFFER after the timed loop: the exchange is broken, the run is invalid")
    times = torch.tensor([ms, ms_e2e, module_dev or 0.0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    ms, ms_e2e, module_dev = float(times[0]), float(times[1]), (float(times[2]) if module_dev else None)
    if rank == 0:
        peaks = load_peaks()
        frames = B * world * args.steps
        value = frames / (ms * 1e-3)
        conv_k = {k: v for k, v in breakdown.items() if k.startswith("conv")}
        dom = max(conv_k, key=conv_k.get)                      # the longest kernel of the step
        names = {"conv1_fwd": "conv1_tp_kernel (tcgen05 Toeplitz implicit GEMM + ReLU + pool3, bf16)",
                 "conv1_wgrad": "conv1_wgrad3_kernel (tcgen05, plane-regrouped Toeplitz wgrad, bf16)"}

        def tensor_roofline(k):
            fl = FLOPS_FWD[int(k[4]) - 1] * B                  # SURVEY 8(d): fwd = dgrad = wgrad FLOPs per layer
            t = conv_k[k] * 1e-6
            tf = fl / t / 1e12
            return {"kernel": names.get(k, k) if args.mode == "bf16" else k + " (exact-f32 FFMA variant)", "bound": "tensor", "achieved": tf,
                    "peak": peaks["tf_burst"], "unit": "TFLOP/s", "frac": tf / peaks["tf_burst"], "traffic": TRAFFIC.get(k) if (args.mode == "bf16" and B == 256) else None,
                    "peak_source": peaks["src"] + " (bf16 cuBLAS burst)", "kernel_ms": conv_k[k] * 1e-3, "flops_per_launch": fl}
        roof = tensor_roofline(dom)
        roof["step_frac_of_dense_flops"] = FLOPS_TRAIN * B / (ms / args.steps * 1e-3) / 1e12 / peaks["tf_sust"]
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3, 2 * NBUF),
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": ("bf16" if args.mode == "bf16" else "f32"), "data": "synthetic",
            "config": {"workload": WORKLOAD.format(B=B),
                       "global_batch": B * world, "parallelism": f"dp{world}", "cuda_graph": not args.no_graph,
                       "overlap_backward": bool(args.overlap), "host_numa_node": numa,
                       "exchange": (None if world == 1 else ("adam kernel reads peer gradient arenas over NVLink"
                                                             + (", [fc..conv2] bucket under conv1's wgrad" if args.dp_overlap else "") if args.dp == "peer" else "nccl 2-bucket all-reduce")),
                       "replicas_identical": same, "arena_checksum": arena_checksum(eng.arena),
                       "l2": f"inputs rotate over {NBUF} x {(B + 4) * FRAME_BYTES / 1e6:.0f} MB device buffers (> 126 MB L2)",
                       "final_loss": loss_dev},
            "e2e": {"value": frames / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e / args.steps,
                    "h2d_bytes_per_step": (B + 4) * FRAME_BYTES + 8 * B, "d2h_bytes_per_step": 4,
                    "api": ("Imitation.training_step -> loss.backward() -> FusedAdam.step fed by data.SequentialFrames from pinned host frames"
                            if e2e_api == "module" else "trainer.TrainStep.step from two pinned host slots"),
                    "final_loss": e2e_loss},
            # per step: stage, 4 conv fwd, head, 3 x (wgrad, dgrad), conv1 wgrad, reduce, adam (tick + operand refresh folded in)
            "gpu_launches": 15 * args.steps,
            "roofline": roof,
            "roofline_conv1_fwd": tensor_roofline("conv1_fwd"),
            "roofline_conv1_wgrad": tensor_roofline("conv1_wgrad"),
            "roofline_hbm": {"kernel": ("stage_gray_tp_kernel" if args.mode == "bf16" else "stage_gray_kernel"), "bound": "hbm", "achieved": stage_bytes / (stage_ms * 1e-3) / 1e9,
                             "peak": peaks["hbm"], "unit": "GB/s", "frac": stage_bytes / (stage_ms * 1e-3) / 1e9 / peaks["hbm"],
                             "bytes_per_launch": stage_bytes, "kernel_ms": stage_ms,
                             "note": "algorithmic bytes (u8 RGB in + staged planes out); input rotated over buffers larger than L2; the staged planes (45 MB) stay in L2 for conv1, see profiles/ for dram__bytes"},
            # every conv kernel against the tensor roofline: algorithmic FLOPs (SURVEY 8d: fwd = dgrad = wgrad per layer) / live time
            "roofline_conv_tflops": {k: round(FLOPS_FWD[int(k[4]) - 1] * B / (v * 1e-6) / 1e12, 1) for k, v in conv_k.items()},
            "breakdown_us": breakdown,
            "clocks": clocks,
        }
        if module_dev:
            out["module_api"] = {"value": frames / (module_dev * 1e-3), "unit": UNIT, "ms_per_step": module_dev / args.steps,
                                 "what": "stage -> Imitation.training_step -> zero_grad -> loss.backward() -> FusedAdam.step, inputs resident in HBM",
                                 "frac_of_engine_value": (frames / (module_dev * 1e-3)) / value}
        if not args.no_cpu:
            out["cpu_baseline"] = cpu_baseline(B)
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ----------------------------------------------------------------------------------------------
def run_infer(args):
    """BASELINE configs[4]: inference-only policy forward + greedy action (imitation.py:34-36, src/data/stat.py:41), batch
    1..4096 on one B200: staging + conv1..4 + head (greedy action inside the head kernel) as ONE CUDA graph per batch size -- up
    to engine.tail_batch conv3, conv4, the head and the argmax are one cluster launch (csrc/policy_tail.cu); p50 / p99 latency over
    `--steps` replays (CUDA events around each replay), frames/s = B / p50. One JSON line; `value` = best frames/s."""
    import ctypes as C
    import numpy as np
    import torch
    from carla_imitation_learning_b200 import _lib, stage_frames, stage_gray, sliding_window
    from src.architectures.nets import ConvNet1
    _lib.build()
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    if int(os.environ.get("RANK", "0")) != 0:
        return
    torch.manual_seed(12345)
    bf16 = args.mode == "bf16"
    net = ConvNet1({"obs_size": 4, "n_actions": 9, "precision": "bf16" if bf16 else "fp32"}).to(dev)
    eng = net.engine()
    rng = np.random.Generator(np.random.PCG64(0))
    peaks = load_peaks()
    sweep, best, launches = [], None, 0
    sampler = ClockSampler(dev.index)
    sampler.start()
    t_host0 = time.time()
    reps = max(50, min(args.steps, 400))
    for B in (1, 2, 4, 8, 16, 32, 64, 128, 256, 512, 1024, 2048, 4096):
        nrot = 4 if (B + 4) * FRAME_BYTES * 4 < (2 << 30) else 2
        frames = [torch.from_numpy(rng.integers(0, 256, size=(B + 4, 256, 256, 3), dtype=np.uint8)).to(dev) for _ in range(nrot)]
        if bf16:
            staged = stage_frames(frames[0])
            bufs = eng.alloc(B, staged, None, False)
        else:
            gray = torch.empty((B + 4, 256, 256), dtype=torch.float32, device=dev)
            bufs = eng.alloc(B, sliding_window(gray), None, False)
        actions = torch.empty(B, dtype=torch.int64, device=dev)

        def measure(tail):
            """p50 / p99 latency (us) of one graph replay: staging + forward + greedy action; tail = conv3..argmax as one launch"""
            def enqueue(fr):
                if bf16:
                    stage_frames(fr, out=staged)
                else:
                    stage_gray(fr, out=gray)
                c = eng.ctx(bufs)
                s = torch.cuda.current_stream().cuda_stream
                _lib.check(eng.lib.bc_forward_act(C.byref(c), actions.data_ptr(), int(tail), s))
            side = torch.cuda.Stream(dev)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for k in range(3):
                    enqueue(frames[k % nrot])
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            graphs = []
            for fr in frames:
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    enqueue(fr)
                graphs.append(g)
            for k in range(5):
                graphs[k % nrot].replay()
            torch.cuda.synchronize()
            ts = []
            for k in range(reps):
                a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a0.record(); graphs[k % nrot].replay(); a1.record()
                torch.cuda.synchronize()
                ts.append(a0.elapsed_time(a1) * 1e3)
            ts = np.sort(np.asarray(ts))
            del graphs
            return float(ts[len(ts) // 2]), float(ts[min(len(ts) - 1, int(len(ts) * 0.99))])
        served_tail = B <= eng.tail_batch                    # the path ConvNet1.act() takes at this batch
        p50, p99 = measure(served_tail)
        row = {"batch": B, "latency_us_p50": round(p50, 1), "latency_us_p99": round(p99, 1), "frames_per_s": round(B / (p50 * 1e-6)),
               "tflops": round(64920128 * B / (p50 * 1e-6) / 1e12, 2), "path": "tail" if served_tail else "layers",
               "launches": 4 if served_tail else 6}
        if B <= 64:                                          # the other path at the same batch, for the crossover
            o50, o99 = measure(not served_tail)
            row["other_path_us_p50"], row["other_path_us_p99"] = round(o50, 1), round(o99, 1)
            launches += reps * (6 if served_tail else 4)
        launches += reps * row["launches"]
        sweep.append(row)
        if best is None or row["frames_per_s"] > best["frames_per_s"]:
            best = row
        del frames, bufs
    eng.check_device_errors()
    t_host1 = time.time()
    time.sleep(0.25)
    sampler.window(t_host0, t_host1)
    clocks = sampler.stop()
    ach = best["tflops"]
    print(json.dumps({
        "metric": "bc_infer_frames_per_sec", "value": best["frames_per_s"], "unit": UNIT, "n_gpus": 1, "steps": reps, "warmup": 8,
        "ms_per_step": best["latency_us_p50"] * 1e-3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16" if bf16 else "f32", "data": "synthetic",
        "config": {"workload": "ConvNet1 policy forward + greedy action (BASELINE configs[4]), obs 4x256x256, batch sweep 1..4096, "
                               "u8 RGB frames staged on the device, one CUDA graph per batch size", "best_batch": best["batch"],
                   "l2": "inputs rotate over 2-4 device buffers per batch size"},
        "sweep": sweep,
        "roofline": {"kernel": "whole forward graph at the best batch (stage + conv1..4 + head with the greedy action)", "bound": "tensor", "achieved": ach,
                     "peak": peaks["tf_sust"], "unit": "TFLOP/s", "frac": ach / peaks["tf_sust"], "traffic": None,
                     "flops_per_frame": 64920128, "peak_source": peaks["src"] + " (bf16 cuBLAS sustained)"},
        "gpu_launches": launches, "clocks": clocks}), flush=True)


def run_stacked12(args):
    """BASELINE configs[3]: the channel-stacked multi-camera variant -- obs_size 12 = 3 cameras x 4 frames, 256x256 (what
    nets.py:14 hard-codes), one B200 per rank, weak scaling. `--mode bf16` (default): every convolution on tcgen05, conv1 as three
    4-frame camera streams accumulated into one result (csrc/conv1_tc.cu); `--mode fp32`: the exact FFMA kernels.
    The three cameras' frames are interleaved frame by frame in the u8 input, so a sample is a zero-copy window of 12
    consecutive gray planes advancing by 3 (stage_frames(frame_skip=12, step=3) / sliding_window(step=3)); stage -> forward ->
    backward -> Adam as one CUDA graph."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from carla_imitation_learning_b200 import FusedAdam, StagedBatch, _lib, sliding_window, stage_frames, stage_gray
    from src.architectures.nets import ConvNet1
    bf16 = args.mode == "bf16"
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.build()
    B = args.batch                                        # 256 per GPU like configs[1] (the exact-f32 mode is ~8x slower per frame: use --batch 64 --mode fp32 for it)
    torch.manual_seed(12345)
    net = ConvNet1({"obs_size": 12, "n_actions": 9, "precision": args.mode}).to(dev)
    eng = net.engine()
    opt = FusedAdam(list(net.parameters()), lr=1e-3)
    nfr = 3 * (B + 4)                                     # 3 cameras x (B + 4) frames: sample b = frames b..b+3 of every camera (+ the frame that carries its label)
    rng = np.random.Generator(np.random.PCG64(7 + rank))
    frames = [torch.from_numpy(rng.integers(0, 256, size=(nfr, 256, 256, 3), dtype=np.uint8)).to(dev) for _ in range(2)]
    labels = torch.from_numpy(rng.integers(0, 9, size=B)).to(dev)
    if bf16:
        x = StagedBatch(torch.empty((nfr, _lib.TP_PLANE_ELEMS), dtype=torch.bfloat16, device=dev), None, 12, 3)
    else:
        gray = torch.empty((nfr, 256, 256), dtype=torch.float32, device=dev)
        x = sliding_window(gray, frame_skip=12, step=3)
    assert x.shape[0] == B
    bufs = eng.alloc(B, x, labels, True)
    opt.prepare()
    xchg = None
    if world > 1:
        from carla_imitation_learning_b200.parallel import PeerExchangeStep
        xchg = PeerExchangeStep(eng, opt)

    def enqueue(fr):
        if bf16:
            stage_frames(fr, out=x, frame_skip=12, step=3)
        else:
            stage_gray(fr, out=gray)
        if xchg is not None:
            xchg(bufs)
        else:
            eng.enqueue_train(bufs)
            opt.step_flat(eng.grads)
    for i in range(3):
        enqueue(frames[i & 1])
    torch.cuda.synchronize()
    graphs = []
    for fr in frames:
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            enqueue(fr)
        graphs.append(g)

    def step(i):
        opt.prepare()
        graphs[i & 1].replay()
        if xchg is not None:
            xchg.peer.host_epoch += 1
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for i in range(max(args.warmup, 3)):
        step(i)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.time()
    e0.record()
    for i in range(args.steps):
        step(i)
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t1 = time.time()
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms[0])
    loss = float(bufs.loss)
    eng.check_device_errors()
    if xchg is not None:
        xchg.peer.check()
    if not (loss == loss and 0.0 < loss < 20.0):
        raise RuntimeError(f"non-finite loss {loss}")
    if rank == 0:
        time.sleep(0.25)
        sampler.window(t0, t1)
        clocks = sampler.stop()
        peaks = load_peaks()
        flops = 327.5e6                                   # SURVEY 8(d): train FLOPs per frame at 12 channels, 256x256
        value = B * world * args.steps / (ms * 1e-3)
        print(json.dumps({
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16" if bf16 else "f32", "data": "synthetic",
            "config": {"workload": f"ConvNet1 BC train step, channel-stacked variant (BASELINE configs[3]): obs 12 = 3 cameras x 4 frames at 256x256, "
                                   f"batch {B}/GPU, " + ("tcgen05 kernels (conv1 = three camera streams)" if bf16 else "exact-f32 FFMA kernels")
                                   + ", u8 RGB frames staged on the device", "global_batch": B * world,
                       "parallelism": f"dp{world}", "cuda_graph": True, "final_loss": loss,
                       "l2": "inputs alternate over 2 device buffers of %d MB" % (nfr * FRAME_BYTES // 1000000)},
            "roofline": {"kernel": "whole step (" + ("tcgen05 kernels" if bf16 else "f32 FFMA kernels") + ")", "bound": "tensor", "achieved": flops * value / 1e12, "peak": peaks["tf_sust"],
                         "unit": "TFLOP/s", "frac": flops * value / 1e12 / peaks["tf_sust"], "traffic": None,
                         "note": "algorithmic FLOPs of the 12-channel step (327.5 MFLOP/frame) against the sustained bf16 tensor peak" + ("" if bf16 else "; the exact-f32 path runs on CUDA cores")},
            "gpu_launches": (19 if bf16 else 15) * args.steps, "clocks": clocks}), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--batch", type=int, default=256, help="frames per GPU per step")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="train", choices=["train", "infer", "stacked12"],
                    help="train = BASELINE configs[1]/[2]; infer = configs[4] batch sweep; stacked12 = configs[3] (12 channels = 3 cameras x 4 frames)")
    ap.add_argument("--mode", default="bf16", choices=["fp32", "bf16"], help="fp32 = exact FFMA kernels; bf16 = tcgen05 kernels")
    ap.add_argument("--nbuf", type=int, default=4)
    ap.add_argument("--dp", default="peer", choices=["peer", "nccl"], help="N>1 gradient exchange: fused peer-memory Adam, or NCCL buckets")
    ap.add_argument("--dp-overlap", type=int, default=0, help="peer exchange: [fc..conv2] bucket on a side stream under conv1's wgrad")
    ap.add_argument("--overlap", type=int, default=0, help="weight-gradient kernels of conv4..conv2 on a side stream (bc_backward_overlap)")
    ap.add_argument("--e2e-api", default="module", choices=["module", "engine"])
    ap.add_argument("--no-module", action="store_true", help="skip the device-resident module-path measurement")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="train workload: write what the last timed step computed (loss, logits, parameters, gradients) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or args.workload != "train"):
        ap.error("--dump-outputs is implemented for --impl b200 --workload train")
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "infer":
        run_infer(args)
    elif args.workload == "stacked12":
        run_stacked12(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
