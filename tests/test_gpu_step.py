"""Parity of the step AS IT IS BENCHED and as the module contract drives it.

bench.py times trainer.TrainStep at B=256: staging into a persistent buffer, CUDA-graph replay, programmatic dependent
launch, the weight-gradient kernels on a side stream, the bf16 operand refresh folded into Adam. These tests run exactly
that object and compare it (a) bitwise with the plain eager enqueue of the same kernels and (b) with the f64 oracle
GIVEN the device's pool routing (oracle.bc_oracle.explicit_backward) at the tolerance BASELINE.json states for bf16 mode:
rel 2e-2 per tensor, outputs and all 14 gradients. (Reference lines: /root/reference/src/models/imitation.py:38-45,82-87.)
"""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from oracle import bc_oracle as O

pytestmark = pytest.mark.gpu

REL_BF16 = 2e-2
HP16 = {"obs_size": 4, "n_actions": 9, "precision": "bf16"}


def _dev():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (no CPU fallback exists to run instead)")
    return torch.device("cuda", 0)


def _net(hp=HP16, seed=12345):
    from src.architectures.nets import ConvNet1
    torch.manual_seed(seed)
    return ConvNet1(dict(hp)).to(_dev())


def _rel(got, ref):
    got, ref = got.detach().double().cpu(), ref.detach().double().cpu()
    return float((got - ref).abs().max() / ref.abs().max().clamp_min(1e-30))


def _named_grads(net, flat):
    return {k: flat[p._bc_offset:p._bc_offset + p.numel()].view(p.shape).detach().cpu() for k, p in net.named_parameters()}


def _uniform_frames(seed, n):
    rng = np.random.Generator(np.random.PCG64(seed))
    return rng.integers(0, 256, size=(n, 256, 256, 3), dtype=np.uint8), rng.integers(0, 9, size=n, dtype=np.int64)


# ------------------------------------------------------------------------------- bf16 whole step vs the oracle
@pytest.mark.parametrize("B,data", [(8, "synth"), (256, "uniform")])
def test_bf16_whole_step_matches_oracle_given_device_decisions(B, data):
    """bf16 (tcgen05) mode, whole step: pooled activations, logits, loss and ALL 14 gradients against the f64 oracle on
    the f32 master weights and f32 gray frames, GIVEN the device's discrete decisions (pool routing and ReLU masks);
    per tensor <= 2e-2 (north_star). Every decision that differs from the oracle's own is shown to be a rounding-level
    near-tie: the oracle's pre-activation of a flipped ReLU unit is within 2e-2 of the layer's scale of zero, and the
    routed element is a window maximum within the same tolerance. B=256 on uniform-noise frames is the benched
    configuration. (With the oracle's own masks the gradients differ by 3-17 % of max|grad|: one flipped unit moves a
    weight gradient by its whole contribution -- printed below for the record.)"""
    from carla_imitation_learning_b200 import stage_frames
    from tests.test_gpu_parity import _check_routing
    dev = _dev()
    net = _net()
    eng = net.engine()
    if data == "synth":
        frames, labels = O.synth_frames(31, B + 4)
    else:
        frames, labels = _uniform_frames(0, B + 4)
    y = torch.from_numpy(labels[4:4 + B].copy())
    bufs = eng.train_forward_backward(stage_frames(torch.from_numpy(frames).to(dev)), y.to(dev))
    torch.cuda.synchronize()
    eng.check_device_errors()
    got = _named_grads(net, eng.grads)
    P = {k: v.detach().cpu() for k, v in net.state_dict().items()}
    x, y2 = O.sequential_samples(frames, labels)
    assert np.array_equal(y2[:B], y.numpy())
    amax = [a.cpu().long() for a in bufs.amax]
    relu = {"pooled": [a.cpu() > 0 for a in bufs.act], "fc": [bufs.hid1.cpu() > 0, bufs.hid2.cpu() > 0]}
    torch.set_num_threads(os.cpu_count() or 1)
    xb = torch.from_numpy(x[:B])
    loss, logits, ref, aux = O.explicit_backward(P, xb, y, dtype=torch.float64, argmax_override=amax, relu_override=relu)
    for li in range(4):
        assert _rel(bufs.act[li], aux["pooled"][li]) <= REL_BF16, (li, _rel(bufs.act[li], aux["pooled"][li]))
        _check_routing(aux["conv_out"][li], bufs.amax[li].cpu(), aux["pooled"][li], O.CONV_SPECS[li][3], tol=REL_BF16)
    assert _rel(bufs.logits, logits) <= REL_BF16
    assert abs(float(bufs.loss) - float(loss)) <= REL_BF16 * float(loss)
    # the ReLU decisions that differ are near-ties at the bf16 rounding level, and they are few
    scale = {O.CONV_SPECS[li][0]: float(aux["conv_out"][li].abs().max()) for li in range(4)}
    scale["fc.0"], scale["fc.2"] = float(bufs.hid1.abs().max()), float(bufs.hid2.abs().max())
    sizes = {O.CONV_SPECS[li][0]: bufs.act[li].numel() for li in range(4)}
    sizes["fc.0"], sizes["fc.2"] = bufs.hid1.numel(), bufs.hid2.numel()
    for name, z in aux["relu_flips"].items():
        if z.numel():
            assert float(z.abs().max()) <= REL_BF16 * scale[name], (name, float(z.abs().max()), scale[name])
        assert z.numel() <= 0.02 * sizes[name] + 2, (name, z.numel(), sizes[name])
    worst = {k: _rel(got[k], ref[k]) for k in O.PARAM_ORDER}
    _, _, ref_own, _ = O.explicit_backward(P, xb, y, dtype=torch.float64, argmax_override=amax)
    own = {k: _rel(got[k], ref_own[k]) for k in O.PARAM_ORDER}
    print("bf16 step vs f64 oracle, B =", B, "given routing + ReLU masks:", {k: f"{v:.2e}" for k, v in worst.items()},
          "| given routing only:", {k: f"{v:.2e}" for k, v in own.items()},
          "| flipped ReLU units:", {k: int(v.numel()) for k, v in aux["relu_flips"].items()})
    assert max(worst.values()) <= REL_BF16, worst


# ------------------------------------------------------------------------------- the benched object
def _run_trainstep(B, steps, nbuf, graph, overlap, hp=HP16, lr_drop_at=None):
    from carla_imitation_learning_b200 import FusedAdam
    from carla_imitation_learning_b200.trainer import TrainStep
    dev = _dev()
    net = _net(hp)
    opt = FusedAdam(list(net.parameters()), lr=1e-3)
    ts = TrainStep(net, opt, B, overlap=overlap, graph=graph)
    data = [_uniform_frames(100 + i, B + 4) for i in range(nbuf)]
    fr = [torch.from_numpy(f).to(dev) for f, _ in data]
    lb = [torch.from_numpy(l[4:4 + B].copy()).to(dev) for _, l in data]
    losses = []
    for i in range(steps):
        if lr_drop_at is not None and i == lr_drop_at:
            opt.param_groups[0]["lr"] = 1e-4                      # what MultiStepLR does at a milestone (imitation.py:84-86)
        losses.append(ts.step(fr[i % nbuf], lb[i % nbuf]).clone())
    torch.cuda.synchronize()
    ts.check()
    return net, opt, ts, torch.stack(losses).cpu(), data


def test_benched_step_graph_pdl_overlap_equals_eager_bitwise_and_oracle():
    """B=256, stage_frames(out=) into the persistent planes, CUDA graph per input slot (every slot: eager pass, capture,
    replays), side-stream weight gradients, Adam with the operand refresh folded in -- after 7 steps over 2 rotating
    buffers the parameter arena, the Adam moments and every loss equal the plain eager serial enqueue BITWISE; and the
    first step's loss / the first update equal the oracle's within the bf16 tolerance."""
    B, steps, nbuf = 256, 7, 2
    net_g, opt_g, ts_g, loss_g, data = _run_trainstep(B, steps, nbuf, graph=True, overlap=True)
    assert len(ts_g._graphs) == nbuf                               # the graphs were really captured and replayed
    net_e, opt_e, ts_e, loss_e, _ = _run_trainstep(B, steps, nbuf, graph=False, overlap=False)
    assert torch.equal(loss_g, loss_e), (loss_g, loss_e)
    assert torch.equal(net_g._arena, net_e._arena)
    for a, b in zip(opt_g._bind()[1:3], opt_e._bind()[1:3]):
        assert torch.equal(a, b)
    assert float(opt_g._bind()[3][4]) == steps                     # the device step counter ticked once per replay
    # the bf16 operand images the Adam kernel maintained == a fresh pack of the final weights
    eng = net_g.engine()
    kept = eng.w_packed.clone()
    eng.pack_weights()
    torch.cuda.synchronize()
    assert torch.equal(kept, eng.w_packed)
    # oracle: loss of step 0 and the direction of the first update (f32 CPU oracle from the same init)
    frames, labels = data[0]
    x, y = O.sequential_samples(frames, labels)
    tr = O.OracleTrainer(O.init_params(12345))
    torch.set_num_threads(os.cpu_count() or 1)
    l0 = tr.step(torch.from_numpy(x[:B]), torch.from_numpy(y[:B]))
    assert abs(float(loss_g[0]) - l0) <= REL_BF16 * l0


def test_backward_overlap_is_bitwise_the_serial_backward():
    from carla_imitation_learning_b200 import stage_frames
    dev = _dev()
    frames, labels = O.synth_frames(5, 41)
    fr, y = torch.from_numpy(frames).to(dev), torch.from_numpy(labels[4:41].copy()).to(dev)
    res = []
    for overlap in (False, True):
        net = _net()
        eng = net.engine()
        eng.overlap = overlap
        b = eng.train_forward_backward(stage_frames(fr), y)
        torch.cuda.synchronize()
        eng.check_device_errors()
        res.append((eng.grads.clone(), b.loss.clone()))
    assert torch.equal(res[0][0], res[1][0]) and torch.equal(res[0][1], res[1][1])


def test_lr_milestone_reaches_the_captured_graph():
    """ADVICE r1: MultiStepLR changes param_groups[0]['lr'] on the host; the captured Adam kernel reads a device scalar.
    A drop between two REPLAYS must take effect: graph run == eager run bitwise, and the device scalar holds the new LR."""
    B = 8
    net_g, opt_g, ts_g, loss_g, _ = _run_trainstep(B, 8, 2, graph=True, overlap=True, lr_drop_at=6)
    net_e, opt_e, _, loss_e, _ = _run_trainstep(B, 8, 2, graph=False, overlap=False, lr_drop_at=6)
    assert len(ts_g._graphs) == 2
    assert float(opt_g._bind()[3][0]) == 1e-4
    assert torch.equal(net_g._arena, net_e._arena) and torch.equal(loss_g, loss_e)
    # and the drop mattered: without it the parameters end elsewhere
    net_n, _, _, _, _ = _run_trainstep(B, 8, 2, graph=True, overlap=True)
    assert not torch.equal(net_n._arena, net_g._arena)


def test_fused_adam_state_cannot_be_created_inside_a_capture():
    from carla_imitation_learning_b200 import FusedAdam
    net = _net()
    opt = FusedAdam(list(net.parameters()), lr=1e-3)
    eng = net.engine()
    g = torch.cuda.CUDAGraph()
    with pytest.raises(RuntimeError, match="before CUDA-graph capture"):
        with torch.cuda.graph(g):
            opt.step_flat(eng.grads)
    torch.cuda.synchronize()


def test_label_out_of_range_raises_at_the_check():
    from carla_imitation_learning_b200 import stage_frames
    dev = _dev()
    net = _net()
    eng = net.engine()
    frames, labels = O.synth_frames(3, 8)
    y = torch.from_numpy(labels[4:8].copy()).to(dev)
    y[2] = 9                                                        # n_actions = 9: one past the last class
    eng.train_forward_backward(stage_frames(torch.from_numpy(frames).to(dev)), y)
    with pytest.raises(RuntimeError, match="label outside"):
        eng.check_device_errors()
    eng.check_device_errors()                                        # the flag is cleared by the report
    with pytest.raises(ValueError):
        eng.train_forward_backward(stage_frames(torch.from_numpy(frames).to(dev)), y.int())     # int32 labels are refused


# ------------------------------------------------------------------------------- the module contract, fast path
def _module_run(hp, steps, B, frames, labels, accumulate=False):
    from carla_imitation_learning_b200.data import SequentialFrames
    from src.architectures.nets import ConvNet1
    from src.models.imitation import Imitation
    dev = _dev()
    torch.manual_seed(12345)
    net = ConvNet1(dict(hp)).to(dev)
    model = Imitation(dict(hp), net, {})
    opt = model.configure_optimizers()[0][0]
    loader = SequentialFrames(frames, labels, batch_size=B, device=dev, layout="tp" if hp.get("precision") == "bf16" else "plain")
    losses, n = [], 0
    while n < steps:
        for x, y in loader:
            if n >= steps:
                break
            loss = model.training_step((x, y), n)
            opt.zero_grad()
            loss.backward()
            opt.step()
            losses.append(loss.detach().clone())
            n += 1
    torch.cuda.synchronize()
    net.engine().check_device_errors()
    return net, opt, torch.stack(losses).cpu()


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_module_fast_path_equals_the_classic_module_path_bitwise(precision):
    """Imitation.training_step -> loss.backward() -> FusedAdam.step with `cuda_graph: true` (fused forward+backward replayed
    as a CUDA graph per loader slot, gradients handed to autograd without a copy) == the classic path (forward in
    training_step, CUDA backward inside loss.backward()): same losses, same parameters, bit for bit, over 9 steps
    (3 passes over a 3-batch loader: every slot is run eagerly, captured, replayed)."""
    B = 16
    frames, labels = O.synth_frames(11, 3 * B + 4)
    hp = {"obs_size": 4, "n_actions": 9, "precision": precision}
    net_c, _, loss_c = _module_run(hp, 9, B, frames, labels)
    net_f, opt_f, loss_f = _module_run(dict(hp, cuda_graph=True), 9, B, frames, labels)
    assert len(net_f._step_graphs.graphs) >= 2
    assert opt_f.stats["zero_copy"] == 9 and opt_f.stats["gathered"] == 0      # autograd adopted the arena views: no gradient copy
    assert torch.equal(loss_c, loss_f), (loss_c, loss_f)
    assert torch.equal(net_c._arena, net_f._arena)


def test_module_fast_path_honours_backward_gradient_and_accumulation():
    """loss.backward(gradient=g) scales the already computed gradients (bc_scale_inplace) and two backward() calls without
    zero_grad accumulate -- the autograd contract survives the fused step."""
    from carla_imitation_learning_b200 import stage_frames
    from src.architectures.nets import ConvNet1
    dev = _dev()
    frames, labels = O.synth_frames(13, 12)
    fr = torch.from_numpy(frames).to(dev)
    y = torch.from_numpy(labels[4:12].copy()).to(dev)
    torch.manual_seed(12345)
    ref_net = ConvNet1(dict(HP16)).to(dev)
    l = ref_net.loss(stage_frames(fr), y)
    l.backward()
    g_ref = {k: p.grad.clone() for k, p in ref_net.named_parameters()}
    torch.manual_seed(12345)
    net = ConvNet1(dict(HP16, fused_step=True)).to(dev)
    x = stage_frames(fr)
    net.loss(x, y).backward(gradient=torch.tensor(0.5, device=dev))
    for k, p in net.named_parameters():
        assert torch.allclose(p.grad, 0.5 * g_ref[k], rtol=1e-6, atol=0), k
    for _ in range(3):                                              # three more micro-steps, no zero_grad: 0.5 g + 3 g
        net.loss(x, y).backward()
    for k, p in net.named_parameters():
        assert torch.allclose(p.grad, 3.5 * g_ref[k], rtol=1e-5, atol=1e-12), k


def test_trainer_fit_writes_a_lightning_layout_checkpoint_that_round_trips(tmp_path):
    """Trainer.fit (the hook order of pl.Trainer for train.py:125-129) for 3 epochs with MultiStepLR milestones moved to
    [1, 2]; the .ckpt has Lightning's keys; a fresh module + optimiser restored from it continues bit-identically."""
    from carla_imitation_learning_b200.data import SequentialFrames
    from carla_imitation_learning_b200.trainer import Trainer, load_checkpoint_into
    from src.architectures.nets import ConvNet1
    from src.models.imitation import Imitation
    dev = _dev()
    B = 8
    hp = dict(HP16, cuda_graph=True)
    ftr, ltr = O.synth_frames(21, 4 * B + 4)
    fva, lva = O.synth_frames(22, 2 * B + 4)

    def build():
        torch.manual_seed(12345)
        net = ConvNet1(dict(hp)).to(dev)
        dl = {"train_dataloader": SequentialFrames(ftr, ltr, B, device=dev, layout="tp"),
              "val_dataloader": SequentialFrames(fva, lva, B, device=dev, layout="tp")}
        return Imitation(dict(hp), net, dl)

    model = build()
    tr = Trainer(max_epochs=2, default_root_dir=str(tmp_path))
    tr.fit(model)
    assert 'val_loss' in model._logged and tr.best_model_path and os.path.exists(tr.best_model_path)
    path = str(tmp_path / "last.ckpt")
    tr.save_checkpoint(model, path)
    ck = torch.load(path, map_location="cpu", weights_only=False)
    assert {"epoch", "global_step", "state_dict", "optimizer_states", "lr_schedulers", "pytorch-lightning_version"} <= set(ck)
    assert list(ck["state_dict"]) == ["net." + k for k in O.PARAM_ORDER]
    assert set(ck["optimizer_states"][0]["state"][0]) == {"step", "exp_avg", "exp_avg_sq"}
    sd_before = {k: v.clone() for k, v in model.state_dict().items()}
    # a fresh module + optimiser restored from the checkpoint
    model2 = build()
    opt2s, sch2s = model2.configure_optimizers()
    load_checkpoint_into(model2, path, opt2s[0], sch2s)
    for k, v in model2.state_dict().items():
        assert torch.equal(v, sd_before[k]), k
    st1, st2 = tr._opt._bind(), opt2s[0]._bind()
    assert torch.equal(st1[1], st2[1]) and torch.equal(st1[2], st2[2]) and float(st1[3][4]) == float(st2[3][4]) == 8.0
    # Imitation.load_from_checkpoint(path, hparams=, net=, data_loader=) as train.py:198-201 calls it
    torch.manual_seed(1)
    m3 = Imitation.load_from_checkpoint(path, hparams=dict(hp), net=ConvNet1(dict(hp)).to(dev), data_loader={})
    for k, v in m3.state_dict().items():
        assert torch.equal(v, sd_before[k]), k


# ------------------------------------------------------------------------------- data parallel
def _dp_worker(rank, world, port, out_dir, mode):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        from carla_imitation_learning_b200 import FusedAdam, stage_frames, stage_gray, sliding_window
        from carla_imitation_learning_b200.parallel import shard_range
        from carla_imitation_learning_b200.trainer import TrainStep, replicas_identical
        from src.architectures.nets import ConvNet1
        Bl, steps = 4, 6
        G = Bl * world
        frames, labels = O.synth_frames(5, steps * G + 4)
        hp = {"obs_size": 4, "n_actions": 9, "precision": mode}
        out = {}
        for kind in ("peer", "peer_serial", "nccl", "single"):
            torch.manual_seed(12345)
            net = ConvNet1(dict(hp)).to(dev)
            opt = FusedAdam(list(net.parameters()), lr=1e-3)
            if kind == "single":                        # the whole global batch on every rank, no exchange
                eng = net.engine()
                for s in range(steps):
                    f = torch.from_numpy(frames[s * G: s * G + G + 4]).to(dev)
                    y = torch.from_numpy(labels[s * G + 4: s * G + G + 4].copy()).to(dev)
                    x = stage_frames(f) if mode == "bf16" else sliding_window(stage_gray(f))
                    eng.train_forward_backward(x, y)
                    opt.step_flat(eng.grads)
            else:
                ts = TrainStep(net, opt, Bl, exchange="nccl" if kind == "nccl" else "peer", dp_overlap=(kind == "peer"), graph=(kind != "nccl"))
                lo, hi = shard_range(G, rank, world)
                slots = [(torch.empty((Bl + 4, 256, 256, 3), dtype=torch.uint8, device=dev), torch.empty(Bl, dtype=torch.int64, device=dev)) for _ in range(2)]
                for s in range(steps):
                    fr, lb = slots[s & 1]
                    fr.copy_(torch.from_numpy(frames[s * G + lo: s * G + hi + 4]))
                    lb.copy_(torch.from_numpy(labels[s * G + lo + 4: s * G + hi + 4].copy()))
                    ts.step(fr, lb)
                torch.cuda.synchronize()
                ts.check()
                assert replicas_identical(net._arena), kind
            torch.cuda.synchronize()
            out[kind] = net._arena.detach().cpu().numpy().copy()
        if rank == 0:
            np.savez(os.path.join(out_dir, f"dp_{mode}.npz"), **out)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_two_rank_peer_exchange_keeps_replicas_identical_and_equals_the_global_batch(tmp_path, mode):
    """2 GPUs (skipped on a 1-GPU box): the fused peer-memory exchange as CUDA graphs, bucket 0 under conv1's wgrad --
    replicas bitwise identical after 6 steps, equal to the un-overlapped exchange bitwise, to the NCCL exchange and to the
    single-process step on the global batch within rounding (train.py:125 `pl.Trainer(gpus=[...])` semantics)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs (tools/dp_check.py is the torchrun version)")
    import socket
    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_dp_worker, args=(2, port, str(tmp_path), mode), nprocs=2, join=True)
    w = np.load(str(tmp_path / f"dp_{mode}.npz"))
    assert np.array_equal(w["peer"], w["peer_serial"])
    # 6 Adam steps move weights by ~6e-3; early Adam is sign-like, so rounding-level gradient differences show up at ~1e-5
    assert np.abs(w["peer"] - w["nccl"]).max() <= 5e-5
    assert np.abs(w["peer"] - w["single"]).max() <= (5e-5 if mode == "fp32" else 4e-3)


def _module_dp_world1(_proc, out_path, port):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    dist.init_process_group("nccl", rank=0, world_size=1, device_id=dev)
    try:
        from carla_imitation_learning_b200.data import SequentialFrames
        from carla_imitation_learning_b200.parallel import ModuleExchange
        from src.architectures.nets import ConvNet1
        from src.models.imitation import Imitation
        B = 8
        frames, labels = O.synth_frames(17, 3 * B + 4)
        res = []
        for dp in (True, False):
            hp = dict(HP16, cuda_graph=True)
            torch.manual_seed(12345)
            net = ConvNet1(dict(hp)).to(dev)
            model = Imitation(dict(hp), net, {})
            opt = model.configure_optimizers()[0][0]
            if dp:
                ModuleExchange(net.engine(), opt)
            loader = SequentialFrames(frames, labels, B, device=dev, layout="tp")
            for _ep in range(3):
                for i, (x, y) in enumerate(loader):
                    loss = model.training_step((x, y), i)
                    opt.zero_grad()
                    loss.backward()
                    opt.step()
            torch.cuda.synchronize()
            net.engine().check_device_errors()
            if dp:
                net.engine().peer.check()
            res.append(net._arena.detach().cpu().numpy().copy())
        np.save(out_path, np.stack(res))
    finally:
        dist.destroy_process_group()


def test_module_path_data_parallel_exchange_degenerates_to_adam_on_one_rank(tmp_path):
    """Data parallelism through the module contract (FusedAdam.step -> ModuleExchange -> bc_adam_step_exchange over the
    double-buffered peer arenas, gradients produced in place by the fused graph step) on a world of one rank == the
    single-process module path, bitwise, after 9 steps."""
    import socket
    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    out = str(tmp_path / "w.npy")
    mp.spawn(_module_dp_world1, args=(out, port), nprocs=1, join=True)
    w = np.load(out)
    assert np.array_equal(w[0], w[1])


# ------------------------------------------------------------------------------- weight operands fetched before the dependency wait
@pytest.mark.parametrize("B", [8, 256])
def test_weights_fetched_before_the_dependency_wait_are_the_updated_ones(B):
    """The conv and head kernels fetch their weight operands BEFORE griddepcontrol.wait, under the previous kernel's tail;
    that is only sound because the kernels that WRITE parameters / operand images (Adam, pack) release their dependents
    after their last write. Worst case for that protocol: Adam directly followed by conv1's forward (pre-staged planes: no
    staging kernel in between) and Adam directly followed by the head, with a learning rate large enough that a stale
    weight changes every output. Back-to-back enqueue == the same sequence with a device synchronisation after every
    launch group, bitwise, over several steps."""
    from carla_imitation_learning_b200 import FusedAdam, _lib, stage_frames
    dev = _dev()
    frames, labels = _uniform_frames(7, B + 4)
    staged = stage_frames(torch.from_numpy(frames).to(dev))
    y = torch.from_numpy(labels[4:4 + B].copy()).to(dev)
    out = []
    for sync in (False, True):
        net = _net()
        eng = net.engine()
        opt = FusedAdam(list(net.parameters()), lr=3e-3)
        opt.prepare()
        eng.ensure_packed()
        b = eng.static_buffers(B, staged, y)
        torch.cuda.synchronize()
        logits = []
        for _ in range(5):
            eng.enqueue_train(b)                 # conv1 forward is the first launch: it follows the previous Adam directly
            if sync:
                torch.cuda.synchronize()
            opt.step_flat(eng.grads)
            if sync:
                torch.cuda.synchronize()
            # Adam -> head: the head's forward on the (old) act3 with the NEW fc weights
            _lib.check(eng.lib.bc_head(C.byref(eng.ctx(b)), 0, torch.cuda.current_stream().cuda_stream), "bc_head")
            if sync:
                torch.cuda.synchronize()
            logits.append(b.logits.clone())
        torch.cuda.synchronize()
        eng.check_device_errors()
        out.append((torch.stack(logits).cpu(), net._arena.clone().cpu(), eng.w_packed.clone().cpu()))
    (la, pa, wa), (lb, pb, wb) = out
    assert torch.isfinite(la).all()
    assert torch.equal(pa, pb) and torch.equal(wa, wb)
    assert torch.equal(la, lb)
    assert not torch.equal(la[0], la[-1])                          # the updates did change the outputs
