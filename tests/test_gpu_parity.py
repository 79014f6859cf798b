"""Parity of the CUDA path (through the C ABI) against the CPU oracle and the golden vectors
the unmodified reference produced. Runs on the B200 box: `pytest -m gpu`.

Tolerances (BASELINE.json north_star): fp32 mode rel 1e-5, bf16-input mode rel 2e-2,
1k-step loss curve within 1 %. Max-pool routing is discontinuous, so gradient parity is
checked GIVEN the device's routing after proving each routed element is a window maximum
to within f32 rounding (see oracle.bc_oracle.explicit_backward).
"""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from oracle import bc_oracle as O

pytestmark = pytest.mark.gpu

REL_F32 = 1e-5
REL_BF16 = 2e-2


def _dev():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (no CPU fallback exists to run instead)")
    return torch.device("cuda", 0)


def _net(seed=12345, obs=4, na=9):
    from src.architectures.nets import ConvNet1
    torch.manual_seed(seed)
    return ConvNet1({"obs_size": obs, "n_actions": na})


def _params_cpu(net):
    return {k: v.detach().cpu() for k, v in net.state_dict().items()}


def _batch(seed, B):
    frames, labels = O.synth_frames(seed, B + 4)
    x, y = O.sequential_samples(frames, labels)
    return torch.from_numpy(x), torch.from_numpy(y), frames, labels


def _relerr(got, ref):
    got = np.asarray(got, np.float64); ref = np.asarray(ref, np.float64)
    return float(np.abs(got - ref).max() / max(np.abs(ref).max(), 1e-30))


def _flat(named):
    return np.concatenate([np.asarray(named[k].detach().cpu().double()).reshape(-1) for k in O.PARAM_ORDER])


def _grads_from_arena(net, flat):
    out = {}
    for (k, p) in net.named_parameters():
        out[k] = flat[p._bc_offset:p._bc_offset + p.numel()].view(p.shape).detach().cpu()
    return out


# ------------------------------------------------------------------------------- K0 staging
def test_stage_gray_bit_exact_all_rgb():
    """Every (R,G,B) triple: device f32 output == numpy's f64 dot /255 -> f32 (imitation_dataset.py:121,130)."""
    from carla_imitation_learning_b200 import stage_gray
    dev = _dev()
    r = np.arange(256, dtype=np.uint8)
    R, G, B = np.meshgrid(r, r, r, indexing="ij")
    rgb = np.stack([R, G, B], -1).reshape(16, 1024, 1024, 3)
    ref = O.gray_stack(rgb)
    got = stage_gray(torch.from_numpy(rgb).to(dev)).cpu().numpy()
    assert np.array_equal(got, ref), f"{int((got != ref).sum())} of 2^24 triples differ"
    got16 = stage_gray(torch.from_numpy(rgb).to(dev), dtype=torch.bfloat16).float().cpu().numpy()
    ref16 = torch.from_numpy(ref).to(torch.bfloat16).float().numpy()
    assert np.array_equal(got16, ref16)


def test_stage_frames_tp_bit_exact_all_rgb():
    """The Toeplitz-ready bf16 staging kernel (its own, cheaper arithmetic: csrc/stage.cu::gray_px_bf16_exact) on every
    (R,G,B) triple: both its outputs -- the plain bf16 planes and the TP planes -- equal bf16_rn(reference f32 gray)."""
    from carla_imitation_learning_b200 import stage_frames, _lib
    dev = _dev()
    r = np.arange(256, dtype=np.uint8)
    R, G, B = np.meshgrid(r, r, r, indexing="ij")
    rgb = np.stack([R, G, B], -1).reshape(256, 256, 256, 3)
    ref16 = torch.from_numpy(O.gray_stack(rgb)).to(torch.bfloat16)
    st = stage_frames(torch.from_numpy(rgb).to(dev), plain=True)
    tp, plain = st.tp, st.plain
    torch.cuda.synchronize()
    assert torch.equal(plain.cpu().view(torch.int16), ref16.view(torch.int16))
    # TP planes = a pure rearrangement of the plain planes (bc_planes_to_tp is the independent re-layout)
    tp2 = torch.empty_like(tp)
    _lib.check(_lib.lib().bc_planes_to_tp(plain.data_ptr(), _lib.BC_BF16, 256, 256 * 256, tp2.data_ptr(), torch.cuda.current_stream().cuda_stream), "bc_planes_to_tp")
    torch.cuda.synchronize()
    assert torch.equal(tp.view(torch.int16), tp2.view(torch.int16))


def test_stage_gray_golden_and_window(golden_dir):
    from carla_imitation_learning_b200 import stage_gray, sliding_window
    dev = _dev()
    g = np.load(os.path.join(golden_dir, "ref_gray.npz"))
    frames, _ = O.synth_frames(3, 5, 64, 48)
    got = stage_gray(torch.from_numpy(frames).to(dev)).cpu().numpy()
    assert np.array_equal(got, g["gray_f32"])
    frames, labels = O.synth_frames(9, 11)
    x_ref, _ = O.sequential_samples(frames, labels)
    win = sliding_window(stage_gray(torch.from_numpy(frames).to(dev)))
    assert tuple(win.shape) == (7, 4, 256, 256)
    assert np.array_equal(win.cpu().numpy(), x_ref)


def test_stage_gray_rejects_bad_input():
    from carla_imitation_learning_b200 import stage_gray
    dev = _dev()
    with pytest.raises(ValueError):
        stage_gray(torch.zeros(2, 8, 8, 4, dtype=torch.uint8, device=dev))
    with pytest.raises(RuntimeError):
        stage_gray(torch.zeros(2, 8, 8, 3, dtype=torch.uint8))          # host tensor: no CPU path
    out = stage_gray(torch.zeros(0, 8, 8, 3, dtype=torch.uint8, device=dev))  # empty is fine
    assert out.shape == (0, 8, 8)


# ------------------------------------------------------------------------------- per-layer forward
@pytest.mark.parametrize("layer,B", [(0, 3), (1, 5), (2, 7), (3, 37), (3, 1), (2, 1)])
def test_conv_relu_pool_layer(layer, B):
    from carla_imitation_learning_b200 import _lib
    dev = _dev()
    net = _net().to(dev)
    eng = net.engine()
    P = _params_cpu(net)
    name, k, s, p = O.CONV_SPECS[layer]
    cin = P[f"{name}.weight"].shape[1]
    hin = (256, 28, 12, 4)[layer]
    gen = torch.Generator().manual_seed(100 + layer)
    xin = torch.rand((B, cin, hin, hin), generator=gen) * (1.0 if layer == 0 else 0.5)
    x0 = xin if layer == 0 else torch.zeros(B, 4, 256, 256)
    bufs = eng.alloc(B, x0.to(dev), None, False)
    if layer > 0:
        bufs.act[layer - 1].copy_(xin.to(dev))
    c = eng.ctx(bufs)
    _lib.check(eng.lib.bc_conv_relu_pool_fwd(C.byref(c), layer, torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    z = torch.nn.functional.conv2d(xin.double(), P[f"{name}.weight"].double(), P[f"{name}.bias"].double(), stride=s)
    ref = torch.nn.functional.max_pool2d(torch.relu(z), p)
    got = bufs.act[layer].cpu().double()
    assert got.shape == ref.shape
    assert _relerr(got, ref) <= REL_F32, (layer, _relerr(got, ref))
    _check_routing(z, bufs.amax[layer].cpu(), got, p)


def _check_routing(z, amax, pooled, p, tol=2e-5):
    """Each routed element is a maximum of its window up to rounding; value equals relu(max)."""
    B, Cc, Hc, Wc = z.shape
    Hp, Wp = Hc // p, Wc // p
    win = z[..., :Hp * p, :Wp * p].reshape(B, Cc, Hp, p, Wp, p).permute(0, 1, 2, 4, 3, 5).reshape(B, Cc, Hp, Wp, p * p)
    assert int(amax.max()) < p * p
    chosen = win.gather(-1, amax.long()[..., None]).squeeze(-1)
    mx = win.max(-1).values
    scale = float(z.abs().max())
    live = pooled > 0
    assert float((mx - chosen)[live].abs().max() if live.any() else 0.0) <= tol * scale
    # exact first-max agreement wherever the window has a clear winner
    srt = win.sort(-1, descending=True).values
    clear = live & ((srt[..., 0] - srt[..., 1]) > tol * scale)
    first = (win == mx[..., None]).long().argmax(-1)
    assert bool((first[clear] == amax.long()[clear]).all())


# ------------------------------------------------------------------------------- whole network
@pytest.mark.parametrize("name", ["ref_step_b4.npz", "ref_step_b1.npz"])
def test_forward_and_loss_vs_reference_golden(golden_dir, name):
    dev = _dev()
    g = np.load(os.path.join(golden_dir, name))
    net = _net().to(dev)
    assert np.array_equal(_flat(dict(net.named_parameters())).astype(np.float32), g["init"])
    x, y, _, _ = _batch(int(g["data_seed"]), int(g["B"]))
    logits = net(x.to(dev)).detach().cpu().numpy()
    assert _relerr(logits, g["logits"]) <= REL_F32
    loss = net.loss(x.to(dev), y.to(dev))
    assert abs(float(loss) - float(g["loss"])) <= REL_F32 * abs(float(g["loss"]))
    torch.manual_seed(12345)
    ex = torch.randn((1, 4, 256, 256))
    assert torch.equal(ex, net.example_input_array)
    ex_logits = net(net.example_input_array).detach().cpu().numpy()     # train.py:120 smoke forward
    assert _relerr(ex_logits, g["example_logits"]) <= REL_F32


@pytest.mark.parametrize("B,seed", [(4, 0), (1, 1), (5, 2), (33, 3), (129, 4), (297, 5)])
def test_gradients_given_device_routing(B, seed, golden_dir):
    dev = _dev()
    net = _net().to(dev)
    eng = net.engine()
    x, y, _, _ = _batch(seed, B)
    bufs = eng.train_forward_backward(x.to(dev), y.to(dev))
    torch.cuda.synchronize()
    grads = _grads_from_arena(net, eng.grads)
    P = _params_cpu(net)
    amax = [a.cpu().long() for a in bufs.amax]
    loss, logits, ref, aux = O.explicit_backward(P, x, y, dtype=torch.float64, argmax_override=amax)
    for li in range(4):
        _check_routing(aux["conv_out"][li], bufs.amax[li].cpu(), bufs.act[li].cpu().double(), O.CONV_SPECS[li][3])
        assert _relerr(bufs.act[li].cpu(), aux["pooled"][li]) <= REL_F32
    assert _relerr(bufs.logits.cpu(), logits) <= REL_F32
    assert abs(float(bufs.loss) - float(loss)) <= REL_F32 * float(loss)
    worst = {}
    for k in O.PARAM_ORDER:
        worst[k] = _relerr(grads[k], ref[k])
    assert max(worst.values()) <= REL_F32, worst
    if B == 4 and seed == 0:   # the reference's own f32 gradients, when its routing matches ours
        g = np.load(os.path.join(golden_dir, "ref_step_b4.npz"))
        _, _, _, aux32 = O.explicit_backward(P, x, y, dtype=torch.float32)
        same = all(bool((a == b).all()) for a, b in zip(aux32["argmax"], amax))
        tol = REL_F32 if same else 5e-3   # one flipped near-tie moves conv1/conv2 grads by ~3e-3 (f32 vs f64 oracle)
        assert _relerr(_flat(grads), g["grads"]) <= tol, (same, _relerr(_flat(grads), g["grads"]))


def test_pool_ties_and_dead_relu_inputs():
    """All-zero and constant-255 frames: every window is an exact tie (SURVEY 8d value distributions)."""
    dev = _dev()
    net = _net().to(dev)
    eng = net.engine()
    P = _params_cpu(net)
    for fill in (0, 255):
        frames = np.full((7, 256, 256, 3), fill, np.uint8)
        labels = np.arange(7) % 9
        x, y = O.sequential_samples(frames, labels)
        x, y = torch.from_numpy(x), torch.from_numpy(y)
        bufs = eng.train_forward_backward(x.to(dev), y.to(dev))
        torch.cuda.synchronize()
        # constant input => every conv1 window is an exact tie; torch routes to element 0
        live = bufs.act[0].cpu() > 0
        assert bool((bufs.amax[0].cpu()[live] == 0).all())
        loss, logits, ref, _ = O.explicit_backward(P, x, y, dtype=torch.float64,
                                                   argmax_override=[a.cpu().long() for a in bufs.amax])
        assert _relerr(bufs.logits.cpu(), logits) <= REL_F32
        grads = _grads_from_arena(net, eng.grads)
        for k in O.PARAM_ORDER:
            assert _relerr(grads[k], ref[k]) <= REL_F32, (fill, k)


def test_sliding_window_view_equals_materialised_batch():
    from carla_imitation_learning_b200 import stage_gray, sliding_window
    dev = _dev()
    net = _net().to(dev)
    eng = net.engine()
    frames, labels = O.synth_frames(21, 13)
    y = torch.from_numpy(labels[4:13]).to(dev)
    win = sliding_window(stage_gray(torch.from_numpy(frames).to(dev)))
    b1 = eng.train_forward_backward(win, y)
    g1 = eng.grads.clone()
    b2 = eng.train_forward_backward(win.contiguous(), y)
    assert torch.equal(b1.logits, b2.logits) and torch.equal(g1, eng.grads)   # same kernels, same order: bitwise


def test_bf16_staged_input_within_bf16_tolerance():
    from carla_imitation_learning_b200 import stage_gray, sliding_window
    dev = _dev()
    net = _net().to(dev)
    eng = net.engine()
    frames, labels = O.synth_frames(5, 20)
    y = torch.from_numpy(labels[4:20]).to(dev)
    fr = torch.from_numpy(frames).to(dev)
    b32 = eng.train_forward_backward(sliding_window(stage_gray(fr)), y)
    g32 = eng.grads.clone()
    b16 = eng.train_forward_backward(sliding_window(stage_gray(fr, dtype=torch.bfloat16)), y)
    assert _relerr(b16.logits.cpu(), b32.logits.cpu()) <= REL_BF16
    assert abs(float(b16.loss) - float(b32.loss)) <= REL_BF16 * float(b32.loss)
    assert _relerr(eng.grads.cpu(), g32.cpu()) <= 5 * REL_BF16   # includes routing flips caused by input rounding


# ------------------------------------------------------------------------------- Adam
def test_fused_adam_three_steps_vs_reference_golden(golden_dir):
    dev = _dev()
    g = np.load(os.path.join(golden_dir, "ref_step_b4.npz"))
    adam = np.load(os.path.join(golden_dir, "ref_step_b4_adam.npz"))
    from src.models.imitation import Imitation
    net = _net().to(dev)
    model = Imitation({"obs_size": 4, "n_actions": 9}, net, {})
    opt = model.configure_optimizers()[0][0]
    x, y, _, _ = _batch(0, 4)
    x, y = x.to(dev), y.to(dev)
    init = g["init"].astype(np.float64)
    # Adam's first update is -lr*sign(g): where |g| is below the f32 noise of the gradient itself
    # (1e-5 of the layer maximum) the sign, hence the update, is not a property of the algorithm.
    # Compare where the reference gradient is resolvable; bound the rest by |update| <= lr.
    gref = np.abs(g["grads"].astype(np.float64))
    solid = np.zeros(gref.shape, bool)
    off = 0
    for shp in O.param_shapes().values():      # per tensor, like the gradient tolerance itself
        n = int(np.prod(shp))
        seg = gref[off:off + n]
        solid[off:off + n] = (seg > 1e-3 * seg.max()) | (seg == 0.0)   # exact zeros (dead ReLU paths) stay exact
        off += n
    assert solid.mean() > 0.6
    for i in range(3):
        loss = model.training_step((x, y), i)
        opt.zero_grad()
        loss.backward()
        opt.step()
        if i == 0:
            d = _flat(dict(net.named_parameters())) - init
            dref = adam["after1"].astype(np.float64) - init
            # a pool-routing flip between f32 CPU and f32 GPU arithmetic (DESIGN.md section 2) can move a few
            # small conv gradients across zero; those elements get the opposite +-lr update. Everything
            # else must match the reference update to f32 rounding.
            match = np.abs(d - dref) <= 2e-6
            assert match[solid].mean() >= 0.999, (match[solid].mean(), match.mean())
            assert match.mean() >= 0.99, match.mean()
            assert np.abs(d).max() <= 1e-3 * (1 + 1e-4)
    a3 = _flat(dict(net.named_parameters()))
    # steps 2 and 3 divide by sqrt(v): elements whose step-1 gradient was exactly 0 (dead paths) or at the
    # noise floor get updates whose sign is decided by rounding, in the reference as much as here
    # (measured: 92.6 % of elements agree to 2e-5 after 3 steps; all stay inside the 3*lr envelope; the
    # loss after 3 steps, asserted below, agrees to 1e-3).
    match3 = np.abs(a3 - adam["after3"].astype(np.float64)) <= 2e-5
    assert match3[solid].mean() >= 0.90, (match3[solid].mean(), match3.mean())
    assert np.abs(a3 - init).max() <= 3e-3 * 1.01      # |update| can exceed lr slightly once m/sqrt(v) > 1
    val = model.validation_step((x, y), 0)
    assert abs(float(val) - float(g["val_loss_after3"])) <= 1e-3 * float(g["val_loss_after3"])
    assert float(model._logged["val_loss"] if hasattr(model, "_logged") else val) == float(val)


def test_fused_adam_matches_oracle_formula_elementwise():
    from carla_imitation_learning_b200 import _lib
    dev = _dev()
    n = 4096
    gen = torch.Generator().manual_seed(5)
    p = torch.randn(n, generator=gen); m = torch.zeros(n); v = torch.zeros(n)
    pd, md, vd = p.to(dev), m.to(dev), v.to(dev)
    st = torch.tensor([1e-3, 0.9, 0.999, 1e-8, 0, 1.0, 0, 0], dtype=torch.float64, device=dev)
    lib, s = _lib.lib(), torch.cuda.current_stream().cuda_stream
    for t in range(1, 6):
        grad = torch.randn(n, generator=gen) * (10.0 ** (t - 3))
        O.adam_update(p, grad, m, v, t)
        gd = grad.to(dev)
        _lib.check(lib.bc_adam_tick(st.data_ptr(), s))
        _lib.check(lib.bc_adam_step(pd.data_ptr(), gd.data_ptr(), md.data_ptr(), vd.data_ptr(), st.data_ptr(), n, s))
        torch.cuda.synchronize()
        assert float(st[4]) == t
        assert float((pd.cpu() - p).abs().max()) <= 2e-7 * float(p.abs().max()) + 1e-9
        assert _relerr(md.cpu(), m) <= 1e-6 and _relerr(vd.cpu(), v) <= 1e-6


# ------------------------------------------------------------------------------- module contract
def test_lightning_contract_on_device():
    dev = _dev()
    from src.models.imitation import Imitation
    net = _net()
    assert next(net.parameters()).is_cuda            # placed on the B200 at construction
    assert list(net.state_dict().keys()) == list(O.PARAM_ORDER)
    out = net(net.example_input_array)               # train.py:120: CPU tensor in, logits out
    assert out.shape == (1, 9) and out.is_cuda
    model = Imitation({"obs_size": 4, "n_actions": 9}, net, {"train_dataloader": 1, "val_dataloader": 2, "test_dataloader": 3})
    assert (model.train_dataloader(), model.val_dataloader(), model.test_dataloader()) == (1, 2, 3)
    x, y, _, _ = _batch(4, 6)
    loss = model.training_step((x.to(dev), y.to(dev)), 0)
    assert loss.dim() == 0 and loss.requires_grad
    loss.backward()
    for k, p in net.named_parameters():
        assert p.grad is not None and p.grad.shape == p.shape, k
    # generic path: logits -> any loss -> autograd
    for p in net.parameters():
        p.grad = None
    logits = model(x.to(dev))
    torch.nn.functional.cross_entropy(logits, y.to(dev)).backward()
    g_generic = torch.cat([p.grad.reshape(-1) for p in net.parameters()])
    for p in net.parameters():
        p.grad = None
    model.training_step((x.to(dev), y.to(dev)), 0).backward()
    g_fused = torch.cat([p.grad.reshape(-1) for p in net.parameters()])
    assert _relerr(g_generic.cpu(), g_fused.cpu()) <= REL_F32
    opt, sch = model.configure_optimizers()
    assert isinstance(opt[0], torch.optim.Optimizer)
    before = net.fc[4].weight.detach().clone()
    opt[0].step(lambda: None)
    assert not torch.equal(before, net.fc[4].weight)
    model.training_epoch_end([{"loss": loss.detach()}])
    sd = opt[0].state_dict()
    assert set(sd["state"][0].keys()) >= {"step", "exp_avg", "exp_avg_sq"}
    # reference-format checkpoint round trip
    cpu_sd = {k: v.cpu() for k, v in net.state_dict().items()}
    net2 = _net(seed=1)
    net2.load_state_dict(cpu_sd)
    assert torch.equal(net2(x.to(dev)), net(x.to(dev)))
    assert torch.equal(net.act(x.to(dev)).cpu(), net(x.to(dev)).argmax(1).cpu())


def test_errors_are_loud():
    dev = _dev()
    net = _net()
    with pytest.raises(ValueError):
        net(torch.zeros(2, 4, 224, 224, device=dev))       # configs/model image_size 224 cannot work (SURVEY 0.1)
    with pytest.raises(ValueError):
        net.loss(torch.zeros(2, 4, 256, 256, device=dev), torch.zeros(3, dtype=torch.int64, device=dev))
    net.cpu()
    with pytest.raises(RuntimeError):
        net(torch.zeros(1, 4, 256, 256))                   # no CPU fallback


# ------------------------------------------------------------------------------- 1k-step loss curve
def test_loss_curve_1k_steps_within_one_percent(golden_dir, tmp_path):
    from carla_imitation_learning_b200 import stage_gray
    from src.models.imitation import Imitation
    dev = _dev()
    g = np.load(os.path.join(golden_dir, "ref_curve_b8_1k.npz"))
    B, steps = int(g["B"]), int(g["steps"])
    frames, labels = O.synth_frames(int(g["data_seed"]), steps * B + 4)
    net = _net().to(dev)
    model = Imitation({"obs_size": 4, "n_actions": 9}, net, {})
    opt = model.configure_optimizers()[0][0]
    lab = torch.from_numpy(labels).to(dev)
    losses = []
    chunk = 50 * B
    for s0 in range(0, steps, 50):
        fr = torch.from_numpy(frames[s0 * B: s0 * B + chunk + 4]).to(dev)
        gray = stage_gray(fr)
        for s in range(s0, s0 + 50):
            o = (s - s0) * B
            x = gray.as_strided((B, 4, 256, 256), (65536, 65536, 256, 1), gray.storage_offset() + o * 65536)
            y = lab[s * B + 4: s * B + 4 + B]
            loss = model.training_step((x, y), s)
            opt.zero_grad()
            loss.backward()
            opt.step()
            losses.append(loss.detach())
    got = torch.stack(losses).cpu().double().numpy()
    ref = g["losses"]
    np.save(os.path.join(os.environ.get("BC_TEST_OUT", str(tmp_path)), "curve_b8_1k_device.npy"), got)
    # (1) while the two trajectories are still the same trajectory, steps agree to rounding
    assert np.abs(got[:70] - ref[:70]).max() <= 1e-3 * ref[:70].max()
    # (2)-(5): within 1 % of the reference's own reproducibility envelope (tests/curve_check.py explains why a
    # bare 1 % band around ONE reference run is not a property the reference itself has)
    from tests.curve_check import check_curve
    check_curve(got, golden_dir, tol=1e-2)


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_inference_sweep_batches_match_oracle(mode):
    """BASELINE configs[4]: inference-only policy forward + greedy action over a batch sweep (1..4096; the closed-loop
    rollout of src/data/stat.py:41 uses B=1). Logits vs the oracle forward on the same weights: rel 1e-5 (fp32 mode) /
    2e-2 (bf16 mode); actions equal wherever the oracle's top-2 margin exceeds the tolerance."""
    from carla_imitation_learning_b200 import stage_frames, stage_gray, sliding_window
    from src.architectures.nets import ConvNet1
    dev = _dev()
    torch.manual_seed(12345)
    net = ConvNet1({"obs_size": 4, "n_actions": 9, "precision": mode}).to(dev)
    params = {k: v.detach().cpu() for k, v in net.state_dict().items()}
    tol = REL_F32 if mode == "fp32" else 2e-2
    frames, _ = O.synth_frames(4242, 4096 + 4)
    fr = torch.from_numpy(frames).to(dev)
    gray = stage_gray(fr)
    ref_all = O.forward(params, torch.from_numpy(O.gray_stack(frames[:132])).unfold(0, 4, 1).permute(0, 3, 1, 2)[:128])
    for B in (1, 2, 8, 9, 31, 128, 1024, 4096):      # up to engine.tail_batch = 8 the serving path is the one-launch tail
        if mode == "bf16":
            x = stage_frames(fr[:B + 4])
        else:
            x = sliding_window(gray[:B + 4])
        with torch.no_grad():
            logits = net(x)
            actions, served = net.engine().forward_act(x)      # what net.act() returns + the logits of that same launch chain
            assert torch.equal(net.act(x), actions)
        assert logits.shape == (B, 9) and actions.shape == (B,) and actions.dtype == torch.int64
        n = min(B, 128)
        ref = ref_all[:n].double()
        for lg in (logits, served.logits):
            got = lg[:n].cpu().double()
            assert float((got - ref).abs().max() / ref.abs().max()) <= tol, (mode, B)
        top2 = ref.topk(2, dim=1).values
        clear = (top2[:, 0] - top2[:, 1]) > 2 * tol * ref.abs().max()
        assert torch.equal(actions[:n].cpu()[clear], ref.argmax(1)[clear])
        assert torch.equal(actions.cpu(), served.logits.argmax(1).cpu())
    net.engine().check_device_errors()


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_policy_tail_matches_layer_kernels_and_oracle(mode):
    """csrc/policy_tail.cu (conv3 + conv4 + head + argmax as one 8-CTA-cluster launch, exact f32 arithmetic) against the
    layer-by-layer kernels and the f64 oracle, both paths forced at the same batch; also replayed from a CUDA graph
    (cluster launch + programmatic dependent launch inside a capture), as the serving loop of bench.py --workload infer does."""
    from carla_imitation_learning_b200 import stage_frames, stage_gray, sliding_window
    from src.architectures.nets import ConvNet1
    dev = _dev()
    torch.manual_seed(4321)
    net = ConvNet1({"obs_size": 4, "n_actions": 9, "precision": mode}).to(dev)
    eng = net.engine()
    params = {k: v.detach().cpu() for k, v in net.state_dict().items()}
    tol = REL_F32 if mode == "fp32" else 2e-2
    frames, _ = O.synth_frames(77, 65 + 4)
    fr = torch.from_numpy(frames).to(dev)
    ref_all = O.forward(params, torch.from_numpy(O.gray_stack(frames)).unfold(0, 4, 1).permute(0, 3, 1, 2)[:64]).double()
    for B in (1, 3, 16, 33, 64):
        x = stage_frames(fr[:B + 4]) if mode == "bf16" else sliding_window(stage_gray(fr[:B + 4]))
        a_tail, b_tail = eng.forward_act(x, tail=True)
        a_std, b_std = eng.forward_act(x, tail=False)
        torch.cuda.synchronize()
        ref = ref_all[:B]
        for lg in (b_tail.logits, b_std.logits):
            assert float((lg.cpu().double() - ref).abs().max() / ref.abs().max()) <= tol, (mode, B)
        assert torch.equal(a_tail.cpu(), b_tail.logits.argmax(1).cpu())
        assert torch.equal(a_std.cpu(), b_std.logits.argmax(1).cpu())
        if mode == "fp32":                     # same operands, different summation order only
            for i in (2, 3):
                assert _relerr(b_tail.act[i].cpu(), b_std.act[i].cpu()) <= REL_F32, (B, i)
            assert _relerr(b_tail.hid1.cpu(), b_std.hid1.cpu()) <= REL_F32 and _relerr(b_tail.hid2.cpu(), b_std.hid2.cpu()) <= REL_F32
            assert _relerr(b_tail.logits.cpu(), b_std.logits.cpu()) <= REL_F32
    with pytest.raises(ValueError):
        eng.forward_act(stage_frames(fr[:65 + 4]) if mode == "bf16" else sliding_window(stage_gray(fr[:65 + 4])), tail=True)
    # graph replay over two inputs written into the same staging buffers
    B = 2
    staged = stage_frames(fr[:B + 4]) if mode == "bf16" else None
    gray = None if mode == "bf16" else stage_gray(fr[:B + 4])
    x = staged if mode == "bf16" else sliding_window(gray)
    bufs = eng.alloc(B, x, None, False)
    out = torch.empty(B, dtype=torch.int64, device=dev)
    src = fr[:B + 4].clone()

    def enqueue():
        if mode == "bf16":
            stage_frames(src, out=staged)
        else:
            stage_gray(src, out=gray)
        eng.forward_act(x, out=out, bufs=bufs, tail=True)
    side = torch.cuda.Stream(dev)
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        enqueue()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        enqueue()
    for off in (10, 20, 0):
        src.copy_(fr[off:off + B + 4])
        g.replay()
        torch.cuda.synchronize()
        ref = ref_all[off:off + B]
        assert float((bufs.logits.cpu().double() - ref).abs().max() / ref.abs().max()) <= tol, (mode, off)
        assert torch.equal(out.cpu(), bufs.logits.argmax(1).cpu())
    eng.check_device_errors()


def test_stacked_12_channel_variant_matches_oracle():
    """BASELINE configs[3]: obs_size = 12 (3 cameras x 4 frames channel-stacked) at the 256x256 the architecture
    hard-codes (nets.py:14), exact-f32 kernels: forward, loss and all 14 gradients vs the f64 oracle given the device's routing.
    (The tensor-core mode of this variant: tests/test_gpu_stacked12.py.)"""
    from src.architectures.nets import ConvNet1
    dev = _dev()
    torch.manual_seed(7)
    net = ConvNet1({"obs_size": 12, "n_actions": 9}).to(dev)
    assert net.engine().conv_mode == 0
    params = {k: v.detach().cpu() for k, v in net.state_dict().items()}
    assert params["cnn_base.0.weight"].shape == (16, 12, 7, 7)
    gen = torch.Generator().manual_seed(3)
    B = 3
    x = torch.rand((B, 12, 256, 256), generator=gen)
    y = torch.randint(0, 9, (B,), generator=gen)
    eng = net.engine()
    bufs = eng.train_forward_backward(x.to(dev), y.to(dev))
    torch.cuda.synchronize()
    amax = [a.cpu().long() for a in bufs.amax]
    ref_loss, ref_logits, ref, _ = O.explicit_backward(params, x, y, dtype=torch.float64, argmax_override=amax)
    assert _relerr(bufs.logits.cpu(), ref_logits) <= REL_F32
    assert abs(float(bufs.loss) - float(ref_loss)) <= REL_F32 * float(ref_loss)
    for k, p in net.named_parameters():
        g = eng.grads[p._bc_offset:p._bc_offset + p.numel()].view(p.shape).cpu()
        assert _relerr(g, ref[k]) <= REL_F32, k


def test_stacked_camera_window_view_equals_materialised_batch():
    """configs[3] input pipeline: 3 cameras interleaved frame by frame -> sliding_window(frame_skip=12, step=3) is a zero-copy
    (B,12,256,256) batch; the step on the view == the step on the materialised copy, bit for bit."""
    from carla_imitation_learning_b200 import sliding_window, stage_gray
    from src.architectures.nets import ConvNet1
    dev = _dev()
    torch.manual_seed(7)
    net = ConvNet1({"obs_size": 12, "n_actions": 9}).to(dev)
    eng = net.engine()
    B = 5
    rng = np.random.Generator(np.random.PCG64(2))
    frames = torch.from_numpy(rng.integers(0, 256, size=(3 * (B + 4), 256, 256, 3), dtype=np.uint8)).to(dev)
    y = torch.from_numpy(rng.integers(0, 9, size=B)).to(dev)
    x = sliding_window(stage_gray(frames), frame_skip=12, step=3)
    assert tuple(x.shape) == (B, 12, 256, 256) and x.stride(0) == 3 * 65536 and x.stride(1) == 65536
    b1 = eng.train_forward_backward(x, y)
    g1 = eng.grads.clone()
    b2 = eng.train_forward_backward(x.contiguous(), y)
    torch.cuda.synchronize()
    assert torch.equal(b1.logits, b2.logits) and torch.equal(g1, eng.grads)
    # sample 1, channel (frame 2, camera 1) is plane 3*1 + 3*2 + 1
    gray = stage_gray(frames)
    assert torch.equal(x[1, 7], gray[3 + 7])


def test_imitation_aux_step_matches_the_reference_golden(golden_dir):
    """ImitationAux.training_step -> backward on the device against the UNMODIFIED reference's ImitationAux + lossCriterion
    (tests/golden/ref_aux_step_b4.npz): loss and all 14 gradients at rel 1e-5 (routing permitting, as for Imitation);
    validation_step returns the loss without logging 'val_loss'."""
    from carla_imitation_learning_b200 import sliding_window, stage_gray
    from src.architectures.nets import ConvNet1
    from src.models.imitation import ImitationAux
    dev = _dev()
    g = np.load(os.path.join(golden_dir, "ref_aux_step_b4.npz"))
    B = int(g["B"])
    frames, _labels = O.synth_frames(int(g["data_seed"]), B + 4)
    torch.manual_seed(12345)
    hp = {"obs_size": 4, "n_actions": 9}
    net = ConvNet1(hp).to(dev)
    model = ImitationAux(hp, net, {})
    x = sliding_window(stage_gray(torch.from_numpy(frames).to(dev)))
    y2 = torch.from_numpy(g["y2"]).to(dev)
    loss = model.training_step((x, y2), 0)
    loss.backward()
    torch.cuda.synchronize()
    assert abs(float(loss.detach()) - float(g["loss"])) <= REL_F32 * abs(float(g["loss"]))
    got = np.concatenate([p.grad.detach().cpu().reshape(-1).numpy() for p in (dict(net.named_parameters())[k] for k in O.PARAM_ORDER)])
    ref = g["grads"]
    # the reference's own f32 run and the device may route a pool window differently (DESIGN.md 2): bound by the routing-flip scale
    assert np.abs(got - ref).max() <= 5e-3 * np.abs(ref).max()
    val = model.validation_step((x, y2), 0)
    assert abs(float(val) - float(g["val_loss"])) <= REL_F32 * abs(float(g["val_loss"]))
    assert "val_loss" not in getattr(model, "_logged", {})


def _peer_exchange_world1(_proc, out_path, port):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    dist.init_process_group("nccl", rank=0, world_size=1, device_id=dev)
    try:
        from carla_imitation_learning_b200 import FusedAdam, stage_frames
        from carla_imitation_learning_b200.parallel import PeerExchangeStep
        from src.architectures.nets import ConvNet1
        frames, labels = O.synth_frames(9, 3 * 6 + 4)
        res = []
        for fused in (True, False):
            torch.manual_seed(12345)
            net = ConvNet1({"obs_size": 4, "n_actions": 9, "precision": "bf16"}).to(dev)
            eng = net.engine()
            opt = FusedAdam(list(net.parameters()), lr=1e-3)
            step = PeerExchangeStep(eng, opt) if fused else None
            for s in range(3):
                x = stage_frames(torch.from_numpy(frames[6 * s: 6 * s + 10]).to(dev))
                y = torch.from_numpy(labels[6 * s + 4: 6 * s + 10]).to(dev)
                eng.pack_weights()
                bufs = eng.alloc(6, x, y, True)
                if fused:
                    step(bufs)
                else:
                    eng.enqueue_train(bufs)
                    opt.step_flat(eng.grads)
            torch.cuda.synchronize()
            if fused:
                step.peer.check()
            res.append(net._arena.detach().cpu().numpy().copy())
        np.save(out_path, np.stack(res))
    finally:
        dist.destroy_process_group()


def test_fused_peer_exchange_adam_degenerates_to_adam_on_one_rank(tmp_path):
    """bc_adam_step_exchange (the data-parallel exchange fused into Adam over peer memory) on a world of ONE rank:
    flag handshakes with itself, one arena summed, grad_scale 1 -> bitwise the plain fused Adam after 3 steps.
    (The 2- and 8-GPU behaviour is checked by tools/dp_check.py; the driver's GPU test box has one GPU.)"""
    import socket
    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    out = str(tmp_path / "w.npy")
    mp.spawn(_peer_exchange_world1, args=(out, port), nprocs=1, join=True)
    w = np.load(out)
    assert np.array_equal(w[0], w[1])
