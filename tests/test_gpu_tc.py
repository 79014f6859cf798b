"""tcgen05 / TMEM building blocks (csrc/tc05.cuh) pinned by a plain bf16 GEMM through the C ABI."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("M,N,K", [(128, 64, 16), (128, 16, 16), (256, 64, 64), (300, 128, 208), (128, 256, 32), (1000, 64, 448)])
def test_tc_gemm_selftest(M, N, K):
    from carla_imitation_learning_b200 import _lib
    assert torch.cuda.is_available()
    dev = torch.device("cuda", 0)
    gen = torch.Generator().manual_seed(M * 7 + N * 3 + K)
    A = torch.randn((M, K), generator=gen).to(torch.bfloat16)
    B = torch.randn((N, K), generator=gen).to(torch.bfloat16)
    Ad, Bd = A.to(dev), B.to(dev)
    D = torch.full((M, N), float("nan"), dtype=torch.float32, device=dev)
    err = torch.zeros(1, dtype=torch.int32, device=dev)
    _lib.check(_lib.lib().bc_tc_gemm_selftest(Ad.data_ptr(), Bd.data_ptr(), D.data_ptr(), M, N, K, err.data_ptr(),
                                             torch.cuda.current_stream().cuda_stream), "bc_tc_gemm_selftest")
    torch.cuda.synchronize()
    assert int(err[0]) == 0, "mbarrier wait timed out inside the kernel"
    ref = A.double() @ B.double().t()
    got = D.cpu().double()
    assert torch.isfinite(got).all()
    # bf16 products are exact in f32; only the f32 accumulation order differs
    assert float((got - ref).abs().max()) <= 1e-5 * float(ref.abs().max()) * max(1, K // 64)


@pytest.mark.parametrize("B", [1, 3, 40])
def test_conv1_tcgen05_matches_bf16_rounded_oracle(B):
    """conv1+ReLU+pool on tensor cores == f64 conv of the bf16-ROUNDED inputs and weights (products of
    bf16 values are exact in f32, so only accumulation order separates the two): rel 1e-5, plus routing."""
    import ctypes as C
    from carla_imitation_learning_b200 import _lib, stage_gray, sliding_window
    from oracle import bc_oracle as O
    from src.architectures.nets import ConvNet1
    from tests.test_gpu_parity import _check_routing
    dev = torch.device("cuda", 0)
    torch.manual_seed(12345)
    net = ConvNet1({"obs_size": 4, "n_actions": 9}).to(dev)
    eng = net.engine()
    eng.set_mode("bf16")
    eng.pack_weights()
    frames, _ = O.synth_frames(50 + B, B + 4)
    gray = stage_gray(torch.from_numpy(frames).to(dev), dtype=torch.bfloat16)
    x = sliding_window(gray)
    bufs = eng.alloc(B, x, None, False)
    c = eng.ctx(bufs)
    _lib.check(eng.lib.bc_conv_relu_pool_fwd(C.byref(c), 0, torch.cuda.current_stream().cuda_stream), "conv1 tc")
    torch.cuda.synchronize()
    eng.check_device_errors()
    w = net.cnn_base[0].weight.detach().to(torch.bfloat16).double().cpu()
    bias = net.cnn_base[0].bias.detach().double().cpu()
    z = torch.nn.functional.conv2d(x.double().cpu(), w, bias, stride=3)
    ref = torch.nn.functional.max_pool2d(torch.relu(z), 3)
    got = bufs.act[0].cpu().double()
    err = float((got - ref).abs().max() / ref.abs().max())
    assert err <= 1e-5, err
    _check_routing(z, bufs.amax[0].cpu(), got, 3)
    # and against the un-rounded f32 network it is inside the bf16 tolerance of the north star
    z32 = torch.nn.functional.conv2d(x.float().cpu().double(), net.cnn_base[0].weight.detach().double().cpu(), bias, stride=3)
    ref32 = torch.nn.functional.max_pool2d(torch.relu(z32), 3)
    assert float((got - ref32).abs().max() / ref32.abs().max()) <= 2e-2


def test_bf16_mode_training_step_within_tolerance():
    from carla_imitation_learning_b200 import stage_gray, sliding_window
    from oracle import bc_oracle as O
    from src.architectures.nets import ConvNet1
    dev = torch.device("cuda", 0)
    torch.manual_seed(12345)
    net = ConvNet1({"obs_size": 4, "n_actions": 9}).to(dev)
    eng = net.engine()
    frames, labels = O.synth_frames(77, 36)
    y = torch.from_numpy(labels[4:36]).to(dev)
    fr = torch.from_numpy(frames).to(dev)
    b32 = eng.train_forward_backward(sliding_window(stage_gray(fr)), y)
    g32 = eng.grads.clone()
    eng.set_mode("bf16")
    eng.pack_weights()
    b16 = eng.train_forward_backward(sliding_window(stage_gray(fr, dtype=torch.bfloat16)), y)
    torch.cuda.synchronize()
    eng.check_device_errors()
    rel = lambda a, b: float((a.double() - b.double()).abs().max() / b.double().abs().max())
    assert rel(b16.logits, b32.logits) <= 2e-2
    assert abs(float(b16.loss) - float(b32.loss)) <= 2e-2 * float(b32.loss)
    assert rel(eng.grads, g32) <= 0.1      # includes pool-routing flips caused by the bf16 rounding


def _to_act_bf16(x_nchw, idx):
    """NCHW -> the layout of bufs.act_bf16[idx]: P8 (B, C/8, H*W, 8) for act1/act2, P8B (C/8, B, H*W, 8) for act3."""
    B, Cc, Hh, Ww = x_nchw.shape
    p8 = x_nchw.reshape(B, Cc // 8, 8, Hh * Ww).permute(0, 1, 3, 2)
    return (p8.permute(1, 0, 2, 3) if idx == 2 else p8).contiguous()


def _from_act_bf16(t, idx, shape):
    B, Cc, Hh, Ww = shape
    if idx == 2:
        t = t.permute(1, 0, 2, 3)
    return t.permute(0, 1, 3, 2).reshape(B, Cc, Hh, Ww)


@pytest.mark.parametrize("layer,B", [(1, 3), (1, 37), (2, 5), (2, 1), (3, 33), (3, 1), (3, 70)])
def test_conv234_tcgen05_matches_bf16_rounded_oracle(layer, B):
    """conv2/3/4 + ReLU + pool as shifted-window tcgen05 GEMMs over P8 / P8B bf16 activations."""
    import ctypes as C
    from carla_imitation_learning_b200 import _lib
    from oracle import bc_oracle as O
    from src.architectures.nets import ConvNet1
    from tests.test_gpu_parity import _check_routing
    dev = torch.device("cuda", 0)
    torch.manual_seed(12345)
    net = ConvNet1({"obs_size": 4, "n_actions": 9}).to(dev)
    eng = net.engine()
    eng.set_mode("bf16")
    eng.pack_weights()
    name, k, s, p = O.CONV_SPECS[layer]
    w = net.state_dict()[f"{name}.weight"].detach().cpu()
    bias = net.state_dict()[f"{name}.bias"].detach().cpu().double()
    cin, hin = w.shape[1], (256, 28, 12, 4)[layer]
    gen = torch.Generator().manual_seed(7 * layer + B)
    xin = (torch.rand((B, cin, hin, hin), generator=gen) - 0.3).to(torch.bfloat16)
    bufs = eng.alloc(B, torch.zeros(B, 4, 256, 256, device=dev, dtype=torch.bfloat16), None, False)
    bufs.act_bf16[layer - 1].copy_(_to_act_bf16(xin, layer - 1).to(dev))
    c = eng.ctx(bufs)
    _lib.check(eng.lib.bc_conv_relu_pool_fwd(C.byref(c), layer, torch.cuda.current_stream().cuda_stream), "conv tc")
    torch.cuda.synchronize()
    eng.check_device_errors()
    z = torch.nn.functional.conv2d(xin.double(), w.to(torch.bfloat16).double(), bias, stride=1)
    ref = torch.nn.functional.max_pool2d(torch.relu(z), 2)
    got = bufs.act[layer].cpu().double()
    assert got.shape == ref.shape
    err = float((got - ref).abs().max() / ref.abs().max())
    assert err <= 1e-5, err
    _check_routing(z, bufs.amax[layer].cpu(), got, 2)
    if layer < 3:   # the bf16 copy handed to the next layer (P8 / P8B)
        back = _from_act_bf16(bufs.act_bf16[layer].float().cpu(), layer, bufs.act[layer].shape)
        assert torch.equal(back, bufs.act[layer].cpu().to(torch.bfloat16).float())


@pytest.mark.parametrize("B", [2, 37])
def test_dgrad_tcgen05_matches_exact_f32_dgrad(B):
    """Dense tensor-core dgrad (routed gradient built in smem -> shifted-window GEMM) vs the exact routing-sparse f32 kernel, same inputs."""
    import ctypes as C
    from carla_imitation_learning_b200 import _lib, stage_gray, sliding_window
    from oracle import bc_oracle as O
    from src.architectures.nets import ConvNet1
    dev = torch.device("cuda", 0)
    torch.manual_seed(12345)
    net = ConvNet1({"obs_size": 4, "n_actions": 9}).to(dev)
    eng = net.engine()
    eng.set_mode("bf16")
    eng.pack_weights()
    frames, labels = O.synth_frames(5 + B, B + 4)
    x = sliding_window(stage_gray(torch.from_numpy(frames).to(dev), dtype=torch.bfloat16))
    y = torch.from_numpy(labels[4:4 + B]).to(dev)
    bufs = eng.train_forward_backward(x, y)          # fills act/amax (tensor-core forward) and allocates backward buffers
    s = torch.cuda.current_stream().cuda_stream
    gen = torch.Generator(device="cpu").manual_seed(3)
    for layer in (3, 2, 1):
        gP = bufs.ghead if layer == 3 else bufs.gact[layer]
        gP.copy_(torch.randn(gP.shape, generator=gen).to(dev))
        eng.conv_mode = 15
        c = eng.ctx(bufs)
        _lib.check(eng.lib.bc_conv_bwd_dgrad(C.byref(c), layer, s), "dgrad tc")
        got = bufs.gact[layer - 1].clone()
        eng.conv_mode = 0
        c = eng.ctx(bufs)
        _lib.check(eng.lib.bc_conv_bwd_dgrad(C.byref(c), layer, s), "dgrad f32")
        torch.cuda.synchronize()
        ref = bufs.gact[layer - 1]
        err = float((got - ref).abs().max() / ref.abs().max())
        assert err <= 1e-2, (layer, err)             # bf16 rounding of dY and W, f32 accumulation
    eng.conv_mode = 15
    eng.check_device_errors()


@pytest.mark.parametrize("B", [2, 37])
def test_wgrad_tcgen05_matches_exact_f32_wgrad(B):
    """Tensor-core wgrad (MN-major operands, ones-chunk bias row) vs the exact routing-sparse f32 kernel."""
    import ctypes as C
    from carla_imitation_learning_b200 import _lib, stage_gray, sliding_window
    from oracle import bc_oracle as O
    from src.architectures.nets import ConvNet1
    dev = torch.device("cuda", 0)
    torch.manual_seed(12345)
    net = ConvNet1({"obs_size": 4, "n_actions": 9}).to(dev)
    eng = net.engine()
    eng.set_mode("bf16")
    eng.pack_weights()
    frames, labels = O.synth_frames(9 + B, B + 4)
    x = sliding_window(stage_gray(torch.from_numpy(frames).to(dev), dtype=torch.bfloat16))
    y = torch.from_numpy(labels[4:4 + B]).to(dev)
    bufs = eng.train_forward_backward(x, y)
    s = torch.cuda.current_stream().cuda_stream
    gen = torch.Generator(device="cpu").manual_seed(4)
    params = dict(net.named_parameters())
    names = ["cnn_base.0", "cnn_base.3", "cnn_base.6", "cnn_base.9"]
    for layer in (3, 2, 1, 0):          # layer 0 = conv1: Toeplitz wgrad with the fold in the epilogue
        gP = bufs.ghead if layer == 3 else bufs.gact[layer]
        gP.copy_(torch.randn(gP.shape, generator=gen).to(dev))
        res = {}
        for mode in (15, 0):
            eng.conv_mode = mode
            c = eng.ctx(bufs)
            _lib.check(eng.lib.bc_conv_bwd_wgrad(C.byref(c), layer, s), "wgrad")
            _lib.check(eng.lib.bc_reduce_partials_range(C.byref(c), 4 - layer, 5 - layer, 0, s), "reduce")
            torch.cuda.synchronize()
            res[mode] = {k: eng.grads[params[f"{names[layer]}.{k}"]._bc_offset:][:params[f"{names[layer]}.{k}"].numel()].clone()
                         for k in ("weight", "bias")}
        for k in ("weight", "bias"):
            err = float((res[15][k] - res[0][k]).abs().max() / res[0][k].abs().max())
            assert err <= 1e-2, (layer, k, err)
    eng.conv_mode = 15
    eng.check_device_errors()


def test_bf16_module_path_trains_like_the_reference(golden_dir, tmp_path):
    """precision='bf16' through the Lightning-contract shells against the reference's 1k-step curve:
    per step on the plateau, then 800 steps from the reference's own state at step 200 (tests/curve_check.py)."""
    import os
    from carla_imitation_learning_b200 import stage_gray
    from oracle import bc_oracle as O
    from src.architectures.nets import ConvNet1
    from src.models.imitation import Imitation
    from tests.curve_check import check_curve
    dev = torch.device("cuda", 0)
    g = np.load(os.path.join(golden_dir, "ref_curve_b8_1k.npz"))
    st = np.load(os.path.join(golden_dir, "ref_state_b8_step200.npz"))
    st_adam = np.load(os.path.join(golden_dir, "ref_state_b8_step200_adam.npz"))
    B, steps, at = int(g["B"]), int(g["steps"]), int(st["at_step"])
    frames, labels = O.synth_frames(int(g["data_seed"]), steps * B + 4)
    lab = torch.from_numpy(labels).to(dev)
    ref = g["losses"]

    def run(model, opt, s_begin, s_end):
        losses = []
        for s0 in range(s_begin, s_end, 50):
            n = min(50, s_end - s0)
            gray = stage_gray(torch.from_numpy(frames[s0 * B: s0 * B + n * B + 4]).to(dev), dtype=torch.bfloat16)
            for s in range(s0, s0 + n):
                o = (s - s0) * B
                x = gray.as_strided((B, 4, 256, 256), (65536, 65536, 256, 1), gray.storage_offset() + o * 65536)
                loss = model.training_step((x, lab[s * B + 4: s * B + 4 + B]), s)
                opt.zero_grad(); loss.backward(); opt.step()
                losses.append(loss.detach())
        return torch.stack(losses).cpu().double().numpy(), x

    # (a) from the common initial state: the same trajectory within the bf16 tolerance while on the plateau
    torch.manual_seed(12345)
    net = ConvNet1({"obs_size": 4, "n_actions": 9, "precision": "bf16"}).to(dev)
    model = Imitation({"obs_size": 4, "n_actions": 9}, net, {})
    opt = model.configure_optimizers()[0][0]
    got, x = run(model, opt, 0, 30)
    # a step's loss is an 8-sample mean after up to 30 Adam steps on bf16-rounded gradients (early Adam moves every
    # weight by ~lr whatever the gradient's size): all steps within 5 %, all but one within the 2 % tolerance
    dev_rel = np.abs(got - ref[:30]) / ref[:30].max()
    assert dev_rel.max() <= 5e-2 and np.sort(dev_rel)[-2] <= 2e-2, dev_rel
    # f32 reference-style batches are accepted too (converted by our kernel) and give the same logits as bf16 planes
    assert torch.equal(net(x.float()), net(x))

    # (b) from the reference's parameters and Adam state after 200 steps
    names = [n for n, _ in net.named_parameters()]
    assert names == list(O.PARAM_ORDER)
    sd, adam, off = {}, {}, 0
    for i, (n, p) in enumerate(net.named_parameters()):
        k = p.numel()
        sd[n] = torch.from_numpy(st["params"][off:off + k].copy()).view(p.shape)
        adam[i] = dict(step=torch.tensor(float(at)), exp_avg=torch.from_numpy(st_adam["exp_avg"][off:off + k].copy()).view(p.shape),
                       exp_avg_sq=torch.from_numpy(st_adam["exp_avg_sq"][off:off + k].copy()).view(p.shape))
        off += k
    net.load_state_dict(sd)
    opt = model.configure_optimizers()[0][0]
    opt.load_state_dict(dict(state=adam, param_groups=[dict(lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0,
                                                            amsgrad=False, params=list(range(len(names))))]))
    got, _ = run(model, opt, at, steps)
    net.engine().check_device_errors()
    np.save(os.path.join(os.environ.get("BC_TEST_OUT", str(tmp_path)), "curve_b8_1k_device_bf16.npy"), got)
    assert np.abs(got[:20] - ref[at:at + 20]).max() <= 5e-2 * ref[at:at + 20].max()       # still the same trajectory right after the resume
    check_curve(got, golden_dir, tol=2e-2, start=at)


def _dense_dy(gP, aP, amax, p, hc):
    """Routed, ReLU-masked conv-output gradient (f64): rounded to bf16 like the dY builders of the kernels, and unrounded."""
    B, Cc, Hp, Wp = gP.shape
    g = torch.where(aP > 0, gP, torch.zeros_like(gP)).double()
    oh = torch.nn.functional.one_hot(amax.long(), p * p).double() * g[..., None]
    dy = torch.zeros(B, Cc, hc, hc, dtype=torch.float64)
    dy[..., :Hp * p, :Wp * p] = oh.reshape(B, Cc, Hp, Wp, p, p).permute(0, 1, 2, 4, 3, 5).reshape(B, Cc, Hp * p, Wp * p)
    return dy.to(torch.bfloat16).double(), dy


@pytest.mark.parametrize("B", [3, 37])
def test_tc_backward_is_exact_on_its_bf16_operands(B):
    """Tensor-core dgrad/wgrad == f64 transposed-conv / correlation of the SAME bf16-rounded operands (rel 2e-5):
    separates kernel correctness from the (expected) bf16 operand rounding."""
    import ctypes as C
    from carla_imitation_learning_b200 import _lib, stage_gray, sliding_window
    from oracle import bc_oracle as O
    from src.architectures.nets import ConvNet1
    F = torch.nn.functional
    dev = torch.device("cuda", 0)
    torch.manual_seed(12345)
    net = ConvNet1({"obs_size": 4, "n_actions": 9}).to(dev)
    eng = net.engine()
    eng.set_mode("bf16")
    eng.pack_weights()
    frames, labels = O.synth_frames(19 + B, B + 4)
    x = sliding_window(stage_gray(torch.from_numpy(frames).to(dev), dtype=torch.bfloat16))
    y = torch.from_numpy(labels[4:4 + B]).to(dev)
    bufs = eng.train_forward_backward(x, y)
    eng.conv_mode = 15        # kernel by kernel on the f32 NCHW gradient buffers this test fills (the compact conv1 path: next test)
    s = torch.cuda.current_stream().cuda_stream
    gen = torch.Generator(device="cpu").manual_seed(6)
    params = dict(net.named_parameters())
    names = ["cnn_base.0", "cnn_base.3", "cnn_base.6", "cnn_base.9"]
    hc = (84, 24, 9, 2)
    pool = (3, 2, 2, 2)
    for layer in (3, 2, 1, 0):
        gP = bufs.ghead.view(B, 128, 1, 1) if layer == 3 else bufs.gact[layer]
        gP.copy_(torch.randn(gP.shape, generator=gen).to(dev))
        c = eng.ctx(bufs)
        _lib.check(eng.lib.bc_conv_bwd_wgrad(C.byref(c), layer, s), "wgrad")
        _lib.check(eng.lib.bc_reduce_partials_range(C.byref(c), 4 - layer, 5 - layer, 0, s), "reduce")
        if layer > 0:
            _lib.check(eng.lib.bc_conv_bwd_dgrad(C.byref(c), layer, s), "dgrad")
        torch.cuda.synchronize()
        dy, dy_f32 = _dense_dy(gP.cpu(), bufs.act[layer].cpu(), bufs.amax[layer].cpu(), pool[layer], hc[layer])
        w = params[f"{names[layer]}.weight"].detach().cpu()
        if layer == 0:
            xin = x.double().cpu()
            stride = 3
        else:
            xin = _from_act_bf16(bufs.act_bf16[layer - 1].double().cpu(), layer - 1, bufs.act[layer - 1].shape)
            stride = 1
        k = w.shape[-1]
        cols = F.unfold(xin, kernel_size=k, stride=stride)                       # (B, Cin*k*k, L) over the full conv map
        L_used = dy.shape[-1]
        ref_w = torch.einsum("bol,bkl->ok", dy.reshape(B, dy.shape[1], -1), cols).reshape(w.shape)
        # conv2-4 (shifted-window wgrad) fold the f32 gradient before its bf16 rounding; conv1 uses a ones row of the GEMM
        ref_b = (dy_f32 if layer >= 1 else dy).sum(dim=(0, 2, 3))
        pw, pb = params[f"{names[layer]}.weight"], params[f"{names[layer]}.bias"]
        got_w = eng.grads[pw._bc_offset:pw._bc_offset + pw.numel()].view(w.shape).cpu().double()
        got_b = eng.grads[pb._bc_offset:pb._bc_offset + pb.numel()].cpu().double()
        ew = float((got_w - ref_w).abs().max() / ref_w.abs().max())
        eb = float((got_b - ref_b).abs().max() / ref_b.abs().max())
        assert ew <= 2e-5 and eb <= 2e-5, (layer, "wgrad", ew, eb)
        if layer > 0:
            ref_d = F.conv_transpose2d(dy, w.to(torch.bfloat16).double(), stride=1)
            got_d = bufs.gact[layer - 1].cpu().double()
            ed = float((got_d - ref_d).abs().max() / ref_d.abs().max())
            assert ed <= 2e-5, (layer, "dgrad", ed)
    eng.check_device_errors()


@pytest.mark.parametrize("B", [3, 37])
def test_compact_conv1_gradient_path_is_bitwise_the_nchw_path(B):
    """conv_mode bit 16 (what set_mode('bf16') enables): conv1's forward also writes its routing in P8 order, conv2's dgrad
    writes the ReLU-masked bf16 gradient in P8 order instead of f32 NCHW, conv1's wgrad (third generation, conv1_wgrad3.cu)
    builds dY from those -- a pure re-layout of the same bf16 operands: the intermediate tensors are bit-identical to the
    f32 NCHW path (conv_mode 15), conv1's gradient differs only by the f32 accumulation order (two issuers' partial sums)."""
    import ctypes as C
    from carla_imitation_learning_b200 import _lib, stage_frames
    from oracle import bc_oracle as O
    from src.architectures.nets import ConvNet1
    dev = torch.device("cuda", 0)
    torch.manual_seed(12345)
    net = ConvNet1({"obs_size": 4, "n_actions": 9, "precision": "bf16"}).to(dev)
    eng = net.engine()
    assert eng.conv_mode == 31
    frames, labels = O.synth_frames(23 + B, B + 4)
    y = torch.from_numpy(labels[4:4 + B].copy()).to(dev)
    bufs = eng.train_forward_backward(stage_frames(torch.from_numpy(frames).to(dev)), y)
    torch.cuda.synchronize()
    eng.check_device_errors()
    g_compact = eng.grads.clone()
    p8 = lambda t: t.reshape(B, 2, 8, 784).permute(0, 1, 3, 2).contiguous()
    assert torch.equal(bufs.amax0_p8, p8(bufs.amax[0]))
    # the same backward through the f32 NCHW buffers
    eng.conv_mode = 15
    c = eng.ctx(bufs)
    _lib.check(eng.lib.bc_backward(C.byref(c), 1, torch.cuda.current_stream().cuda_stream), "bc_backward")
    torch.cuda.synchronize()
    eng.check_device_errors()
    w1 = dict(net.named_parameters())["cnn_base.0.weight"]._bc_offset       # conv1 is the last arena segment
    assert torch.equal(eng.grads[:w1], g_compact[:w1])
    d1 = (eng.grads[w1:] - g_compact[w1:]).abs().max() / eng.grads[w1:].abs().max()
    assert float(d1) <= 2e-5, float(d1)
    # the third-generation kernel is deterministic: the same step again gives the same bits
    eng.conv_mode = 31
    c = eng.ctx(bufs)
    _lib.check(eng.lib.bc_backward(C.byref(c), 1, torch.cuda.current_stream().cuda_stream), "bc_backward")
    torch.cuda.synchronize()
    assert torch.equal(eng.grads, g_compact)
    eng.conv_mode = 15
    c = eng.ctx(bufs)
    _lib.check(eng.lib.bc_backward(C.byref(c), 1, torch.cuda.current_stream().cuda_stream), "bc_backward")
    torch.cuda.synchronize()
    masked = torch.where(bufs.act[0] > 0, bufs.gact[0], torch.zeros_like(bufs.gact[0])).to(torch.bfloat16)
    assert torch.equal(bufs.gact0_p8.view(torch.int16), p8(masked).view(torch.int16))


def _tp_reference(planes):
    """(n,256,256) -> (n, 3, 2, 86, 21, 8): TP[c][h][q][g][i] = plane[3q+c][12g+8h+i], zero rows beyond 255
    (the layout include/bc_b200.h documents for BC_BF16_TP)."""
    n = planes.shape[0]
    pad = torch.zeros((n, 258, 256), dtype=planes.dtype, device=planes.device)
    pad[:, :256] = planes
    R = (3 * torch.arange(86)[None, :] + torch.arange(3)[:, None]).to(planes.device)                     # (3,86)
    px = (12 * torch.arange(21)[None, :, None] + 8 * torch.arange(2)[:, None, None] + torch.arange(8)[None, None, :]).to(planes.device)  # (2,21,8)
    return pad[:, R[:, None, :, None, None], px[None, :, None, :, :]]


@pytest.mark.parametrize("n", [1, 5])
def test_toeplitz_ready_planes_are_a_pure_rearrangement(n):
    """bc_planes_to_tp (f32 and bf16 input) and bc_stage_gray(..., BC_BF16_TP) == the plain bf16 planes re-indexed."""
    from carla_imitation_learning_b200 import _lib, stage_gray
    from oracle import bc_oracle as O
    dev = torch.device("cuda", 0)
    frames, _ = O.synth_frames(90 + n, n)
    fr = torch.from_numpy(frames).to(dev)
    plain16 = stage_gray(fr, dtype=torch.bfloat16)
    plain32 = stage_gray(fr)
    ref = _tp_reference(plain16).reshape(n, -1)
    assert ref.shape[1] == _lib.TP_PLANE_ELEMS
    s = torch.cuda.current_stream().cuda_stream
    for src, code in ((plain16, _lib.BC_BF16), (plain32, _lib.BC_F32)):
        out = torch.full((n, _lib.TP_PLANE_ELEMS), float("nan"), dtype=torch.bfloat16, device=dev)
        _lib.check(_lib.lib().bc_planes_to_tp(src.data_ptr(), code, n, 65536, out.data_ptr(), s), "bc_planes_to_tp")
        assert torch.equal(out.view(torch.int16), ref.view(torch.int16))
    out = torch.full((n, _lib.TP_PLANE_ELEMS), float("nan"), dtype=torch.bfloat16, device=dev)
    _lib.check(_lib.lib().bc_stage_gray(fr.data_ptr(), out.data_ptr(), n * 65536, _lib.BC_BF16_TP, s), "bc_stage_gray TP")
    assert torch.equal(out.view(torch.int16), ref.view(torch.int16))


@pytest.mark.parametrize("B", [1, 2, 7, 37])
def test_conv1_tcgen05_materialised_batch_equals_sliding_view(B):
    """The plane-sharing path (sliding view: one load feeds 4 samples) and the per-sample path (contiguous batch)
    of conv1_tp_kernel produce identical bits, for batch sizes that leave partial sample groups."""
    import ctypes as C
    from carla_imitation_learning_b200 import _lib, stage_gray, sliding_window
    from oracle import bc_oracle as O
    from src.architectures.nets import ConvNet1
    dev = torch.device("cuda", 0)
    torch.manual_seed(12345)
    net = ConvNet1({"obs_size": 4, "n_actions": 9}).to(dev)
    eng = net.engine()
    eng.set_mode("bf16")
    eng.pack_weights()
    frames, _ = O.synth_frames(150 + B, B + 4)
    x = sliding_window(stage_gray(torch.from_numpy(frames).to(dev), dtype=torch.bfloat16))[:B]
    outs = []
    for xx in (x, x.contiguous()):
        bufs = eng.alloc(B, xx, None, False)
        assert (bufs.x_tp_strides[0] == bufs.x_tp_strides[1]) == (xx is x)
        c = eng.ctx(bufs)
        _lib.check(eng.lib.bc_conv_relu_pool_fwd(C.byref(c), 0, torch.cuda.current_stream().cuda_stream), "conv1 tc")
        torch.cuda.synchronize()
        outs.append((bufs.act[0].clone(), bufs.amax[0].clone(), bufs.act_bf16[0].clone()))
    eng.check_device_errors()
    for a, b in zip(*outs):
        assert torch.equal(a, b)


def test_stage_frames_feeds_both_layouts_and_matches_the_plain_path():
    """stage_frames (one fused pass: u8 -> Toeplitz-ready + plain bf16) == stage_gray + bc_planes_to_tp, and a training
    step driven by the StagedBatch is bitwise the step driven by the plain sliding view."""
    from carla_imitation_learning_b200 import stage_frames, stage_gray, sliding_window
    from oracle import bc_oracle as O
    from src.architectures.nets import ConvNet1
    dev = torch.device("cuda", 0)
    B = 9
    frames, labels = O.synth_frames(321, B + 4)
    fr = torch.from_numpy(frames).to(dev)
    y = torch.from_numpy(labels[4:4 + B]).to(dev)
    sb = stage_frames(fr, plain=True)
    plain = stage_gray(fr, dtype=torch.bfloat16)
    assert torch.equal(sb.plain.view(torch.int16), plain.view(torch.int16))
    assert torch.equal(sb.tp.view(torch.int16), _tp_reference(plain).reshape(B + 4, -1).view(torch.int16))
    assert stage_frames(fr).plain is None and torch.equal(stage_frames(fr).tp.view(torch.int16), sb.tp.view(torch.int16))
    sb = stage_frames(fr)                       # the product path: Toeplitz-ready planes only
    assert tuple(sb.shape) == (B, 4, 256, 256)
    torch.manual_seed(12345)
    net = ConvNet1({"obs_size": 4, "n_actions": 9, "precision": "bf16"}).to(dev)
    eng = net.engine()
    b1 = eng.train_forward_backward(sb, y)
    g1, l1 = eng.grads.clone(), b1.loss.clone()
    b2 = eng.train_forward_backward(sliding_window(plain), y)
    torch.cuda.synchronize()
    eng.check_device_errors()
    assert torch.equal(l1, b2.loss) and torch.equal(g1, eng.grads)
    # the module shells take it too
    assert torch.equal(net(sb), b2.logits)
    with pytest.raises(ValueError):
        ConvNet1({"obs_size": 4, "n_actions": 9}).to(dev).engine().forward(sb)      # fp32 mode reads plain f32/bf16 planes


def test_sequential_loader_feeds_the_bf16_mode_with_staged_batches():
    """SequentialFrames(layout='tp') (the device-side SequentialTorchDataset for precision='bf16') yields StagedBatch
    windows, short last batch included; a training step on them is bitwise the step on the plain-plane loader's batch."""
    from carla_imitation_learning_b200 import StagedBatch
    from carla_imitation_learning_b200.data import SequentialFrames, synthetic_sequence
    from src.architectures.nets import ConvNet1
    dev = torch.device("cuda", 0)
    frames, labels = synthetic_sequence(3, 23)                       # 19 samples: batches of 8, 8, 3
    tp = SequentialFrames(frames, labels, batch_size=8, layout="tp")
    plain = SequentialFrames(frames, labels, batch_size=8, dtype=torch.bfloat16)
    assert len(tp) == 3
    torch.manual_seed(12345)
    net = ConvNet1({"obs_size": 4, "n_actions": 9, "precision": "bf16"}).to(dev)
    eng = net.engine()
    sizes = []
    for (xa, ya), (xb, yb) in zip(tp, plain):
        assert isinstance(xa, StagedBatch) and torch.equal(ya, yb) and tuple(xa.shape) == tuple(xb.shape)
        la = eng.train_forward_backward(xa, ya).loss.clone()
        ga = eng.grads.clone()
        lb = eng.train_forward_backward(xb, yb).loss.clone()
        assert torch.equal(la, lb) and torch.equal(ga, eng.grads)
        sizes.append(xa.shape[0])
    torch.cuda.synchronize()
    eng.check_device_errors()
    assert sizes == [8, 8, 3]


@pytest.mark.parametrize("B", [1, 5, 8, 255, 257])
def test_bf16_step_tail_batches(B):
    """Batch sizes that leave partial tiles / empty partial-sum slots in every tensor-core kernel: the bf16 step stays
    within the bf16 tolerance of the exact-f32 step and no pipeline wait times out."""
    from carla_imitation_learning_b200 import stage_frames, stage_gray, sliding_window
    from oracle import bc_oracle as O
    from src.architectures.nets import ConvNet1
    dev = torch.device("cuda", 0)
    frames, labels = O.synth_frames(1000 + B, B + 4)
    fr = torch.from_numpy(frames).to(dev)
    y = torch.from_numpy(labels[4:4 + B]).to(dev)
    res = {}
    for mode in ("fp32", "bf16"):
        torch.manual_seed(12345)
        net = ConvNet1({"obs_size": 4, "n_actions": 9, "precision": mode}).to(dev)
        eng = net.engine()
        x = stage_frames(fr) if mode == "bf16" else sliding_window(stage_gray(fr))
        b = eng.train_forward_backward(x, y)
        torch.cuda.synchronize()
        eng.check_device_errors()
        res[mode] = (b.logits.clone(), float(b.loss), eng.grads.clone())
    rel = lambda a, r: float((a.double() - r.double()).abs().max() / r.double().abs().max())
    assert rel(res["bf16"][0], res["fp32"][0]) <= 2e-2
    assert abs(res["bf16"][1] - res["fp32"][1]) <= 2e-2 * res["fp32"][1]
    assert torch.isfinite(res["bf16"][2]).all()
    assert rel(res["bf16"][2], res["fp32"][2]) <= 0.15      # includes pool-routing flips caused by the bf16 rounding
