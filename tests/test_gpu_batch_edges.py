"""Every kernel of a training step at the batch sizes the product runs, against an exact reference on its own operands.

Each output y = sum a*b (+ bias) is compared element-wise with the f64 sum over the operands the kernel actually read from
the buffers of the same run, with the bound |got - ref| <= TAU * S (+ 2^-8 |ref| where the kernel writes bf16), where
S = the same f64 sum over |a|*|b| (+ |bias|). The bound has power: for every sample b some element of its f64
contribution exceeds the bound, so a kernel that lost one sample (a tile, a partial-sum slot, a head CTA's second sample)
fails. Batch sizes are where the persistent kernels change how they split the work: conv1 forward gives a CTA a second
tile from B = 11, conv1 wgrad3 splits tile rows into segments from B = 8, a head CTA holds two samples from B = 129,
conv4 dgrad starts a second wave at B = 297. `pytest -s` prints the smallest headroom (bound / error) and power margin
(contribution / bound) per tensor.
"""
import os

import numpy as np
import pytest
import torch

from oracle import bc_oracle as O
from tests.test_gpu_parity import _check_routing
from tests.test_gpu_tc import _dense_dy, _from_act_bf16, _tp_reference

pytestmark = pytest.mark.gpu

F = torch.nn.functional
TAU = 1e-5
BF16_HALF_ULP = 2.0 ** -8
CONV_NAMES = [c[0] for c in O.CONV_SPECS]
CONV_HC = (84, 24, 9, 2)               # conv output maps before pooling


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (no CPU fallback exists to run instead)")
    torch.set_num_threads(os.cpu_count() or 1)
    return torch.device("cuda", 0)


def _net(hp, seed=12345):
    from src.architectures.nets import ConvNet1
    torch.manual_seed(seed)
    return ConvNet1(dict(hp)).to(torch.device("cuda", 0))


def _uniform_frames(seed, n):
    rng = np.random.Generator(np.random.PCG64(seed))
    return rng.integers(0, 256, size=(n, 256, 256, 3), dtype=np.uint8)


def _cpu64(t):
    return t.detach().cpu().double()


def _bound(tag, got, ref, S, per_sample=None, bf16=False, power=True):
    """|got - ref| <= TAU*S (+ 2^-8 |ref| for a bf16 output), element-wise. With `power`, every sample must matter: its
    contribution exceeds the bound somewhere. per_sample = (B, *ref.shape) contributions of each sample to a batch sum;
    None = ref's first axis is the sample. Returns (headroom, power margin)."""
    got, ref, S = _cpu64(got).reshape(ref.shape), ref.double(), S.double()
    tol = TAU * S + (BF16_HALF_ULP * ref.abs() if bf16 else 0.0)
    err = (got - ref).abs()
    bad = err > tol
    assert not bool(bad.any()), (f"{tag}: {int(bad.sum())} of {err.numel()} elements outside the bound, "
                                 f"worst err/bound {float((err / tol.clamp_min(1e-300))[bad].max()):.3g}")
    nz = err > 0
    headroom = float((tol[nz] / err[nz]).min()) if bool(nz.any()) else float("inf")
    margin = float("nan")
    if power:
        c = (per_sample if per_sample is not None else ref).double().abs()
        B = c.shape[0]
        c = c.reshape(B, -1)
        t = tol.reshape(1, -1) if per_sample is not None else tol.reshape(B, -1)
        ratio = torch.where(t > 0, c / t.clamp_min(1e-300), torch.where(c > 0, float("inf"), 0.0))
        per_b = ratio.max(dim=1).values
        margin = float(per_b.min())
        assert margin > 1, f"{tag}: sample {int(per_b.argmin())} could be dropped unnoticed (power margin {margin:.3g})"
    print(f"  {tag:<34s} headroom {headroom:10.3g}   power {margin:10.3g}")
    return headroom, margin


def _at_routing(z, amax, p):
    """Value of each pool window of z at the window-local index the device routed to."""
    B, Cc, Hc, Wc = z.shape
    Hp, Wp = Hc // p, Wc // p
    win = z[..., :Hp * p, :Wp * p].reshape(B, Cc, Hp, p, Wp, p).permute(0, 1, 2, 4, 3, 5).reshape(B, Cc, Hp, Wp, p * p)
    return win.gather(-1, amax.long()[..., None]).squeeze(-1)


def _planes_from_tp(tp):
    """Toeplitz-ready planes (n, TP_PLANE_ELEMS) -> the plain (n, 256, 256) planes they hold; a round trip through the
    documented layout proves the decode complete, so these are exactly the values conv1 read."""
    tp = tp.cpu()
    n = tp.shape[0]
    out = torch.zeros((n, 258, 256), dtype=tp.dtype)
    R = 3 * torch.arange(86)[None, :] + torch.arange(3)[:, None]
    px = 12 * torch.arange(21)[None, :, None] + 8 * torch.arange(2)[:, None, None] + torch.arange(8)[None, None, :]
    out[:, R[:, None, :, None, None], px[None, :, None, :, :]] = tp.view(n, 3, 2, 86, 21, 8)
    planes = out[:, :256].contiguous()
    assert torch.equal(_tp_reference(planes).reshape(n, -1).view(torch.int16), tp.view(torch.int16))
    return planes


def _grads(net, eng):
    return {k: _cpu64(eng.grads[p._bc_offset:p._bc_offset + p.numel()].view(p.shape)) for k, p in net.named_parameters()}


def _p8_to_nchw(t):
    """(B, C/8, H*W, 8) P8 -> (B, C, 28, 28) for conv1's output map."""
    return _from_act_bf16(t, 0, (t.shape[0], 16, 28, 28))


# ------------------------------------------------------------------------------- per-kernel checks
def _conv_in(bufs, layer, bf16):
    """The activation conv `layer` (1..3) read: the bf16 copy in tensor-core mode, the f32 map otherwise."""
    if bf16:
        return _from_act_bf16(_cpu64(bufs.act_bf16[layer - 1]), layer - 1, bufs.act[layer - 1].shape)
    return _cpu64(bufs.act[layer - 1])


def _conv_w(P, layer, bf16):
    w = P[f"{CONV_NAMES[layer]}.weight"]
    return (w.float().to(torch.bfloat16) if bf16 else w).double()


def _check_conv1(tag, bufs, x, w, bias, B, dy=None, chunk=16):
    """conv1 forward (act[0] at the device's routing) and, given dY, its weight gradient; f64 in sample chunks."""
    refs, Ss, cw, sw, cb, sb = [], [], [], [], [], []
    act0, amax0 = bufs.act[0].cpu(), bufs.amax[0].cpu()
    for b0 in range(0, B, chunk):
        xc = x[b0:b0 + chunk].double().contiguous()
        z = F.conv2d(xc, w, bias, stride=3)
        Sz = F.conv2d(xc.abs(), w.abs(), bias.abs(), stride=3)
        am = amax0[b0:b0 + chunk]
        _check_routing(z, am, act0[b0:b0 + chunk].double(), 3)
        refs.append(torch.relu(_at_routing(z, am, 3)))
        Ss.append(_at_routing(Sz, am, 3))
        del z, Sz
        if dy is not None:
            cols = F.unfold(xc, kernel_size=7, stride=3)                  # (n, obs*49, 84*84); gray planes are >= 0
            d = dy[b0:b0 + chunk].reshape(xc.shape[0], 16, -1)
            cw.append(torch.einsum("bol,bkl->bok", d, cols))
            sw.append(torch.einsum("bol,bkl->ok", d.abs(), cols))
            cb.append(d.sum(-1))
            sb.append(d.abs().sum(-1).sum(0))
            del cols
    _bound(f"{tag} conv1 fwd act[0]", act0, torch.cat(refs), torch.cat(Ss))
    if dy is None:
        return None
    return torch.cat(cw), sum(sw), torch.cat(cb), sum(sb)


def _check_conv_fwd(tag, bufs, P, B, bf16):
    """conv2..conv4 forward on the activation they read, at the device's routing; bf16 copies handed on bitwise."""
    for layer in (1, 2, 3):
        name, k, s, p = O.CONV_SPECS[layer]
        xin = _conv_in(bufs, layer, bf16)
        w, bias = _conv_w(P, layer, bf16), P[f"{name}.bias"]
        z = F.conv2d(xin, w, bias, stride=s)
        Sz = F.conv2d(xin.abs(), w.abs(), bias.abs(), stride=s)
        am = bufs.amax[layer].cpu()
        got = bufs.act[layer].cpu()
        _check_routing(z, am, got.double(), p)
        _bound(f"{tag} conv{layer + 1} fwd act[{layer}]", got, torch.relu(_at_routing(z, am, p)), _at_routing(Sz, am, p))
    if bf16:
        for i in range(3):
            back = _from_act_bf16(bufs.act_bf16[i].float().cpu(), i, bufs.act[i].shape)
            assert torch.equal(back, bufs.act[i].cpu().to(torch.bfloat16).float()), (tag, "act_bf16", i)


def _check_head_fwd(tag, bufs, P, B, NA):
    a3 = _cpu64(bufs.act[3]).reshape(B, 128)
    h1, h2 = _cpu64(bufs.hid1), _cpu64(bufs.hid2)
    for name, inp, out, relu in (("fc.0", a3, h1, True), ("fc.2", h1, h2, True), ("fc.4", h2, bufs.logits, False)):
        W, b = P[f"{name}.weight"], P[f"{name}.bias"]
        ref = inp @ W.t() + b
        _bound(f"{tag} {name} fwd", out, torch.relu(ref) if relu else ref, inp.abs() @ W.abs().t() + b.abs())
    assert bufs.logits.shape == (B, NA)


def _check_head_bwd(tag, bufs, P, G, y, B, NA, power=True):
    """CE loss, dlogits, the fc gradients and ghead, each from the device's own inputs to it (exact f32 kernel)."""
    a3 = _cpu64(bufs.act[3]).reshape(B, 128)
    h1, h2, z, dl = _cpu64(bufs.hid1), _cpu64(bufs.hid2), _cpu64(bufs.logits), _cpu64(bufs.dlogits)
    y = y.cpu()
    m = z.max(1).values
    lsum = torch.log(torch.exp(z - m[:, None]).sum(1))
    zy = z.gather(1, y[:, None]).squeeze(1)
    per = (lsum + m - zy) / B
    _bound(f"{tag} loss", bufs.loss.reshape(1), per.sum().reshape(1), ((lsum.abs() + m.abs() + zy.abs()) / B).sum().reshape(1),
           per_sample=per.reshape(B, 1), power=power)
    sm, oh = torch.softmax(z, 1), F.one_hot(y, NA).double()
    _bound(f"{tag} dlogits", dl, (sm - oh) / B, (sm + oh) / B, power=power)
    W0, W2, W4 = (P[f"{n}.weight"] for n in ("fc.0", "fc.2", "fc.4"))
    m2, m1 = (h2 > 0).double(), (h1 > 0).double()
    dh2, dh2a = (dl @ W4) * m2, (dl.abs() @ W4.abs()) * m2
    dh1, dh1a = (dh2 @ W2) * m1, (dh2a @ W2.abs()) * m1
    for name, d, da, inp in (("fc.4", dl, dl.abs(), h2), ("fc.2", dh2, dh2a, h1), ("fc.0", dh1, dh1a, a3)):
        _bound(f"{tag} {name}.weight grad", G[f"{name}.weight"], d.t() @ inp, da.t() @ inp.abs(),
               per_sample=torch.einsum("bo,bi->boi", d, inp), power=power)
        _bound(f"{tag} {name}.bias grad", G[f"{name}.bias"], d.sum(0), da.sum(0), per_sample=d, power=power)
    _bound(f"{tag} ghead", bufs.ghead, dh1 @ W0, dh1a @ W0.abs(), power=power)


def _check_tc_backward(tag, bufs, P, G, B):
    """bf16 (tcgen05) dgrad conv4..conv2 and wgrad conv4..conv2 on the bf16-rounded routed dY and W they consume."""
    for layer in (3, 2, 1):
        name, k, _s, p = O.CONV_SPECS[layer]
        gP = bufs.ghead.view(B, 128, 1, 1) if layer == 3 else bufs.gact[layer]
        dy, dy32 = _dense_dy(gP.cpu(), bufs.act[layer].cpu(), bufs.amax[layer].cpu(), p, CONV_HC[layer])
        wb = _conv_w(P, layer, True)
        ref = F.conv_transpose2d(dy, wb)
        S = F.conv_transpose2d(dy.abs(), wb.abs())
        if layer > 1:
            _bound(f"{tag} conv{layer + 1} dgrad gact[{layer - 1}]", bufs.gact[layer - 1], ref, S)
        else:       # the compact path: ReLU-masked bf16 gradient w.r.t. act1 in P8 order
            mask = (bufs.act[0].cpu() > 0).double()
            _bound(f"{tag} conv2 dgrad gact0_p8", _p8_to_nchw(bufs.gact0_p8.float().cpu()), ref * mask, S * mask, bf16=True)
        cols = F.unfold(_conv_in(bufs, layer, True), kernel_size=k)            # pooled ReLU activations: >= 0
        d = dy.reshape(B, dy.shape[1], -1)
        cw = torch.einsum("bol,bkl->bok", d, cols)
        shape = P[f"{name}.weight"].shape
        _bound(f"{tag} conv{layer + 1} wgrad weight", G[f"{name}.weight"], cw.sum(0).reshape(shape),
               torch.einsum("bol,bkl->ok", d.abs(), cols).reshape(shape), per_sample=cw.reshape(B, *shape))
        d32 = dy32.reshape(B, dy.shape[1], -1)                                  # the bias is folded before the bf16 rounding
        _bound(f"{tag} conv{layer + 1} wgrad bias", G[f"{name}.bias"], d32.sum((0, 2)), d32.abs().sum((0, 2)), per_sample=d32.sum(2))


def _check_forward(tag, bufs, P, x, B, NA, bf16):
    """Every forward kernel; x = the (B, obs, 256, 256) planes conv1 read."""
    _check_conv1(tag, bufs, x, _conv_w(P, 0, bf16), P["cnn_base.0.bias"], B)
    _check_conv_fwd(tag, bufs, P, B, bf16)
    _check_head_fwd(tag, bufs, P, B, NA)


# ------------------------------------------------------------------------------- the product bf16 step, kernel by kernel
def _check_bf16_kernels(tag, net, eng, bufs, sb, y, B, obs, NA):
    """Every kernel of a bf16-mode training step (conv_mode 31) against f64 on the operands it read from `bufs`."""
    step = obs // 4
    P = {k: _cpu64(v) for k, v in net.state_dict().items()}
    G = _grads(net, eng)
    planes = _planes_from_tp(sb.tp).double()
    x = planes.as_strided((B, obs, 256, 256), (step * 65536, 65536, 256, 1))
    print(f"\n{tag}")
    # conv1's routing handed to its weight gradient in P8 order, and its bf16 output
    p8 = lambda t: t.reshape(B, 2, 8, 784).permute(0, 1, 3, 2).contiguous()
    assert torch.equal(bufs.amax0_p8.cpu(), p8(bufs.amax[0].cpu()))
    # conv1 forward + wgrad3 (dY decoded from gact0_p8 / amax0_p8, one f64 pass in sample chunks)
    g0 = _p8_to_nchw(bufs.gact0_p8.float().cpu())
    am0 = _p8_to_nchw(bufs.amax0_p8.cpu())
    dy1, _ = _dense_dy(g0, torch.ones_like(g0), am0, 3, 84)
    cw, sw, cb, sbias = _check_conv1(tag, bufs, x, _conv_w(P, 0, True), P["cnn_base.0.bias"], B, dy=dy1,
                                     chunk=16 if obs == 4 else 6)
    shape = P["cnn_base.0.weight"].shape
    _check_conv_fwd(tag, bufs, P, B, True)
    _check_head_fwd(tag, bufs, P, B, NA)
    _check_head_bwd(tag, bufs, P, G, y, B, NA)
    _check_tc_backward(tag, bufs, P, G, B)
    _bound(f"{tag} conv1 wgrad3 weight", G["cnn_base.0.weight"], cw.sum(0).reshape(shape), sw.reshape(shape),
           per_sample=cw.reshape(B, *shape))
    _bound(f"{tag} conv1 wgrad3 bias", G["cnn_base.0.bias"], cb.sum(0), sbias, per_sample=cb)


@pytest.mark.parametrize("B,obs", [(1, 4), (7, 4), (8, 4), (10, 4), (11, 4), (129, 4), (256, 4), (297, 4), (129, 12)])
def test_bf16_step_every_kernel_is_exact_on_its_operands(dev, B, obs):
    from carla_imitation_learning_b200 import stage_frames
    step = obs // 4
    net = _net({"obs_size": obs, "n_actions": 9, "precision": "bf16"})
    eng = net.engine()
    assert eng.conv_mode == 31
    n_frames = step * (B - 1) + obs + step
    frames = _uniform_frames(1000 + 13 * B + obs, n_frames)
    y = torch.from_numpy(np.random.Generator(np.random.PCG64(B)).integers(0, 9, size=B))
    sb = stage_frames(torch.from_numpy(frames).to(dev), frame_skip=obs, step=step)
    assert sb.shape[0] == B
    bufs = eng.train_forward_backward(sb, y.to(dev))
    torch.cuda.synchronize()
    eng.check_device_errors()
    _check_bf16_kernels(f"bf16 B={B} obs={obs}", net, eng, bufs, sb, y, B, obs, 9)


# ------------------------------------------------------------------------------- head widths
def _whole_step_vs_oracle(net, bufs, G, frames, y, B, mode):
    """The whole step against the f64 oracle on the f32 master weights and gray frames, given the device's routing
    (and, in bf16 mode, its ReLU decisions, each of which must be a near-tie when it differs from the oracle's)."""
    P = {k: v.detach().cpu() for k, v in net.state_dict().items()}
    x, _ = O.sequential_samples(frames, np.zeros(len(frames), np.int64))
    amax = [a.cpu().long() for a in bufs.amax]
    relu = None if mode == "fp32" else {"pooled": [a.cpu() > 0 for a in bufs.act], "fc": [bufs.hid1.cpu() > 0, bufs.hid2.cpu() > 0]}
    loss, logits, ref, aux = O.explicit_backward(P, torch.from_numpy(x[:B]), y, dtype=torch.float64, argmax_override=amax, relu_override=relu)
    tol = 1e-5 if mode == "fp32" else 2e-2
    rel = lambda g, r: float((_cpu64(g) - r).abs().max() / r.abs().max().clamp_min(1e-30))
    assert rel(bufs.logits, logits) <= tol
    assert abs(float(bufs.loss) - float(loss)) <= tol * float(loss)
    worst = {k: rel(G[k], ref[k]) for k in O.PARAM_ORDER}
    print(f"  whole step vs f64 oracle ({mode}), worst rel per tensor:", {k: f"{v:.2e}" for k, v in worst.items()})
    # bf16 mode: the conv gradients carry the bf16 rounding of the frames, the weights, the activations handed on and dY.
    # With few classes the per-sample gradients cancel more in the batch sum, so that rounding weighs more against
    # max|grad| (measured on a B200: 2.7e-2 at n_actions = 2). Those kernels are held to TAU on their own operands at this
    # width by _check_bf16_kernels; here they only have to stay on the oracle's trajectory.
    conv_tol = tol if mode == "fp32" else 5e-2
    assert max(v for k, v in worst.items() if k.startswith("fc.")) <= tol, worst
    assert max(v for k, v in worst.items() if k.startswith("cnn_base.")) <= conv_tol, worst
    for name, zf in aux.get("relu_flips", {}).items():
        scale = float(bufs.hid1.abs().max()) if name == "fc.0" else float(bufs.hid2.abs().max()) if name == "fc.2" else \
            float(aux["conv_out"][CONV_NAMES.index(name)].abs().max())
        assert zf.numel() == 0 or float(zf.abs().max()) <= tol * scale, name


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("NA", [1, 2, 15, 16])
def test_head_widths(dev, NA, mode):
    """n_actions other than 9 moves every conv offset in the arena and every lane count of the head: the whole step, the
    head kernel element-wise (bf16 mode: every kernel of the step), the serving paths, the label check and (bf16) the
    operand-image refresh of the fused Adam."""
    from carla_imitation_learning_b200 import FusedAdam, stage_frames, stage_gray, sliding_window
    B = 129
    net = _net({"obs_size": 4, "n_actions": NA, "precision": mode})
    eng = net.engine()
    frames = _uniform_frames(500 + NA, B + 4)
    rng = np.random.Generator(np.random.PCG64(NA))
    yn = rng.integers(0, NA, size=B)
    yn[0], yn[-1] = 0, NA - 1
    y = torch.from_numpy(yn)
    fr = torch.from_numpy(frames).to(dev)
    stage = (lambda f: stage_frames(f)) if mode == "bf16" else (lambda f: sliding_window(stage_gray(f)))
    x = stage(fr)
    bufs = eng.train_forward_backward(x, y.to(dev))
    torch.cuda.synchronize()
    eng.check_device_errors()
    P = {k: _cpu64(v) for k, v in net.state_dict().items()}
    G = _grads(net, eng)
    tag = f"{mode} NA={NA} B={B}"
    if mode == "bf16" and NA > 1:       # every kernel of the step, the head's included, at this arena layout
        _check_bf16_kernels(tag, net, eng, bufs, x, y, B, 4, NA)
    else:
        print(f"\n{tag}")
        _check_head_fwd(tag, bufs, P, B, NA)
        _check_head_bwd(tag, bufs, P, G, y, B, NA, power=NA > 1)
    if NA == 1:         # softmax over one class: exactly zero loss and gradients
        assert float(bufs.loss) == 0.0
        assert int(torch.count_nonzero(bufs.dlogits)) == 0
        assert int(torch.count_nonzero(eng.grads)) == 0
    else:
        _whole_step_vs_oracle(net, bufs, G, frames, y, B, mode)
    # serving: the one-launch tail and the layer-by-layer chain return the first maximum of their own logits
    with torch.no_grad():
        for xs, tails in ((stage(fr[:7]), (True, False)), (x, (False,))):
            for tail in tails:
                actions, sb = eng.forward_act(xs, tail=tail)
                torch.cuda.synchronize()
                assert sb.logits.shape == (xs.shape[0], NA)
                assert torch.equal(actions.cpu(), sb.logits.cpu().argmax(1)), (tail, xs.shape[0])
    # a label equal to n_actions is reported through the device flag
    bad = y.clone()
    bad[5] = NA
    eng.train_forward_backward(x, bad.to(dev))
    with pytest.raises(RuntimeError, match="label outside"):
        eng.check_device_errors()
    if mode == "bf16":
        bufs = eng.train_forward_backward(x, y.to(dev))
        opt = FusedAdam(list(net.parameters()), lr=1e-3)
        p0, g0 = net._arena.detach().cpu().clone(), eng.grads.cpu().clone()
        opt.step_flat(eng.grads)
        torch.cuda.synchronize()
        kept = eng.w_packed.clone()
        eng.pack_weights()
        torch.cuda.synchronize()
        assert torch.equal(kept, eng.w_packed)
        p = p0.clone()
        O.adam_update(p, g0, torch.zeros_like(p), torch.zeros_like(p), 1)
        assert float((net._arena.detach().cpu() - p).abs().max()) <= 2e-7 * float(p.abs().max()) + 1e-9
    eng.check_device_errors()


# ------------------------------------------------------------------------------- batch invariance of the forward
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_forward_is_batch_invariant(dev, mode):
    """B = 4096 puts conv4's forward into a second wave and 32 samples on each head CTA; chunks of 128 give one sample per
    head CTA and a single wave everywhere. act[3] and the logits of every sample are bitwise the same either way, and the
    first chunk is bounded against f64 on its own operands."""
    from carla_imitation_learning_b200 import stage_frames, stage_gray, sliding_window
    B, CH = 4096, 128
    net = _net({"obs_size": 4, "n_actions": 9, "precision": mode})
    eng = net.engine()
    fr = torch.from_numpy(_uniform_frames(4096, B + 4)).to(dev)
    stage = (lambda f: stage_frames(f)) if mode == "bf16" else (lambda f: sliding_window(stage_gray(f)))
    with torch.no_grad():
        big = eng.forward(stage(fr))
        torch.cuda.synchronize()
        a3, lg = big.act[3].clone(), big.logits.clone()
        del big
        for i in range(B // CH):
            xi = stage(fr[i * CH:i * CH + CH + 4])
            b = eng.forward(xi)
            torch.cuda.synchronize()
            assert torch.equal(b.act[3], a3[i * CH:(i + 1) * CH]), (mode, i)
            assert torch.equal(b.logits, lg[i * CH:(i + 1) * CH]), (mode, i)
            if i == 0:
                if mode == "bf16":
                    planes = _planes_from_tp(xi.tp).double()
                else:
                    planes = stage_gray(fr[:CH + 4]).cpu().double()
                x = planes.as_strided((CH, 4, 256, 256), (65536, 65536, 256, 1))
                P = {k: _cpu64(v) for k, v in net.state_dict().items()}
                print(f"\n{mode} B={B}, first chunk of {CH}")
                _check_forward(f"{mode} chunk0", b, P, x, CH, 9, mode == "bf16")
    eng.check_device_errors()
