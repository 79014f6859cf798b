"""The serving path -- ConvNet1.act(), engine.forward_act(), bench.py --workload infer -- against exact references.

Every stage is compared element-wise with the f64 computation on exactly the operands it read from the buffers of the same
run, with the bound of tests/test_gpu_batch_edges.py: |got - ref| <= TAU * S, S = the f64 sum of the absolute terms.
The one-launch tail (csrc/policy_tail.cu: conv3, conv4, the three Linear layers and the argmax, an 8-CTA cluster per
sample) is checked stage by stage on its own output of the stage before, at every head width and at batches around the
point where its clusters no longer fit on the GPU at once. Every output buffer is filled with NaN (actions with -1) before
a launch, so an element the kernel failed to write fails. Mix-up power: the f64 reference of sample b is farther than the
bound from every other sample's device output in some element, so output written to another sample's slot fails.
The greedy action is checked on crafted logits (ties, +-inf, NaN) on all three paths against torch.argmax on the CPU.
`pytest -s` prints the smallest headroom (bound / error) and the power margins per tensor.
"""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from tests.test_gpu_batch_edges import (TAU, _at_routing, _bound, _check_conv1, _check_forward, _conv_in, _conv_w, _cpu64,
                                        _net, _planes_from_tp, _uniform_frames)
from tests.test_gpu_parity import _check_routing

pytestmark = pytest.mark.gpu

F = torch.nn.functional
PLANE = 256 * 256
NAN = float("nan")


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (no CPU fallback exists to run instead)")
    torch.set_num_threads(os.cpu_count() or 1)
    return torch.device("cuda", 0)


def _frames(seed, n):
    """Uniform frames, each scaled by its own gain in [0.25, 1]: samples then differ in their mean brightness, so that every
    sample's outputs stand apart from every other sample's by far more than the bound (the mix-up power check)."""
    gain = np.random.Generator(np.random.PCG64(seed + 1)).uniform(0.25, 1.0, size=(n, 1, 1, 1))
    return (_uniform_frames(seed, n) * gain.astype(np.float32)).astype(np.uint8)


def _stage(mode, fr, obs=4):
    """(the batch forward_act takes, the (B, obs, 256, 256) f64 CPU planes conv1 reads from it)."""
    from carla_imitation_learning_b200 import stage_frames, stage_gray, sliding_window
    step = obs // 4
    if mode == "bf16":
        x = stage_frames(fr, frame_skip=obs, step=step)
        planes = lambda: _planes_from_tp(x.tp).double()
    else:
        gray = stage_gray(fr)
        x = sliding_window(gray, obs, step)
        planes = lambda: _cpu64(gray)
    B = x.shape[0]
    return x, lambda: planes().as_strided((B, obs, 256, 256), (step * PLANE, PLANE, 256, 1))


def _poison(bufs, out):
    """Every output of the serving forward NaN (pool routing 255), the actions -1."""
    for t in (*bufs.act, bufs.hid1, bufs.hid2, bufs.logits):
        t.fill_(NAN)
    for t in bufs.amax:
        t.fill_(255)
    out.fill_(-1)


def _mixup(tag, got, ref, S):
    """For every sample b, ref[b] differs from got[b'] (b' != b) by more than the bound in some element. Returns the margin."""
    B = ref.shape[0]
    if B == 1:
        return float("inf")
    g, r, t = _cpu64(got).reshape(B, -1), ref.double().reshape(B, -1), TAU * S.double().reshape(B, -1)
    d = ((r[:, None, :] - g[None, :, :]).abs() / t[:, None, :]).amax(-1)
    d.fill_diagonal_(float("inf"))
    margin = float(d.min())
    assert margin > 1, f"{tag}: the reference of sample {int(d.min(1).values.argmin())} matches another sample's output"
    return margin


def _stage_check(tag, got, ref, S, mixup=True):
    _bound(tag, got, ref, S)
    if mixup:
        print(f"  {tag:<34s} mix-up power {_mixup(tag, got, ref, S):10.3g}")


def _conv_pool(xin, w, bias):
    """relu(maxpool2(conv(x))) in f64 and its bound S pooled the same way: the tail adds the bias after the 2x2 maximum, and
    |max a - max b| <= max |a - b|, so the bound of a pooled value is TAU times the largest S of its window."""
    z = F.conv2d(xin, w, bias)
    S = F.conv2d(xin.abs(), w.abs(), bias.abs())
    return torch.relu(F.max_pool2d(z, 2)), F.max_pool2d(S, 2)


def _check_tail(tag, bufs, P, B, NA, actions):
    """conv3 on act[1] as read (f32 master weights in both modes), conv4 on the device's act[2], the Linear layers on the
    device's act[3] / hid1 / hid2, and the action = the first maximum of the device's logits."""
    a1 = _cpu64(bufs.act[1])
    ref, S = _conv_pool(a1, P["cnn_base.6.weight"], P["cnn_base.6.bias"])
    _stage_check(f"{tag} tail act[2]", bufs.act[2], ref, S)
    ref, S = _conv_pool(_cpu64(bufs.act[2]), P["cnn_base.9.weight"], P["cnn_base.9.bias"])
    _stage_check(f"{tag} tail act[3]", bufs.act[3], ref, S)
    inp = _cpu64(bufs.act[3]).reshape(B, 128)
    for name, out, relu in (("fc.0", bufs.hid1, True), ("fc.2", bufs.hid2, True), ("fc.4", bufs.logits, False)):
        W, b = P[f"{name}.weight"], P[f"{name}.bias"]
        ref = inp @ W.t() + b
        # one logit per sample (NA = 1) cannot tell 64 samples apart at this bound; the logits' sample indexing is the same
        # code at every width and is held to the mix-up check from NA = 2
        _stage_check(f"{tag} tail {name}", out, torch.relu(ref) if relu else ref, inp.abs() @ W.abs().t() + b.abs(),
                     mixup=name != "fc.4" or NA > 1)
        inp = _cpu64(out)
    assert bufs.logits.shape == (B, NA)
    _check_action(tag, actions, bufs.logits)


def _check_action(tag, actions, logits):
    lg = logits.cpu()
    assert bool(torch.isfinite(lg).all()), f"{tag}: logits not written"
    assert torch.equal(actions.cpu(), lg.argmax(1)), f"{tag}: the action is not the first maximum of the logits"


def _check_conv12(tag, bufs, P, planes, B, bf16):
    """conv1 and conv2 as the chain runs them, ahead of the tail (which writes no pool routing of its own)."""
    _check_conv1(tag, bufs, planes, _conv_w(P, 0, bf16), P["cnn_base.0.bias"], B)
    xin, w, bias = _conv_in(bufs, 1, bf16), _conv_w(P, 1, bf16), P["cnn_base.3.bias"]
    z, Sz = F.conv2d(xin, w, bias), F.conv2d(xin.abs(), w.abs(), bias.abs())
    am, got = bufs.amax[1].cpu(), bufs.act[1].cpu()
    _check_routing(z, am, got.double(), 2)
    _bound(f"{tag} conv2 fwd act[1]", got, torch.relu(_at_routing(z, am, 2)), _at_routing(Sz, am, 2))


_NETS = {}


def _cached_net(mode, NA, obs=4):
    key = (mode, NA, obs)
    if key not in _NETS:
        _NETS[key] = _net({"obs_size": obs, "n_actions": NA, "precision": mode}, seed=777 + NA + obs)
    return _NETS[key]


def _params(net):
    return {k: _cpu64(v) for k, v in net.state_dict().items()}


# ------------------------------------------------------------------------------- 1. the tail on its own operands
TAIL_CASES = [(B, 9) for B in (1, 2, 7, 8, 9, 16, 17, 18, 19, 20, 33, 63, 64)] + \
             [(B, NA) for NA in (1, 2, 15, 16) for B in (1, 8, 64)]


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("B,NA", TAIL_CASES)
def test_policy_tail_is_exact_on_its_operands(dev, B, NA, mode):
    """Up to 18 clusters of 8 CTAs (one CTA per SM) run at once: B = 16..20 bracket the second wave, 64 is the largest
    batch the tail takes."""
    net = _cached_net(mode, NA)
    eng = net.engine()
    fr = torch.from_numpy(_frames(100 * B + NA, B + 4)).to(dev)
    x, planes = _stage(mode, fr)
    bufs = eng.alloc(B, x, None, False)
    out = torch.empty(B, dtype=torch.int64, device=dev)
    _poison(bufs, out)
    with torch.no_grad():
        eng.forward_act(x, out=out, bufs=bufs, tail=True)
    torch.cuda.synchronize()
    eng.check_device_errors()
    tag = f"{mode} NA={NA} B={B}"
    print(f"\n{tag}")
    P = _params(net)
    if (B, NA) == (8, 9):                   # conv1 and conv2 ahead of the tail, once per mode
        _check_conv12(tag, bufs, P, planes(), B, mode == "bf16")
    _check_tail(tag, bufs, P, B, NA, out)


# ------------------------------------------------------------------------------- 2. the layer-by-layer serving chain
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("B", [1, 9, 64, 65, 129, 300])
def test_serving_chain_is_exact_on_its_operands(dev, B, mode):
    """tail=False: conv1..conv4 and head_kernel with the action taken inside it; a head CTA serves two samples from B = 129."""
    net = _cached_net(mode, 9)
    eng = net.engine()
    fr = torch.from_numpy(_frames(5000 + B, B + 4)).to(dev)
    x, planes = _stage(mode, fr)
    bufs = eng.alloc(B, x, None, False)
    out = torch.empty(B, dtype=torch.int64, device=dev)
    _poison(bufs, out)
    with torch.no_grad():
        eng.forward_act(x, out=out, bufs=bufs, tail=False)
    torch.cuda.synchronize()
    eng.check_device_errors()
    tag = f"{mode} chain B={B}"
    print(f"\n{tag}")
    _check_forward(tag, bufs, _params(net), planes(), B, 9, mode == "bf16")
    _check_action(tag, out, bufs.logits)


# ------------------------------------------------------------------------------- 3. greedy-action semantics
def _bias_cases(NA):
    """Named logit rows of width NA: ties, +-inf and NaN where the greedy action's rule is decided."""
    inf = float("inf")
    base = torch.linspace(-1.0, 1.0, NA)[torch.randperm(NA, generator=torch.Generator().manual_seed(NA))] + 0.125
    top = float(base.max()) + 1.0
    cases = {}

    def case(name, *sets, fill=None):
        t = base.clone() if fill is None else torch.full((NA,), fill)
        for idx, v in sets:
            t[idx] = v
        cases[name] = t
    case("tie at 0 and 1", (0, top), (1, top))
    case("tie at the last two", (NA - 2, top), (NA - 1, top))
    case("all equal", fill=0.375)
    case("unique maximum last", (NA - 1, top))
    case("-inf entries", (slice(0, NA, 2), -inf))
    case("all -inf", fill=-inf)
    case("two +inf", (NA // 2 - 1, inf), (NA - 1, inf))
    case("NaN after a larger value", (0, top), (1, NAN))
    case("NaN after +inf", (0, inf), (NA - 1, NAN))
    case("NaN at 0", (0, NAN))
    case("all NaN", fill=NAN)
    return cases


def _same_logits(got, ref):
    got, ref = got.cpu(), ref.cpu().expand_as(got)
    nan = torch.isnan(ref)
    return torch.equal(torch.isnan(got), nan) and torch.equal(got[~nan], ref[~nan])


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("NA", [2, 9, 16])
def test_greedy_action_follows_torch_argmax(dev, NA, mode):
    """fc.4.weight = 0 makes every sample's logits exactly fc.4.bias (0 * h + b, h finite). Each crafted row through the
    tail (B = 1, 8), the chain (B = 9) and engine.argmax gives torch.argmax's answer on the CPU: the first maximum, and the
    first NaN where there is one."""
    net = _net({"obs_size": 4, "n_actions": NA, "precision": mode}, seed=31 + NA)
    eng = net.engine()
    prm = dict(net.named_parameters())
    with torch.no_grad():
        prm["fc.4.weight"].zero_()
    fr = torch.from_numpy(_frames(900 + NA, 9 + 4)).to(dev)
    runs = []
    for B, tail in ((1, True), (8, True), (9, False)):
        x, _ = _stage(mode, fr[:B + 4])
        runs.append((B, tail, x, eng.alloc(B, x, None, False), torch.empty(B, dtype=torch.int64, device=dev)))
    failed = []
    for name, row in _bias_cases(NA).items():
        with torch.no_grad():
            prm["fc.4.bias"].copy_(row.to(dev))
        want = int(row[None].argmax(1))
        for B, tail, x, bufs, out in runs:
            _poison(bufs, out)
            with torch.no_grad():
                eng.forward_act(x, out=out, bufs=bufs, tail=tail)
            got_eng = eng.argmax(bufs.logits)
            torch.cuda.synchronize()
            assert _same_logits(bufs.logits, row[None]), (name, B, tail, bufs.logits.cpu())
            for path, a in (("tail" if tail else "chain", out), ("engine.argmax", got_eng)):
                if not torch.equal(a.cpu(), torch.full((B,), want)):
                    failed.append(f"{name!r} {path} B={B}: {a.cpu().tolist()} (torch.argmax {want})")
    eng.check_device_errors()
    assert not failed, "\n".join(failed)


def test_bc_argmax_rows_over_several_blocks(dev):
    """bc_argmax through the C ABI on one (320, NA) tensor of all the crafted rows (3 blocks of 128 threads)."""
    from carla_imitation_learning_b200 import _lib
    lib = _lib.lib()
    for NA in (2, 9, 16):
        rows = torch.stack(list(_bias_cases(NA).values()))
        z = torch.randn(320, NA, generator=torch.Generator().manual_seed(NA))
        for r0 in (0, 150, 305):                                     # every crafted row in each of the three blocks
            z[r0:r0 + len(rows)] = rows
        zd = z.to(dev)
        out = torch.full((320,), -1, dtype=torch.int64, device=dev)
        _lib.check(lib.bc_argmax(zd.data_ptr(), out.data_ptr(), 320, NA, torch.cuda.current_stream().cuda_stream), "bc_argmax")
        torch.cuda.synchronize()
        want = z.argmax(1)
        bad = (out.cpu() != want).nonzero().flatten()
        assert bad.numel() == 0, [(int(i), z[i].tolist(), int(out[i]), int(want[i])) for i in bad[:8]]


# ------------------------------------------------------------------------------- 5. Adam -> tail launch ordering
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_weights_fetched_before_the_dependency_wait_reach_the_tail(dev, mode):
    """The tail, like the head, loads its weights (conv3, conv4, fc) before griddepcontrol.wait. Worst case: Adam directly
    followed by bc_policy_tail on an act[1] computed earlier, and Adam followed by forward_act(tail=True), as an evaluation
    rollout between training steps does. lr 3e-3 changes every logit each step. Back to back == the same sequence with a
    device synchronisation after every launch group, bitwise, over 5 steps."""
    from carla_imitation_learning_b200 import FusedAdam, _lib
    B = 8
    fr = torch.from_numpy(_frames(31337, B + 4)).to(dev)
    y = torch.from_numpy(np.random.Generator(np.random.PCG64(5)).integers(0, 9, size=B)).to(dev)
    runs = []
    for sync in (False, True):
        net = _net({"obs_size": 4, "n_actions": 9, "precision": mode}, seed=99)
        eng = net.engine()
        opt = FusedAdam(list(net.parameters()), lr=3e-3)
        opt.prepare()
        eng.ensure_packed()
        x, _ = _stage(mode, fr)
        train = eng.train_forward_backward(x, y)             # gradients + the act[1] the direct tail launches read
        serve = eng.alloc(B, x, None, False)
        a_direct = torch.empty(B, dtype=torch.int64, device=dev)
        a_served = torch.empty(B, dtype=torch.int64, device=dev)
        torch.cuda.synchronize()
        s = torch.cuda.current_stream().cuda_stream
        got = []
        for _ in range(5):
            opt.step_flat(eng.grads)
            if sync:
                torch.cuda.synchronize()
            _lib.check(eng.lib.bc_policy_tail(C.byref(eng.ctx(train)), a_direct.data_ptr(), s), "bc_policy_tail")
            if sync:
                torch.cuda.synchronize()
            got += [train.logits.clone(), train.hid1.clone(), a_direct.clone()]
            opt.step_flat(eng.grads)
            if sync:
                torch.cuda.synchronize()
            with torch.no_grad():
                eng.forward_act(x, out=a_served, bufs=serve, tail=True)
            if sync:
                torch.cuda.synchronize()
            got += [serve.logits.clone(), serve.act[2].clone(), a_served.clone()]
        torch.cuda.synchronize()
        eng.check_device_errors()
        runs.append(([t.cpu() for t in got], net._arena.detach().cpu().clone()))
    (ga, pa), (gb, pb) = runs
    assert torch.equal(pa, pb)
    for i, (a, b) in enumerate(zip(ga, gb)):
        assert torch.equal(a, b), (mode, "step", i // 6, "tensor", i % 6)
    assert all(bool(torch.isfinite(t).all()) for t in ga[0::6] + ga[3::6])
    for k in (0, 3):                                           # the updates did change the logits, step after step
        assert all(not torch.equal(ga[k + 6 * i], ga[k + 6 * (i + 1)]) for i in range(4)), k


# ------------------------------------------------------------------------------- 6. captured serving == eager
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("B,tail", [(1, True), (8, True), (9, False), (64, False), (256, False)])
def test_captured_serving_equals_eager(dev, B, tail, mode):
    """As bench.py --workload infer builds it: staging with out= and forward_act on persistent buffers, one CUDA graph per
    input over 3 rotating inputs. Every replay's actions and logits equal an eager call on the same input, bitwise."""
    from carla_imitation_learning_b200 import stage_frames, stage_gray, sliding_window
    net = _cached_net(mode, 9)
    eng = net.engine()
    frames = [torch.from_numpy(_frames(7000 + 10 * B + k, B + 4)).to(dev) for k in range(3)]
    if mode == "bf16":
        staged = stage_frames(frames[0])
        x = staged
    else:
        gray = torch.empty((B + 4, 256, 256), dtype=torch.float32, device=dev)
        x = sliding_window(gray)
    bufs = eng.alloc(B, x, None, False)
    out = torch.empty(B, dtype=torch.int64, device=dev)

    def enqueue(fr):
        if mode == "bf16":
            stage_frames(fr, out=staged)
        else:
            stage_gray(fr, out=gray)
        eng.forward_act(x, out=out, bufs=bufs, tail=tail)
    with torch.no_grad():
        eager = []
        for fr in frames:
            a, sb = eng.forward_act(_stage(mode, fr)[0], tail=tail)
            eager.append((a.clone(), sb.logits.clone()))
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for fr in frames:
                enqueue(fr)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graphs = []
        for fr in frames:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                enqueue(fr)
            graphs.append(g)
    for k in (0, 1, 2, 1, 0, 2, 2):
        out.fill_(-1)
        bufs.logits.fill_(NAN)
        graphs[k].replay()
        torch.cuda.synchronize()
        assert torch.equal(out, eager[k][0]), (mode, B, k)
        assert torch.equal(bufs.logits, eager[k][1]), (mode, B, k)
    del graphs
    eng.check_device_errors()


# ------------------------------------------------------------------------------- 7. the stacked-camera network
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_stacked_camera_serving_is_exact_on_its_operands(dev, mode):
    """obs_size 12 (3 cameras x 4 frames, channel = 3 * frame + camera): sample i = planes [3i, 3i + 12). The tail at B = 1
    and 8 and the chain at B = 9 and 64, each stage on its own operands; net.act() returns the same actions."""
    net = _cached_net(mode, 9, obs=12)
    eng = net.engine()
    P = _params(net)
    fr_all = torch.from_numpy(_frames(1212, 3 * 64 + 12)).to(dev)
    for B, tail in ((1, True), (8, True), (9, False), (64, False)):
        x, planes = _stage(mode, fr_all[:3 * B + 12], obs=12)
        assert x.shape[0] == B
        bufs = eng.alloc(B, x, None, False)
        out = torch.empty(B, dtype=torch.int64, device=dev)
        _poison(bufs, out)
        with torch.no_grad():
            eng.forward_act(x, out=out, bufs=bufs, tail=tail)
            acted = net.act(x)
        torch.cuda.synchronize()
        eng.check_device_errors()
        tag = f"{mode} obs=12 {'tail' if tail else 'chain'} B={B}"
        print(f"\n{tag}")
        if tail:
            _check_conv12(tag, bufs, P, planes(), B, mode == "bf16")
            _check_tail(tag, bufs, P, B, 9, out)
        else:
            _check_forward(tag, bufs, P, planes(), B, 9, mode == "bf16")
            _check_action(tag, out, bufs.logits)
        assert torch.equal(acted, out), tag
