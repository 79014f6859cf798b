"""EXTENSION -- NO REFERENCE PARITY. Serving the command-conditioned branched policy (ConvNet1Branched.act,
trainer.BranchedActStep, bc_forward_branched_act) against exact references.

Two paths: the one-launch tail (bc_policy_tail_branched: conv3, conv4 and the commanded branch's three Linear layers in one
8-CTA cluster per sample) and the layer path (conv1..conv4, then head_branched_kernel with the greedy action taken inside
it). Each stage is bounded element-wise against f64 on the operands it read, with the bound of tests/test_gpu_batch_edges.py:
|got - ref| <= TAU * S, S = the f64 sum of the absolute terms. Every output buffer is filled with NaN before a launch and
the actions with -1, so an element the kernels failed to write fails. Mix-up power: per sample (another sample's output
in b's slot fails) and per branch (the device's out[b] is farther than the bound from every other branch's f64 output on the
same features, so a tail that read the wrong branch fails). `pytest -s` prints the headroom and the margins.
"""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from oracle import ext_oracle as X
from tests.test_gpu_batch_edges import TAU, _bound, _cpu64
from tests.test_gpu_serving import NAN, _bias_cases, _conv_pool, _frames, _same_logits, _stage, _stage_check

pytestmark = pytest.mark.gpu

SRC_HW = (288, 320)


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (no CPU fallback exists to run instead)")
    torch.set_num_threads(os.cpu_count() or 1)
    return torch.device("cuda", 0)


def _bnet(mode, G, NA, kind="ce", seed=0):
    from src.architectures.branched import ConvNet1Branched
    torch.manual_seed(4242 + 97 * G + NA + seed)
    return ConvNet1Branched({"obs_size": 4, "n_actions": NA, "n_branches": G, "branch_loss": kind,
                             "precision": mode}).to(torch.device("cuda", 0))


_NETS = {}


def _cached(mode, G, NA):
    key = (mode, G, NA)
    if key not in _NETS:
        _NETS[key] = _bnet(mode, G, NA)
    return _NETS[key]


def _params(net):
    return {k: _cpu64(v) for k, v in net.state_dict().items()}


def _alternating(B, G, dev, shift=0):
    """Neighbouring samples carry different commands (for G > 1)."""
    return ((torch.arange(B) + shift) % G).to(dev)


def _serve(net, x, command, tail):
    """One bc_forward_branched_act on fresh buffers, every output NaN (actions -1) beforehand."""
    eng = net.engine()
    B = command.shape[0]
    bufs = eng.alloc(B, x, None, False)
    for t in (*bufs.act, bufs.hid1, bufs.hid2):
        t.fill_(NAN)
    out = torch.full((B, net.n_actions), NAN, device=command.device)
    actions = torch.full((B,), -1, dtype=torch.int64, device=command.device)
    with torch.no_grad():
        net._serve(bufs, out, actions, command, tail)
    torch.cuda.synchronize()
    return bufs, out, actions


def _branch_w(P, cmd, name):
    """(B, out, in) weights and (B, out) biases of each sample's commanded branch."""
    W = torch.stack([P[f"branches.{int(g)}.{name}.weight"] for g in cmd])
    b = torch.stack([P[f"branches.{int(g)}.{name}.bias"] for g in cmd])
    return W, b


def _linear(W, b, inp):
    return torch.einsum("boi,bi->bo", W, inp) + b, torch.einsum("boi,bi->bo", W.abs(), inp.abs()) + b.abs()


def _head_chain(P, cmd, a3):
    """The commanded branches' MLP in f64 on features a3 (B, 128): (out, S of the whole chain: the absolute values of every
    weight, bias and input carried through the three layers)."""
    inp, S = a3, a3.abs()
    for name, relu in (("0", True), ("2", True), ("4", False)):
        W, b = _branch_w(P, cmd, name)
        z, _ = _linear(W, b, inp)
        S = torch.einsum("boi,bi->bo", W.abs(), S) + b.abs()
        inp = torch.relu(z) if relu else z
    return inp, S


def _branch_mixup(tag, out, a3, P, cmd, G):
    """out[b] is farther than the bound from every other branch's f64 output on the same features a3[b]. Skipped for one
    output per sample (NA = 1), where two of up to 16 x 64 random values may fall within 1e-5 of each other; the branch
    indexing is the same code at every width and is held to the check from NA = 2."""
    if G == 1 or out.shape[1] == 1:
        return float("inf")
    got = _cpu64(out)
    margin = float("inf")
    for g in range(G):
        ref, S = _head_chain(P, torch.full_like(cmd, g), a3)
        d = ((got - ref).abs() / (TAU * S)).amax(1)
        other = cmd != g
        if bool(other.any()):
            margin = min(margin, float(d[other].min()))
    assert margin > 1, f"{tag}: some sample's output is within the bound of another branch's output"
    return margin


def _check_tail(tag, bufs, out, actions, P, cmd, G, NA):
    """conv3 on act[1] (f32 master weights in both modes), conv4 on the device's act[2], the commanded branch's fc.0, fc.2
    and fc.4 on the device's act[3] / hid1 / hid2, the action = the first maximum of the device's out."""
    B = cmd.shape[0]
    cmd = cmd.cpu()
    ref, S = _conv_pool(_cpu64(bufs.act[1]), P["cnn_base.6.weight"], P["cnn_base.6.bias"])
    _stage_check(f"{tag} act[2]", bufs.act[2], ref, S)
    ref, S = _conv_pool(_cpu64(bufs.act[2]), P["cnn_base.9.weight"], P["cnn_base.9.bias"])
    _stage_check(f"{tag} act[3]", bufs.act[3], ref, S)
    a3 = _cpu64(bufs.act[3]).reshape(B, 128)
    inp = a3
    for name, got, relu in (("0", bufs.hid1, True), ("2", bufs.hid2, True), ("4", out, False)):
        W, b = _branch_w(P, cmd, name)
        ref, S = _linear(W, b, inp)
        # per-sample mix-up of out from NA = 3: one or two outputs of 64 samples spread over the branches can fall within the
        # bound of another sample's; out's sample indexing is the same code at every width
        _stage_check(f"{tag} fc.{name}", got, torch.relu(ref) if relu else ref, S, mixup=name != "4" or NA > 2)
        inp = _cpu64(got)
    print(f"  {tag + ' branch mix-up':<34s} margin {_branch_mixup(tag, out, a3, P, cmd, G):10.3g}")
    _check_action(tag, actions, out)


def _check_action(tag, actions, out):
    o = out.cpu()
    assert bool(torch.isfinite(o).all()), f"{tag}: out not written"
    assert torch.equal(actions.cpu(), o.argmax(1)), f"{tag}: the action is not the first maximum of out"


# ------------------------------------------------------------------------------- 1. the tail on its own operands
TAIL_CASES = ([(B, 4, 9) for B in (1, 2, 7, 8, 9, 16, 17, 18, 19, 20, 33, 63, 64)]
              + [(B, G, NA) for G in (1, 16) for NA in (1, 2, 3, 9, 15, 16) for B in (1, 8, 64)]
              + [(B, 4, NA) for NA in (1, 2, 3, 15, 16) for B in (8, 64)])


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("B,G,NA", TAIL_CASES)
def test_branched_tail_is_exact_on_its_operands(dev, B, G, NA, mode):
    """Commands alternate between neighbouring samples, then one batch where every sample has the same command (G - 1)."""
    net = _cached(mode, G, NA)
    fr = torch.from_numpy(_frames(300 * B + 7 * G + NA, B + 4)).to(dev)
    x, _ = _stage(mode, fr)
    P = _params(net)
    for name, cmd in (("alternating", _alternating(B, G, dev)), ("all same", torch.full((B,), G - 1, dtype=torch.int64, device=dev))):
        bufs, out, actions = _serve(net, x, cmd, True)
        net.engine().check_device_errors()
        tag = f"{mode} G={G} NA={NA} B={B} {name}"
        print(f"\n{tag}")
        _check_tail(tag, bufs, out, actions, P, cmd, G, NA)


# ------------------------------------------------------------------------------- 2. the layer path with actions
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("B", [1, 9, 64, 65, 129, 300, 1023, 1024, 1025, 4096])
def test_layer_path_actions(dev, B, mode):
    """tail = 0: head_branched_kernel reads the commands in chunks of 1024. out is bitwise net.forward(x, command) (the
    existing path, no actions), bounded against the f64 chain of the commanded branch on the device's act[3] (3 TAU S: each
    Linear layer adds at most TAU times its own S, and ReLU is 1-Lipschitz), and the action is the first maximum of out. Up
    to B = 64 the tail agrees with it: each path is within 5 TAU S of the f64 chain from act[1] in fp32; in bf16 the layer
    path's conv3 and conv4 read bf16 operands, so the agreement is to 2^-5 S."""
    G, NA = 4, 9
    net = _cached(mode, G, NA)
    fr = torch.from_numpy(_frames(5000 + B, B + 4)).to(dev)
    x, _ = _stage(mode, fr)
    cmd = _alternating(B, G, dev)
    bufs, out, actions = _serve(net, x, cmd, False)
    net.engine().check_device_errors()
    with torch.no_grad():
        fwd = net(x, cmd).clone()
    torch.cuda.synchronize()
    assert torch.equal(out, fwd), "the layer path differs from net.forward"
    P = _params(net)
    tag = f"{mode} layers B={B}"
    print(f"\n{tag}")
    a3 = _cpu64(bufs.act[3]).reshape(B, 128)
    ref, S = _head_chain(P, cmd.cpu(), a3)
    if B <= 300:
        _stage_check(f"{tag} out (3 TAU S)", out, ref, 3 * S)
    else:                          # from ~1000 samples two of them can have all 9 outputs within 3 TAU S of each other
        _bound(f"{tag} out (3 TAU S)", out, ref, 3 * S)
    print(f"  {tag + ' branch mix-up':<34s} margin {_branch_mixup(tag, out, a3, P, cmd.cpu(), G):10.3g}")
    _check_action(tag, actions, out)
    if B <= 64:
        _t, out_t, act_t = _serve(net, x, cmd, True)
        Sc3 = _conv_pool(_cpu64(bufs.act[1]).abs(), P["cnn_base.6.weight"].abs(), P["cnn_base.6.bias"].abs())[0]
        Sc4 = _conv_pool(Sc3, P["cnn_base.9.weight"].abs(), P["cnn_base.9.bias"].abs())[0].reshape(B, 128)
        _z, S_full = _head_chain({k: v.abs() for k, v in P.items()}, cmd.cpu(), Sc4)
        tol = 10 * TAU * S_full if mode == "fp32" else 2.0 ** -5 * S_full
        err = (_cpu64(out_t) - _cpu64(out)).abs()
        assert bool((err <= tol).all()), f"{tag}: tail and layer path disagree by {float((err / tol).max()):.3g} x the bound"
        print(f"  {tag + ' tail vs layers':<34s} headroom {float((tol / err.clamp_min(1e-300)).min()):10.3g}")


# ------------------------------------------------------------------------------- 3. the greedy rule
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("NA", [2, 9, 16])
def test_greedy_action_follows_torch_argmax_per_branch(dev, NA, mode):
    """Every branch's fc.4.weight = 0 makes out exactly its fc.4.bias. The crafted rows of test_gpu_serving (ties, +-inf,
    NaN) are dealt to the branches, a different row per branch, and rotated so that every row reaches every branch. Tail
    at B = 1 and 8, layers at B = 9 and 300, commands alternating: each sample's action is torch.argmax on the CPU of its
    commanded branch's row."""
    G = 4
    net = _bnet(mode, G, NA, seed=1)
    prm = dict(net.named_parameters())
    with torch.no_grad():
        for g in range(G):
            prm[f"branches.{g}.4.weight"].zero_()
    rows = list(_bias_cases(NA).items())
    fr = torch.from_numpy(_frames(900 + NA, 300 + 4)).to(dev)
    runs = [(B, tail, _stage(mode, fr[:B + 4])[0], _alternating(B, G, dev, shift=B)) for B, tail in ((1, True), (8, True), (9, False), (300, False))]
    failed = []
    for i in range(len(rows)):
        picked = [rows[(i + g) % len(rows)] for g in range(G)]
        with torch.no_grad():
            for g, (_n, row) in enumerate(picked):
                prm[f"branches.{g}.4.bias"].copy_(row.to(dev))
        for B, tail, x, cmd in runs:
            _b, out, actions = _serve(net, x, cmd, tail)
            for b, g in enumerate(cmd.cpu().tolist()):
                name, row = picked[g]
                assert _same_logits(out[b:b + 1], row[None]), (name, B, tail, b, out[b].cpu())
                want = int(row[None].argmax(1))
                if int(actions[b]) != want:
                    failed.append(f"{name!r} branch {g} {'tail' if tail else 'layers'} B={B} b={b}: {int(actions[b])} (torch.argmax {want})")
    net.engine().check_device_errors()
    assert not failed, "\n".join(failed[:20])


# ------------------------------------------------------------------------------- 4. out-of-range commands
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("B,tail", [(8, True), (64, True), (300, False), (1100, False)])
def test_out_of_range_commands(dev, B, tail, mode):
    """-1, G and 2^40 mixed into a valid batch: flag 4 at check_device_errors(), a zero row and action 0 for those samples,
    and every other sample bitwise what it is with the bad commands replaced by valid ones."""
    G, NA = 4, 9
    net = _cached(mode, G, NA)
    eng = net.engine()
    fr = torch.from_numpy(_frames(77 + B, B + 4)).to(dev)
    x, _ = _stage(mode, fr)
    good = _alternating(B, G, dev)
    bad_at = torch.tensor([0, 3, B // 2, B - 1])
    bad = good.clone()
    bad[bad_at.to(dev)] = torch.tensor([-1, G, 2 ** 40, -(2 ** 40)], device=dev)
    eng.check_device_errors()
    _b, out_ok, act_ok = _serve(net, x, good, tail)
    eng.check_device_errors()
    _b, out_bad, act_bad = _serve(net, x, bad, tail)
    with pytest.raises(RuntimeError, match="command"):
        eng.check_device_errors()
    eng.check_device_errors()                                   # the flag was cleared by the raise
    keep = torch.ones(B, dtype=torch.bool)
    keep[bad_at] = False
    assert torch.equal(out_bad.cpu()[bad_at], torch.zeros(len(bad_at), NA))
    assert torch.equal(act_bad.cpu()[bad_at], torch.zeros(len(bad_at), dtype=torch.int64))
    assert torch.equal(out_bad.cpu()[keep], out_ok.cpu()[keep])
    assert torch.equal(act_bad.cpu()[keep], act_ok.cpu()[keep])


# ------------------------------------------------------------------------------- 5. ordering
def _step_inputs(B, G, src_hw, seed, dev, NA=3):
    gen = torch.Generator().manual_seed(seed)
    hw = src_hw or (256, 256)
    frames = torch.randint(0, 256, (B + 4, hw[0], hw[1], 3), generator=gen, dtype=torch.uint8).to(dev)
    command = torch.randint(0, G, (B,), generator=gen).to(dev)
    target = (torch.rand((B, NA), generator=gen) * 2 - 1).to(dev)
    return frames, command, target


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("B", [8, 64])
def test_replays_follow_a_rewritten_command_buffer(dev, B, mode):
    """A captured BranchedActStep replayed 5 times; before each replay a torch op rewrites the command buffer in place, with
    no synchronisation. Every replay equals an eager net.act with that command, bitwise."""
    from carla_imitation_learning_b200.trainer import BranchedActStep
    G = 4
    net = _cached(mode, G, 9)
    step = BranchedActStep(net, B)
    frames, command, _t = _step_inputs(B, G, None, 11 + B, dev)
    x, _ = _stage(mode, frames)
    cmds = [torch.randint(0, G, (B,), generator=torch.Generator().manual_seed(k)).to(dev) for k in range(5)]
    step.act(frames, None, command)
    step.act(frames, None, command)                              # captured
    assert len(step._graphs) == 1
    got = []
    for k in range(5):
        command.copy_(cmds[k])
        out, actions = step.act(frames, None, command)
        got.append((out.clone(), actions.clone()))
    torch.cuda.synchronize()
    step.check()
    for k in range(5):
        want = net.act(x, cmds[k])
        _b, want_out, _a = _serve(net, x, cmds[k], B <= net.tail_batch)
        assert torch.equal(got[k][1], want), (mode, B, k)
        assert torch.equal(got[k][0], want_out), (mode, B, k)
    assert any(not torch.equal(got[0][0], got[k][0]) for k in range(1, 5))


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_training_step_directly_followed_by_serving(dev, mode):
    """BranchedTrainStep.step then BranchedActStep.act (tail at B = 8, layers at B = 64), back to back for 5 steps, equals
    the same sequence with a synchronisation after every call, bitwise: the branch weights the serving kernels fetch before
    griddepcontrol.wait are the ones the Adam launch just wrote."""
    from carla_imitation_learning_b200.trainer import BranchedActStep, BranchedTrainStep
    G, NA, B = 4, 3, 8
    frames, command, target = _step_inputs(B, G, None, 5, dev)
    sf8, sc8, _ = _step_inputs(8, G, None, 6, dev)
    sf64, sc64, _ = _step_inputs(64, G, None, 7, dev)
    runs = []
    for sync in (False, True):
        net = _bnet(mode, G, NA, kind="l1", seed=2)
        tr = BranchedTrainStep(net, net.configure_optimizer(lr=3e-3), B)
        serve = [BranchedActStep(net, 8), BranchedActStep(net, 64)]
        torch.cuda.synchronize()
        got = []
        for _ in range(5):
            tr.step(frames, None, command, target)
            for st, f, c in ((serve[0], sf8, sc8), (serve[1], sf64, sc64)):
                if sync:
                    torch.cuda.synchronize()
                out, _a = st.act(f, None, c)
                if sync:
                    torch.cuda.synchronize()
                got.append(out.clone())
                tr.step(frames, None, command, target)
        torch.cuda.synchronize()
        tr.check()
        runs.append(([t.cpu() for t in got], net._barena.detach().cpu().clone()))
    (ga, pa), (gb, pb) = runs
    assert torch.equal(pa, pb)
    for i, (a, b) in enumerate(zip(ga, gb)):
        assert torch.equal(a, b), (mode, i)
    assert all(not torch.equal(ga[i], ga[i + 2]) for i in range(len(ga) - 2))    # the updates did change the outputs


# ------------------------------------------------------------------------------- 6. captured serving == eager
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("src_hw", [None, SRC_HW])
@pytest.mark.parametrize("B", [1, 8, 9, 64, 256])
def test_captured_serving_equals_eager(dev, B, src_hw, mode):
    """BranchedActStep over 3 rotating input slots (eager, capture, replays) == eager net.act on the same staged input,
    bitwise, for an L1 and a CE net. From 288x320 frames through center_crop_table the staged planes are X.stage_augmented's
    bit for bit, and within 4 f32 ulp of the 256x256 centre slice staged plainly (fp32 mode)."""
    from carla_imitation_learning_b200 import stage_augmented
    from carla_imitation_learning_b200.data import center_crop_table
    from carla_imitation_learning_b200.trainer import BranchedActStep
    G = 4
    for kind, NA in (("l1", 3), ("ce", 9)):
        net = _bnet(mode, G, NA, kind=kind, seed=3)
        step = BranchedActStep(net, B, src_hw=src_hw)
        assert step.tail == (B <= net.tail_batch)
        slots = [_step_inputs(B, G, src_hw, 100 * B + k, dev) for k in range(3)]
        table = None if src_hw is None else torch.from_numpy(center_crop_table(B + 4, src_hw)).to(dev)
        eager = []
        for f, c, _t in slots:
            x = (_stage(mode, f)[0] if src_hw is None
                 else stage_augmented(f, table, layout="tp" if mode == "bf16" else "plain"))
            if src_hw is not None and mode == "fp32":
                from carla_imitation_learning_b200 import sliding_window
                x = sliding_window(x)
            eager.append(net.act(x, c).clone())
        for k in (0, 1, 2, 0, 1, 2, 2, 1, 0):
            f, c, _t = slots[k]
            step.out.fill_(NAN)
            if step.actions is not None:
                step.actions.fill_(-1)
            out, actions = step.act(f, table, c)
            torch.cuda.synchronize()
            assert torch.equal(actions if kind == "ce" else out, eager[k]), (kind, mode, B, k)
            assert (actions is None) == (kind != "ce")
        assert len(step._graphs) == 3
        step.check()
        if src_hw is not None and mode == "fp32":
            f = slots[0][0]                                     # the slot staged last
            got = step.gray.cpu().numpy()
            ref = X.stage_augmented(f.cpu().numpy(), table.cpu().numpy())
            assert np.array_equal(got, ref)
            (cy, cx) = ((src_hw[0] - 256) // 2, (src_hw[1] - 256) // 2)
            from carla_imitation_learning_b200 import stage_gray
            plain = stage_gray(f[:, cy:cy + 256, cx:cx + 256].contiguous()).cpu().numpy()
            assert np.abs(got - plain).max() <= 2.0 ** -21                 # 4 f32 ulp of 1.0: the planes are in [0, 1]


# ------------------------------------------------------------------------------- 7. after training and reloading
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_serving_follows_training_and_reloaded_weights(dev, mode):
    """A few BranchedTrainStep steps, then load_state_dict of another net's weights (in bf16 mode the operand images are
    re-packed): the captured BranchedActStep follows both, on the tail (B = 8) and the layers (B = 64), and equals eager
    net.act on a net holding the same weights, bitwise."""
    from carla_imitation_learning_b200.trainer import BranchedActStep, BranchedTrainStep
    G, NA = 4, 3
    net = _bnet(mode, G, NA, kind="l1", seed=4)
    other = _bnet(mode, G, NA, kind="l1", seed=5)
    tr = BranchedTrainStep(net, net.configure_optimizer(lr=3e-3), 8)
    tf, tc, tt = _step_inputs(8, G, None, 9, dev)
    cases = []
    for B in (8, 64):
        f, c, _t = _step_inputs(B, G, None, 20 + B, dev)
        st = BranchedActStep(net, B)
        for _ in range(3):                                       # eager, capture, replay
            before = st.act(f, None, c)[0].clone()
        cases.append((st, f, c, _stage(mode, f)[0], before))
    for _ in range(3):
        tr.step(tf, None, tc, tt)
    for st, f, c, x, before in cases:
        out = st.act(f, None, c)[0].clone()
        assert not torch.equal(out, before)
        assert torch.equal(out, net.act(x, c))
    net.load_state_dict(other.state_dict())
    for st, f, c, x, _before in cases:
        out = st.act(f, None, c)[0].clone()
        assert torch.equal(out, other.act(_stage(mode, f)[0], c)), (mode, st.batch)
    tr.check()


# ------------------------------------------------------------------------------- 8. arguments
def test_arguments_are_checked(dev):
    from carla_imitation_learning_b200 import _lib
    from carla_imitation_learning_b200.trainer import BranchedActStep
    net = _cached("fp32", 4, 9)
    eng = net.engine()
    lib = eng.lib
    s = torch.cuda.current_stream().cuda_stream

    def call(B, hbatch=None, arena_off=0, tail=1):
        fr = torch.from_numpy(_frames(1, B + 4)).to(dev)
        x, _ = _stage("fp32", fr)
        bufs = eng.alloc(B, x, None, False)
        c = eng.ctx(bufs)
        h = _lib.BcBranched()
        h.n_branches, h.n_out, h.batch = 4, 9, B if hbatch is None else hbatch
        cmd = torch.zeros(B, dtype=torch.int64, device=dev)
        out = torch.empty((B, 9), device=dev)
        h.command, h.params, h.out = cmd.data_ptr(), net._barena.data_ptr() + 4 * arena_off, out.data_ptr()
        h.err_flag = eng.err_flag.data_ptr()
        act = torch.empty(B, dtype=torch.int64, device=dev)
        rc = lib.bc_forward_branched_act(C.byref(c), C.byref(h), act.data_ptr(), tail, s)
        torch.cuda.synchronize()
        return rc, lib.bc_last_error_string().decode()
    assert call(8)[0] == 0
    rc, msg = call(65)
    assert rc != 0 and "64" in msg, msg
    rc, msg = call(8, hbatch=7)
    assert rc != 0 and "batch" in msg, msg
    for tail in (0, 1):
        rc, msg = call(8, arena_off=1, tail=tail)
        assert rc != 0 and "16 B" in msg, msg
    x, _ = _stage("fp32", torch.from_numpy(_frames(2, 12)).to(dev))
    for bad in (torch.zeros(8, dtype=torch.int32, device=dev), torch.zeros((8, 1), dtype=torch.int64, device=dev),
                torch.zeros(7, dtype=torch.int64, device=dev)):
        with pytest.raises(ValueError, match="command"):
            net.act(x, bad)
    st = BranchedActStep(net, 8)
    f, c, _t = _step_inputs(8, 4, None, 3, dev)
    with pytest.raises(ValueError, match="command"):
        st.act(f, None, c.int())
    with pytest.raises(ValueError):
        st.act(f, torch.zeros((12, 8), device=dev), c)             # built without a crop: no table
    eng.check_device_errors()
