"""EXTENSION -- NO REFERENCE PARITY. The command-conditioned branched policy's training step (trainer.BranchedTrainStep) and
the branched head kernel it runs (csrc/head_branched.cu), against their specification in oracle/ext_oracle.py and against
the module path: graph == eager and step == module path bitwise, the head exact on its own operands, batch and branch
edges, the launch ordering of the branch Adam and the head, and LR milestones reaching both arenas."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import bc_oracle as O
from oracle import ext_oracle as X

pytestmark = pytest.mark.gpu

SRC_HW = (288, 320)


def _dev():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (no CPU fallback exists to run instead)")
    return torch.device("cuda", 0)


def _rel(got, ref):
    got, ref = got.detach().double().cpu(), ref.detach().double().cpu()
    return float((got - ref).abs().max() / ref.abs().max().clamp_min(1e-30))


def _net(G=4, n_out=3, kind="l1", precision="fp32"):
    from src.architectures.branched import ConvNet1Branched
    torch.manual_seed(12345)
    return ConvNet1Branched({"obs_size": 4, "n_actions": n_out, "n_branches": G, "branch_loss": kind,
                             "precision": precision}).to(_dev())


def _step(net, B, src_hw=None, graph=True, lr=1e-3):
    from carla_imitation_learning_b200.trainer import BranchedTrainStep
    opt = net.configure_optimizer(lr=lr)
    return BranchedTrainStep(net, opt, B, src_hw=src_hw, graph=graph), opt


def _inputs(B, G, n_out, kind, src_hw, seed, frames=None):
    """Seeded device inputs of one slot: frames, table (or None), command, target."""
    from carla_imitation_learning_b200.data import augment_table
    dev = _dev()
    gen = torch.Generator().manual_seed(seed)
    hw = src_hw or (256, 256)
    if frames is None:
        frames = torch.randint(0, 256, (B + 4, hw[0], hw[1], 3), generator=gen, dtype=torch.uint8)
    table = None if src_hw is None else torch.from_numpy(augment_table(seed, B + 4, src_hw))
    command = torch.randint(0, G, (B,), generator=gen)
    target = torch.randint(0, n_out, (B,), generator=gen) if kind == "ce" else torch.rand((B, n_out), generator=gen) * 2 - 1
    return tuple(None if t is None else t.to(dev).contiguous() for t in (frames, table, command, target))


def _branch_grads(net, flat):
    return {k: flat[p._bc_offset:p._bc_offset + p.numel()].view(p.shape)
            for k, p in net.named_parameters() if k.startswith("branches.")}


def _trunk_grads(net, flat):
    return {k: flat[p._bc_offset:p._bc_offset + p.numel()].view(p.shape)
            for k, p in net.named_parameters() if k.startswith("cnn_base.")}


def _state(opt):
    """Both arenas' parameters and Adam moments (copies)."""
    return [t.clone() for c in opt.children_ for t in (c._bound[0], c._bound[1], c._bound[2])]


def _head_f64(P, feat, command, target, G, kind):
    """The branched MLP in f64 on given features: (out, loss, branch grads, d loss / d feat)."""
    leaf = {k: v.detach().double().cpu().clone().requires_grad_(True) for k, v in P.items() if k.startswith("branches.")}
    f = feat.detach().double().cpu().clone().requires_grad_(True)
    cmd = command.cpu()
    outs = []
    for g in range(G):
        h = F.relu(F.linear(f, leaf[f"branches.{g}.0.weight"], leaf[f"branches.{g}.0.bias"]))
        h = F.relu(F.linear(h, leaf[f"branches.{g}.2.weight"], leaf[f"branches.{g}.2.bias"]))
        outs.append(F.linear(h, leaf[f"branches.{g}.4.weight"], leaf[f"branches.{g}.4.bias"]))
    allb = torch.stack(outs, 1)
    out = allb.gather(1, cmd.view(-1, 1, 1).expand(-1, 1, allb.shape[-1])).squeeze(1)
    if target is None:
        return out.detach(), None, None, None
    loss = X.branched_loss(out, target.cpu() if kind == "ce" else target.double().cpu(), kind)
    grads = torch.autograd.grad(loss, list(leaf.values()) + [f], allow_unused=True)
    named = {k: (torch.zeros_like(v) if g is None else g) for (k, v), g in zip(leaf.items(), grads[:-1])}
    return out.detach(), loss.detach(), named, grads[-1]


# ------------------------------------------------------------------------------- 1. the rewritten kernel, new cases
@pytest.mark.parametrize("case", ["g16", "one_branch", "b_not_multiple_of_nb", "b1"])
def test_rewritten_head_matches_the_specification(case):
    """net.loss(...).backward() and net(x, command) against the f64 specification, to the tolerances of the existing
    branched test (1e-5 for outputs, loss and branch gradients; 5e-3 for the trunk's routing-dependent gradients), at the
    cases the serial command scan never met: 16 branches, every sample on one branch, a batch that is not a multiple of
    the CTAs per branch, and one sample."""
    G, B, kind, n_out = {"g16": (16, 40, "ce", 9), "one_branch": (4, 33, "l1", 3),
                         "b_not_multiple_of_nb": (4, 37, "mse", 3), "b1": (3, 1, "l1", 3)}[case]
    dev = _dev()
    net = _net(G, n_out, kind)
    P = {k: v.detach().cpu() for k, v in net.state_dict().items()}
    frames, labels = O.synth_frames(60 + G, B + 4)
    x, y = O.sequential_samples(frames, labels)
    x = torch.from_numpy(x)
    gen = torch.Generator().manual_seed(9)
    command = torch.full((B,), 2) if case == "one_branch" else torch.randint(0, G, (B,), generator=gen)
    target = torch.randint(0, n_out, (B,), generator=gen) if kind == "ce" else torch.randn((B, n_out), generator=gen)
    loss = net.loss(x.to(dev), command.to(dev), target.to(dev))
    loss.backward()
    out = net(x.to(dev), command.to(dev))
    torch.cuda.synchronize()
    net.engine().check_device_errors()
    ref_loss, ref_out, ref = X.branched_loss_and_grads(P, x, command, target, G, kind)
    assert _rel(out, ref_out) <= 1e-5
    assert abs(float(loss) - float(ref_loss)) <= 1e-5 * abs(float(ref_loss))
    got = {k: p.grad for k, p in net.named_parameters()}
    for k in ref:
        tol = 1e-5 if k.startswith("branches.") else 5e-3
        if float(ref[k].abs().max()) == 0.0:
            assert float(got[k].abs().max()) == 0.0, k
        else:
            assert _rel(got[k], ref[k]) <= tol, (k, _rel(got[k], ref[k]))


# ------------------------------------------------------------------------------- 2. graph == eager
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("aug", [False, True])
def test_graph_replays_equal_eager_steps_bitwise(precision, aug):
    """BranchedTrainStep with graph=True (eager pass, capture, replays) over 8 steps rotating over 3 input slots ==
    graph=False on the same inputs: every loss, both parameter arenas and both sets of Adam moments, bit for bit."""
    B, G, n_out, kind = 16, 4, 3, "l1"
    src_hw = SRC_HW if aug else None
    slots = [_inputs(B, G, n_out, kind, src_hw, 30 + s) for s in range(3)]
    res = []
    for graph in (True, False):
        net = _net(G, n_out, kind, precision)
        st, opt = _step(net, B, src_hw, graph=graph)
        losses = []
        for i in range(8):
            losses.append(st.step(*slots[i % 3]).clone())
        torch.cuda.synchronize()
        st.check()
        res.append((torch.stack(losses).cpu(), _state(opt)))
    (la, sa), (lb, sb) = res
    assert torch.isfinite(la).all() and torch.equal(la, lb)
    for a, b in zip(sa, sb):
        assert torch.equal(a, b)
    assert not torch.equal(la[0], la[3])


# ------------------------------------------------------------------------------- 3. step == module path
@pytest.mark.parametrize("precision,kind,n_out", [("fp32", "ce", 9), ("bf16", "l1", 3)])
def test_step_equals_the_module_path_bitwise(precision, kind, n_out):
    """One BranchedTrainStep == stage_augmented -> net.loss -> backward -> MultiArenaAdam.step on the same frames: the step
    adds no arithmetic of its own (loss, both arenas and both sets of moments, bit for bit)."""
    from carla_imitation_learning_b200 import sliding_window, stage_augmented
    B, G = 12, 4
    f, t, c, y = _inputs(B, G, n_out, kind, SRC_HW, 5)
    net = _net(G, n_out, kind, precision)
    st, opt = _step(net, B, SRC_HW)
    loss_s = st.step(f, t, c, y).clone()
    torch.cuda.synchronize()
    st.check()
    net_m = _net(G, n_out, kind, precision)
    opt_m = net_m.configure_optimizer(lr=1e-3)
    x = stage_augmented(f, t, layout="tp") if precision == "bf16" else sliding_window(stage_augmented(f, t))
    loss_m = net_m.loss(x, c, y)
    opt_m.zero_grad()
    loss_m.backward()
    opt_m.step()
    torch.cuda.synchronize()
    assert torch.equal(loss_s, loss_m.detach())
    for a, b in zip(_state(opt), _state(opt_m)):
        assert torch.equal(a, b)


# ------------------------------------------------------------------------------- 4. against the specification
@pytest.mark.parametrize("B", [7, 256])
def test_fp32_step_matches_the_specification(B):
    """fp32, one step: the commanded outputs, the loss and every branch gradient against the f64 specification (rel 1e-5),
    the trunk's conv gradients within the routing-dependent 5e-3 of the existing branched test."""
    G, n_out, kind = 4, 3, "l1"
    frames, labels = O.synth_frames(70, B + 4)
    f, _t, c, y = _inputs(B, G, n_out, kind, None, 8, frames=torch.from_numpy(frames))
    net = _net(G, n_out, kind)
    P = {k: v.detach().cpu() for k, v in net.state_dict().items()}
    st, _opt = _step(net, B)
    loss = st.step(f, None, c, y)
    torch.cuda.synchronize()
    st.check()
    x = torch.from_numpy(O.sequential_samples(frames, labels)[0])
    ref_loss, ref_out, ref = X.branched_loss_and_grads(P, x, c.cpu(), y.cpu(), G, kind)
    assert _rel(st.out, ref_out) <= 1e-5
    assert abs(float(loss) - float(ref_loss)) <= 1e-5 * abs(float(ref_loss))
    got = {**_branch_grads(net, st.hb["grads"]), **_trunk_grads(net, st.eng.grads)}
    for k in ref:
        tol = 1e-5 if k.startswith("branches.") else 5e-3
        if float(ref[k].abs().max()) == 0.0:
            assert float(got[k].abs().max()) == 0.0, k
        else:
            assert _rel(got[k], ref[k]) <= tol, (k, _rel(got[k], ref[k]))


@pytest.mark.parametrize("aug", [False, True])
def test_bf16_step_head_is_exact_on_its_own_operands(aug):
    """bf16: the head is exact f32 arithmetic on the device's own act[3]: outputs, loss, branch gradients and d loss / d act4
    equal the f64 branched MLP evaluated on those features, rel 1e-5."""
    B, G, n_out, kind = 64, 4, 3, "l1"
    src_hw = SRC_HW if aug else None
    f, t, c, y = _inputs(B, G, n_out, kind, src_hw, 12)
    net = _net(G, n_out, kind, "bf16")
    P = {k: v.detach().clone() for k, v in net.state_dict().items()}
    st, _opt = _step(net, B, src_hw)
    loss = st.step(f, t, c, y)
    torch.cuda.synchronize()
    st.check()
    out, rloss, rg, rgfeat = _head_f64(P, st.bufs.act[3].view(B, 128), c, y, G, kind)
    assert _rel(st.out, out) <= 1e-5
    assert abs(float(loss) - float(rloss)) <= 1e-5 * abs(float(rloss))
    got = _branch_grads(net, st.hb["grads"])
    for k, r in rg.items():
        assert _rel(got[k], r) <= 1e-5, k
    assert _rel(st.bufs.ghead, rgfeat) <= 1e-5


def test_augmented_staging_inside_the_step_is_the_specification():
    """The f32 planes the step stages from 288x320 sources == X.stage_augmented bit for bit."""
    B = 6
    f, t, c, y = _inputs(B, 4, 3, "l1", SRC_HW, 21)
    net = _net()
    st, _opt = _step(net, B, SRC_HW)
    st.step(f, t, c, y)
    torch.cuda.synchronize()
    ref = X.stage_augmented(f.cpu().numpy(), t.cpu().numpy())
    assert np.array_equal(st.gray.cpu().numpy(), ref)


# ------------------------------------------------------------------------------- 5. batch and branch edges
def test_large_batch_head_against_the_specification_on_given_features():
    """B = 4096 (four command chunks): forward-only outputs (mode 0), then loss, branch gradients and d loss / d feat
    (mode 3), against the f64 branched MLP on the same features."""
    from carla_imitation_learning_b200 import _lib
    B, G, n_out, kind = 4096, 5, 3, "mse"
    dev = _dev()
    net = _net(G, n_out, kind)
    P = {k: v.detach().clone() for k, v in net.state_dict().items()}
    gen = torch.Generator().manual_seed(4)
    feat = torch.rand((B, 128), generator=gen).to(dev)
    command = torch.randint(0, G, (B,), generator=gen).to(dev)
    target = torch.randn((B, n_out), generator=gen).to(dev)
    bufs = SimpleNamespace(batch=B, act=[None, None, None, feat], ghead=torch.full((B, 128), float("nan"), device=dev))
    n = int(_lib.lib().bc_head_branched_partials_floats(G, n_out))
    hb = dict(out=torch.full((B, n_out), float("nan"), device=dev), dout=torch.empty((B, n_out), device=dev),
              loss=torch.zeros((), device=dev), grads=torch.zeros_like(net._barena), partials=torch.zeros(n, device=dev))
    net._head(bufs, hb, command, None, 0)
    torch.cuda.synchronize()
    out, _, _, _ = _head_f64(P, feat, command, None, G, kind)
    assert _rel(hb["out"], out) <= 1e-5
    hb["out"].fill_(float("nan"))
    net._head(bufs, hb, command, target, 3)
    torch.cuda.synchronize()
    net.engine().check_device_errors()
    out, rloss, rg, rgfeat = _head_f64(P, feat, command, target, G, kind)
    assert _rel(hb["out"], out) <= 1e-5
    assert abs(float(hb["loss"]) - float(rloss)) <= 1e-5 * abs(float(rloss))
    got = _branch_grads(net, hb["grads"])
    for k, r in rg.items():
        assert _rel(got[k], r) <= 1e-5, k
    assert _rel(bufs.ghead, rgfeat) <= 1e-5


def test_a_branch_without_samples_gets_zero_gradient_and_keeps_its_parameters():
    B, G = 24, 4
    f, t, c, y = _inputs(B, G, 3, "l1", None, 13)
    c = (c % (G - 1)).contiguous()                          # branch G-1 gets no sample
    net = _net(G)
    st, _opt = _step(net, B)
    before = net._barena.clone()
    st.step(f, t, c, y)
    torch.cuda.synchronize()
    st.check()
    L = net._head_len
    assert float(st.hb["grads"][(G - 1) * L:].abs().max()) == 0.0
    assert torch.equal(net._barena[(G - 1) * L:], before[(G - 1) * L:])
    assert not torch.equal(net._barena[:L], before[:L])


def test_out_of_range_command_raises_at_check_and_leaves_zero_rows():
    B, G = 20, 4
    f, t, c, y = _inputs(B, G, 3, "l1", None, 14)
    c[5], c[11] = G, -1
    net = _net(G)
    st, _opt = _step(net, B)
    st.hb["out"].fill_(float("nan"))
    st.bufs.ghead.fill_(float("nan"))
    st.step(f, t, c, y)
    torch.cuda.synchronize()
    with pytest.raises(RuntimeError, match="command"):
        st.check()
    for b in (5, 11):
        assert float(st.out[b].abs().max()) == 0.0 and float(st.bufs.ghead[b].abs().max()) == 0.0
    assert torch.isfinite(st.out).all() and torch.isfinite(st.bufs.ghead).all()
    st.check()                                              # the flag was cleared by the raise


def test_step_rejects_wrong_inputs():
    B = 8
    net = _net()
    st, _opt = _step(net, B, SRC_HW)
    f, t, c, y = _inputs(B, 4, 3, "l1", SRC_HW, 1)
    with pytest.raises(ValueError):
        st.step(f, None, c, y)                              # augmentation needs its table
    with pytest.raises(ValueError):
        st.step(f, t, c.int(), y)                           # command dtype
    with pytest.raises(ValueError):
        st.step(f, t, c, y[:, :2].contiguous())             # target shape
    with pytest.raises(ValueError):
        st.step(f.cpu(), t, c, y)                           # device
    with pytest.raises(ValueError):
        st.step(f[:-1].contiguous(), t, c, y)               # B + 4 frames


# ------------------------------------------------------------------------------- 6. launch ordering
def test_branch_weights_fetched_before_the_dependency_wait_are_the_updated_ones():
    """The branched head fetches its branch's weights BEFORE griddepcontrol.wait; that is sound only because the branch
    Adam (bc_adam_tick_step) releases its dependents after its last write. Worst case: the branch Adam directly followed
    by the head (lr 3e-3, nothing in between), bitwise against the same sequence with a device synchronisation after
    every launch, over several steps. Branch-arena counterpart of test_gpu_step's single-head ordering test."""
    B, G, n_out, kind = 256, 4, 3, "l1"
    f, _t, c, y = _inputs(B, G, n_out, kind, None, 15)
    from carla_imitation_learning_b200 import stage_frames
    out = []
    for sync in (False, True):
        net = _net(G, n_out, kind, "bf16")
        opt = net.configure_optimizer(lr=3e-3)
        opt.prepare()
        badam = opt.children_[1]
        bufs = net._trunk_forward(net.engine().check_input(stage_frames(f)), True)
        hb = net._bbufs(B)
        torch.cuda.synchronize()
        outs = []
        for _ in range(5):
            net._head(bufs, hb, c, y, 3)
            if sync:
                torch.cuda.synchronize()
            badam.step_flat(hb["grads"])
            if sync:
                torch.cuda.synchronize()
            net._head(bufs, hb, c, None, 0)              # follows the branch Adam directly
            if sync:
                torch.cuda.synchronize()
            outs.append(hb["out"].clone())
        torch.cuda.synchronize()
        net.engine().check_device_errors()
        out.append((torch.stack(outs).cpu(), net._barena.clone().cpu()))
    (oa, pa), (ob, pb) = out
    assert torch.isfinite(oa).all()
    assert torch.equal(pa, pb) and torch.equal(oa, ob)
    assert not torch.equal(oa[0], oa[-1])


# ------------------------------------------------------------------------------- 7. LR milestone
def test_lr_change_between_replays_reaches_both_arenas():
    """param_groups[0]['lr'] changed between two graph replays (a MultiStepLR milestone) reaches the device scalars of
    both captured Adam kernels: the graph run equals the eager run with the same change, bitwise."""
    B, G = 16, 4
    slots = [_inputs(B, G, 3, "l1", None, 40 + s) for s in range(2)]
    res = []
    for graph in (True, False):
        net = _net(G)
        st, opt = _step(net, B, graph=graph)
        for i in range(6):                                  # per slot: eager, capture, replay
            st.step(*slots[i % 2])
        opt.param_groups[0]["lr"] = 1e-4
        for i in range(2):
            st.step(*slots[i % 2])
        torch.cuda.synchronize()
        assert [float(c._bound[3][0]) for c in opt.children_] == [1e-4, 1e-4]
        res.append(_state(opt))
    for a, b in zip(*res):
        assert torch.equal(a, b)
