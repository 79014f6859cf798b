"""EXTENSION -- NO REFERENCE PARITY. Training of the command-conditioned branched policy beyond one step, against exact
references that share no code with the product:

A. bc_adam_tick_step, the Adam launch of every training path, against the Adam formula in f64, elementwise, at every
   arena size the product launches and across its grid-stride loop;
B. both arenas' Adam inside BranchedTrainStep (eager, capture, replay) against that formula on the step's own gradients,
   and the bits the update must never touch (the trunk's unused head, the arenas' padding);
C. a checkpoint of ImitationBranched: the Adam state of both arenas in torch.optim.Adam's layout, restored exactly;
D. a 40-step BranchedTrainStep loss curve against the f64 specification run live on the CPU;
E. the augmented staging kernels at crop corners, odd source sizes, every clamp and their grid-stride loops, and the
   host-side check of the augmentation table.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import bc_oracle as O
from oracle import ext_oracle as X

pytestmark = pytest.mark.gpu

SRC_HW = (288, 320)
EPS32 = 2.0 ** -24            # unit roundoff of f32


def _dev():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (no CPU fallback exists to run instead)")
    return torch.device("cuda", 0)


def _net(G=4, n_out=3, kind="l1", precision="fp32", seed=12345):
    from src.architectures.branched import ConvNet1Branched
    torch.manual_seed(seed)
    return ConvNet1Branched({"obs_size": 4, "n_actions": n_out, "n_branches": G, "branch_loss": kind,
                             "precision": precision}).to(_dev())


def _inputs(B, G, n_out, src_hw, seed):
    """Seeded device inputs of one slot for an L1 step: frames, augmentation table, command, target."""
    from carla_imitation_learning_b200.data import augment_table
    gen = torch.Generator().manual_seed(seed)
    frames = torch.randint(0, 256, (B + 4, src_hw[0], src_hw[1], 3), generator=gen, dtype=torch.uint8)
    table = torch.from_numpy(augment_table(seed, B + 4, src_hw, mean=0.45, std=0.22))
    command = torch.randint(0, G, (B,), generator=gen)
    target = torch.rand((B, n_out), generator=gen) * 2 - 1
    return tuple(t.to(_dev()).contiguous() for t in (frames, table, command, target))


def _children_state(opt):
    """[(params, exp_avg, exp_avg_sq, scalars)] of each arena's FusedAdam, copied to the host."""
    return [tuple(t.detach().cpu().clone() for t in c._bound[:4]) for c in opt.children_]


def _branch_len(n_out):
    from carla_imitation_learning_b200 import _lib
    off, siz = (C.c_int64 * 6)(), (C.c_int64 * 6)()
    return int(_lib.lib().bc_head_branched_layout(n_out, off, siz)), list(off), list(siz)


def _padding_mask(total, regions):
    """True on the floats of an arena that no tensor occupies."""
    pad = torch.ones(total, dtype=torch.bool)
    for o, n in regions:
        pad[o:o + n] = False
    return pad


# ------------------------------------------------------------------------------- the Adam formula and its bound
def _adam_check(before, grads, after, t, lr, gs=1.0, what=""):
    """`after` (p, m, v) == O.adam_update in f64 on the f32 values `before` and `grads` * gs, elementwise, within the
    rounding the kernel's f32 chain can add. Each bound is a few f32 roundoffs of the terms that enter the element:
      m = fma(1-b1, g-m, m):                 |dm| <= 2 eps (b1 |m0| + (1-b1) |g| + |m1|)
      v = fma((1-b2) g, g, b2 v):            |dv| <= 2 eps (b2 v0 + (1-b2) g^2 + v1)
      p = fma(-lr/bc1, m / (sqrt(v)/bc2 + e), p):  |dp| <= 2 eps |p1| + lr/bc1 (|dm| + 8 eps |m1|) / denom1
    (1-b2 = 0.001 is 0.8 eps away from its f32 rounding, b2 and 1-b1 less; sqrt, the two divides, the add and the
    rounding of the f64 scalars to f32 are 0.5 eps each). Returns the largest |error| / bound of p, m, v."""
    p0, m0, v0 = (x.double() for x in before)
    g = grads.detach().cpu().double() * gs
    p1, m1, v1 = p0.clone(), m0.clone(), v0.clone()
    O.adam_update(p1, g, m1, v1, t, lr=lr)
    b1, b2 = 0.9, 0.999
    tol_m = 2 * EPS32 * (b1 * m0.abs() + (1 - b1) * g.abs() + m1.abs())
    tol_v = 2 * EPS32 * (b2 * v0 + (1 - b2) * g * g + v1)
    step_size = lr / (1 - b1 ** t)
    denom = v1.sqrt() / (1 - b2 ** t) ** 0.5 + 1e-8
    tol_p = 2 * EPS32 * p1.abs() + step_size * (tol_m + 8 * EPS32 * m1.abs()) / denom
    worst = []
    for name, got, ref, tol in (("p", after[0], p1, tol_p), ("m", after[1], m1, tol_m), ("v", after[2], v1, tol_v)):
        err = (got.double() - ref).abs()
        bad = err > tol
        assert not bool(bad.any()), (what, name, t, int(bad.sum()), int(bad.nonzero()[0]), float(err.max()))
        nz = tol > 0
        worst.append(float((err[nz] / tol[nz]).max()) if bool(nz.any()) else 0.0)
    return worst


def _grads(gen, n, always_zero):
    """Gradients spanning 1e-12..1e3 in magnitude, both signs, ~5 % exact zeros, and exact zeros on `always_zero`."""
    mag = 10.0 ** (torch.rand(n, generator=gen, dtype=torch.float64) * 15 - 12)
    sign = torch.where(torch.rand(n, generator=gen) < 0.5, -1.0, 1.0).double()
    g = (mag * sign).float()
    g[torch.rand(n, generator=gen) < 0.05] = 0.0
    g[always_zero] = 0.0
    return g


def _adam_sizes():
    from carla_imitation_learning_b200 import _lib
    sizes = {"empty": 0, "one_vector": 4, "partial_last_cta": 3 * 1024 + 516}
    for n_out in (1, 3, 9):
        L = _branch_len(n_out)[0]
        for G in (1, 5, 16):
            sizes[f"branches_g{G}_nout{n_out}"] = G * L
    sizes["trunk"] = _lib.arena_layout(4, 9)[0]
    sizes["above_grid_cap"] = 5_000_004          # > 8 CTAs/SM x 148 SMs x 1024 floats: the grid-stride loop runs
    return sizes


ADAM_SIZES = ["empty", "one_vector", "partial_last_cta"] + [f"branches_g{G}_nout{n}" for n in (1, 3, 9) for G in (1, 5, 16)] \
    + ["trunk", "above_grid_cap"]


# ------------------------------------------------------------------------------- A. bc_adam_tick_step
@pytest.mark.parametrize("size", ADAM_SIZES)
def test_adam_tick_step_matches_the_adam_formula_elementwise(size):
    """bc_adam_tick_step (tick folded into the update, grad_scale read from st[5]) called directly, six launches on one
    state vector with grad_scale 0.5 and the learning rate changed between launches 3 and 4. After every launch, against
    O.adam_update in f64 on the same f32 inputs: p, m and v elementwise within the bound _adam_check derives (a few f32
    roundoffs of each element's own terms, not of the arena's maximum), an element whose gradient is always 0 bit for
    bit unchanged, st[4] == t, st[6] / st[7] == the f64 bias-correction formulas, the CTA counter st[8] back to 0.
    n = 0 still ticks and leaves its (non-null) buffers alone. On an NVIDIA B200 (1000 W limit) the largest error / bound
    over all sizes was 0.51 for p and m and 0.69 for v.
    The kernel is NOT bitwise torch.optim.Adam(foreach=False) on the same CUDA tensors: m is, but torch rounds
    v * beta2 before its addcmul where the kernel fuses both into one fma, so v differs in the last bit in about a third
    of the elements and p in under 1 % (measured at the sizes above). Hence the formula bound, not bit equality."""
    from carla_imitation_learning_b200 import _lib
    dev = _dev()
    n = _adam_sizes()[size]
    gen = torch.Generator().manual_seed(1000 + n % 997)
    cap = max(n, 4)                                              # n = 0: valid pointers, nothing may be touched
    p = torch.randn(cap, generator=gen)
    m, v = torch.zeros(cap), torch.zeros(cap)
    always_zero = torch.rand(cap, generator=gen) < 0.01
    pd, md, vd = p.to(dev), m.to(dev), v.to(dev)
    gd = torch.empty(cap, device=dev)
    st = torch.tensor([1e-3, 0.9, 0.999, 1e-8, 0, 0.5, 0, 0, 0], dtype=torch.float64, device=dev)
    lib, s = _lib.lib(), torch.cuda.current_stream().cuda_stream
    lr, worst = 1e-3, [0.0, 0.0, 0.0]
    for t in range(1, 7):
        if t == 4:
            lr = 3e-4
            st[0] = lr
        g = _grads(gen, cap, always_zero)
        gd.copy_(g)
        before = (pd.cpu(), md.cpu(), vd.cpu())
        _lib.check(lib.bc_adam_tick_step(pd.data_ptr(), gd.data_ptr(), md.data_ptr(), vd.data_ptr(), st.data_ptr(), n,
                                         None, 0, 0, s), "bc_adam_tick_step")
        torch.cuda.synchronize()
        after = (pd.cpu(), md.cpu(), vd.cpu())
        sc = st.cpu()
        assert float(sc[4]) == t
        assert float(sc[6]) == pytest.approx(lr / (1 - 0.9 ** t), rel=1e-14, abs=0)
        assert float(sc[7]) == pytest.approx((1 - 0.999 ** t) ** 0.5, rel=1e-14, abs=0)
        assert sc[8:9].view(torch.int64).item() & 0xFFFFFFFF == 0
        if n == 0:
            for a, b in zip(before, after):
                assert torch.equal(a, b)
            continue
        worst = [max(a, b) for a, b in zip(worst, _adam_check(before, g, after, t, lr, gs=0.5, what=size))]
        for a, b in zip(before, after):
            assert torch.equal(a[always_zero], b[always_zero])
    print(f"bc_adam_tick_step n={n}: largest error / bound of p, m, v: {worst[0]:.3f} {worst[1]:.3f} {worst[2]:.3f}")


# ------------------------------------------------------------------------------- B. both arenas inside the step
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("G", [1, 16])
def test_step_applies_the_adam_formula_to_both_arenas_on_its_own_gradients(precision, G):
    """BranchedTrainStep with augmentation from 288x320, 6 steps over 2 input slots (eager, eager, capture, capture,
    replay, replay), the learning rate lowered before the fifth step as a MultiStepLR milestone would. Before each step
    both arenas and both sets of moments are copied; after it, the update is recomputed in f64 from that copy and the
    gradients the step left in its buffers (eng.grads, hb['grads']): parameters and moments of both arenas elementwise
    within _adam_check's rounding bound, whatever the trajectory's sign noise. The trunk arena's unregistered fc region
    and the padding of both arenas stay bit for bit unchanged through all six steps, and their gradients are zero."""
    from carla_imitation_learning_b200 import _lib
    from carla_imitation_learning_b200.trainer import BranchedTrainStep
    B, n_out = 16, 3
    net = _net(G, n_out, "l1", precision)
    opt = net.configure_optimizer(lr=1e-3)
    stp = BranchedTrainStep(net, opt, B, src_hw=SRC_HW)
    slots = [_inputs(B, G, n_out, SRC_HW, 70 + s) for s in range(2)]
    total, off, siz = _lib.arena_layout(4, n_out)
    assert total == net._arena.numel()
    fixed_t = _padding_mask(total, zip(off[:8], siz[:8]))          # fc region (never registered) + padding
    L, boff, bsiz = _branch_len(n_out)
    pad_b = _padding_mask(G * L, [(g * L + o, n) for g in range(G) for o, n in zip(boff, bsiz)])
    assert fixed_t.any() and pad_b.any()
    p0 = (net._arena.detach().cpu().clone(), net._barena.detach().cpu().clone())
    lr, worst = 1e-3, [0.0, 0.0, 0.0]
    for i in range(6):
        if i == 4:
            lr = opt.param_groups[0]["lr"] = 1e-4
        before = _children_state(opt)
        stp.step(*slots[i % 2])
        torch.cuda.synchronize()
        stp.check()
        after = _children_state(opt)
        for k, (grads, fixed) in enumerate(((stp.eng.grads, fixed_t), (stp.hb["grads"], pad_b))):
            gk = grads.detach().cpu()
            assert torch.isfinite(gk).all() and float(gk[fixed].abs().max()) == 0.0, (k, i)
            w = _adam_check(before[k][:3], gk, after[k][:3], i + 1, lr, what=("trunk", "branches")[k])
            worst = [max(a, b) for a, b in zip(worst, w)]
            assert float(after[k][3][4]) == i + 1 and float(after[k][3][0]) == lr
            assert torch.equal(after[k][0][fixed], p0[k][fixed])
            assert float(after[k][1][fixed].abs().max()) == 0.0 and float(after[k][2][fixed].abs().max()) == 0.0
    assert (net._arena.cpu() != p0[0]).any() and (net._barena.cpu() != p0[1]).any()
    print(f"step Adam ({precision}, G={G}): largest error / bound of p, m, v: {worst[0]:.3f} {worst[1]:.3f} {worst[2]:.3f}")


# ------------------------------------------------------------------------------- C. checkpoint round trip
def _branched_model(G):
    from src.models.imitation_branched import ImitationBranched
    from torch.optim import lr_scheduler

    class _Model(ImitationBranched):
        def configure_optimizers(self):                 # milestones moved to [1, 2]: both epochs' LR changes are in play
            optimizer = self.net.configure_optimizer(lr=1e-3)
            scheduler = lr_scheduler.MultiStepLR(optimizer, milestones=[1, 2], gamma=0.1)
            self._schedulers = scheduler
            return [optimizer], [scheduler]

    hp = {"obs_size": 4, "n_actions": 3, "n_branches": G, "branch_loss": "l1"}
    return _Model, hp


def _loader(seed, n_batches, B, G, dev):
    frames, _ = O.synth_frames(seed, n_batches * B + 4)
    x = torch.from_numpy(O.sequential_samples(frames, np.zeros(len(frames), np.int64))[0]).to(dev)
    gen = torch.Generator().manual_seed(seed)
    command = torch.randint(0, G, (n_batches * B,), generator=gen).to(dev)
    target = (torch.rand((n_batches * B, 3), generator=gen) * 2 - 1).to(dev)
    return [(x[i * B:(i + 1) * B], command[i * B:(i + 1) * B], target[i * B:(i + 1) * B]) for i in range(n_batches)]


def _one_epoch(model, opt, sch, loader):
    """Trainer.fit's hook order for one epoch, on a given optimiser and scheduler."""
    for i, batch in enumerate(loader):
        loss = model.training_step(batch, i)
        opt.zero_grad()
        loss.backward()
        opt.step()
    sch.step()
    torch.cuda.synchronize()
    model.net.engine().check_device_errors()


def test_branched_checkpoint_round_trips_both_arenas_adam_state(tmp_path):
    """Trainer.fit(ImitationBranched) for 2 epochs (L1, 4 branches, MultiStepLR milestones at [1, 2]), then
    save_checkpoint: optimizer_states[0]['state'] holds {step, exp_avg, exp_avg_sq} for all 8 + 6G parameters under the
    indices of param_groups[0]['params'] -- the layout torch.optim.Adam(list(net.parameters())) writes -- with each
    parameter's own arena slice of the moments. load_checkpoint_into a fresh module, optimiser and scheduler restores both
    children's moments, step count and device learning rate; one more epoch on both runs is then bit for bit the same.
    A torch.optim.Adam state_dict over the same parameters lands in the right arena slices, and
    ImitationBranched.load_from_checkpoint restores the weights."""
    from carla_imitation_learning_b200.trainer import Trainer, load_checkpoint_into
    from src.architectures.branched import ConvNet1Branched
    dev = _dev()
    B, G = 8, 4
    Model, hp = _branched_model(G)
    dl = {"train_dataloader": _loader(31, 3, B, G, dev), "val_dataloader": _loader(32, 1, B, G, dev)}

    def build():
        torch.manual_seed(12345)
        return Model(dict(hp), ConvNet1Branched(dict(hp)).to(dev), dl)

    model = build()
    tr = Trainer(max_epochs=2, default_root_dir=str(tmp_path))
    tr.fit(model)
    opt, sch = tr._opt, tr._schedulers[0]
    assert opt.param_groups[0]["lr"] == pytest.approx(1e-5)
    path = str(tmp_path / "last.ckpt")
    tr.save_checkpoint(model, path)
    ck = torch.load(path, map_location="cpu", weights_only=False)
    params = list(model.net.parameters())
    assert len(params) == 8 + 6 * G and all(a is b for a, b in zip(opt.param_groups[0]["params"], params))
    osd = ck["optimizer_states"][0]
    assert osd["param_groups"][0]["params"] == list(range(len(params)))
    assert sorted(osd["state"]) == list(range(len(params)))
    owner = {id(p): c for c in opt.children_ for p in c._params}
    for i, p in enumerate(params):
        s = osd["state"][i]
        assert set(s) == {"step", "exp_avg", "exp_avg_sq"}, i
        _a, m, v, st, _g = owner[id(p)]._bound
        o, n = p._bc_offset, p.numel()
        assert float(s["step"]) == 6.0
        assert torch.equal(s["exp_avg"], m[o:o + n].view(p.shape).cpu()), i
        assert torch.equal(s["exp_avg_sq"], v[o:o + n].view(p.shape).cpu()), i
        assert float(s["exp_avg_sq"].abs().max()) > 0, i
    # a fresh module, optimiser and scheduler restored from the checkpoint
    model2 = build()
    opts2, schs2 = model2.configure_optimizers()
    opt2, sch2 = opts2[0], schs2[0]
    load_checkpoint_into(model2, path, opt2, schs2)
    assert opt2.param_groups[0]["lr"] == pytest.approx(1e-5) and sch2.last_epoch == sch.last_epoch
    opt.prepare()                                   # the original's device LR catches up with its last milestone
    for c1, c2 in zip(opt.children_, opt2.children_):
        a1, a2 = c1._bound, c2._bound
        assert torch.equal(a1[0], a2[0]) and torch.equal(a1[1], a2[1]) and torch.equal(a1[2], a2[2])
        assert torch.equal(a1[3][:6], a2[3][:6])    # lr beta1 beta2 eps step grad_scale
        assert float(a2[3][4]) == 6.0 and float(a2[3][0]) == pytest.approx(1e-5)
    for i, p in enumerate(model2.net.parameters()):
        assert torch.equal(opt2.state[p]["exp_avg"].cpu(), osd["state"][i]["exp_avg"]), i
    # one more epoch on both: bit for bit the same run
    _one_epoch(model, opt, sch, dl["train_dataloader"])
    _one_epoch(model2, opt2, sch2, dl["train_dataloader"])
    for c1, c2 in zip(opt.children_, opt2.children_):
        for a, b in zip(c1._bound[:3], c2._bound[:3]):
            assert torch.equal(a, b)
        assert float(c1._bound[3][4]) == float(c2._bound[3][4]) == 9.0
    # a torch.optim.Adam state_dict over the same parameter list
    net_a = ConvNet1Branched(dict(hp)).to(dev)
    gen = torch.Generator().manual_seed(3)
    for p in net_a.parameters():
        p.grad = torch.randn(p.shape, generator=gen).to(dev)
    adam = torch.optim.Adam(list(net_a.parameters()), lr=2e-4, foreach=False)
    adam.step()
    net_b = ConvNet1Branched(dict(hp)).to(dev)
    opt_b = net_b.configure_optimizer(lr=1e-3)
    opt_b.load_state_dict(adam.state_dict())
    assert opt_b.param_groups[0]["lr"] == 2e-4
    for pa, pb in zip(net_a.parameters(), net_b.parameters()):
        c = next(c for c in opt_b.children_ if any(q is pb for q in c._params))
        _a, m, v, st, _g = c._bound
        o, n = pb._bc_offset, pb.numel()
        assert torch.equal(m[o:o + n].view(pb.shape), adam.state[pa]["exp_avg"])
        assert torch.equal(v[o:o + n].view(pb.shape), adam.state[pa]["exp_avg_sq"])
        assert float(st[4]) == 1.0 and float(st[0]) == 2e-4
    # ImitationBranched.load_from_checkpoint(path, hparams=, net=, data_loader=)
    torch.manual_seed(1)
    m3 = Model.load_from_checkpoint(path, hparams=dict(hp), net=ConvNet1Branched(dict(hp)).to(dev), data_loader={})
    for k, v in m3.state_dict().items():
        assert torch.equal(v.cpu(), ck["state_dict"][k]), k


# ------------------------------------------------------------------------------- D. trajectory against the f64 spec
def test_branched_step_loss_curve_follows_the_f64_specification():
    """fp32 BranchedTrainStep with augmentation from 288x320, B = 8, G = 4, L1, 40 steps over 3 input slots, against the
    f64 specification run live on the CPU: X.stage_augmented (bit-exact host planes) -> sliding windows ->
    X.branched_loss_and_grads -> O.adam_update on both parameter sets. Steps 0..14, while the two runs are still the same
    trajectory, agree to rel 1e-4 of the loss; all 40 steps to rel 2e-2, which leaves room for the f32-vs-f64 difference
    that L1's sign(out - target) and the pooling argmax amplify once trajectories part. Measured on an NVIDIA B200 (1000 W
    limit): at most 7.5e-6 over steps 0..14 and 7.7e-3 over all 40. A captured step that skipped the branch Adam moved
    the loss by 2.7e-3 at step 4 (the first loss after a captured step) and by up to 0.1 within steps 0..14."""
    from carla_imitation_learning_b200.trainer import BranchedTrainStep
    B, G, n_out, steps = 8, 4, 3, 40
    net = _net(G, n_out, "l1", "fp32")
    P = {k: v.detach().cpu().double() for k, v in net.state_dict().items()}
    opt = net.configure_optimizer(lr=1e-3)
    stp = BranchedTrainStep(net, opt, B, src_hw=SRC_HW)
    slots = [_inputs(B, G, n_out, SRC_HW, 80 + s) for s in range(3)]
    ref_x = []
    for f, t, _c, _y in slots:
        planes = torch.from_numpy(X.stage_augmented(f.cpu().numpy(), t.cpu().numpy()))
        ref_x.append(torch.stack([planes[i:i + 4] for i in range(B)]))
    M = {k: torch.zeros_like(v) for k, v in P.items()}
    V = {k: torch.zeros_like(v) for k, v in P.items()}
    got, ref = [], []
    for i in range(steps):
        f, t, c, y = slots[i % 3]
        got.append(stp.step(f, t, c, y).clone())
        loss, _out, grads = X.branched_loss_and_grads(P, ref_x[i % 3], c.cpu(), y.cpu(), G, "l1")
        ref.append(float(loss))
        for k in P:
            O.adam_update(P[k], grads[k], M[k], V[k], i + 1)
    torch.cuda.synchronize()
    stp.check()
    got = torch.stack(got).double().cpu().numpy()
    ref = np.asarray(ref)
    dev_rel = np.abs(got - ref) / np.abs(ref)
    print("branched 40-step curve: max rel deviation steps 0..14 %.3e, all %.3e; per step %s"
          % (dev_rel[:15].max(), dev_rel.max(), np.array2string(dev_rel, precision=1)))
    assert dev_rel[:15].max() <= 1e-4, dev_rel
    assert dev_rel.max() <= 2e-2, dev_rel
    assert ref[-1] < ref[0] and got[-1] < got[0]


# ------------------------------------------------------------------------------- E. augmented staging edges
def _edge_table(n, src_hw, seed):
    """Rows cycling through the four crop corners and interior crops, brightness / contrast / saturation from {0, 2.5,
    ordinary} in every combination (so each clamp is reached from both sides), mean / std away from (0, 1)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    hs, ws = src_hw
    t = np.zeros((n, 8), np.float32)
    corners = [(0, 0), (0, ws - 256), (hs - 256, 0), (hs - 256, ws - 256)]
    for i in range(n):
        if i % 5 < 4:
            t[i, 0], t[i, 1] = corners[i % 5]
        else:
            t[i, 0], t[i, 1] = rng.integers(0, hs - 255), rng.integers(0, ws - 255)
        k = i // 5
        for j in range(3):
            choice = (k // 3 ** j) % 3
            t[i, 2 + j] = (0.0, 2.5, rng.uniform(0.6, 1.4))[choice]
        t[i, 5] = rng.uniform(-0.5, 0.7)
        t[i, 6] = 1.0 / rng.uniform(0.1, 2.0)
    return t


@pytest.mark.parametrize("src_hw", [(257, 259), (301, 263), (288, 320)])
def test_augmented_staging_edges_are_bit_exact(src_hw):
    """stage_augmented, plain f32 and Toeplitz-ready bf16, == X.stage_augmented (and its bf16 rounding) bit for bit at
    n = 300 frames (both kernels run their grid-stride loops: 19200 and 6652 CTAs of work against the 16-CTA-per-SM
    cap), crops at all four corners, odd source sizes whose rows are not 4-byte aligned, every jitter clamp from both
    sides and non-trivial mean / std."""
    from carla_imitation_learning_b200 import stage_augmented
    from tests.test_gpu_tc import _tp_reference
    dev = _dev()
    n = 300
    rng = np.random.Generator(np.random.PCG64(src_hw[0] * 1000 + src_hw[1]))
    frames = rng.integers(0, 256, size=(n, src_hw[0], src_hw[1], 3), dtype=np.uint8)
    table = _edge_table(n, src_hw, 5)
    ref = X.stage_augmented(frames, table)
    f32 = np.float32
    white = ((f32(0.299) * f32(255) + f32(0.587) * f32(255)) + f32(0.114) * f32(255)) * f32(1.0 / 255.0)
    for gray in (f32(0), white):                     # every channel clamped to 0, and to 255, somewhere in the batch
        assert (ref == (gray - table[:, 5, None, None]) * table[:, 6, None, None]).any()
    fr = torch.from_numpy(frames).to(dev)
    got = stage_augmented(fr, torch.from_numpy(table), layout="plain")
    assert np.array_equal(got.cpu().numpy().view(np.uint32), ref.view(np.uint32))
    tp = stage_augmented(fr, torch.from_numpy(table), layout="tp")
    want = _tp_reference(torch.from_numpy(ref).to(torch.bfloat16))
    assert torch.equal(tp.tp.cpu().view(torch.int16), want.view(torch.int16).reshape(n, -1))


@pytest.mark.parametrize("bad", ["crop_y_negative", "crop_y_past_end", "crop_x_past_end", "crop_fractional",
                                 "crop_nan", "brightness_inf", "mean_nan", "inv_std_inf"])
def test_host_augmentation_table_is_checked_before_any_launch(bad):
    """A host table with a crop outside [0, Hs-256] x [0, Ws-256], a fractional crop or a non-finite factor raises
    ValueError in stage_augmented before anything is copied or launched: the output buffer keeps its contents. The
    same table with the entry put back stages normally."""
    from carla_imitation_learning_b200 import stage_augmented
    from carla_imitation_learning_b200.data import augment_table
    dev = _dev()
    n, hs, ws = 3, 260, 270
    frames = torch.randint(0, 256, (n, hs, ws, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(2)).to(dev)
    good = torch.from_numpy(augment_table(4, n, (hs, ws)))
    row, col, val = {"crop_y_negative": (1, 0, -1.0), "crop_y_past_end": (2, 0, hs - 255.0), "crop_x_past_end": (0, 1, ws - 255.0),
                     "crop_fractional": (1, 1, 2.5), "crop_nan": (0, 0, float("nan")), "brightness_inf": (2, 2, float("inf")),
                     "mean_nan": (1, 5, float("nan")), "inv_std_inf": (0, 6, float("inf"))}[bad]
    table = good.clone()
    table[row, col] = val
    out = torch.full((n, 256, 256), 7.0, device=dev)
    torch.cuda.synchronize()
    with pytest.raises(ValueError, match="augmentation table"):
        stage_augmented(frames, table, out=out)
    torch.cuda.synchronize()
    assert bool((out == 7.0).all())
    stage_augmented(frames, good, out=out)
    torch.cuda.synchronize()
    assert np.array_equal(out.cpu().numpy(), X.stage_augmented(frames.cpu().numpy(), good.numpy()))
