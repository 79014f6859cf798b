"""Generate tests/golden/*.npz from the UNMODIFIED reference (run in the build container only).

    python oracle/make_golden.py

Imports /root/reference/src/architectures/nets.py::ConvNet1 and
/root/reference/src/models/imitation.py::Imitation through the import stubs in
oracle/_stubs (pytorch_lightning, matplotlib are not installed here), seeds as
train.py:103 does, and records what the reference produces for seeded synthetic
inputs. The GPU box has no /root/reference, so these files are how the reference's
behaviour travels. TEST INFRASTRUCTURE ONLY.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = os.environ.get("BC_REFERENCE", "/root/reference")
sys.path[:0] = [os.path.join(HERE, "_stubs"), REF, ROOT]

from src.architectures.nets import ConvNet1 as RefNet  # noqa: E402  (reference)
from src.models.imitation import Imitation as RefImitation  # noqa: E402  (reference)
from src.dataset.imitation_dataset import continous_to_discreet  # noqa: E402 (reference; needs pandas only)

from oracle import bc_oracle as O  # noqa: E402

HP = dict(obs_size=4, n_actions=9)
SEED = 12345  # configs/seeds/default_seeds.yaml:3


def build_ref():
    torch.manual_seed(SEED)
    net = RefNet(HP)
    return net, RefImitation(HP, net, {})


def flat(named):
    return np.concatenate([named[k].detach().reshape(-1).numpy() for k in O.PARAM_ORDER])


def golden_step(B, data_seed, path):
    frames, labels = O.synth_frames(data_seed, B + 4)
    x_np, y_np = O.sequential_samples(frames, labels)
    x, y = torch.from_numpy(x_np), torch.from_numpy(y_np)
    net, model = build_ref()
    init = flat(dict(net.named_parameters()))
    example = net.example_input_array.numpy().copy()
    example_logits = net(net.example_input_array).detach().numpy()
    opt, _ = model.configure_optimizers()
    opt = opt[0]
    loss = model.training_step((x, y), 0)
    logits = model(x).detach().numpy()
    opt.zero_grad()
    loss.backward()
    grads = flat({k: p.grad for k, p in net.named_parameters()})
    opt.step()
    after1 = flat(dict(net.named_parameters()))
    # two more steps so bias-correction with t>1 is pinned as well
    for i in range(2):
        l2 = model.training_step((x, y), i + 1)
        opt.zero_grad(); l2.backward(); opt.step()
    after3 = flat(dict(net.named_parameters()))
    val = model.validation_step((x, y), 0)
    # the parameters after the Adam steps go to a second file so that each stays under 1 MB
    np.savez_compressed(
        path, B=B, data_seed=data_seed, init=init, loss=float(loss.detach()), logits=logits, grads=grads,
        val_loss_after3=float(val),
        example_checksum=float(np.abs(example).sum()), example_logits=example_logits,
        logged_val=float(model.logged["val_loss"]))
    np.savez_compressed(path.replace(".npz", "_adam.npz"), after1=after1, after3=after3)
    print(path, "loss", float(loss), "val", float(val))


def golden_curve(B, steps, data_seed, path):
    """Loss curve of the reference over `steps` optimiser steps on a synthetic frame stream."""
    net, model = build_ref()
    opt = model.configure_optimizers()[0][0]
    frames, labels = O.synth_frames(data_seed, steps * B + 4)
    gray = torch.from_numpy(O.gray_stack(frames))
    lab = torch.from_numpy(labels)
    losses = []
    for s in range(steps):
        x = torch.stack([gray[s * B + i: s * B + i + 4] for i in range(B)])
        y = lab[s * B + 4: s * B + 4 + B]
        loss = model.training_step((x, y), s)
        opt.zero_grad(); loss.backward(); opt.step()
        losses.append(float(loss))
    np.savez_compressed(path, B=B, steps=steps, data_seed=data_seed, losses=np.asarray(losses, np.float64))
    print(path, losses[0], losses[steps // 2], losses[-1])


def golden_curve_ensemble(B, steps, data_seed, path, members=8):
    """The reference's OWN reproducibility envelope: the same 1k-step run of the unmodified reference,
    re-run `members` times with every initial weight moved by about one f32 ulp (w *= 1 + 6e-8 * N(0,1))
    and with different intra-op thread counts (different f32 summation orders). Any independent
    implementation differs from the reference by at least this much rounding, so the spread of these curves
    is what 'the loss curves agree' can mean; the tests bound the device curve by it."""
    frames, labels = O.synth_frames(data_seed, steps * B + 4)
    gray = torch.from_numpy(O.gray_stack(frames))
    lab = torch.from_numpy(labels)
    curves, meta = [], []
    for m in range(members):
        threads = (1, 2, 4, 8)[m % 4]
        torch.set_num_threads(threads)
        net, model = build_ref()
        gen = torch.Generator().manual_seed(1000 + m)
        with torch.no_grad():
            for p_ in net.parameters():
                p_.mul_(1.0 + 6e-8 * torch.randn(p_.shape, generator=gen))
        opt = model.configure_optimizers()[0][0]
        losses = []
        for s in range(steps):
            x = torch.stack([gray[s * B + i: s * B + i + 4] for i in range(B)])
            y = lab[s * B + 4: s * B + 4 + B]
            loss = model.training_step((x, y), s)
            opt.zero_grad(); loss.backward(); opt.step()
            losses.append(float(loss))
        curves.append(losses); meta.append(threads)
        print("member", m, "threads", threads, "mean", np.mean(losses), flush=True)
    torch.set_num_threads(os.cpu_count())
    np.savez_compressed(path, B=B, steps=steps, data_seed=data_seed, threads=np.asarray(meta),
                        losses=np.asarray(curves, np.float64))


def golden_resume_state(B, at_step, data_seed, path):
    """Parameters and Adam state of the canonical reference run (golden_curve) after `at_step` steps, i.e. past the
    ln 9 plateau. The plateau exit is a saddle escape whose timing amplifies bf16-sized (4e-3) gradient rounding into
    +-100 steps or no exit at all (measured on the unmodified reference with that noise injected, DESIGN.md 2), so
    the bf16 mode's 1k-step curve is compared from this common state, where the dynamics are contractive again."""
    net, model = build_ref()
    opt = model.configure_optimizers()[0][0]
    frames, labels = O.synth_frames(data_seed, 1000 * B + 4)
    gray = torch.from_numpy(O.gray_stack(frames[:at_step * B + 4]))
    lab = torch.from_numpy(labels)
    for s in range(at_step):
        x = torch.stack([gray[s * B + i: s * B + i + 4] for i in range(B)])
        loss = model.training_step((x, lab[s * B + 4: s * B + 4 + B]), s)
        opt.zero_grad(); loss.backward(); opt.step()
    named = dict(net.named_parameters())
    st = opt.state
    # the Adam moments go to a second file so that each stays under 1 MB
    np.savez_compressed(path, B=B, at_step=at_step, data_seed=data_seed, params=flat(named), last_loss=float(loss.detach()))
    np.savez_compressed(
        path.replace(".npz", "_adam.npz"),
        exp_avg=np.concatenate([st[named[k]]["exp_avg"].reshape(-1).numpy() for k in O.PARAM_ORDER]),
        exp_avg_sq=np.concatenate([st[named[k]]["exp_avg_sq"].reshape(-1).numpy() for k in O.PARAM_ORDER]))
    print(path, "loss at resume", float(loss.detach()))


def golden_labels(path):
    # pandas 3 (this image) returns read-only `.values` under copy-on-write, which the
    # reference's in-place writes (imitation_dataset.py:322-324) predate; feed it a
    # column holder with the 2021-era semantics (writable arrays) instead of a DataFrame.
    class _Col:
        def __init__(self, a):
            self.values = a

    rng = np.random.Generator(np.random.PCG64(7))
    n = 512
    steer = rng.choice([0.0, 2.0, 0.05, -0.05, 0.051, -0.051, 0.3, -0.7, 0.01, -0.02], size=n)
    throttle = rng.choice([0.0, 0.5, 1.0, 0.75], size=n)
    brake = rng.choice([0.0, 1.0, 0.5], size=n)
    df = dict(steer=_Col(steer.copy()), throttle=_Col(throttle.copy()), brake=_Col(brake.copy()))
    out = continous_to_discreet(df)
    np.savez_compressed(path, steer=steer, throttle=throttle, brake=brake, action=np.asarray(out, np.float64))
    print(path, np.unique(out))


def golden_gray(path):
    frames, _ = O.synth_frames(3, 5, 64, 48)
    ref = np.dot(frames[..., :], [0.299, 0.587, 0.114]) / 255.0   # imitation_dataset.py:121, verbatim formula
    np.savez_compressed(path, gray_f64=ref, gray_f32=ref.astype(np.float32))


def oracle_curve_f64(B, steps, data_seed, path):
    """The same 1k-step run with the ORACLE in f64 (~5 min): measures how far rounding alone moves the
    curve, which bounds what 'loss curves agree' can mean for any independent implementation."""
    frames, labels = O.synth_frames(data_seed, steps * B + 4)
    gray = torch.from_numpy(O.gray_stack(frames)); lab = torch.from_numpy(labels)
    tr = O.OracleTrainer(O.init_params(SEED), dtype=torch.float64)
    out = [tr.step(torch.stack([gray[s * B + i: s * B + i + 4] for i in range(B)]), lab[s * B + 4: s * B + 4 + B])
           for s in range(steps)]
    np.save(path, np.asarray(out, np.float64))


def golden_aux(B, data_seed, path):
    """ImitationAux + lossCriterion of the UNMODIFIED reference (imitation.py:11-24, 94-159) on a net whose third output is the
    reference ConvNet1's logits (CNNAuxNet is not shipped): two-column labels [traffic light, action], loss = CE(out[2], y[:, 1]).
    Also records that the reference's ConvNetRawSegment cannot be constructed (nets.py:44)."""
    from src.models.imitation import ImitationAux as RefAux  # noqa: E402 (reference)
    from src.architectures.nets import ConvNetRawSegment as RefRaw  # noqa: E402 (reference)

    class AuxNet(torch.nn.Module):
        def __init__(self, base):
            super().__init__()
            self.base = base

        def forward(self, x):
            return None, None, self.base(x)

    frames, labels = O.synth_frames(data_seed, B + 4)
    x_np, y_np = O.sequential_samples(frames, labels)
    rng = np.random.Generator(np.random.PCG64(data_seed + 99))
    y2 = np.stack([rng.integers(0, 3, size=B), y_np], axis=1).astype(np.int64)       # column 0: traffic-light status (unused by the loss)
    x, y = torch.from_numpy(x_np), torch.from_numpy(y2)
    net, _ = build_ref()
    model = RefAux(HP, AuxNet(net), {})
    loss = model.training_step((x, y), 0)
    loss.backward()
    grads = flat({k: p.grad for k, p in net.named_parameters()})
    val = model.validation_step((x, y), 0)
    try:
        RefRaw(HP)
        raw_error = ""
    except Exception as e:  # noqa: BLE001
        raw_error = type(e).__name__
    np.savez_compressed(path, B=B, data_seed=data_seed, y2=y2, loss=float(loss.detach()), val_loss=float(val), grads=grads,
                        logged_val_loss=("val_loss" in model.logged), raw_segment_error=raw_error)
    print(path, "aux loss", float(loss), "ConvNetRawSegment(hp) raises", raw_error)


if __name__ == "__main__":
    g = os.path.join(ROOT, "tests", "golden")
    os.makedirs(g, exist_ok=True)
    torch.set_num_threads(os.cpu_count())
    if "--aux-only" in sys.argv:
        golden_aux(4, 0, os.path.join(g, "ref_aux_step_b4.npz"))
        sys.exit(0)
    golden_step(4, 0, os.path.join(g, "ref_step_b4.npz"))
    golden_aux(4, 0, os.path.join(g, "ref_aux_step_b4.npz"))
    golden_step(1, 1, os.path.join(g, "ref_step_b1.npz"))
    golden_labels(os.path.join(g, "ref_labels.npz"))
    golden_gray(os.path.join(g, "ref_gray.npz"))
    golden_curve(8, 1000, 11, os.path.join(g, "ref_curve_b8_1k.npz"))
    if "--resume-state" in sys.argv:
        golden_resume_state(8, 200, 11, os.path.join(g, "ref_state_b8_step200.npz"))
    if "--ensemble" in sys.argv:
        golden_curve_ensemble(8, 1000, 11, os.path.join(g, "ref_curve_b8_1k_ensemble.npz"))
    if "--f64-curve" in sys.argv:
        oracle_curve_f64(8, 1000, 11, os.path.join(g, "oracle_curve_b8_1k_f64.npy"))
