"""The oracle restatement vs. the golden vectors the unmodified reference produced
(oracle/make_golden.py). CPU only."""
import os

import numpy as np
import pytest
import torch

from oracle import bc_oracle as O


def _flat(named):
    return np.concatenate([named[k].detach().reshape(-1).double().numpy() for k in O.PARAM_ORDER])


def _unflat(vec):
    out, off = {}, 0
    for k, shp in O.param_shapes().items():
        n = int(np.prod(shp))
        out[k] = torch.from_numpy(np.asarray(vec[off:off + n], dtype=np.float32).reshape(shp).copy())
        off += n
    assert off == vec.size == 133305
    return out


def _batch(g):
    frames, labels = O.synth_frames(int(g["data_seed"]), int(g["B"]) + 4)
    x, y = O.sequential_samples(frames, labels)
    return torch.from_numpy(x), torch.from_numpy(y)


@pytest.mark.parametrize("name", ["ref_step_b4.npz", "ref_step_b1.npz"])
def test_init_matches_reference_bitwise(golden_dir, name):
    g = np.load(os.path.join(golden_dir, name))
    p = O.init_params(12345)
    assert np.array_equal(_flat(p).astype(np.float32), g["init"])
    ex_logits = O.forward(p, _example()).numpy()
    np.testing.assert_allclose(ex_logits, g["example_logits"], rtol=1e-5, atol=1e-6)


def _example():
    torch.manual_seed(12345)
    return torch.randn((1, 4, 256, 256))


@pytest.mark.parametrize("name", ["ref_step_b4.npz", "ref_step_b1.npz"])
def test_forward_loss_grads(golden_dir, name):
    g = np.load(os.path.join(golden_dir, name))
    x, y = _batch(g)
    p = _unflat(g["init"])
    loss, logits, grads = O.loss_and_grads(p, x, y)
    np.testing.assert_allclose(logits.numpy(), g["logits"], rtol=1e-5, atol=1e-6)
    assert abs(float(loss) - float(g["loss"])) <= 1e-6 * abs(float(g["loss"]))
    ref = g["grads"].astype(np.float64)
    got = _flat(grads)
    assert np.abs(got - ref).max() <= 1e-5 * np.abs(ref).max()


@pytest.mark.parametrize("name", ["ref_step_b4.npz", "ref_step_b1.npz"])
def test_explicit_backward_is_the_same_function(golden_dir, name):
    g = np.load(os.path.join(golden_dir, name))
    x, y = _batch(g)
    p = _unflat(g["init"])
    # f32 explicit formulas reproduce the reference's f32 pool routing; the f64 run is then
    # given that routing (see explicit_backward docstring: routing flips are discontinuous)
    _, _, g32, aux = O.explicit_backward(p, x, y, dtype=torch.float32)
    loss, logits, grads, _ = O.explicit_backward(p, x, y, dtype=torch.float64, argmax_override=aux["argmax"])
    ref = g["grads"].astype(np.float64)
    assert np.abs(_flat(g32) - ref).max() <= 1e-5 * np.abs(ref).max()
    got = _flat(grads)
    off = 0
    for k, shp in O.param_shapes().items():
        n = int(np.prod(shp))
        r, t = ref[off:off + n], got[off:off + n]
        assert np.abs(r - t).max() <= 2e-5 * max(np.abs(r).max(), 1e-12), k
        off += n
    assert abs(float(loss) - float(g["loss"])) < 1e-6


@pytest.mark.parametrize("name", ["ref_step_b4.npz", "ref_step_b1.npz"])
def test_adam_three_steps(golden_dir, name):
    g = np.load(os.path.join(golden_dir, name))
    adam = np.load(os.path.join(golden_dir, name.replace(".npz", "_adam.npz")))
    x, y = _batch(g)
    tr = O.OracleTrainer(_unflat(g["init"]))
    tr.step(x, y)
    a1 = _flat(tr.p)
    # Adam's first step moves every weight by ~lr*sign(g): compare the UPDATE, not just the value
    d_ref = adam["after1"].astype(np.float64) - g["init"].astype(np.float64)
    d_got = a1 - g["init"].astype(np.float64)
    assert np.abs(d_got - d_ref).max() <= 2e-6  # |update| = 1e-3; f32 ulp of the params ~6e-8
    tr.step(x, y)
    tr.step(x, y)
    assert np.abs(_flat(tr.p) - adam["after3"].astype(np.float64)).max() <= 2e-5
    val = float(O.cross_entropy(O.forward(tr.p, x), y))
    assert abs(val - float(g["val_loss_after3"])) <= 1e-4 * abs(float(g["val_loss_after3"]))
    assert float(g["logged_val"]) == float(g["val_loss_after3"])


def test_gray_formula(golden_dir):
    g = np.load(os.path.join(golden_dir, "ref_gray.npz"))
    frames, _ = O.synth_frames(3, 5, 64, 48)
    assert np.array_equal(O.gray_stack(frames), g["gray_f32"])


def test_label_discretisation(golden_dir):
    g = np.load(os.path.join(golden_dir, "ref_labels.npz"))
    got = O.discretise_actions(g["steer"], g["throttle"], g["brake"])
    assert np.array_equal(got, g["action"])


def test_sequential_window_contract():
    frames, labels = O.synth_frames(5, 9, 32, 32)
    x, y = O.sequential_samples(frames, labels)
    assert x.shape == (5, 4, 32, 32) and x.dtype == np.float32 and y.dtype == np.int64
    g = O.gray_stack(frames)
    for i in range(5):
        assert np.array_equal(x[i], g[i:i + 4]) and y[i] == labels[i + 4]


def test_lr_schedule():
    assert O.lr_at_epoch(0) == 1e-3 and O.lr_at_epoch(19) == 1e-3
    assert abs(O.lr_at_epoch(20) - 1e-4) < 1e-12 and abs(O.lr_at_epoch(30) - 1e-5) < 1e-12


def test_loss_curve_first_steps(golden_dir):
    """First 40 steps of the reference's 1k-step curve (the full curve is checked on the GPU)."""
    g = np.load(os.path.join(golden_dir, "ref_curve_b8_1k.npz"))
    B, n = int(g["B"]), 40
    frames, labels = O.synth_frames(int(g["data_seed"]), int(g["steps"]) * B + 4)
    frames, labels = frames[:n * B + 4], labels[:n * B + 4]
    gray = torch.from_numpy(O.gray_stack(frames))
    lab = torch.from_numpy(labels)
    tr = O.OracleTrainer(O.init_params(12345))
    for s in range(n):
        xb = torch.stack([gray[s * B + i:s * B + i + 4] for i in range(B)])
        loss = tr.step(xb, lab[s * B + 4:s * B + 4 + B])
        assert abs(loss - g["losses"][s]) <= 2e-3 * g["losses"][s], s


def test_oracle_f64_curve_sits_inside_the_reference_reproducibility_envelope(golden_dir):
    """The f64 oracle run and every ensemble member pass the same curve check the device curves get
    (tests/curve_check.py); a curve stuck on the ln 9 plateau does not."""
    import pytest
    from tests.curve_check import check_curve
    f64 = np.load(os.path.join(golden_dir, "oracle_curve_b8_1k_f64.npy"))
    check_curve(f64, golden_dir, tol=1e-2)
    ens = np.load(os.path.join(golden_dir, "ref_curve_b8_1k_ensemble.npz"))["losses"]
    assert ens.shape == (8, 1000)
    for c in ens:
        check_curve(c, golden_dir, tol=1e-2)
    with pytest.raises(AssertionError):
        check_curve(np.full(1000, 2.1972), golden_dir, tol=2e-2)


def test_oracle_aux_criterion_matches_the_reference_imitation_aux(golden_dir):
    """ImitationAux + lossCriterion of the unmodified reference (golden ref_aux_step_b4.npz, oracle/make_golden.py::golden_aux)."""
    g = np.load(os.path.join(golden_dir, "ref_aux_step_b4.npz"))
    frames, labels = O.synth_frames(int(g["data_seed"]), int(g["B"]) + 4)
    x, _y = O.sequential_samples(frames, labels)
    P = O.init_params(12345)
    loss, _logits, grads = O.aux_criterion(P, torch.from_numpy(x), torch.from_numpy(g["y2"]))
    assert abs(float(loss) - float(g["loss"])) <= 1e-6
    got = np.concatenate([grads[k].detach().reshape(-1).numpy() for k in O.PARAM_ORDER])
    assert np.abs(got - g["grads"]).max() <= 1e-6 * np.abs(g["grads"]).max()
    assert not bool(g["logged_val_loss"])                   # the reference's ImitationAux.validation_step does not log
    assert str(g["raw_segment_error"]) == "TypeError"       # ConvNetRawSegment(hparams) cannot be constructed (nets.py:44)
