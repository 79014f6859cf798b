"""What feeds the training step and what Trainer.fit runs on it, against the reference dataset and exact references.

data.SequentialFrames is the device-side SequentialTorchDataset + DataLoader: it rotates two device slots, uploads batch
k + 1 on a copy stream while the consumer runs batch k, and hands out views of the slots. A consumer slower than the next
upload is modelled by a bounded device delay (torch.cuda._sleep, ~10 ms against the ~0.1 ms a 12-frame chunk takes to
upload) enqueued on the consumer's stream before the batch is read. Each batch is read when it is handed out and again
after the next one has been, which the loader allows: by then an upload that overwrites the slot early has been enqueued,
so the check does not depend on the host's timing. Every comparison with the reference batches is bitwise.

The forward-only loss (net.loss under no_grad, the validation_step path: head CE mode 1, then bc_loss_reduce) is bounded
against the f64 mean cross-entropy of the device's own logits, with per-sample power: every sample's contribution
exceeds the bound, so a lost head CTA or loss partial fails. Batch sizes are where the head kernel splits the work
differently: one sample per CTA up to B = 128, two from B = 129, 32 at B = 4096.
"""
import itertools
import os

import numpy as np
import pytest
import torch

from oracle import bc_oracle as O
from tests.test_gpu_batch_edges import _bound, _check_head_fwd, _cpu64, _planes_from_tp, _uniform_frames

pytestmark = pytest.mark.gpu

DELAY_CYCLES = 20_000_000       # ~10 ms at the B200's ~2 GHz SM clock


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (no CPU fallback exists to run instead)")
    torch.set_num_threads(os.cpu_count() or 1)
    return torch.device("cuda", 0)


def _slow_consumer():
    torch.cuda._sleep(DELAY_CYCLES)


def _net(hp, seed=12345):
    from src.architectures.nets import ConvNet1
    torch.manual_seed(seed)
    return ConvNet1(dict(hp)).to(torch.device("cuda", 0))


# ------------------------------------------------------------------------------- loader batches vs the reference dataset
def _loader(frames, labels, bs, fs, kind, dev):
    from carla_imitation_learning_b200.data import SequentialFrames
    if kind == "tp":
        return SequentialFrames(frames, labels, bs, fs, device=dev, layout="tp")
    return SequentialFrames(frames, labels, bs, fs, device=dev, dtype=torch.bfloat16 if kind == "bf16" else torch.float32)


def _snapshots(batches, n):
    """n batches of one iterator, each read by a slow consumer (the delay, then a copy of x and y on the consumer's
    stream) when it is handed out, and again after the next batch has been (a batch stays valid until two more have
    been asked for). The second read comes after the upload of batch k + 2 was enqueued, so a slot overwritten early is
    seen whatever the host's timing. Returns the first reads and the second reads of batches 0 .. n-2."""
    from carla_imitation_learning_b200 import StagedBatch
    snap = lambda x, y: (x.tp.clone() if isinstance(x, StagedBatch) else x.clone(), y.clone())
    now, later, prev = [], [], None
    for x, y in itertools.islice(batches, n):
        _slow_consumer()
        if prev is not None:
            later.append(snap(*prev))
        now.append(snap(x, y))
        prev = (x, y)
    torch.cuda.synchronize()
    assert len(now) == n
    return now, later


def _check_batches(tag, reads, frames, labels, bs, fs, kind):
    """reads = _snapshots(...) of one iterator: snapshot i must be sequence batch i % len(loader) of
    O.sequential_samples; bf16 planes = bf16_rn(reference f32), Toeplitz-ready planes decoded first."""
    xr, yr = O.sequential_samples(frames, labels, fs)
    nb = (len(yr) + bs - 1) // bs
    now, later = reads
    for i, (xs, ys), when in [(i, s, "read") for i, s in enumerate(now)] + [(i, s, "read after the next batch")
                                                                           for i, s in enumerate(later)]:
        k = i % nb
        lo, hi = k * bs, min(k * bs + bs, len(yr))
        b = hi - lo
        ref = torch.from_numpy(xr[lo:hi])
        if kind == "tp":
            planes = _planes_from_tp(xs)
            assert planes.shape[0] == b + fs, (tag, i)
            xs = planes.as_strided((b, fs, 256, 256), (65536, 65536, 256, 1))
        if kind != "f32":
            ref = ref.to(torch.bfloat16)
        got_y = ys.cpu()
        if not torch.equal(got_y, torch.from_numpy(yr[lo:hi])):
            # labels = 1000 + frame index: a wrong label names the sample it belongs to
            samples = (got_y - 1000 - fs).tolist()
            raise AssertionError(f"{tag}: batch {i} (sequence batch {k}, samples {lo}..{hi - 1}), {when}, holds the labels "
                                 f"of samples {samples}, i.e. of sequence batches {sorted({s // bs for s in samples})}")
        assert xs.dtype == ref.dtype and tuple(xs.shape) == tuple(ref.shape), (tag, i, xs.dtype, tuple(xs.shape))
        assert torch.equal(xs.cpu(), ref), f"{tag}: batch {i} (sequence batch {k}), {when}: planes differ from the reference"


LAYOUTS = [("f32", 4), ("f32", 12), ("bf16", 4), ("bf16", 12), ("tp", 4)]
SHAPES = {"8-8-3": (19, 8), "3-full": (24, 8), "one-short": (5, 8), "bs1": (7, 1)}     # (samples, batch_size)


@pytest.mark.parametrize("iteration", ["epochs", "cycle"])
@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("kind,fs", LAYOUTS)
def test_loader_batches_equal_the_reference_dataset_under_a_slow_consumer(dev, kind, fs, shape, iteration):
    """Every batch a slow consumer reads is the reference dataset's batch: `epochs` = __iter__ twice, `cycle` = cycle()
    over 2.5 passes of an odd batch count, so the slot parity flips at the wrap. Labels are unique per frame, so batch k
    and batch k + 2 always differ."""
    n, bs = SHAPES[shape]
    frames, _ = O.synth_frames(40 + fs + bs, n + fs)
    labels = 1000 + np.arange(n + fs, dtype=np.int64)
    loader = _loader(frames, labels, bs, fs, kind, dev)
    nb = len(loader)
    assert nb == (n + bs - 1) // bs
    tag = f"{kind} fs={fs} {shape} {iteration}"
    if iteration == "epochs":
        for epoch in range(2):
            _check_batches(f"{tag} {epoch}", _snapshots(iter(loader), nb), frames, labels, bs, fs, kind)
    else:
        assert nb % 2 == 1
        _check_batches(tag, _snapshots(loader.cycle(), (5 * nb + 1) // 2), frames, labels, bs, fs, kind)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_train_val_test_iterator_hands_out_the_reference_batches(dev, precision):
    """sequential_train_val_test_iterator builds f32 gray-plane loaders for fp32 and Toeplitz-ready ones for bf16; a pass
    over each split is the reference dataset of the synthetic sequence it was built from."""
    from carla_imitation_learning_b200.data import sequential_train_val_test_iterator, synthetic_sequence
    bs, fs = 8, 4
    dls = sequential_train_val_test_iterator({"BATCH_SIZE": bs, "frame_skip": fs, "n_actions": 9, "precision": precision})
    kind = "tp" if precision == "bf16" else "f32"
    for i, split in enumerate(("train", "val", "test")):
        dl = dls[f"{split}_dataloader"]
        assert dl.layout == ("tp" if precision == "bf16" else "plain") and dl.dtype == torch.float32
        frames, labels = synthetic_sequence(i, (8 if split == "train" else 2) * bs + fs, n_actions=9)
        assert len(dl) == (8 if split == "train" else 2)
        _check_batches(f"{precision} {split}", _snapshots(iter(dl), len(dl)), frames, labels, bs, fs, kind)


# ------------------------------------------------------------------------------- Trainer.fit through the loader
def _slow_model_class():
    from src.models.imitation import Imitation

    class SlowImitation(Imitation):
        """Imitation whose steps start behind a device delay; it records every loss it returns."""

        def __init__(self, *a, **k):
            super().__init__(*a, **k)
            self.train_losses, self.val_losses = [], []

        def training_step(self, batch, batch_idx):
            _slow_consumer()
            loss = super().training_step(batch, batch_idx)
            self.train_losses.append(loss.detach().clone())
            return loss

        def validation_step(self, batch, batch_idx):
            _slow_consumer()
            loss = super().validation_step(batch, batch_idx)
            self.val_losses.append(loss.clone())
            return loss

    return SlowImitation


def _reference_batches(frames, labels, bs, mode, dev):
    """The loader's batches built straight from the frames: fresh device tensors per batch."""
    from carla_imitation_learning_b200 import sliding_window, stage_frames, stage_gray
    n = len(frames) - 4
    out = []
    for lo in range(0, n, bs):
        b = min(bs, n - lo)
        fr = torch.from_numpy(frames[lo:lo + b + 4]).to(dev)
        x = stage_frames(fr) if mode == "bf16" else sliding_window(stage_gray(fr))
        out.append((x, torch.from_numpy(labels[lo + 4:lo + 4 + b].copy()).to(dev)))
    return out


def _adam_state(opt):
    _arena, m, v, st, _ = opt._bind()
    return m, v, float(st[4])


@pytest.mark.parametrize("graph", [False, True])
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_fit_through_the_loader_equals_the_steps_on_reference_batches(dev, mode, graph):
    """Trainer.fit for 2 epochs over train (4 batches) and val (3) SequentialFrames, short last batches, every step behind
    the delay, == the same steps on batches built straight from the frames (train_forward_backward + FusedAdam.step_flat,
    net.loss under no_grad): every training and validation loss, the final parameters and both Adam moments, bitwise;
    callback_metrics['val_loss'] is the mean of the last epoch's reference validation losses."""
    from carla_imitation_learning_b200 import FusedAdam
    from carla_imitation_learning_b200.data import SequentialFrames
    from carla_imitation_learning_b200.trainer import Trainer
    B, epochs = 8, 2
    ftr, ltr = O.synth_frames(61, 27 + 4)                           # 8, 8, 8, 3: an even count repeats graph keys
    fva, lva = O.synth_frames(62, 21 + 4)                           # 8, 8, 5
    hp = {"obs_size": 4, "n_actions": 9, "precision": mode}
    layout = "tp" if mode == "bf16" else "plain"
    dl = {"train_dataloader": SequentialFrames(ftr, ltr, B, device=dev, layout=layout),
          "val_dataloader": SequentialFrames(fva, lva, B, device=dev, layout=layout)}
    model = _slow_model_class()(dict(hp), _net(dict(hp, cuda_graph=graph)), dl)
    tr = Trainer(max_epochs=epochs)
    tr.fit(model)
    torch.cuda.synchronize()
    if graph:
        assert model.net._step_graphs.graphs                        # the second epoch replayed captured steps

    net = _net(hp)
    opt = FusedAdam(list(net.parameters()), lr=1e-3)
    eng = net.engine()
    train_ref, val_ref = _reference_batches(ftr, ltr, B, mode, dev), _reference_batches(fva, lva, B, mode, dev)
    losses, vals = [], []
    for _ in range(epochs):
        for x, y in train_ref:
            losses.append(eng.train_forward_backward(x, y).loss.clone())
            opt.step_flat(eng.grads)
        with torch.no_grad():
            vals.append([net.loss(x, y) for x, y in val_ref])
    torch.cuda.synchronize()
    eng.check_device_errors()

    got, ref = torch.stack(model.train_losses).cpu(), torch.stack(losses).cpu()
    assert torch.equal(got, ref), (got, ref)
    got_v, ref_v = torch.stack(model.val_losses).cpu(), torch.stack([v for e in vals for v in e]).cpu()
    assert torch.equal(got_v, ref_v), (got_v, ref_v)
    assert torch.equal(tr.callback_metrics["val_loss"].cpu(), torch.stack(vals[-1]).mean().cpu())
    assert torch.equal(model.net._arena, net._arena)
    m_got, v_got, t_got = _adam_state(tr._opt)
    m_ref, v_ref, t_ref = _adam_state(opt)
    assert torch.equal(m_got, m_ref) and torch.equal(v_got, v_ref) and t_got == t_ref == epochs * len(train_ref)


@pytest.mark.parametrize("graph", [False, True])
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_micro_batches_accumulated_across_one_next_equal_reference_batches(dev, mode, graph):
    """A batch stays valid until the consumer has asked for two more: loss_a on batch 0, next(), loss_b on batch 1,
    (loss_a + loss_b).backward(), one optimiser step -- through the loader == the same on reference batches, bitwise
    (both losses, every accumulated gradient, the parameters after the step). The classic path reads batch 0's planes
    again in its backward, after the next()."""
    from carla_imitation_learning_b200.data import SequentialFrames
    B = 8
    frames, labels = O.synth_frames(63, 3 * B + 4)
    hp = {"obs_size": 4, "n_actions": 9, "precision": mode, "cuda_graph": graph}
    Slow = _slow_model_class()
    res = []
    for source in ("loader", "reference"):
        model = Slow(dict(hp), _net(hp), {})
        opt = model.configure_optimizers()[0][0]
        if source == "loader":
            batches = iter(SequentialFrames(frames, labels, B, device=dev, layout="tp" if mode == "bf16" else "plain"))
        else:
            batches = iter(_reference_batches(frames, labels, B, mode, dev))
        loss_a = model.training_step(next(batches), 0)
        loss_b = model.training_step(next(batches), 1)
        (loss_a + loss_b).backward()
        grads = torch.cat([p.grad.detach().reshape(-1) for p in model.net.parameters()]).clone()
        opt.step()
        torch.cuda.synchronize()
        model.net.engine().check_device_errors()
        res.append((torch.stack([loss_a.detach(), loss_b.detach()]).cpu(), grads.cpu(), model.net._arena.detach().cpu()))
    (la, ga, pa), (lr_, gr, pr) = res
    assert torch.equal(la, lr_), (la, lr_)
    assert torch.equal(ga, gr)
    assert torch.equal(pa, pr)


# ------------------------------------------------------------------------------- the forward-only loss
def _check_loss(tag, loss, logits, y, B, NA):
    """Mean CE against its f64 value on the device's own logits; every sample's term must exceed the bound."""
    z, y = _cpu64(logits), y.cpu()
    m = z.max(1).values
    lsum = torch.log(torch.exp(z - m[:, None]).sum(1))
    zy = z.gather(1, y[:, None]).squeeze(1)
    per = (lsum + m - zy) / B
    S = ((lsum.abs() + m.abs() + zy.abs()) / B).sum()
    _bound(f"{tag} loss", loss.reshape(1), per.sum().reshape(1), S.reshape(1), per_sample=per.reshape(B, 1), power=NA > 1)


def _oracle_loss(P, frames, y, B, chunk=256):
    """The f64 oracle forward on the f32 master weights and the reference gray planes, in sample chunks."""
    logits = []
    for lo in range(0, B, chunk):
        b = min(chunk, B - lo)
        g = torch.from_numpy(O.gray_stack(frames[lo:lo + b + 4])).double()
        logits.append(O.forward(P, g.as_strided((b, 4, 256, 256), (65536, 65536, 256, 1))))
    return float(O.cross_entropy(torch.cat(logits), y))


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("B,NA", [(1, 9), (128, 9), (129, 9), (256, 9), (257, 9), (4096, 9), (129, 1), (129, 2), (129, 16)])
def test_forward_only_loss_is_exact_on_its_logits(dev, monkeypatch, B, NA, mode):
    """net.loss(x, y) under no_grad (validation_step): the head's forward element-wise on its own inputs, the loss
    bounded on its own logits with per-sample power, and in fp32 mode within 1e-5 of the f64 oracle; n_actions = 1 gives
    exactly 0. The training step's loss on the same batch (the bc_backward with-loss reduction) meets the same bound.
    A label equal to n_actions in a validation batch is reported at check_device_errors()."""
    from carla_imitation_learning_b200 import sliding_window, stage_frames, stage_gray
    net = _net({"obs_size": 4, "n_actions": NA, "precision": mode})
    eng = net.engine()
    frames = _uniform_frames(7000 + B + NA, B + 4)
    rng = np.random.Generator(np.random.PCG64(B * 31 + NA))
    yn = rng.integers(0, NA, size=B)
    yn[0], yn[-1] = 0, NA - 1
    y = torch.from_numpy(yn)
    fr = torch.from_numpy(frames).to(dev)
    x = stage_frames(fr) if mode == "bf16" else sliding_window(stage_gray(fr))
    seen = []
    forward = eng.forward
    monkeypatch.setattr(eng, "forward", lambda *a, **k: seen.append(forward(*a, **k)) or seen[-1])
    with torch.no_grad():
        loss = net.loss(x, y.to(dev))
    torch.cuda.synchronize()
    eng.check_device_errors()
    assert len(seen) == 1 and torch.equal(loss, seen[0].loss)
    bufs = seen[0]
    P = {k: _cpu64(v) for k, v in net.state_dict().items()}
    tag = f"{mode} B={B} NA={NA}"
    print(f"\n{tag}")
    _check_head_fwd(tag, bufs, P, B, NA)
    _check_loss(f"{tag} forward-only", loss, bufs.logits, y, B, NA)
    if NA == 1:
        assert float(loss) == 0.0
    if mode == "fp32":
        ref = _oracle_loss(P, frames, y, B)
        assert abs(float(loss) - ref) <= 1e-5 * abs(ref), (float(loss), ref)
    step = eng.train_forward_backward(x, y.to(dev))
    torch.cuda.synchronize()
    eng.check_device_errors()
    _check_loss(f"{tag} training step", step.loss, step.logits, y, B, NA)
    bad = y.clone()
    bad[B // 2] = NA
    with torch.no_grad():
        net.loss(x, bad.to(dev))
    with pytest.raises(RuntimeError, match="label outside"):
        eng.check_device_errors()
