"""Sequential frame pipeline: pinned host frames -> H2D -> fused staging kernel -> window views.

Replaces the per-sample host work of SequentialTorchDataset + DataLoader
(/root/reference/src/dataset/imitation_dataset.py:90-136, 263-288): there every sample
re-reads and re-converts its 4 frames in numpy (`np.dot(...)/255.0`, :121) inside worker
processes and ships (B,4,256,256) f32 = 1 MB/sample to the trainer. Because the loader is
`shuffle=False` and sample i = frames [i, i+4) with the label of frame i+4 (:117,:125,:131),
a batch of B samples is B+3 distinct frames: this pipeline copies those B+frame_skip u8
frames once (196 KB each), converts each ONCE on the device, and hands the model a
zero-copy strided view -- 5.4x fewer PCIe bytes than f32 samples, 4x fewer conversions.
"""
from __future__ import annotations

from typing import Iterator, Optional, Tuple

import numpy as np
import torch

from . import _lib
from .engine import StagedBatch, sliding_window, stage_frames, stage_gray


def synthetic_sequence(seed: int, n_frames: int, h: int = 256, w: int = 256, n_actions: int = 9,
                       label_noise: float = 0.25) -> Tuple[np.ndarray, np.ndarray]:
    """Deterministic CARLA-shaped frames + labels (numpy PCG64): noise in [0,128) plus a +100 band
    whose row announces the next frame's label (wrong with probability `label_noise`)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    labels = rng.integers(0, n_actions, size=n_frames + 1, dtype=np.int64)
    shown = labels.copy()
    flip = rng.random(n_frames + 1) < label_noise
    shown[flip] = rng.integers(0, n_actions, size=int(flip.sum()))
    frames = rng.integers(0, 128, size=(n_frames, h, w, 3), dtype=np.uint8)
    band = h // n_actions
    for i in range(n_frames):
        r0 = int(shown[i + 1]) * band
        frames[i, r0:r0 + band] += 100
    return frames, labels[:n_frames]


def continous_to_discreet(steer, throttle, brake, steer_threshold: float = 0.05) -> np.ndarray:
    """(steer, throttle, brake) -> class id acc*3 + steer, the label contract of
    /root/reference/src/dataset/imitation_dataset.py:317-339 (name kept, spelling included).
    Takes the three columns as arrays instead of a DataFrame."""
    steer = np.asarray(steer, np.float64)
    throttle = np.asarray(throttle, np.float64)
    brake = np.asarray(brake, np.float64)
    right, left = steer > steer_threshold, steer < -steer_threshold
    s = np.where(right, 2.0, np.where(left, 0.0, 1.0))
    # inside the dead band the reference leaves raw values equal to 0.0 (or 2.0) untouched
    s = np.where(~right & ~left & (steer == 0.0), 0.0, s)
    acc = brake.copy()
    acc[(brake == 0.0) & (throttle == 1.0)] = 2.0
    acc[(brake == 0.0) & (throttle == 0.5)] = 1.0
    acc[(brake == 1.0) & (throttle == 0.0)] = 0.0
    return acc * 3 + s


def augment_table(seed: int, n_frames: int, src_hw, out_hw=(256, 256), brightness: float = 0.2, contrast: float = 0.2,
                  saturation: float = 0.2, mean: float = 0.0, std: float = 1.0) -> np.ndarray:
    """EXTENSION (no counterpart in the reference): the per-frame table of engine.stage_augmented, reproducible from `seed`
    on the host (numpy PCG64): (n_frames, 8) f32 rows [crop_y, crop_x, brightness, contrast, saturation, mean, 1/std, 0] --
    crop offsets uniform over the valid range, jitter factors uniform in [1 - a, 1 + a]."""
    rng = np.random.Generator(np.random.PCG64(seed))
    t = np.zeros((n_frames, 8), np.float32)
    t[:, 0] = rng.integers(0, src_hw[0] - out_hw[0] + 1, size=n_frames)
    t[:, 1] = rng.integers(0, src_hw[1] - out_hw[1] + 1, size=n_frames)
    t[:, 2] = rng.uniform(1 - brightness, 1 + brightness, size=n_frames)
    t[:, 3] = rng.uniform(1 - contrast, 1 + contrast, size=n_frames)
    t[:, 4] = rng.uniform(1 - saturation, 1 + saturation, size=n_frames)
    t[:, 5] = mean
    t[:, 6] = 1.0 / std
    return t


def center_crop_table(n_frames: int, src_hw, mean: float = 0.0, std: float = 1.0, out_hw=(256, 256)) -> np.ndarray:
    """EXTENSION: the deterministic serving counterpart of augment_table -- rows of the same (n_frames, 8) f32 layout with
    the centre crop ((Hs - 256) // 2, (Ws - 256) // 2), brightness, contrast and saturation factors of exactly 1 and the
    training normalisation (mean, 1/std). A policy trained on augment_table(..., mean, std) rows is served on these."""
    if src_hw[0] < out_hw[0] or src_hw[1] < out_hw[1]:
        raise ValueError(f"source frames {tuple(src_hw)} are smaller than the {out_hw[0]}x{out_hw[1]} crop")
    t = np.zeros((n_frames, 8), np.float32)
    t[:, 0] = (src_hw[0] - out_hw[0]) // 2
    t[:, 1] = (src_hw[1] - out_hw[1]) // 2
    t[:, 2:5] = 1.0
    t[:, 5] = mean
    t[:, 6] = 1.0 / std
    return t


class SequentialFrames:
    """Iterable of (x, y) batches over one frame sequence, staged on the device.

    x is a (b, frame_skip, H, W) strided view into the staged gray planes (f32 or bf16) or, with
    layout='tp' (the bf16 tensor-core mode), a StagedBatch of Toeplitz-ready planes written by the same
    single staging pass; y the (b,) int64 labels of the frames that follow each window. The last batch may be
    short (the reference's DataLoader has no drop_last). Host frames are pinned; chunk k+1's
    H2D copy runs on a side stream while the trainer consumes chunk k.

    x and y are views of two rotating device slots, not copies. A yielded batch stays valid until the consumer has asked
    the same iterator for two more: work enqueued on the consumer's current stream before that second request reads
    batch k (so two micro-batches may be accumulated across one next()); the request that hands out batch k + 2
    restages the slot, and a new iterator starts again from the first slot. Keep a batch longer, or read it from another
    stream, and clone it first.
    """

    def __init__(self, frames_u8: np.ndarray, labels: np.ndarray, batch_size: int = 64, frame_skip: int = 4,
                 device: Optional[torch.device] = None, dtype: torch.dtype = torch.float32, layout: str = "plain"):
        if frames_u8.dtype != np.uint8 or frames_u8.ndim != 4 or frames_u8.shape[-1] != 3:
            raise ValueError("frames must be (N,H,W,3) uint8")
        if len(labels) != len(frames_u8):
            raise ValueError("one label per frame (state.csv rows, imitation_dataset.py:108-111)")
        if len(frames_u8) <= frame_skip:
            raise ValueError(f"need more than frame_skip={frame_skip} frames")
        self.device = device if device is not None else torch.device("cuda", torch.cuda.current_device())
        if self.device.type != "cuda":
            raise RuntimeError("SequentialFrames stages on a CUDA device; there is no CPU path")
        self.frames = torch.from_numpy(np.ascontiguousarray(frames_u8)).pin_memory()
        self.labels = torch.from_numpy(np.asarray(labels, np.int64)).to(self.device)
        self.batch_size, self.frame_skip, self.dtype = int(batch_size), int(frame_skip), dtype
        self.n_samples = len(frames_u8) - frame_skip
        self._copy_stream = torch.cuda.Stream(self.device)
        self._staged = [None, None]
        n, h, w, _ = frames_u8.shape
        rows = self.batch_size + frame_skip
        self._raw = [torch.empty((rows, h, w, 3), dtype=torch.uint8, device=self.device) for _ in range(2)]
        # labels travel through per-slot buffers too: a batch then has the same (input, label) addresses every time its slot
        # comes round, which is what lets the training step be a replayed CUDA graph (autograd.FusedStepFunction, trainer.TrainStep)
        self._lab = [torch.zeros(self.batch_size, dtype=torch.int64, device=self.device) for _ in range(2)]
        if layout not in ("plain", "tp"):
            raise ValueError("layout is 'plain' (gray planes) or 'tp' (Toeplitz-ready bf16 planes for precision='bf16')")
        if layout == "tp" and (h, w, frame_skip) != (256, 256, 4):
            raise ValueError("the Toeplitz-ready layout is defined for 256x256 frames and frame_skip 4")
        self.layout = layout
        if layout == "tp":
            self._gray = [torch.empty((rows, _lib.TP_PLANE_ELEMS), dtype=torch.bfloat16, device=self.device) for _ in range(2)]
        else:
            self._gray = [torch.empty((rows, h, w), dtype=dtype, device=self.device) for _ in range(2)]

    def __len__(self) -> int:
        return (self.n_samples + self.batch_size - 1) // self.batch_size

    def _produce(self, k: int, slot: int) -> torch.cuda.Event:
        """H2D of chunk k's frames into raw slot `slot` on the copy stream (nothing else runs there: uploads go back to
        back; the staging kernel runs on the consumer's stream right before the batch is handed out)."""
        lo = k * self.batch_size
        hi = min(lo + self.batch_size, self.n_samples) + self.frame_skip
        with torch.cuda.stream(self._copy_stream):
            if self._staged[slot] is not None:
                self._copy_stream.wait_event(self._staged[slot])       # the staging pass that last read this raw slot
            self._raw[slot][:hi - lo].copy_(self.frames[lo:hi], non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(self._copy_stream)
        return ev

    def _stage(self, k: int, slot: int, cur) -> None:
        lo = k * self.batch_size
        hi = min(lo + self.batch_size, self.n_samples) + self.frame_skip
        if self.layout == "tp":
            stage_frames(self._raw[slot][:hi - lo], out=StagedBatch(self._gray[slot][:hi - lo], None, self.frame_skip))
        else:
            stage_gray(self._raw[slot][:hi - lo], out=self._gray[slot][:hi - lo])
        # the labels are copied on the consumer's stream too (device to device): a step of batch k - 2 still queued there
        # reads this slot's previous labels, and the copy stream would not wait for it
        nb = hi - lo - self.frame_skip
        self._lab[slot][:nb].copy_(self.labels[lo + self.frame_skip: lo + self.frame_skip + nb])
        if self._staged[slot] is None:
            self._staged[slot] = torch.cuda.Event()
        self._staged[slot].record(cur)

    def __iter__(self) -> Iterator[Tuple[torch.Tensor, torch.Tensor]]:
        return self._batches(loop=False)

    def cycle(self) -> Iterator[Tuple[torch.Tensor, torch.Tensor]]:
        """Endless iteration over the sequence; the first batch of the next pass is uploaded under the last batch of the
        current one (a fresh __iter__ per epoch would start every pass with an exposed H2D copy)."""
        return self._batches(loop=True)

    def _batches(self, loop: bool) -> Iterator[Tuple[torch.Tensor, torch.Tensor]]:
        nb = len(self)
        self._staged = [None, None]
        cur = torch.cuda.current_stream(self.device)
        self._copy_stream.wait_stream(cur)      # whatever still reads the slots from a previous pass
        ev = self._produce(0, 0)
        n = 0                                   # batches produced so far: slot = n & 1
        while True:
            k, slot = n % nb, n & 1
            cur = torch.cuda.current_stream(self.device)
            cur.wait_event(ev)
            self._stage(k, slot, cur)           # on the consumer's stream: ordered before the step that reads the planes
            if loop or k + 1 < nb:
                ev = self._produce((k + 1) % nb, slot ^ 1)
            lo = k * self.batch_size
            b = min(self.batch_size, self.n_samples - lo)
            if self.layout == "tp":
                x = StagedBatch(self._gray[slot][:b + self.frame_skip], None, self.frame_skip)
            else:
                x = sliding_window(self._gray[slot][:b + self.frame_skip], self.frame_skip)
            yield x, self._lab[slot][:b]
            n += 1
            if not loop and n == nb:
                return


def sequential_train_val_test_iterator(hparams, frames_by_split=None):
    """{'train_dataloader','val_dataloader','test_dataloader'} like
    imitation_dataset.sequential_train_val_test_iterator (imitation_dataset.py:263-288).
    `frames_by_split` maps split -> (frames_u8, labels); without it a synthetic sequence is
    generated (the reference ships no data, BASELINE.json asks for synthetic frames)."""
    bs = int(hparams['BATCH_SIZE'])
    fs = int(hparams.get('frame_skip', 4)) if hasattr(hparams, 'get') else int(hparams['frame_skip'])
    out = {}
    for i, split in enumerate(("train", "val", "test")):
        if frames_by_split is not None:
            frames, labels = frames_by_split[split]
        else:
            frames, labels = synthetic_sequence(i, (8 if split == "train" else 2) * bs + fs,
                                                n_actions=int(hparams['n_actions']))
        bf16 = (hparams.get('precision', 'fp32') if hasattr(hparams, 'get') else 'fp32') == 'bf16'
        out[f"{split}_dataloader"] = SequentialFrames(frames, labels, bs, fs, layout="tp" if bf16 else "plain")
    return out
