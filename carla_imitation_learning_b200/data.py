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

from typing import Callable, Iterator, Optional, Tuple

import numpy as np
import torch

from . import _lib
from .engine import StagedBatch, _check_augment_table, _ptr, sliding_window, stage_frames, stage_gather, stage_gray


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


def valid_starts(episode_lengths, frame_skip: int = 4) -> np.ndarray:
    """EXTENSION: the sample indices of a store of episodes laid end to end (episode e holds time steps [o_e, o_e + L_e)) whose
    window [i, i + frame_skip) and label frame i + frame_skip lie inside one episode: o_e .. o_e + L_e - frame_skip - 1 for
    every episode, in order. This is what a ConcatDataset of per-episode SequentialTorchDatasets exposes
    (imitation_dataset.py:90-136: L - frame_skip samples per episode); an episode of frame_skip frames or fewer has none."""
    lengths = np.asarray(episode_lengths, dtype=np.int64).reshape(-1)
    if (lengths < 0).any():
        raise ValueError("episode lengths are non-negative")
    offsets = np.concatenate([[0], np.cumsum(lengths)[:-1]]).astype(np.int64)
    parts = [o + np.arange(max(int(n) - frame_skip, 0), dtype=np.int64) for o, n in zip(offsets, lengths)]
    return np.concatenate(parts) if parts else np.zeros(0, np.int64)


class FrameStore:
    """EXTENSION: a dataset's frames and side data in device memory, the source of shuffled minibatches (engine.stage_gather,
    ShuffledFrames, TrainStep.step_gather). A B200 holds 200 K CARLA frames of 256 x 256 u8 RGB (39 GB).

    frames_u8: (n_frames*cams, Hs, Ws, 3) u8, row t*cams + k = camera k at time t, Hs, Ws >= 256 (larger frames are cropped
    by an augmentation table); labels (n_frames,) int64 class ids, commands (n_frames,) int64 branch ids, targets
    (n_frames, n_out) f32 regression targets, each optional. numpy arrays or host tensors are uploaded once; CUDA tensors on
    `device` are wrapped without a copy (they must then stay alive and unchanged while the store is in use). Several
    episodes are laid end to end; valid_starts() names the samples that do not straddle two of them."""

    def __init__(self, frames_u8, labels=None, commands=None, targets=None, cams: int = 1, device: Optional[torch.device] = None):
        if cams not in (1, 3):
            raise ValueError("cams is 1 (obs_size 4) or 3 (obs_size 12)")
        if device is None:
            device = frames_u8.device if isinstance(frames_u8, torch.Tensor) and frames_u8.is_cuda else \
                torch.device("cuda", torch.cuda.current_device())
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("FrameStore lives in device memory; there is no CPU path")
        fr = self._upload(frames_u8, torch.uint8, "frames")
        if fr.dim() != 4 or fr.shape[-1] != 3 or fr.shape[1] < 256 or fr.shape[2] < 256 or fr.shape[0] % cams:
            raise ValueError("frames must be (n_frames*cams, Hs, Ws, 3) uint8 with Hs, Ws >= 256")
        self.frames, self.cams = fr, int(cams)
        self.n_frames = fr.shape[0] // cams
        if self.n_frames < 5:
            raise ValueError("a store holds at least 5 time steps (one 4-frame window and the label after it)")
        self.src_hw = (int(fr.shape[1]), int(fr.shape[2]))
        self.labels = None if labels is None else self._upload(labels, torch.int64, "labels")
        self.commands = None if commands is None else self._upload(commands, torch.int64, "commands")
        self.targets = None if targets is None else self._upload(targets, torch.float32, "targets")
        for name, t in (("labels", self.labels), ("commands", self.commands)):
            if t is not None and tuple(t.shape) != (self.n_frames,):
                raise ValueError(f"{name} are ({self.n_frames},): one per time step")
        if self.targets is not None and (self.targets.dim() != 2 or self.targets.shape[0] != self.n_frames):
            raise ValueError(f"targets are ({self.n_frames}, n_out): one row per time step")
        self.n_out = 0 if self.targets is None else int(self.targets.shape[1])
        self.n_samples = self.n_frames - 4
        self.err_flag = torch.zeros(1, dtype=torch.int32, device=self.device)
        self.struct = _lib.BcFrameStore(self.frames.data_ptr(), self.n_frames, self.cams, self.src_hw[0], self.src_hw[1],
                                        _ptr(self.labels), _ptr(self.commands), _ptr(self.targets), self.n_out)

    def _upload(self, a, dtype: torch.dtype, what: str) -> torch.Tensor:
        t = torch.from_numpy(np.ascontiguousarray(a)) if isinstance(a, np.ndarray) else a
        if not isinstance(t, torch.Tensor):
            raise ValueError(f"{what} must be a numpy array or a tensor")
        if t.is_cuda:
            if t.device != self.device or t.dtype != dtype or not t.is_contiguous():
                raise ValueError(f"device {what} must be a contiguous {dtype} tensor on {self.device}")
            return t
        return t.to(dtype=dtype).contiguous().to(self.device)

    def check(self) -> None:
        """Raise if a staging launch met a sample index outside [0, n_frames - 5] (synchronises)."""
        code = int(self.err_flag.item())
        if code != 0:
            self.err_flag.zero_()
            raise RuntimeError(f"bc_stage_gather: a sample index outside [0, {self.n_frames - 5}] was staged (device flag {code})")


class ShuffledFrames:
    """EXTENSION: the shuffled counterpart of SequentialFrames -- minibatches of samples drawn at random from a FrameStore,
    staged by ONE bc_stage_gather launch per batch (conditional imitation trains on such batches; a sequential batch is
    ~13 s of one drive and may straddle two episodes).

    Yields (x, y) like SequentialFrames, or (x, command, target) when the store has commands (the branched policy: target =
    the store's targets when it has them, else its labels). x holds the windows materialised: layout 'plain' = a contiguous
    (b, 4*cams, 256, 256) f32 tensor, 'tp' = a StagedBatch of Toeplitz-ready bf16 planes (precision='bf16').

    Order: epoch e visits `starts` (default: every sample of the store; valid_starts() for episodes) in the order of a host
    numpy PCG64 permutation seeded with seed + e, so it is reproducible and checkable on the CPU. Rank r of `world` takes
    the disjoint shard permutation[r::world] (DistributedSampler's interleaving, without padding: shards differ by at most
    one sample). The last batch may be short (no drop_last, as in the reference). Each __iter__ runs epoch `self.epoch`
    and advances it (set it to resume at an epoch). table_fn(epoch, batch_idx, rows) -> (rows, 8) f32 rows of data.augment_table (rows =
    b*cams), required for frames larger than 256x256: row b*cams + k applies to all four frames of camera k of sample b.

    Index, side data, table and staging buffers rotate over two persistent device slots, as in SequentialFrames: a batch is
    valid until the consumer has asked for two more, and its addresses repeat, so a CUDA-graph module step keeps replaying.
    Everything is enqueued on the consumer's current stream; nothing synchronises the host."""

    def __init__(self, store: FrameStore, batch_size: int, seed: int = 0, layout: str = "plain", starts=None,
                 table_fn: Optional[Callable] = None, rank: int = 0, world: int = 1):
        if layout not in ("plain", "tp"):
            raise ValueError("layout is 'plain' (f32 planes) or 'tp' (Toeplitz-ready bf16 planes for precision='bf16')")
        if not 0 <= rank < world:
            raise ValueError(f"rank {rank} outside [0, {world})")
        if int(batch_size) < 1:
            raise ValueError("batch_size must be at least 1")
        self.store, self.batch_size, self.seed, self.layout = store, int(batch_size), int(seed), layout
        self.rank, self.world, self.table_fn, self.epoch = int(rank), int(world), table_fn, 0
        self.starts = (np.arange(store.n_samples, dtype=np.int64) if starts is None
                       else np.asarray(starts, dtype=np.int64).reshape(-1))
        if self.starts.size == 0:
            raise ValueError("no sample to draw")
        if self.starts.min() < 0 or self.starts.max() > store.n_frames - 5:
            raise ValueError(f"sample indices lie in [0, {store.n_frames - 5}]")
        if store.src_hw != (256, 256) and table_fn is None:
            raise ValueError(f"{store.src_hw[0]}x{store.src_hw[1]} frames need table_fn (crop rows, data.augment_table)")
        dev, B, cams = store.device, self.batch_size, store.cams
        self.branched = store.commands is not None
        i64 = dict(dtype=torch.int64, device=dev)
        self._idx = [torch.zeros(B, **i64) for _ in range(2)]
        self._lab = [torch.zeros(B, **i64) for _ in range(2)] if store.labels is not None else None
        self._cmd = [torch.zeros(B, **i64) for _ in range(2)] if self.branched else None
        self._tgt = ([torch.zeros((B, store.n_out), dtype=torch.float32, device=dev) for _ in range(2)]
                     if store.targets is not None else None)
        self._tab = [torch.zeros((B * cams, 8), dtype=torch.float32, device=dev) for _ in range(2)] if table_fn else None
        if layout == "tp":
            self._x = [torch.empty((B * 4 * cams, _lib.TP_PLANE_ELEMS), dtype=torch.bfloat16, device=dev) for _ in range(2)]
        else:
            self._x = [torch.empty((B, 4 * cams, 256, 256), dtype=torch.float32, device=dev) for _ in range(2)]
        if self.branched and self._tgt is None and self._lab is None:
            raise ValueError("a store with commands needs labels (CE) or targets (L1 / MSE)")
        if not self.branched and self._lab is None:
            raise ValueError("a store without commands needs labels")

    def permutation(self, epoch: int) -> np.ndarray:
        """Every start, in epoch `epoch`'s order (all ranks)."""
        rng = np.random.Generator(np.random.PCG64(self.seed + int(epoch)))
        return self.starts[rng.permutation(self.starts.size)]

    def shard(self, epoch: int) -> np.ndarray:
        """This rank's sample indices of epoch `epoch`, in the order they are staged."""
        return self.permutation(epoch)[self.rank::self.world]

    def __len__(self) -> int:
        n = (self.starts.size - self.rank + self.world - 1) // self.world
        return (n + self.batch_size - 1) // self.batch_size

    def __iter__(self):
        epoch = self.epoch
        self.epoch += 1
        order = self.shard(epoch)
        store, B, cams = self.store, self.batch_size, self.store.cams
        dev_order = torch.from_numpy(np.ascontiguousarray(order)).to(store.device)
        for k in range((order.size + B - 1) // B):
            slot, lo = k & 1, k * B
            b = min(B, order.size - lo)
            idx = self._idx[slot][:b]
            idx.copy_(dev_order[lo:lo + b])
            table = None
            if self.table_fn is not None:
                rows = self.table_fn(epoch, k, b * cams)
                rows = torch.as_tensor(rows, dtype=torch.float32)
                if tuple(rows.shape) != (b * cams, 8):
                    raise ValueError(f"table_fn must return ({b * cams}, 8) float32 rows")
                if rows.device.type == "cpu":
                    _check_augment_table(rows, *store.src_hw)
                table = self._tab[slot][:b * cams]
                table.copy_(rows)
            out = (StagedBatch(self._x[slot][:b * 4 * cams], None, 4 * cams, 4 * cams) if self.layout == "tp"
                   else self._x[slot][:b])
            lab = None if self._lab is None else self._lab[slot][:b]
            cmd = None if self._cmd is None else self._cmd[slot][:b]
            tgt = None if self._tgt is None else self._tgt[slot][:b]
            x = stage_gather(store, idx, self.layout, out=out, table=table, y=lab, command=cmd, target=tgt)
            if self.branched:
                yield x, cmd, (tgt if tgt is not None else lab)
            else:
                yield x, lab


def _datamodule_key(hparams, key: str, default):
    """A configs/datamodule key: at the root of flat hparams, else in the composed config's `datamodule` group."""
    if not hasattr(hparams, 'get'):
        return default
    if key in hparams:
        return hparams[key]
    group = hparams.get('datamodule')
    return group.get(key, default) if hasattr(group, 'get') else default


def sequential_train_val_test_iterator(hparams, frames_by_split=None):
    """{'train_dataloader','val_dataloader','test_dataloader'} like
    imitation_dataset.sequential_train_val_test_iterator (imitation_dataset.py:263-288).
    `frames_by_split` maps split -> (frames_u8, labels); without it a synthetic sequence is
    generated (the reference ships no data, BASELINE.json asks for synthetic frames).
    With `shuffle: true` (configs/datamodule) the train split is a ShuffledFrames over a device FrameStore of its frames,
    permuted per epoch from `shuffle_seed`; validation and test stay sequential."""
    bs = int(hparams['BATCH_SIZE'])
    fs = int(hparams.get('frame_skip', 4)) if hasattr(hparams, 'get') else int(hparams['frame_skip'])
    bf16 = (hparams.get('precision', 'fp32') if hasattr(hparams, 'get') else 'fp32') == 'bf16'
    shuffle, seed = bool(_datamodule_key(hparams, 'shuffle', False)), int(_datamodule_key(hparams, 'shuffle_seed', 0))
    if shuffle and fs != 4:
        raise ValueError("shuffled batches stage 4-frame windows: frame_skip must be 4")
    out = {}
    for i, split in enumerate(("train", "val", "test")):
        if frames_by_split is not None:
            frames, labels = frames_by_split[split]
        else:
            frames, labels = synthetic_sequence(i, (8 if split == "train" else 2) * bs + fs,
                                                n_actions=int(hparams['n_actions']))
        if shuffle and split == "train":
            out["train_dataloader"] = ShuffledFrames(FrameStore(frames, labels), bs, seed, layout="tp" if bf16 else "plain")
        else:
            out[f"{split}_dataloader"] = SequentialFrames(frames, labels, bs, fs, layout="tp" if bf16 else "plain")
    return out
