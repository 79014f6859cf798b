"""Host side of the hot path: buffer management and kernel sequencing for one device.

Mirrors what torch autograd + ATen do for the reference's
`ConvNet1.forward` (/root/reference/src/architectures/nets.py:35-39) and
`Imitation.training_step` (/root/reference/src/models/imitation.py:38-45), but every
numeric op is a call into libbc_b200.so. PyTorch provides device memory and streams only.
"""
from __future__ import annotations

import contextlib
import ctypes as C
from dataclasses import dataclass, field
from typing import List, Optional

import torch

from . import _lib

ACT_SHAPES = ((16, 28, 28), (32, 12, 12), (64, 4, 4), (128, 1, 1))
H = W = 256


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def _stream_ptr() -> int:
    """cudaStream_t of the current stream of the current device. The raw getter skips building a torch.cuda.Stream object:
    the module path is host-bound once the device step is shorter than the Python loop (tools/module_host_profile.py)."""
    if _raw_stream is not None:
        return _raw_stream(torch.cuda.current_device())
    return torch.cuda.current_stream().cuda_stream


_NO_SWITCH = contextlib.nullcontext()


def on_device(dev: torch.device):
    """`with torch.cuda.device(dev)` when another device is current, nothing otherwise (the context manager costs ~10 us of
    Python per use; one process per GPU means the device is already current in every hot call)."""
    return _NO_SWITCH if dev.index is None or torch.cuda.current_device() == dev.index else torch.cuda.device(dev)


def _require_cuda(t: torch.Tensor, what: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(f"{what} must live on a CUDA (sm_100) device: the BC hot path has no CPU fallback")


def stage_gray(frames_u8: torch.Tensor, dtype: torch.dtype = torch.float32, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """(n,H,W,3) u8 RGB on the device -> (n,H,W) gray planes, (0.299R+0.587G+0.114B)/255.

    The device version of SequentialTorchDataset._load_file
    (/root/reference/src/dataset/imitation_dataset.py:120-121,130); f32 output is bit-exact."""
    _require_cuda(frames_u8, "frames")
    if frames_u8.dtype != torch.uint8 or frames_u8.dim() != 4 or frames_u8.shape[-1] != 3 or not frames_u8.is_contiguous():
        raise ValueError("frames must be a contiguous (n,H,W,3) uint8 tensor")
    n, h, w, _ = frames_u8.shape
    if out is None:
        out = torch.empty((n, h, w), dtype=dtype, device=frames_u8.device)
    code = {torch.float32: _lib.BC_F32, torch.bfloat16: _lib.BC_BF16}[out.dtype]
    if n * h * w == 0:
        return out
    _lib.check(_lib.lib().bc_stage_gray(frames_u8.data_ptr(), out.data_ptr(), n * h * w, code, _stream_ptr()), "bc_stage_gray")
    return out


def sliding_window(gray: torch.Tensor, frame_skip: int = 4, step: int = 1) -> torch.Tensor:
    """Zero-copy ((n-frame_skip)/step, frame_skip, H, W) view: sample i = planes [i*step, i*step+frame_skip).

    The reference's loader is shuffle=False (imitation_dataset.py:270-274) with
    files[index-frame_skip:index], index=i+4 (:117,:125), so consecutive samples share 3 of 4
    planes; the view hands that overlap to the conv1 kernels without materialising it.
    step > 1 is the multi-camera stacking of BASELINE configs[3]: with the planes of `step` cameras interleaved frame by
    frame (plane = t*step + cam), sample i = window of frame_skip = step*frames planes starting at plane i*step, i.e.
    channels ordered (frame, camera)."""
    n, h, w = gray.shape
    if n <= frame_skip:
        raise ValueError(f"need more than {frame_skip} frames, got {n}")
    return gray.as_strided(((n - frame_skip) // step, frame_skip, h, w), (step * h * w, h * w, w, 1))


class StagedBatch:
    """bf16-mode input produced by stage_frames(): n staged frames = n - frame_skip samples as `tp`
    (n, TP_PLANE_ELEMS) Toeplitz-ready bf16 planes, the layout both tcgen05 conv1 kernels consume as it is
    (include/bc_b200.h, BC_BF16_TP). `plain` (n,256,256) bf16 is optional: the same gray values as ordinary
    planes (diagnostics, or the exact-f32 kernels), written by the same pass of the staging kernel."""

    def __init__(self, tp: torch.Tensor, plain: Optional[torch.Tensor] = None, frame_skip: int = 4, step: int = 1):
        # step = planes a sample advances by: 1 = the reference's 4-frame window; 3 with frame_skip 12 = BASELINE configs[3],
        # three cameras interleaved frame by frame (sample i = planes [3i, 3i+12), channel = 3*frame + camera);
        # step == frame_skip = materialised windows that share no plane (stage_gather: shuffled samples)
        self.tp, self.plain, self.frame_skip, self.step = tp, plain, frame_skip, step

    @property
    def materialised(self) -> bool:
        return self.step == self.frame_skip

    @property
    def x(self) -> Optional[torch.Tensor]:
        if self.plain is None:
            return None
        if self.materialised:
            return self.plain.view(-1, self.frame_skip, H, W)
        return sliding_window(self.plain, self.frame_skip, self.step)

    @property
    def shape(self):
        if self.materialised:
            return (self.tp.shape[0] // self.step, self.frame_skip, H, W)
        return ((self.tp.shape[0] - self.frame_skip) // self.step, self.frame_skip, H, W)

    @property
    def device(self):
        return self.tp.device

    def to(self, *_a, **_k):
        return self


def stage_frames(frames_u8: torch.Tensor, out: Optional[StagedBatch] = None, frame_skip: int = 4,
                 plain: bool = False, step: int = 1) -> StagedBatch:
    """(n,256,256,3) u8 RGB on the device -> StagedBatch. The bf16-mode replacement of SequentialTorchDataset's
    per-sample numpy work (imitation_dataset.py:115-133): gray conversion, /255, 4-frame stacking (as a view) and
    the MMA operand layout of conv1 in one fused kernel."""
    _require_cuda(frames_u8, "frames")
    if frames_u8.dtype != torch.uint8 or frames_u8.dim() != 4 or tuple(frames_u8.shape[1:]) != (H, W, 3) or not frames_u8.is_contiguous():
        raise ValueError("frames must be a contiguous (n,256,256,3) uint8 tensor")
    n = frames_u8.shape[0]
    if n <= frame_skip:
        raise ValueError(f"need more than {frame_skip} frames, got {n}")
    if out is None:
        out = StagedBatch(torch.empty((n, _lib.TP_PLANE_ELEMS), dtype=torch.bfloat16, device=frames_u8.device),
                          torch.empty((n, H, W), dtype=torch.bfloat16, device=frames_u8.device) if plain else None, frame_skip, step)
    elif out.tp.shape[0] != n:
        raise ValueError("out was staged for a different number of frames")
    _lib.check(_lib.lib().bc_stage_gray_tp(frames_u8.data_ptr(), out.tp.data_ptr(),
                                           out.plain.data_ptr() if out.plain is not None else None, n, _stream_ptr()), "bc_stage_gray_tp")
    return out


def _check_augment_table(table: torch.Tensor, hs: int, ws: int) -> None:
    """Rows {crop_y, crop_x, brightness, contrast, saturation, mean, 1/std, -} of a host f32 table: a crop outside the
    source would make the staging kernel read outside the frames."""
    t = table[:, :7].double()
    if not bool(torch.isfinite(t).all()):
        raise ValueError("the augmentation table has a non-finite entry")
    crop = t[:, :2]
    if not torch.equal(crop, crop.floor()):
        raise ValueError("the augmentation table's crop offsets must be integers")
    if t.shape[0] and (float(crop.min()) < 0 or float(crop[:, 0].max()) > hs - H or float(crop[:, 1].max()) > ws - W):
        raise ValueError(f"the augmentation table's crop offsets must lie in [0, {hs - H}] x [0, {ws - W}] for {hs}x{ws} sources")


def stage_augmented(frames_u8: torch.Tensor, table: torch.Tensor, layout: str = "plain", frame_skip: int = 4, out=None):
    """EXTENSION (no counterpart in the reference): crop + colour jitter + normalise fused into the staging pass.
    frames (n, Hs, Ws, 3) u8 on the device with Hs, Ws >= 256; table (n, 8) f32 = data.augment_table(seed, ...) rows
    {crop_y, crop_x, brightness, contrast, saturation, mean, 1/std, -}. layout 'plain' -> (n,256,256) f32 gray planes
    (use sliding_window() on them), 'tp' -> StagedBatch of Toeplitz-ready bf16 planes for precision='bf16'.
    `out` = persistent destination (a (n,256,256) f32 tensor for 'plain', a StagedBatch for 'tp'): a fixed-shape training
    loop or a CUDA graph stages into the same buffers every step.
    A host table is checked before it is copied: integral crop offsets in [0, Hs-256] x [0, Ws-256] and finite factors,
    else ValueError and nothing is launched. A device table is not read back (that would synchronise every step): its
    rows are the caller's contract, as for BranchedTrainStep."""
    _require_cuda(frames_u8, "frames")
    if frames_u8.dtype != torch.uint8 or frames_u8.dim() != 4 or frames_u8.shape[-1] != 3 or not frames_u8.is_contiguous():
        raise ValueError("frames must be a contiguous (n,Hs,Ws,3) uint8 tensor")
    n, hs, ws, _ = frames_u8.shape
    if hs < H or ws < W:
        raise ValueError(f"source frames {hs}x{ws} are smaller than the {H}x{W} crop")
    if tuple(table.shape) != (n, 8):
        raise ValueError("the augmentation table is (n_frames, 8) float32")
    if table.device.type == "cpu":
        table = table.to(dtype=torch.float32)
        _check_augment_table(table, hs, ws)
    table = table.to(device=frames_u8.device, dtype=torch.float32).contiguous()
    if layout == "plain":
        if out is None:
            out = torch.empty((n, H, W), dtype=torch.float32, device=frames_u8.device)
        elif (not isinstance(out, torch.Tensor) or out.dtype != torch.float32 or tuple(out.shape) != (n, H, W)
              or not out.is_contiguous() or out.device != frames_u8.device):
            raise ValueError(f"out for layout 'plain' is a contiguous ({n},{H},{W}) float32 tensor on the frames' device")
        code, res = _lib.BC_F32, out
    elif layout == "tp":
        if out is None:
            res = StagedBatch(torch.empty((n, _lib.TP_PLANE_ELEMS), dtype=torch.bfloat16, device=frames_u8.device), None, frame_skip)
        elif (not isinstance(out, StagedBatch) or tuple(out.tp.shape) != (n, _lib.TP_PLANE_ELEMS)
              or out.tp.dtype != torch.bfloat16 or out.tp.device != frames_u8.device):
            raise ValueError(f"out for layout 'tp' is a StagedBatch of {n} frames on the frames' device")
        else:
            res = out
        code, out = _lib.BC_BF16_TP, res.tp
    else:
        raise ValueError("layout is 'plain' or 'tp'")
    if n:
        _lib.check(_lib.lib().bc_stage_augment(frames_u8.data_ptr(), n, hs, ws, table.data_ptr(), out.data_ptr(), code, _stream_ptr()), "bc_stage_augment")
    return res


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def stage_gather(store, index: torch.Tensor, layout: str = "tp", out=None, table: Optional[torch.Tensor] = None,
                 y: Optional[torch.Tensor] = None, command: Optional[torch.Tensor] = None,
                 target: Optional[torch.Tensor] = None, err_flag: Optional[torch.Tensor] = None):
    """EXTENSION: B shuffled samples from a device-resident data.FrameStore in ONE staging launch (bc_stage_gather).
    index (B,) int64 on the store's device: index[b] = i is the reference's sample i (frames i .. i+3, side data of frame
    i+4). Returns the windows materialised, channel cams*j + k = camera k of frame i+j: layout 'tp' -> StagedBatch of B*4*cams
    Toeplitz-ready bf16 planes (precision='bf16'), 'plain' -> a contiguous (B, 4*cams, 256, 256) f32 tensor. `out` = a
    persistent destination of that form. table = (B*cams, 8) f32 rows (data.augment_table / center_crop_table layout), row
    b*cams + k for all four frames of camera k of sample b; required for stores of frames larger than 256x256. y, command
    (B,) int64 and target (B, n_out) f32 are filled from the store's labels / commands / targets in the same launch when
    given. An index outside [0, n_frames - 5] zeroes that sample and sets err_flag (default: store.err_flag) to 5.
    A host table is checked like stage_augmented's; device tensors are not read back."""
    dev = store.device
    if not isinstance(index, torch.Tensor) or index.device != dev or index.dtype != torch.int64 or index.dim() != 1 \
            or not index.is_contiguous():
        raise ValueError(f"index must be a contiguous (B,) int64 tensor on {dev}")
    B, cams = index.shape[0], store.cams
    if B < 1:
        raise ValueError("index holds no sample")
    hs, ws = store.src_hw
    if table is not None:
        if tuple(table.shape) != (B * cams, 8):
            raise ValueError(f"the augmentation table is ({B * cams}, 8) float32: one row per sample and camera")
        if table.device.type == "cpu":
            table = table.to(dtype=torch.float32)
            _check_augment_table(table, hs, ws)
            table = table.to(dev)
        if table.device != dev or table.dtype != torch.float32 or not table.is_contiguous():
            raise ValueError(f"table must be a contiguous float32 tensor on {dev}")
    elif (hs, ws) != (H, W):
        raise ValueError(f"{hs}x{ws} frames need a crop table (data.augment_table / center_crop_table rows)")
    n_planes = B * 4 * cams
    if layout == "tp":
        if out is None:
            out = StagedBatch(torch.empty((n_planes, _lib.TP_PLANE_ELEMS), dtype=torch.bfloat16, device=dev), None, 4 * cams, 4 * cams)
        elif (not isinstance(out, StagedBatch) or tuple(out.tp.shape) != (n_planes, _lib.TP_PLANE_ELEMS) or not out.materialised
              or out.frame_skip != 4 * cams or out.tp.dtype != torch.bfloat16 or out.tp.device != dev or not out.tp.is_contiguous()):
            raise ValueError(f"out for layout 'tp' is a materialised StagedBatch of {n_planes} planes on {dev}")
        code, dst = _lib.BC_BF16_TP, out.tp
    elif layout == "plain":
        if out is None:
            out = torch.empty((B, 4 * cams, H, W), dtype=torch.float32, device=dev)
        elif (not isinstance(out, torch.Tensor) or out.dtype != torch.float32 or tuple(out.shape) != (B, 4 * cams, H, W)
              or not out.is_contiguous() or out.device != dev):
            raise ValueError(f"out for layout 'plain' is a contiguous ({B}, {4 * cams}, {H}, {W}) float32 tensor on {dev}")
        code, dst = _lib.BC_F32, out
    else:
        raise ValueError("layout is 'plain' or 'tp'")
    for name, t, dt, shape in (("y", y, torch.int64, (B,)), ("command", command, torch.int64, (B,)),
                               ("target", target, torch.float32, (B, store.n_out))):
        if t is not None and (not isinstance(t, torch.Tensor) or t.device != dev or t.dtype != dt
                              or tuple(t.shape) != shape or not t.is_contiguous()):
            raise ValueError(f"{name} must be a contiguous {shape} {dt} tensor on {dev}")
    flag = store.err_flag if err_flag is None else err_flag
    with on_device(dev):
        _lib.check(_lib.lib().bc_stage_gather(C.byref(store.struct), index.data_ptr(), B, _ptr(table), dst.data_ptr(), code,
                                              _ptr(y), _ptr(command), _ptr(target), flag.data_ptr(), _stream_ptr()),
                   "bc_stage_gather")
    return out


@dataclass
class StepBuffers:
    """Everything one forward produces and one backward consumes."""
    batch: int
    x: Optional[torch.Tensor]         # None when the input exists only as Toeplitz-ready planes (x_tp)
    y: Optional[torch.Tensor]
    act: List[torch.Tensor]
    amax: List[torch.Tensor]
    hid1: torch.Tensor
    hid2: torch.Tensor
    logits: torch.Tensor
    dlogits: torch.Tensor
    loss: torch.Tensor
    ghead: Optional[torch.Tensor] = None
    gact: List[torch.Tensor] = field(default_factory=list)
    act_bf16: List[torch.Tensor] = field(default_factory=list)   # bf16 mode: bf16 copies feeding the next layer's MMA
    gact0_p8: Optional[torch.Tensor] = None                      # bf16 mode: masked gradient w.r.t. act1, P8 bf16 (conv2 dgrad -> conv1 wgrad)
    amax0_p8: Optional[torch.Tensor] = None                      # bf16 mode: conv1's pool routing again in P8 order
    x_tp: Optional[torch.Tensor] = None                          # bf16 mode: the input as Toeplitz-ready planes
    x_tp_strides: tuple = (0, 0)                                 # (sample, channel) element strides into x_tp
    c1_acc: Optional[torch.Tensor] = None                        # bf16 mode, obs_size 12: raw conv1 accumulators between the camera launches


class BCEngine:
    """Kernel sequencing for one parameter arena on one device."""

    def __init__(self, arena: torch.Tensor, obs_size: int, n_actions: int):
        _require_cuda(arena, "parameter arena")
        if arena.dtype != torch.float32 or not arena.is_contiguous():
            raise ValueError("the parameter arena is a contiguous float32 tensor")
        self.lib = _lib.lib()
        with torch.cuda.device(arena.device):
            _lib.check(self.lib.bc_device_check(), "bc_device_check")
        self.arena = arena
        self.device = arena.device
        self.obs_size, self.n_actions = int(obs_size), int(n_actions)
        total, self.offsets, self.sizes = _lib.arena_layout(self.obs_size, self.n_actions)
        if arena.numel() != total:
            raise ValueError(f"arena has {arena.numel()} floats, layout needs {total}")
        self.grads = torch.zeros_like(arena)
        self.grads_epoch: Optional[torch.Tensor] = None    # peer exchange: device word selecting the half of a double-buffered arena (bc_ctx.grads_epoch)
        self.grads_stride = 0
        # partial-sum workspace: pads are never written, so it must start zeroed
        self.partials = torch.zeros(int(self.lib.bc_partials_floats(self.obs_size, self.n_actions)),
                                    dtype=torch.float32, device=self.device)
        # bf16 tensor-core mode: packed MMA operand images + the device error flag of the bounded waits
        self.w_packed = torch.zeros(int(self.lib.bc_packed_weight_bytes()), dtype=torch.uint8, device=self.device)
        self.err_flag = torch.zeros(1, dtype=torch.int32, device=self.device)
        self.conv_mode = 0            # bit mask, see bc_ctx.conv_mode: 0 = exact f32 FFMA kernels, 15 = all tcgen05 kernels
        self._packed_version = None   # weights_version() the bf16 operand images were last derived from (None = never)
        self.weights_version = lambda: self.arena._version     # ConvNet1 widens it to every Parameter view (p.copy_ bumps p's own counter)
        self.overlap = False          # backward with the conv4..conv2 weight-gradient kernels on a side stream (bc_backward_overlap)
        self._side = None             # (side stream, 4 events, ctypes array of their handles)
        self._static = {}             # batch -> StepBuffers reused by the static-shape paths (no per-step allocation)
        self.peer = None              # parallel.PeerGrads once the gradients live in peer-visible memory
        self._slots, self._slot_i = None, 0

    # ------------------------------------------------------------------ buffers
    def alloc(self, batch: int, x, y: Optional[torch.Tensor], backward: bool) -> StepBuffers:
        dev, f32 = self.device, torch.float32
        staged = x if isinstance(x, StagedBatch) else None
        if staged is not None:
            x = staged.x
        e = lambda *s, dt=f32: torch.empty(s, dtype=dt, device=dev)
        bufs = StepBuffers(
            batch=batch, x=x, y=y,
            act=[e(batch, *s) for s in ACT_SHAPES],
            amax=[e(batch, *s, dt=torch.uint8) for s in ACT_SHAPES],
            hid1=e(batch, 64), hid2=e(batch, 32), logits=e(batch, self.n_actions),
            dlogits=e(batch, self.n_actions), loss=torch.zeros((), dtype=f32, device=dev))
        if staged is not None:
            bufs.x_tp, bufs.x_tp_strides = staged.tp, (staged.step * _lib.TP_PLANE_ELEMS, _lib.TP_PLANE_ELEMS)
        elif (self.conv_mode & 1) and batch:
            bufs.x_tp, bufs.x_tp_strides = self.to_tp(x)
        if (self.conv_mode & 1) and self.obs_size == 12:
            # the raw conv1 accumulators the three camera launches hand to each other (bc_ctx.c1_acc)
            bufs.c1_acc = torch.empty((max(batch, 1), 14, 126, 64), dtype=f32, device=dev)
        if self.conv_mode & 1:
            # bf16 copies feeding the next layer's MMAs: act1, act2 as P8 = (B, C/8, H*W, 8) for the shifted-window
            # kernels (csrc/conv_sw.cu), act3 as P8B = (C/8, B, H*W, 8) for conv4 (csrc/conv4_sw.cu)
            bufs.act_bf16 = [torch.empty((batch, 2, 784, 8), dtype=torch.bfloat16, device=dev),
                             torch.empty((batch, 4, 144, 8), dtype=torch.bfloat16, device=dev),
                             torch.empty((8, batch, 16, 8), dtype=torch.bfloat16, device=dev)]
        if self.conv_mode & 16:
            bufs.gact0_p8 = torch.zeros((batch, 2, 784, 8), dtype=torch.bfloat16, device=dev)
            bufs.amax0_p8 = torch.zeros((batch, 2, 784, 8), dtype=torch.uint8, device=dev)
        if backward:
            self._alloc_bwd(bufs)
        return bufs

    def _alloc_bwd(self, bufs: StepBuffers) -> None:
        if bufs.ghead is None:
            e = lambda *s: torch.empty(s, dtype=torch.float32, device=self.device)
            bufs.ghead = e(bufs.batch, 128)
            bufs.gact = [e(bufs.batch, *s) for s in ACT_SHAPES[:3]]

    def to_tp(self, x: torch.Tensor, out: Optional[torch.Tensor] = None):
        """(B,4,256,256) f32/bf16 batch -> Toeplitz-ready bf16 planes (include/bc_b200.h BC_BF16_TP) + strides.
        A sliding-window view (sliding_window()) is converted once per PLANE, not per sample."""
        B = x.shape[0]
        P = H * W
        step = self.obs_size // 4                                   # planes per sample step of the (stacked) sliding window: 1, or 3 for obs 12
        sliding = x.stride(0) == step * P and x.stride(1) == P
        if not sliding and not (x.stride(1) == P and x.stride(0) == self.obs_size * P):
            x = x.contiguous()
        n_planes = step * (B - 1) + self.obs_size if sliding else B * self.obs_size
        tp = out if out is not None else torch.empty((n_planes, _lib.TP_PLANE_ELEMS), dtype=torch.bfloat16, device=x.device)
        code = _lib.BC_F32 if x.dtype == torch.float32 else _lib.BC_BF16
        _lib.check(self.lib.bc_planes_to_tp(x.data_ptr(), code, n_planes, P, tp.data_ptr(), _stream_ptr()), "bc_planes_to_tp")
        e = _lib.TP_PLANE_ELEMS
        return tp, ((step * e, e) if sliding else (self.obs_size * e, e))

    def check_input(self, x):
        if isinstance(x, StagedBatch):
            if not (self.conv_mode & 1) or x.frame_skip != self.obs_size or x.step not in (self.obs_size // 4, self.obs_size):
                raise ValueError("a StagedBatch feeds the bf16 tensor-core mode (precision='bf16'): frame_skip 4 for obs_size 4, "
                                 "stage_frames(frame_skip=12, step=3) for obs_size 12, or stage_gather's materialised windows")
            if x.device != self.device:
                raise RuntimeError(f"x is on {x.device}, parameters on {self.device}")
            return x
        _require_cuda(x, "x")
        if x.device != self.device:
            raise RuntimeError(f"x is on {x.device}, parameters on {self.device}")
        if x.dim() != 4 or x.shape[1] != self.obs_size or x.shape[2] != H or x.shape[3] != W:
            raise ValueError(f"x must be (B,{self.obs_size},{H},{W}) like nets.py:14, got {tuple(x.shape)}")
        if x.dtype not in (torch.float32, torch.bfloat16):
            x = x.float()
        esz = x.element_size()
        ok = (x.stride(3) == 1 and x.stride(2) == W and (x.stride(0) * esz) % 16 == 0 and (x.stride(1) * esz) % 16 == 0
              and x.data_ptr() % 16 == 0)
        return x if ok else x.contiguous()

    def ctx(self, b: StepBuffers, loss_scale: Optional[float] = None) -> _lib.BcCtx:
        c = _lib.BcCtx()
        c.obs_size, c.n_actions, c.batch = self.obs_size, self.n_actions, b.batch
        if b.x is None:
            c.x, c.x_dtype, c.x_stride_n, c.x_stride_c = None, _lib.BC_BF16_TP, 0, 0
        else:
            c.x_dtype = _lib.BC_F32 if b.x.dtype == torch.float32 else _lib.BC_BF16
            c.x_stride_n, c.x_stride_c = (b.x.stride(0), b.x.stride(1)) if b.batch else (0, 0)
            c.x = b.x.data_ptr()
        c.y = b.y.data_ptr() if b.y is not None else None
        c.params, c.grads = self.arena.data_ptr(), self.grads.data_ptr()
        for i in range(4):
            c.act[i], c.amax[i] = b.act[i].data_ptr(), b.amax[i].data_ptr()
        for i in range(3):
            c.gact[i] = b.gact[i].data_ptr() if b.gact else None
        c.ghead = b.ghead.data_ptr() if b.ghead is not None else None
        c.hid1, c.hid2 = b.hid1.data_ptr(), b.hid2.data_ptr()
        c.logits, c.dlogits, c.loss = b.logits.data_ptr(), b.dlogits.data_ptr(), b.loss.data_ptr()
        c.partials = self.partials.data_ptr()
        c.loss_scale = (1.0 / max(b.batch, 1)) if loss_scale is None else float(loss_scale)
        c.conv_mode = self.conv_mode
        for i in range(3):
            c.act_bf16[i] = b.act_bf16[i].data_ptr() if b.act_bf16 else None
        c.w_packed, c.err_flag = self.w_packed.data_ptr(), self.err_flag.data_ptr()
        if b.x_tp is not None:
            c.x_tp, (c.x_tp_stride_n, c.x_tp_stride_c) = b.x_tp.data_ptr(), b.x_tp_strides
        if self.grads_epoch is not None:
            c.grads_epoch, c.grads_stride = self.grads_epoch.data_ptr(), self.grads_stride
        if b.gact0_p8 is not None:
            c.gact0_p8, c.amax0_p8 = b.gact0_p8.data_ptr(), b.amax0_p8.data_ptr()
        if b.c1_acc is not None:
            c.c1_acc = b.c1_acc.data_ptr()
        return c

    def static_buffers(self, batch: int, x, y: Optional[torch.Tensor]) -> StepBuffers:
        """One persistent StepBuffers per batch size (training: with the backward buffers); only the input and label
        pointers are re-pointed. What a fixed-shape training loop uses instead of alloc() every step."""
        b = self._static.get(batch)
        if b is None:
            b = self._static[batch] = self.alloc(batch, x, y, True)
            return b
        staged = x if isinstance(x, StagedBatch) else None
        if staged is not None:
            b.x, b.x_tp, b.x_tp_strides = staged.x, staged.tp, (staged.step * _lib.TP_PLANE_ELEMS, _lib.TP_PLANE_ELEMS)
        else:
            b.x = x
            if (self.conv_mode & 1) and batch:
                # a plain batch in bf16 mode: converted per call into a persistent plane buffer (stable pointer for graphs)
                step = self.obs_size // 4
                sliding = x.stride(0) == step * H * W and x.stride(1) == H * W
                n_planes = step * (batch - 1) + self.obs_size if sliding else batch * self.obs_size
                own = getattr(b, "_tp_own", None)
                if own is None or own.shape[0] != n_planes:
                    own = b._tp_own = torch.empty((n_planes, _lib.TP_PLANE_ELEMS), dtype=torch.bfloat16, device=self.device)
                b.x_tp, b.x_tp_strides = self.to_tp(x, out=own)
        b.y = y
        return b

    def grad_view(self) -> torch.Tensor:
        """The arena-shaped buffer the backward of the current step writes (peer exchange: the half the epoch selects)."""
        return self.peer.current() if self.peer is not None else self.grads

    def grad_arena_at(self, ptr: int) -> Optional[torch.Tensor]:
        """The engine-owned arena-shaped gradient buffer starting at device address `ptr` (None if there is none): lets the
        optimiser recognise .grad tensors that are views of one arena and consume it without a copy."""
        cands = [self.grads] + (self._slots or []) + ([self._last_flat] if getattr(self, "_last_flat", None) is not None else [])
        if self.peer is not None:
            S = self.peer.stride
            cands = [self.peer.buf[:S], self.peer.buf[S:]] + cands[1:]
        for t in cands:
            if t.data_ptr() == ptr and t.numel() >= self.arena.numel():
                return t[:self.arena.numel()]
        return None

    def _views_of(self, flat: torch.Tensor, params):
        """Per-parameter views of an arena-shaped gradient buffer, cached per buffer address."""
        cache = self.__dict__.setdefault("_grad_views", {})
        key = flat.data_ptr()
        v = cache.get(key)
        if v is None:
            v = cache[key] = (flat, [flat[p._bc_offset:p._bc_offset + p.numel()].view(p.shape) for p in params])
        return v

    def next_grad_slot(self, params):
        """(arena, per-parameter views) for the next fused step. Two arenas alternate, so the .grad tensors of the previous
        step stay intact until zero_grad() drops them (Lightning runs training_step BEFORE zero_grad); should a live .grad
        still alias the arena about to be rewritten (gradient accumulation over more than two micro-steps), it is copied
        out first."""
        if self.peer is not None:
            flat = self.peer.current()
        else:
            if self._slots is None:
                self._slots = [self.grads, torch.zeros_like(self.grads)]
            self._slot_i ^= 1
            flat = self.grads = self._slots[self._slot_i]
        flat, views = self._views_of(flat, params)
        for p, v in zip(params, views):
            if p.grad is v:
                p.grad = v.clone()
        return flat, views

    def grads_as_arena(self, params) -> Optional[torch.Tensor]:
        """The gradient arena whose cached views ARE the .grad tensors of `params` (identity), else None."""
        first = params[0].grad
        if first is None:
            return None
        for flat, views in self.__dict__.get("_grad_views", {}).values():
            if views[0] is first:
                return flat if all(p.grad is v for p, v in zip(params, views)) else None
        return None

    def side_handles(self):
        """(side stream, events, ctypes void*[4]) of the overlapped backward; created outside any graph capture."""
        if self._side is None:
            if torch.cuda.is_current_stream_capturing():
                raise RuntimeError("create the engine's side stream before capturing (run one eager step first)")
            with on_device(self.device):
                # torch hands out pool streams round robin, 32 per priority: a default-priority side stream becomes the
                # CUDA-graph capture stream again once 32 more streams have been created (one per SequentialFrames
                # loader), and bc_backward_overlap refuses side == main. The high-priority pool holds no such stream.
                side = torch.cuda.Stream(self.device, priority=-1)
                evs = [torch.cuda.Event() for _ in range(4)]
                for e in evs:
                    e.record()                      # torch creates the cudaEvent lazily: force it now
                arr = (C.c_void_p * 4)(*[e.cuda_event for e in evs])
            self._side = (side, evs, arr)
        return self._side

    def set_mode(self, mode: str) -> None:
        """'fp32' = exact FFMA kernels (rel 1e-5); 'bf16' = tcgen05 kernels on bf16-staged frames (rel 2e-2)."""
        self.conv_mode = {"fp32": 0, "bf16": 31}[mode]     # 31 = every tcgen05 kernel + the compact conv1 gradient path

    def pack_weights(self) -> None:
        """Derive the bf16 operand images from the f32 master weights (one launch). The fused Adam kernels keep the images
        current afterwards (bc_adam_tick_step / bc_adam_step_exchange with w_packed), so a training loop calls this once."""
        c = _lib.BcCtx()
        c.obs_size, c.n_actions = self.obs_size, self.n_actions
        c.params, c.w_packed = self.arena.data_ptr(), self.w_packed.data_ptr()
        with on_device(self.device):
            _lib.check(self.lib.bc_pack_weights(C.byref(c), _stream_ptr()), "bc_pack_weights")
        self._packed_version = self.weights_version()

    def ensure_packed(self) -> None:
        """Re-pack only when the master weights changed behind the kernels' back (torch in-place ops bump the version
        counters: load_state_dict, p.copy_, p.data.add_, a foreign optimiser). FusedAdam refreshes the images itself."""
        if self.conv_mode and self._packed_version != self.weights_version():
            self.pack_weights()

    def packed_ptr(self) -> Optional[int]:
        """w_packed for the optimiser kernels: the images follow the weights only in bf16 mode."""
        return self.w_packed.data_ptr() if self.conv_mode else None

    _ERRORS = {1: "a tcgen05 pipeline wait timed out inside a kernel (mbarrier protocol error)",
               3: "a label outside [0, n_actions) reached the CrossEntropy kernel (nn.CrossEntropyLoss raises on it too)",
               4: "a command outside [0, n_branches) reached the branched heads (its output and gradient rows are zero)",
               5: "a sample index outside [0, n_frames - 5] reached bc_stage_gather (its planes and side data are zero)"}

    def check_device_errors(self) -> None:
        """Host-side check of the device error flag (synchronises; call outside the hot loop, e.g. at epoch end)."""
        code = int(self.err_flag.item())
        if code != 0:
            self.err_flag.zero_()
            raise RuntimeError(self._ERRORS.get(code, f"device error flag {code}"))

    # ------------------------------------------------------------------ kernels
    def forward(self, x: torch.Tensor, y: Optional[torch.Tensor] = None, backward: bool = False,
                loss_scale: Optional[float] = None) -> StepBuffers:
        """conv1..4 (+ReLU+pool) and the head; with `y` also CE loss and dlogits, in the same head launch."""
        x = self.check_input(x)
        self.ensure_packed()
        if y is not None:
            _require_cuda(y, "y")
            if y.dtype != torch.int64 or y.shape != (x.shape[0],):
                raise ValueError("y must be (B,) int64 class ids (imitation_dataset.py:131)")
            y = y.contiguous()
        b = self.alloc(x.shape[0], x, y, backward)
        c = self.ctx(b, loss_scale)
        s = _stream_ptr()
        with on_device(self.device):
            for layer in range(4):
                _lib.check(self.lib.bc_conv_relu_pool_fwd(C.byref(c), layer, s), f"conv{layer + 1} forward")
            _lib.check(self.lib.bc_head(C.byref(c), 1 if y is not None else 0, s), "head forward")
            if y is not None:
                _lib.check(self.lib.bc_loss_reduce(C.byref(c), s), "loss reduce")
        return b

    def backward(self, b: StepBuffers, loss_scale: Optional[float] = None) -> torch.Tensor:
        """Gradients of every parameter from b.dlogits (already holding d loss / d logits). Returns self.grads."""
        self._alloc_bwd(b)
        c = self.ctx(b, loss_scale)
        with on_device(self.device):
            _lib.check(self.lib.bc_backward(C.byref(c), 0, _stream_ptr()), "bc_backward")
        return self.grads

    def train_forward_backward(self, x: torch.Tensor, y: torch.Tensor, loss_scale: Optional[float] = None) -> StepBuffers:
        """Forward, CE loss and full backward in one enqueue (no autograd). grads land in self.grads."""
        x = self.check_input(x)
        self.ensure_packed()
        b = self.alloc(x.shape[0], x, y.contiguous(), True)
        self.enqueue_train(b, loss_scale)
        return b

    def _check_labels(self, b: StepBuffers) -> None:
        y = b.y
        if y is None or not y.is_cuda or y.dtype != torch.int64 or tuple(y.shape) != (b.batch,) or not y.is_contiguous():
            raise ValueError("y must be a contiguous (B,) int64 CUDA tensor of class ids (imitation_dataset.py:131)")

    def enqueue_train(self, b: StepBuffers, loss_scale: Optional[float] = None, dp_split: bool = False) -> None:
        """Forward, CE loss and the whole backward on the current stream (gradients -> self.grads). With self.overlap the
        weight-gradient kernels of conv4..conv2 run on the engine's side stream under the dgrad chain; dp_split is the
        data-parallel variant (parallel.PeerExchangeStep): [fc..conv2] reduced on the side stream, join left to the caller."""
        self._check_labels(b)
        c = self.ctx(b, loss_scale)
        s = _stream_ptr()
        with on_device(self.device):
            for layer in range(4):   # the head's forward is fused into bc_backward's first launch
                _lib.check(self.lib.bc_conv_relu_pool_fwd(C.byref(c), layer, s), f"conv{layer + 1} forward")
            if self.overlap or dp_split:
                side, _evs, arr = self.side_handles()
                flags = (1 if dp_split else 0) | (0 if self.overlap else 2)
                _lib.check(self.lib.bc_backward_overlap(C.byref(c), 1, s, side.cuda_stream, arr, flags), "bc_backward_overlap")
            else:
                _lib.check(self.lib.bc_backward(C.byref(c), 1, s), "bc_backward")

    def enqueue_trunk_forward(self, b: StepBuffers) -> None:
        """conv1..4 (+ReLU+pool) of b's input into b.act on the current stream; no head (the branched heads follow)."""
        c = self.ctx(b)
        s = _stream_ptr()
        with on_device(self.device):
            for layer in range(4):
                _lib.check(self.lib.bc_conv_relu_pool_fwd(C.byref(c), layer, s), f"conv{layer + 1} forward")

    def enqueue_trunk_backward(self, b: StepBuffers) -> None:
        """The conv trunk's backward from b.ghead (d loss / d act4, written by a head of the caller's: the branched heads)
        on the current stream: weight and input gradients of conv4..conv2, conv1's weight gradient, and the reduction of
        their partials into the engine's gradient arena. The arena's fc head segment is left untouched."""
        c = self.ctx(b)
        s = _stream_ptr()
        with on_device(self.device):
            for layer in (3, 2, 1):
                _lib.check(self.lib.bc_conv_bwd_wgrad(C.byref(c), layer, s), "wgrad")
                _lib.check(self.lib.bc_conv_bwd_dgrad(C.byref(c), layer, s), "dgrad")
            _lib.check(self.lib.bc_conv_bwd_wgrad(C.byref(c), 0, s), "conv1 wgrad")
            _lib.check(self.lib.bc_reduce_partials_range(C.byref(c), 1, 5, 0, s), "reduce [conv4..conv1]")

    tail_batch = 8       # serving: up to this batch conv3..head + argmax run as ONE cluster launch (bc_policy_tail). Measured crossover
                         # (bench.py --workload infer, profiles/r2G): 20.6-22.3 us against 26.3-26.6 us up to B = 8, 30.6 against 28.6 at B = 16

    def forward_act(self, x, out: Optional[torch.Tensor] = None, bufs: Optional[StepBuffers] = None,
                    tail: Optional[bool] = None):
        """The serving forward (imitation.py:34-36 + the argmax of src/data/stat.py:41): logits AND greedy actions without a
        separate argmax launch; at small batch conv3, conv4, the head and the argmax are one launch (csrc/policy_tail.cu).
        Returns (actions (B,) int64, StepBuffers with .logits). `bufs` = persistent buffers (eng.alloc(B, x, None, False)) for
        a fixed-shape serving loop / CUDA graph; `tail` forces the path (None = by batch size)."""
        x = self.check_input(x)
        self.ensure_packed()
        B = x.shape[0]
        b = bufs if bufs is not None else self.alloc(B, x, None, False)
        if b.batch != B or (out is not None and (out.dtype != torch.int64 or out.numel() != B or not out.is_cuda)):
            raise ValueError(f"bufs / out were built for another batch (x has {B} samples): out is (B,) int64 on the device")
        if bufs is not None:                     # persistent buffers: only the input is re-pointed
            staged = x if isinstance(x, StagedBatch) else None
            if staged is not None:
                b.x, b.x_tp, b.x_tp_strides = staged.x, staged.tp, (staged.step * _lib.TP_PLANE_ELEMS, _lib.TP_PLANE_ELEMS)
            elif self.conv_mode & 1:
                raise ValueError("persistent serving buffers in bf16 mode take a StagedBatch (stage_frames(out=...)): a plain batch would be re-converted per call")
            else:
                b.x = x
        if out is None:
            out = torch.empty(B, dtype=torch.int64, device=self.device)
        if B == 0:
            return out, b
        if tail is None:
            tail = B <= self.tail_batch
        if tail and B > _lib.POLICY_TAIL_MAX_BATCH:
            raise ValueError(f"the one-launch tail serves batches up to {_lib.POLICY_TAIL_MAX_BATCH}")
        c = self.ctx(b)
        with on_device(self.device):
            _lib.check(self.lib.bc_forward_act(C.byref(c), out.data_ptr(), int(bool(tail)), _stream_ptr()), "bc_forward_act")
        return out, b

    def argmax(self, logits: torch.Tensor) -> torch.Tensor:
        out = torch.empty(logits.shape[0], dtype=torch.int64, device=logits.device)
        _lib.check(self.lib.bc_argmax(logits.data_ptr(), out.data_ptr(), logits.shape[0], logits.shape[1], _stream_ptr()), "bc_argmax")
        return out
