"""B200-native behaviour-cloning hot path (ConvNet1 forward/backward, CE loss, Adam, DDP exchange)
behind the module/constructor contract of HemuManju/carla-imitation-learning.

Everything numeric runs in the hand-written sm_100a kernels of csrc/ through the C ABI in
include/bc_b200.h; this package is the thin host side (buffers, streams, autograd glue)."""
from . import _lib  # noqa: F401
from .engine import BCEngine, StagedBatch, StepBuffers, stage_augmented, stage_frames, stage_gather, stage_gray, sliding_window  # noqa: F401
from .optim import FusedAdam  # noqa: F401

__all__ = ["BCEngine", "StagedBatch", "StepBuffers", "FusedAdam", "stage_augmented", "stage_frames", "stage_gather", "stage_gray", "sliding_window"]
