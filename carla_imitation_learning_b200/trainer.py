"""The training loop around the hot path: what `pl.Trainer(gpus=..., max_epochs=...).fit(model)` does for the
behaviour-cloning block of the reference (/root/reference/train.py:106-129), for boxes without Lightning.

Three layers:

* TrainStep -- one optimisation step for a static batch shape, straight on the engine (no autograd): stage -> conv1..4 ->
  head + CE -> backward -> [peer exchange] -> Adam as ONE CUDA graph per input slot. This is what bench.py times as `value`
  and what Trainer.fit uses when the module is a ConvNet1-backed Imitation with `cuda_graph: true`.
* BranchedTrainStep -- the same for the command-conditioned ConvNet1Branched (one GPU): stage [+ augment] -> conv1..4 ->
  branched heads + CE / L1 / MSE -> trunk backward -> Adam on the trunk and the branch arena, one CUDA graph per input slot.
* BranchedActStep -- its serving counterpart: stage [+ centre crop] -> conv1..4 -> the commanded branches -> greedy action,
  with the one-launch tail at small batch, one CUDA graph per input slot.
* Trainer -- epochs over model.train_dataloader() / val_dataloader() with the LightningModule hook order
  (training_step -> zero_grad -> backward -> optimizer.step; validation_step; *_epoch_end; scheduler.step once per epoch
  from training_epoch_end, imitation.py:57-60), ModelCheckpoint(monitor='val_loss', mode='min') in Lightning's .ckpt layout
  (train.py:106-111, 198-201), data parallel = one process per GPU with the fused peer exchange or NCCL buckets
  (configs/trainer/b200_ddp.yaml: strategy / ddp_backend / ddp_exchange).
"""
from __future__ import annotations

import os
from typing import Callable, Dict, List, Optional

import torch
import torch.distributed as dist

from . import _lib
from .engine import BCEngine, StagedBatch, StepBuffers, stage_augmented, stage_frames, stage_gray, sliding_window
from .optim import FusedAdam


class TrainStep:
    """stage -> forward -> backward -> [exchange] -> Adam on one engine, captured per input slot.

    `step(frames_u8, labels)`: frames (B+frame_skip, 256, 256, 3) u8 and labels (B,) int64 already on the device. The
    first call for a given (frames, labels) buffer pair runs eagerly, the second captures a CUDA graph, later calls
    replay it -- so a caller that rotates over a few device slots pays one graph launch per step."""

    def __init__(self, net, optimizer: FusedAdam, batch: int, *, group=None, exchange: Optional[str] = None,
                 overlap: Optional[bool] = None, graph: bool = True, dp_overlap: bool = False):
        self.net, self.opt, self.batch, self.graph = net, optimizer, int(batch), graph
        self.eng: BCEngine = net.engine()
        if overlap is not None:
            self.eng.overlap = bool(overlap)
        eng = self.eng
        self.bf16 = bool(eng.conv_mode)
        dev = eng.device
        B = self.batch
        if self.bf16:
            self.staged = StagedBatch(torch.empty((B + 4, _lib.TP_PLANE_ELEMS), dtype=torch.bfloat16, device=dev), None, 4)
            self.bufs: StepBuffers = eng.alloc(B, self.staged, torch.zeros(B, dtype=torch.int64, device=dev), True)
        else:
            self.gray = torch.empty((B + 4, 256, 256), dtype=torch.float32, device=dev)
            self.bufs = eng.alloc(B, sliding_window(self.gray), torch.zeros(B, dtype=torch.int64, device=dev), True)
        self.dp = None
        world = dist.get_world_size(group) if dist.is_initialized() else 1
        if world > 1:
            from .parallel import DataParallelStep, PeerExchangeStep
            kind = exchange or "peer"
            if kind not in ("peer", "nccl"):
                raise ValueError("ddp_exchange is 'peer' (fused into the Adam kernel over NVLink peer memory) or 'nccl'")
            self.dp = PeerExchangeStep(eng, optimizer, group, overlap=dp_overlap) if kind == "peer" else DataParallelStep(eng, optimizer, group)
        self.world = world
        optimizer.prepare()
        if eng.overlap:
            eng.side_handles()
        self._seen, self._graphs = set(), {}

    # ------------------------------------------------------------------ pieces
    def _stage(self, frames_u8: torch.Tensor) -> None:
        if self.bf16:
            stage_frames(frames_u8, out=self.staged)
        else:
            stage_gray(frames_u8, out=self.gray)

    def _enqueue(self, frames_u8: torch.Tensor, labels: torch.Tensor) -> None:
        self._stage(frames_u8)
        self.bufs.y = labels
        if self.dp is not None:
            self.dp(self.bufs)
        else:
            self.eng.enqueue_train(self.bufs)
            self.opt.step_flat(self.eng.grads)

    # ------------------------------------------------------------------ step
    def step(self, frames_u8: torch.Tensor, labels: torch.Tensor) -> torch.Tensor:
        """Enqueue one optimisation step; returns the (device) loss cell, rewritten by the next step."""
        if frames_u8.shape[0] != self.batch + 4 or labels.shape[0] != self.batch:
            raise ValueError(f"TrainStep was built for {self.batch} samples ({self.batch + 4} frames)")
        self.eng.ensure_packed()
        key = (frames_u8.data_ptr(), labels.data_ptr())
        g = self._graphs.get(key) if self.graph else None
        if g is not None:
            self._replay(g)
        elif self.graph and key in self._seen:
            g = self._graphs[key] = self._capture(frames_u8, labels)
            self._replay(g)
        else:
            self._seen.add(key)
            self._enqueue(frames_u8, labels)
        return self.bufs.loss

    def _capture(self, frames_u8, labels):
        from .parallel import DataParallelStep
        self.opt.prepare()
        if isinstance(self.dp, DataParallelStep):        # NCCL stays outside the graphs: three segments
            def pre():
                self._stage(frames_u8)
                self.bufs.y = labels
            return self.dp.capture(self.bufs, pre)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            self._enqueue(frames_u8, labels)
        return g

    def _replay(self, g) -> None:
        from .parallel import DataParallelStep
        if isinstance(self.dp, DataParallelStep):
            self.dp.replay(g)
            return
        self.opt.prepare()            # an LR milestone reaches the device scalar the captured kernels read
        g.replay()
        if self.dp is not None:
            self.dp.peer.host_epoch += 1

    def check(self) -> None:
        """Raise if a device-side bounded wait expired or a label was out of range (synchronises)."""
        self.eng.check_device_errors()
        if self.dp is not None and hasattr(self.dp, "peer"):
            self.dp.peer.check()


class _BranchedInput:
    """The input side BranchedTrainStep and BranchedActStep share: a ConvNet1Branched at a static batch, its staging buffer
    (f32 planes, or Toeplitz-ready bf16 planes in bf16 mode) and trunk buffers, the checks of frames / table / command, and
    the staging pass (plain, or crop + jitter + normalise from src_hw sources through a device table)."""

    def _init_input(self, net, batch: int, src_hw, backward: bool) -> None:
        self.net, self.batch = net, int(batch)
        if self.batch < 1:
            raise ValueError("batch must be at least 1")
        self.src_hw = None if src_hw is None else (int(src_hw[0]), int(src_hw[1]))
        if self.src_hw is not None and (self.src_hw[0] < 256 or self.src_hw[1] < 256):
            raise ValueError(f"source frames {self.src_hw} are smaller than the 256x256 crop")
        self.eng: BCEngine = net.engine()
        eng, dev, B = self.eng, self.eng.device, self.batch
        if eng.obs_size != 4:
            raise ValueError(f"{type(self).__name__} stages 4-frame windows: obs_size must be 4")
        if not net._barena.is_cuda or net._barena.device != dev:
            raise RuntimeError("the branch arena must live on the trunk's device (net.to(device))")
        self.bf16 = bool(eng.conv_mode)
        if self.bf16:
            self.staged = StagedBatch(torch.empty((B + 4, _lib.TP_PLANE_ELEMS), dtype=torch.bfloat16, device=dev), None, 4)
            self.bufs: StepBuffers = eng.alloc(B, self.staged, None, backward)
        else:
            self.gray = torch.empty((B + 4, 256, 256), dtype=torch.float32, device=dev)
            self.bufs = eng.alloc(B, sliding_window(self.gray), None, backward)

    def _check_input(self, frames_u8, table, command) -> None:
        B, dev = self.batch, self.eng.device
        hw = self.src_hw or (256, 256)
        for t, what in ((frames_u8, "frames"), (command, "command")):
            if not isinstance(t, torch.Tensor) or t.device != dev:
                raise ValueError(f"{what} must be a tensor on {dev}")
        if frames_u8.dtype != torch.uint8 or tuple(frames_u8.shape) != (B + 4, *hw, 3) or not frames_u8.is_contiguous():
            raise ValueError(f"frames must be a contiguous ({B + 4}, {hw[0]}, {hw[1]}, 3) uint8 tensor")
        if self.src_hw is None:
            if table is not None:
                raise ValueError("this step was built without augmentation (src_hw=None): table must be None")
        elif (not isinstance(table, torch.Tensor) or table.device != dev or table.dtype != torch.float32
              or tuple(table.shape) != (B + 4, 8) or not table.is_contiguous()):
            raise ValueError(f"table must be a contiguous ({B + 4}, 8) float32 tensor on {dev} (data.augment_table rows)")
        if command.dtype != torch.int64 or tuple(command.shape) != (B,) or not command.is_contiguous():
            raise ValueError(f"command must be a contiguous ({B},) int64 tensor of branch ids")

    def _stage(self, frames_u8, table) -> None:
        if self.src_hw is not None:
            stage_augmented(frames_u8, table, layout="tp" if self.bf16 else "plain", out=self.staged if self.bf16 else self.gray)
        elif self.bf16:
            stage_frames(frames_u8, out=self.staged)
        else:
            stage_gray(frames_u8, out=self.gray)


class BranchedTrainStep(_BranchedInput):
    """stage [+ augment] -> conv1..4 -> branched heads + loss + backward -> trunk backward -> Adam on both arenas, for a
    ConvNet1Branched and its MultiArenaAdam at a static batch, captured per input slot like TrainStep.

    `step(frames_u8, table, command, target)`, all on the device: frames (B+4, Hs, Ws, 3) u8; table (B+4, 8) f32 rows of
    data.augment_table when the step was built with src_hw = (Hs, Ws) (crop + colour jitter + normalise in the staging
    kernel), None when src_hw is None (plain staging of 256x256 frames); command (B,) int64 branch ids; target (B,) int64
    class ids for branch_loss 'ce', (B, n_out) f32 for 'l1' / 'mse'. The first call for a given buffer tuple runs
    eagerly, the second captures a CUDA graph, later calls replay it. Returns the device loss cell, rewritten by the next
    step. Nothing in step() synchronises the host; check() does."""

    def __init__(self, net, optimizer, batch: int, *, src_hw=None, graph: bool = True, group=None):
        if dist.is_initialized() and dist.get_world_size(group) > 1:
            raise RuntimeError("BranchedTrainStep trains on one GPU: data-parallel training of the branched policy is not "
                               "supported (the peer exchange drives a single parameter arena)")
        children = getattr(optimizer, "children_", None)
        if (children is None or len(children) != 2 or children[0]._arena_of is not net
                or children[1]._arena_of is not net._bowner):
            raise ValueError("BranchedTrainStep takes the net's MultiArenaAdam (net.configure_optimizer())")
        self.opt, self.graph = optimizer, graph
        self.trunk_opt, self.branch_opt = children
        self._init_input(net, batch, src_hw, True)
        B, dev = self.batch, self.eng.device
        n_part = int(_lib.lib().bc_head_branched_partials_floats(net.n_branches, net.n_actions))
        f32 = dict(dtype=torch.float32, device=dev)
        self.hb = dict(out=torch.empty((B, net.n_actions), **f32), dout=torch.empty((B, net.n_actions), **f32),
                       loss=torch.zeros((), **f32), grads=torch.zeros_like(net._barena),
                       partials=torch.zeros(n_part, **f32))     # partial pads are never written: zeroed once
        optimizer.prepare()
        self._seen, self._graphs = set(), {}

    # ------------------------------------------------------------------ pieces
    def _check_inputs(self, frames_u8, table, command, target) -> None:
        B, dev = self.batch, self.eng.device
        self._check_input(frames_u8, table, command)
        if not isinstance(target, torch.Tensor) or target.device != dev:
            raise ValueError(f"target must be a tensor on {dev}")
        if self.net.branch_loss == "ce":
            if target.dtype != torch.int64 or tuple(target.shape) != (B,) or not target.is_contiguous():
                raise ValueError(f"CE targets are a contiguous ({B},) int64 tensor of class ids")
        elif target.dtype != torch.float32 or tuple(target.shape) != (B, self.net.n_actions) or not target.is_contiguous():
            raise ValueError(f"{self.net.branch_loss} targets are a contiguous ({B}, {self.net.n_actions}) float32 tensor")

    def _enqueue(self, frames_u8, table, command, target) -> None:
        self._stage(frames_u8, table)
        self.eng.enqueue_trunk_forward(self.bufs)
        self.net._head(self.bufs, self.hb, command, target, 3)      # outputs, loss, dout, branch gradients, ghead
        self.eng.enqueue_trunk_backward(self.bufs)
        self.trunk_opt.step_flat(self.eng.grads)
        self.branch_opt.step_flat(self.hb["grads"])

    # ------------------------------------------------------------------ step
    def step(self, frames_u8: torch.Tensor, table: Optional[torch.Tensor], command: torch.Tensor,
             target: torch.Tensor) -> torch.Tensor:
        """Enqueue one optimisation step; returns the (device) loss cell, rewritten by the next step."""
        self._check_inputs(frames_u8, table, command, target)
        self.eng.ensure_packed()
        key = (frames_u8.data_ptr(), None if table is None else table.data_ptr(), command.data_ptr(), target.data_ptr())
        g = self._graphs.get(key) if self.graph else None
        if g is None and self.graph and key in self._seen:
            self.opt.prepare()
            g = self._graphs[key] = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._enqueue(frames_u8, table, command, target)
        if g is not None:
            self.opt.prepare()            # an LR milestone reaches the device scalars the captured Adam kernels read
            g.replay()
        else:
            self._seen.add(key)
            self.opt.prepare()
            self._enqueue(frames_u8, table, command, target)
        return self.hb["loss"]

    @property
    def out(self) -> torch.Tensor:
        """(B, n_out) outputs of the commanded branches in the last step (before its update)."""
        return self.hb["out"]

    def check(self) -> None:
        """Raise if a device-side bounded wait expired, a label (CE) or a command was out of range (synchronises)."""
        self.eng.check_device_errors()


class BranchedActStep(_BranchedInput):
    """The serving counterpart of BranchedTrainStep: stage [+ centre crop] -> the policy forward of a ConvNet1Branched ->
    the commanded branches' outputs and, for branch_loss 'ce', the greedy actions, at a static batch, on persistent buffers.

    `act(frames_u8, table, command)`, all on the device: frames (B+4, Hs, Ws, 3) u8; table (B+4, 8) f32 rows when built with
    src_hw = (Hs, Ws) -- data.center_crop_table(B + 4, src_hw, mean, std) serves a policy trained on augment_table rows --
    else None; command (B,) int64 branch ids. Returns (out (B, n_out) f32, actions (B,) int64 or None for 'l1' / 'mse'),
    both persistent, rewritten by the next call. Up to net.tail_batch samples, conv3, conv4 and the head run as one
    cluster launch (bc_policy_tail_branched). The first call for a given buffer tuple runs eagerly, the second captures a
    CUDA graph, later calls replay it. The graph holds the command buffer's ADDRESS: the kernels read its contents on
    every replay, so a caller rewrites it in place per tick (a host copy or a torch op on the stream) and needs no new
    graph. Nothing in act() synchronises the host; check() does."""

    def __init__(self, net, batch: int, *, src_hw=None, graph: bool = True):
        self.graph = graph
        self._init_input(net, batch, src_hw, False)
        B, dev = self.batch, self.eng.device
        self.tail = B <= net.tail_batch
        self.out = torch.empty((B, net.n_actions), dtype=torch.float32, device=dev)
        self.actions = torch.empty(B, dtype=torch.int64, device=dev) if net.branch_loss == "ce" else None
        self._seen, self._graphs = set(), {}

    def _enqueue(self, frames_u8, table, command) -> None:
        self._stage(frames_u8, table)
        self.net._serve(self.bufs, self.out, self.actions, command, self.tail)

    def act(self, frames_u8: torch.Tensor, table: Optional[torch.Tensor], command: torch.Tensor):
        """Enqueue one serving forward; returns (out, actions or None)."""
        self._check_input(frames_u8, table, command)
        self.eng.ensure_packed()
        key = (frames_u8.data_ptr(), None if table is None else table.data_ptr(), command.data_ptr())
        g = self._graphs.get(key) if self.graph else None
        if g is None and self.graph and key in self._seen:
            g = self._graphs[key] = torch.cuda.CUDAGraph()
            with torch.no_grad(), torch.cuda.graph(g):
                self._enqueue(frames_u8, table, command)
        if g is not None:
            g.replay()
        else:
            self._seen.add(key)
            with torch.no_grad():
                self._enqueue(frames_u8, table, command)
        return self.out, self.actions

    def check(self) -> None:
        """Raise if a device-side bounded wait expired or a command was out of range (synchronises)."""
        self.eng.check_device_errors()


def arena_checksum(arena: torch.Tensor) -> int:
    """Position-weighted fingerprint of the parameter arena's BITS (reported next to the replica check)."""
    bits = arena.detach().contiguous().view(torch.int32).to(torch.int64) & 0xFFFFFFFF
    idx = torch.arange(1, bits.numel() + 1, dtype=torch.int64, device=bits.device)
    return int(((bits * 40503 + idx * 2654435761) % 2147483647).sum().item())


def replicas_identical(arena: torch.Tensor, group=None) -> bool:
    """All ranks hold bitwise the same parameters (the rank-ordered peer sum guarantees it; this verifies it by
    gathering every replica's arena -- 533 KB each -- and comparing the bits)."""
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return True
    mine = arena.detach().contiguous().view(torch.int32)
    allv = [torch.empty_like(mine) for _ in range(dist.get_world_size(group))]
    dist.all_gather(allv, mine, group=group)
    return all(bool(torch.equal(v, allv[0])) for v in allv)


class Trainer:
    """fit(model): the hook order and checkpoint layout of pl.Trainer for the reference's BC block."""

    def __init__(self, max_epochs: int = 50, default_root_dir: Optional[str] = None, limit_train_batches: Optional[int] = None,
                 limit_val_batches: Optional[int] = None, monitor: str = "val_loss", ddp_exchange: str = "peer",
                 ddp_backend: str = "nccl", strategy: str = "ddp", check_errors_every_n_epochs: int = 1, **_ignored):
        if strategy != "ddp":
            raise ValueError("the BC policy (133 K parameters) trains data-parallel only: strategy must be 'ddp'")
        self.max_epochs, self.root = int(max_epochs), default_root_dir
        self.limit_train_batches, self.limit_val_batches = limit_train_batches, limit_val_batches
        self.monitor, self.ddp_exchange, self.ddp_backend = monitor, ddp_exchange, ddp_backend
        self.check_every = max(1, int(check_errors_every_n_epochs))
        self.current_epoch, self.global_step = 0, 0
        self.best_score: Optional[float] = None
        self.best_model_path: Optional[str] = None
        self.callback_metrics: Dict[str, torch.Tensor] = {}

    @classmethod
    def from_hparams(cls, hparams, **kw):
        """Built from the configs/trainer + configs/model keys (max_epochs / NUM_EPOCHS, ddp_exchange, ...)."""
        get = (lambda k, d=None: hparams[k] if k in hparams else d)
        return cls(max_epochs=get("max_epochs", get("NUM_EPOCHS", 50)), default_root_dir=get("default_root_dir"),
                   ddp_exchange=get("ddp_exchange", "peer"), ddp_backend=get("ddp_backend", "nccl"),
                   strategy=get("strategy", "ddp"), **kw)

    # ------------------------------------------------------------------ fit
    def fit(self, model) -> None:
        optimizers, schedulers = model.configure_optimizers()
        opt, self._opt, self._schedulers = optimizers[0], optimizers[0], schedulers
        net = getattr(model, "net", None)
        world = dist.get_world_size() if dist.is_initialized() else 1
        if world > 1:
            if not isinstance(opt, FusedAdam):
                raise RuntimeError("data-parallel training needs the arena-backed FusedAdam (ConvNet1 parameters)")
            if self.ddp_exchange == "peer":
                from .parallel import ModuleExchange
                ModuleExchange(net.engine(), opt)
            else:
                from .parallel import GradExchange
                xchg = GradExchange(net.obs_size, net.n_actions)
                opt.set_grad_scale(xchg.grad_scale)
                opt.exchange = _NcclModuleExchange(opt, xchg)
        model.trainer = self
        for epoch in range(self.current_epoch, self.max_epochs):
            self.current_epoch = model.current_epoch = epoch
            outputs: List[dict] = []
            for i, batch in enumerate(model.train_dataloader()):
                if self.limit_train_batches is not None and i >= self.limit_train_batches:
                    break
                loss = model.training_step(batch, i)
                opt.zero_grad()
                loss.backward()
                opt.step()
                outputs.append({"loss": loss.detach()})
                self.global_step += 1
            model.training_epoch_end(outputs)
            val_out = []
            vl = model.val_dataloader() if "val_dataloader" in getattr(model, "data_loader", {}) else None
            if vl is not None:
                for i, batch in enumerate(vl):
                    if self.limit_val_batches is not None and i >= self.limit_val_batches:
                        break
                    val_out.append(model.validation_step(batch, i))
                if val_out:
                    model.validation_epoch_end(val_out)
                    self.callback_metrics[self.monitor] = torch.stack([v.detach() for v in val_out]).mean()
            if (epoch + 1) % self.check_every == 0 and net is not None and hasattr(net, "engine"):
                net.engine().check_device_errors()
                if getattr(net.engine(), "peer", None) is not None:
                    net.engine().peer.check()
            if self.root and self.monitor in self.callback_metrics and (not dist.is_initialized() or dist.get_rank() == 0):
                score = float(self.callback_metrics[self.monitor])
                if self.best_score is None or score < self.best_score:
                    self.best_score = score
                    self.best_model_path = os.path.join(self.root, "imitation.ckpt")   # ModelCheckpoint(filename='imitation'), train.py:106-111
                    self.save_checkpoint(model, self.best_model_path)
        self.current_epoch = self.max_epochs

    # ------------------------------------------------------------------ checkpoints (Lightning layout)
    def save_checkpoint(self, model, path: str) -> None:
        os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
        ckpt = {
            "epoch": self.current_epoch, "global_step": self.global_step, "pytorch-lightning_version": "1.3.8",
            "state_dict": {k: v.detach().cpu().clone() for k, v in model.state_dict().items()},
            "optimizer_states": [_to_cpu(self._opt.state_dict())] if getattr(self, "_opt", None) is not None else [],
            "lr_schedulers": [s.state_dict() for s in getattr(self, "_schedulers", [])],
            "callbacks": {"ModelCheckpoint": {"monitor": self.monitor, "best_model_score": self.best_score,
                                              "best_model_path": self.best_model_path}},
        }
        torch.save(ckpt, path)


class _NcclModuleExchange:
    """NCCL all-reduce of the arena-shaped gradients, then the fused Adam (module path, ddp_exchange: nccl)."""

    def __init__(self, opt, xchg):
        self.opt, self.xchg = opt, xchg

    def step_from(self, flat_grads: torch.Tensor) -> None:
        self.xchg.all(flat_grads)
        self.opt.step_flat(flat_grads)


def _to_cpu(obj):
    if torch.is_tensor(obj):
        return obj.detach().cpu().clone()
    if isinstance(obj, dict):
        return {k: _to_cpu(v) for k, v in obj.items()}
    if isinstance(obj, (list, tuple)):
        return type(obj)(_to_cpu(v) for v in obj)
    return obj


def load_checkpoint_into(model, path: str, optimizer=None, schedulers=None, strict: bool = True) -> dict:
    """`Imitation.load_from_checkpoint(path, hparams=, net=, data_loader=)` (train.py:198-201) for a module that has
    already been constructed: model weights, and optionally the optimiser / scheduler state, from a Lightning .ckpt
    (written by Trainer.save_checkpoint here or by the reference's ModelCheckpoint: same keys)."""
    ckpt = torch.load(path, map_location="cpu", weights_only=False)
    model.load_state_dict(ckpt["state_dict"], strict=strict)
    if optimizer is not None and ckpt.get("optimizer_states"):
        optimizer.load_state_dict(ckpt["optimizer_states"][0])
    if schedulers is not None:
        for s, sd in zip(schedulers, ckpt.get("lr_schedulers", [])):
            s.load_state_dict(sd)
    return ckpt
