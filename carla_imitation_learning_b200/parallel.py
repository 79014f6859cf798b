"""Data-parallel gradient exchange for the BC step: one process per GPU, NCCL over NVLink.

The reference gets data parallelism implicitly from `pl.Trainer(gpus=[0..n-1])`
(/root/reference/train.py:125, /root/reference/utils.py:60-64), i.e. torch DDP averaging the
533 KB of gradients. Here the gradients already live in ONE flat arena ordered by reverse
completion time [fc | conv4 | conv3 | conv2 || conv1], so the exchange is two all-reduces:
  bucket 0 = everything except conv1 (ready before conv1's wgrad, which is the longest backward
             kernel, starts)  -> reduced while conv1-wgrad runs
  bucket 1 = conv1 (12.7 KB)
and the 1/world mean is folded into the fused Adam's gradient read (FusedAdam.set_grad_scale),
so no separate scaling pass exists. No model sharding: 133 K parameters replicate.

The bucket arithmetic and the exchange are backend-agnostic (tested with gloo on CPU tensors);
on the GPU the all-reduce is NCCL and overlaps with compute because torch enqueues it on its
own communication stream behind the current stream's work.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence, Tuple

import torch
import torch.distributed as dist

from . import _lib
from .engine import on_device


def grad_buckets(obs_size: int, n_actions: int) -> List[Tuple[int, int]]:
    """[(start, end)) float ranges of the two gradient buckets in the arena."""
    total, offsets, _sizes = _lib.arena_layout(obs_size, n_actions)
    conv1_w = offsets[0]          # cnn_base.0.weight is the first tensor of the last segment
    return [(0, conv1_w), (conv1_w, total)]


def shard_range(n_items: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous shard [lo, hi) of a global batch: rank r owns frames [r*B/n, (r+1)*B/n)."""
    if n_items % world != 0:
        raise ValueError(f"global batch {n_items} must divide evenly over {world} ranks "
                         "(equal local batches make mean-of-means the global mean, as DDP assumes)")
    per = n_items // world
    return rank * per, (rank + 1) * per


class GradExchange:
    """All-reduce (sum) of the gradient arena in buckets; the mean's 1/world goes to the optimiser."""

    def __init__(self, obs_size: int, n_actions: int, group: Optional[dist.ProcessGroup] = None):
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.buckets = grad_buckets(obs_size, n_actions)
        self._pending = []

    @property
    def grad_scale(self) -> float:
        return 1.0 / self.world

    def start(self, flat_grads: torch.Tensor, bucket: int) -> None:
        """Launch the (async) all-reduce of one bucket; call when that bucket's gradients are final."""
        if self.world == 1:
            return
        lo, hi = self.buckets[bucket]
        self._pending.append(dist.all_reduce(flat_grads[lo:hi], op=dist.ReduceOp.SUM, group=self.group, async_op=True))

    def finish(self) -> None:
        """Make the current stream (or the host, for gloo) wait for every launched bucket."""
        for w in self._pending:
            w.wait()
        self._pending.clear()

    def all(self, flat_grads: torch.Tensor) -> None:
        for b in range(len(self.buckets)):
            self.start(flat_grads, b)
        self.finish()


class PeerGrads:
    """This rank's gradients in a symmetric allocation every rank maps (torch symmetric memory = cudaIpc / fabric handles;
    plumbing): TWO halves back to back -- step e writes and exchanges half e & 1, so no "done reading" handshake is needed
    (csrc/abi.cu) -- plus the per-rank signal pad and the private sync words of bc_adam_step_exchange.

    A half is the engine's arena (n floats), followed by `extra` floats of a second arena when one exchange covers two
    (the branched policy's branch arena, BranchedPeerExchange): stride = n + extra floats between the halves."""

    def __init__(self, engine, group: Optional[dist.ProcessGroup] = None, extra: int = 0):
        import torch.distributed._symmetric_memory as symm
        group = group if group is not None else dist.group.WORLD
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        self.n = n = engine.arena.numel()
        self.stride = S = n + int(extra)
        self.buf = symm.empty(2 * S, dtype=torch.float32, device=engine.device)
        self.hdl = symm.rendezvous(self.buf, group.group_name)
        self.buf.zero_()
        self.hdl.get_signal_pad(self.rank).zero_()
        self.sync = torch.zeros(4, dtype=torch.int32, device=engine.device)     # [0] completed epochs, [1] CTA counter
        self.err = torch.zeros(1, dtype=torch.int32, device=engine.device)
        self.c_struct = _lib.BcPeer(int(self.hdl.buffer_ptrs_dev), int(self.hdl.signal_pad_ptrs_dev), self.sync.data_ptr(),
                                    self.err.data_ptr(), self.rank, self.world)
        self.host_epoch = 0                           # mirrors sync[0]: one per completed (publishing) exchange launch
        # backward now reduces its partial sums straight into peer-visible memory, into the half the device epoch selects
        engine.grads, engine.grads_epoch, engine.grads_stride, engine.peer = self.buf, self.sync, S, self
        self.buckets = grad_buckets(engine.obs_size, engine.n_actions)
        torch.cuda.synchronize(engine.device)
        dist.barrier(group)                           # every pad is zero before anybody signals

    def current(self) -> torch.Tensor:
        """The half the NEXT exchange reads (= the one the backward of the current step writes): stride floats."""
        half = (self.host_epoch + 1) & 1
        return self.buf[half * self.stride:(half + 1) * self.stride]

    def check(self) -> None:
        if int(self.err.item()) != 0:
            raise RuntimeError("bc_adam_step_exchange: a peer rank never signalled (rank died, or the ranks ran different step "
                               "counts); the parameters were left untouched from that step on")


class PeerExchangeStep:
    """One optimisation step on this rank's shard with the gradient exchange FUSED into the Adam kernel over NVLink
    peer memory: after the backward ONE kernel sums all ranks' arenas and applies Adam (default). overlap=True: the
    [fc..conv2] bucket is reduced, exchanged and applied on the engine's side stream UNDER conv1's wgrad and only the
    12.6 KB conv1 bucket is exchanged after the backward -- measured on 2 x B200 the fork/join costs more than the overlap
    hides (0.2599 vs 0.2455 ms/step, profiles/README.md), so it is off by default. No NCCL call and no host round trip
    inside the step either way: the whole step is one CUDA graph."""

    def __init__(self, engine, optimizer, group: Optional[dist.ProcessGroup] = None, overlap: bool = False):
        self.eng, self.opt, self.overlap = engine, optimizer, overlap
        self.peer = PeerGrads(engine, group)
        optimizer.set_grad_scale(1.0 / self.peer.world)
        optimizer.prepare()
        if overlap:
            engine.side_handles()

    def exchange(self) -> None:
        """The exchange + Adam launches that follow a backward enqueued with dp_split (overlap) or without."""
        eng, opt, peer = self.eng, self.opt, self.peer
        if self.overlap:
            (lo0, hi0), (lo1, hi1) = peer.buckets
            side, evs, _arr = eng.side_handles()
            main = torch.cuda.current_stream(eng.device)
            opt.step_exchange(peer, lo0, hi0, bucket=0, publish=False, stream=side.cuda_stream)   # under conv1's wgrad
            c = eng.ctx(self._bufs)
            with on_device(eng.device):
                _lib.check(eng.lib.bc_reduce_partials_range(C.byref(c), 4, 5, 0, main.cuda_stream), "reduce [conv1]")
            evs[3].record(side)
            main.wait_event(evs[3])
            opt.step_exchange(peer, lo1, hi1, bucket=1, publish=True)
        else:
            opt.step_exchange(peer)
        if not torch.cuda.is_current_stream_capturing():
            peer.host_epoch += 1

    def __call__(self, bufs, loss_scale: Optional[float] = None) -> None:
        self._bufs = bufs
        self.eng.enqueue_train(bufs, loss_scale, dp_split=self.overlap)
        self.exchange()

    def capture(self, bufs, pre=None):
        self.opt.prepare()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            if pre is not None:
                pre()
            self(bufs)
        return g

    def replay(self, graph) -> None:
        self.opt.prepare()                   # a MultiStepLR milestone reaches the device scalar the captured kernels read
        graph.replay()
        self.peer.host_epoch += 1


class ModuleExchange:
    """Data parallelism THROUGH the module contract (Imitation.training_step -> loss.backward() -> FusedAdam.step, the loop
    train.py:125-129 hands to pl.Trainer(gpus=[...])): FusedAdam.step calls step_from() with this rank's arena-shaped
    gradients; they already sit in the peer-visible arena when the fused step produced them (zero-copy), else they are
    copied there; then one bc_adam_step_exchange launch sums all ranks' arenas and applies Adam."""

    def __init__(self, engine, optimizer, group: Optional[dist.ProcessGroup] = None):
        self.eng, self.opt = engine, optimizer
        self.peer = PeerGrads(engine, group)
        optimizer.set_grad_scale(1.0 / self.peer.world)
        optimizer.exchange = self

    def step_from(self, flat_grads: torch.Tensor) -> None:
        cur = self.peer.current()
        if flat_grads.data_ptr() != cur.data_ptr():
            cur.copy_(flat_grads)
        self.opt.step_exchange(self.peer)
        self.peer.host_epoch += 1


class BranchedPeerExchange:
    """The peer exchange of the command-conditioned branched policy (ConvNet1Branched + its MultiArenaAdam): each half of
    the peer-visible gradient buffer is [trunk arena | branch arena]. The trunk backward (bc_ctx.grads_epoch) and the
    branched heads' reduction (bc_branched.grads_epoch) write their gradients straight into the half the next exchange
    reads; one bc_adam_step_exchange_arenas launch then sums all ranks' halves in rank order, folds the 1/world mean and
    applies Adam to both arenas. Used by BranchedTrainStep (inside its CUDA graph) and, through MultiArenaAdam.step, by
    the module path."""

    def __init__(self, net, optimizer, group: Optional[dist.ProcessGroup] = None):
        self.trunk_opt, self.branch_opt = optimizer.children_
        self.peer = PeerGrads(net.engine(), group, extra=net._barena.numel())
        for c in optimizer.children_:
            c.set_grad_scale(1.0 / self.peer.world)
        optimizer.prepare()
        optimizer.exchange = self

    def head_grads(self) -> dict:
        """The bc_branched gradient fields of the heads' backward: the branch arena of half 0 + the epoch word."""
        p = self.peer
        return dict(grads=p.buf[p.n:], grads_epoch=p.sync, grads_stride=p.stride)

    def exchange(self) -> None:
        """Enqueue the two-arena exchange + Adam launch (after both arenas' gradients of this step are complete)."""
        (pt, mt, vt, st, _), (pb, mb, vb, sb, _) = self.trunk_opt._bind(), self.branch_opt._bind()
        if not torch.cuda.is_current_stream_capturing():
            self.trunk_opt._sync_scalars(st)
            self.branch_opt._sync_scalars(sb)
        wp, obs, na = self.trunk_opt._packed()
        with on_device(pt.device):
            _lib.check(_lib.lib().bc_adam_step_exchange_arenas(
                pt.data_ptr(), mt.data_ptr(), vt.data_ptr(), st.data_ptr(), pb.data_ptr(), mb.data_ptr(), vb.data_ptr(),
                sb.data_ptr(), self.peer.stride, self.peer.n, self.peer.c_struct, wp, obs, na,
                torch.cuda.current_stream(pt.device).cuda_stream), "bc_adam_step_exchange_arenas")

    def step_from(self, trunk_grads: torch.Tensor, branch_grads: torch.Tensor) -> None:
        """Module path (MultiArenaAdam.step): this rank's gradients of both arenas -> the current half (copied unless they
        already sit there), then one exchange launch."""
        cur, n = self.peer.current(), self.peer.n
        for dst, g in ((cur[:n], trunk_grads), (cur[n:], branch_grads)):
            if g.data_ptr() != dst.data_ptr():
                dst.copy_(g)
        self.exchange()
        self.peer.host_epoch += 1


class DataParallelStep:
    """One optimisation step on this rank's shard: forward, backward with the NCCL exchange overlapped, Adam.
    (The baseline exchange; PeerExchangeStep above is the fused one.)"""

    def __init__(self, engine, optimizer, group: Optional[dist.ProcessGroup] = None):
        self.eng, self.opt = engine, optimizer
        self.xchg = GradExchange(engine.obs_size, engine.n_actions, group)
        optimizer.set_grad_scale(self.xchg.grad_scale)

    # the step as three kernel segments; the exchange is launched between them
    def _seg_a(self, bufs, loss_scale=None) -> None:
        from .engine import on_device, _stream_ptr
        eng, lib = self.eng, self.eng.lib
        c = eng.ctx(bufs, loss_scale)
        s, ref = _stream_ptr(), None
        ref = C.byref(c)
        with on_device(eng.device):
            for layer in range(4):
                _lib.check(lib.bc_conv_relu_pool_fwd(ref, layer, s), "conv forward")
            _lib.check(lib.bc_head(ref, 3, s), "head")
            for layer in (3, 2, 1):
                _lib.check(lib.bc_conv_bwd_wgrad(ref, layer, s), "wgrad")
                _lib.check(lib.bc_conv_bwd_dgrad(ref, layer, s), "dgrad")
            _lib.check(lib.bc_reduce_partials_range(ref, 0, 4, 1, s), "reduce [fc..conv2]")

    def _seg_b(self, bufs, loss_scale=None) -> None:
        from .engine import _stream_ptr
        eng, lib = self.eng, self.eng.lib
        c = eng.ctx(bufs, loss_scale)
        with on_device(eng.device):
            _lib.check(lib.bc_conv_bwd_wgrad(C.byref(c), 0, _stream_ptr()), "conv1 wgrad")
            _lib.check(lib.bc_reduce_partials_range(C.byref(c), 4, 5, 0, _stream_ptr()), "reduce [conv1]")

    def __call__(self, bufs, loss_scale: Optional[float] = None) -> None:
        self._seg_a(bufs, loss_scale)
        self.xchg.start(self.eng.grads, 0)                 # overlaps with conv1's wgrad below
        self._seg_b(bufs, loss_scale)
        self.xchg.start(self.eng.grads, 1)
        self.xchg.finish()
        self.opt.step_flat(self.eng.grads)

    def capture(self, bufs, pre=None):
        """Capture the three kernel segments as CUDA graphs (NCCL stays outside). `pre` = optional callable
        enqueuing work that precedes the step (staging, weight packing) into the first segment."""
        self.opt.prepare()
        ga, gb, gc = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
        with torch.cuda.graph(ga):
            if pre is not None:
                pre()
            self._seg_a(bufs)
        with torch.cuda.graph(gb):
            self._seg_b(bufs)
        with torch.cuda.graph(gc):
            self.opt.step_flat(self.eng.grads)
        return ga, gb, gc

    def replay(self, graphs) -> None:
        ga, gb, gc = graphs
        self.opt.prepare()
        ga.replay()
        self.xchg.start(self.eng.grads, 0)
        gb.replay()
        self.xchg.start(self.eng.grads, 1)
        self.xchg.finish()
        gc.replay()
