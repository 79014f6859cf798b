"""ConvNet1Branched -- EXTENSION (no counterpart in the reference): the ConvNet1 trunk with command-conditioned heads.

BASELINE.json's north_star asks for "command-conditioned action heads": G per-command MLP branches of the reference's head
shape 128 -> 64 -> 32 -> n_out (/root/reference/src/architectures/nets.py:31-33 has one), a branch-select mask (sample b
is evaluated, and differentiated, only by branch command[b]) and CE or L1 / MSE (steer, throttle, brake) loss
(/root/reference/src/models/imitation.py:43-44 has CE only). Specification and tests: oracle/ext_oracle.py.

    net = ConvNet1Branched({'obs_size': 4, 'n_actions': 3, 'n_branches': 4, 'branch_loss': 'l1'})
    out = net(x, command)                      # (B, n_out): the commanded branch's outputs
    act = net.act(x, command)                  # serving: greedy actions (CE) or the branch's controls (L1 / MSE)
    loss = net.loss(x, command, target)        # fused trunk forward + grouped heads + loss; .backward() runs the CUDA backward

The conv trunk is the ConvNet1 arena and kernels unchanged (its single `fc` head stays in the arena, unregistered and
unused); the branches live in a second flat arena [G][fc.4 fc.2 fc.0] driven by csrc/head_branched.cu. state_dict keys:
`cnn_base.{0,3,6,9}.*` and `branches.{g}.{0,2,4}.*`.
"""
from __future__ import annotations

import ctypes as C
import math

import torch
from torch import nn

from carla_imitation_learning_b200 import _lib
from carla_imitation_learning_b200.engine import BCEngine, _stream_ptr, on_device
from carla_imitation_learning_b200.optim import FusedAdam
from .nets import ConvNet1, _Slot, _Stack

LOSS_KINDS = {"ce": 0, "l1": 1, "mse": 2}


class _BranchOwner:
    """What FusedAdam needs to know about a flat arena (the branch arena has no engine of its own)."""

    def __init__(self, obs_size, n_actions):
        self._arena, self._engine, self.obs_size, self.n_actions = None, None, obs_size, n_actions


class ConvNet1Branched(ConvNet1):
    # serving: up to this batch conv3, conv4 and the commanded branch run as ONE cluster launch (bc_policy_tail_branched),
    # above it conv3, conv4 and the branched head kernel. Measured crossover (tools/branched_serve_bench.py, B200 at 1000 W,
    # profiles/r3b_bench_branched_serve.json, p50): tail 22.0-24.0 us against 30.1-32.2 us up to B = 8, 34.24 against
    # 34.27 at B = 16, 44.5 against 38.4 at B = 32 -- the single head's threshold (BCEngine.tail_batch) again.
    tail_batch = BCEngine.tail_batch

    def __init__(self, hparams):
        super().__init__(hparams)
        self.n_branches = int(hparams['n_branches'])
        kind = str(hparams['branch_loss']) if 'branch_loss' in hparams else 'ce'
        if kind not in LOSS_KINDS:
            raise ValueError(f"branch_loss must be one of {sorted(LOSS_KINDS)}, got {kind!r}")
        if not 1 <= self.n_branches <= 16:
            raise ValueError("n_branches must be in 1..16")
        self.branch_loss = kind
        del self._modules['fc']            # the trunk's single head stays in the arena but is neither registered nor used
        off = (C.c_int64 * 6)()
        siz = (C.c_int64 * 6)()
        self._head_len = int(_lib.lib().bc_head_branched_layout(self.n_actions, off, siz))
        shapes = ((64, 128), (64,), (32, 64), (32,), (self.n_actions, 32), (self.n_actions,))
        barena = torch.zeros(self.n_branches * self._head_len, dtype=torch.float32)
        self._bowner = _BranchOwner(self.obs_size, self.n_actions)
        self.branches = _Stack()
        self._branch_params = []
        for g in range(self.n_branches):
            stack = _Stack()
            for li, slot in enumerate((0, 2, 4)):
                fan_in = shapes[2 * li][1]
                w = torch.empty(shapes[2 * li])
                nn.init.kaiming_uniform_(w, a=math.sqrt(5))               # nn.Linear.reset_parameters
                b = torch.empty(shapes[2 * li + 1])
                nn.init.uniform_(b, -1 / math.sqrt(fan_in), 1 / math.sqrt(fan_in))
                holder = _Slot("linear")
                for j, (name, t) in enumerate((("weight", w), ("bias", b))):
                    o = g * self._head_len + int(off[2 * li + j])
                    barena[o:o + t.numel()] = t.reshape(-1)
                    p = nn.Parameter(barena[o:o + t.numel()].view(t.shape))
                    p._bc_offset, p._bc_owner = o, self._bowner
                    holder.register_parameter(name, p)
                    self._branch_params.append(p)
                stack.add_module(str(slot), holder)
            self.branches.add_module(str(g), stack)
        self._rebind_branches(barena if not self._arena.is_cuda else barena.to(self._arena.device))
        self._bstate = None

    # ------------------------------------------------------------------ arenas
    def _rebind_branches(self, barena: torch.Tensor) -> None:
        self._barena = self._bowner._arena = barena
        for p in self._branch_params:
            p.data = barena[p._bc_offset:p._bc_offset + p.numel()].view(p.shape)
            p._bc_arena = barena
            p.grad = None
        self._bstate = None

    def _apply(self, fn, recurse=True):
        super()._apply(fn, recurse)
        if hasattr(self, "_barena"):
            new = fn(self._barena)
            if new is not self._barena:
                self._rebind_branches(new.contiguous())
        return self

    def load_state_dict(self, state_dict, strict=True, **kw):
        own = dict(self.named_parameters())
        missing = [k for k in own if k not in state_dict]
        unexpected = [k for k in state_dict if k not in own]
        if strict and (missing or unexpected):
            raise RuntimeError(f"state_dict mismatch: missing {missing}, unexpected {unexpected}")
        with torch.no_grad():
            for k, p in own.items():
                if k in state_dict:
                    p.copy_(state_dict[k])
        return torch.nn.modules.module._IncompatibleKeys(missing, unexpected)

    def trunk_parameters(self):
        return self._ordered_params[:8]

    def branch_parameters(self):
        return list(self._branch_params)

    def configure_optimizer(self, lr: float = 1e-3):
        """Adam over both arenas (one fused launch each) behind one torch.optim.Optimizer."""
        return MultiArenaAdam([self.trunk_parameters(), self.branch_parameters()], lr=lr)

    # ------------------------------------------------------------------ compute
    def _bbufs(self, B: int):
        st = self._bstate
        dev = self._barena.device
        if st is None:
            n = int(_lib.lib().bc_head_branched_partials_floats(self.n_branches, self.n_actions))
            st = self._bstate = dict(grads=torch.zeros_like(self._barena), partials=torch.zeros(n, dtype=torch.float32, device=dev))
        e = lambda *s: torch.empty(s, dtype=torch.float32, device=dev)
        return dict(out=e(B, self.n_actions), dout=e(B, self.n_actions), loss=torch.zeros((), dtype=torch.float32, device=dev), **st)

    def _head(self, bufs, hb, command, target, mode: int) -> None:
        eng = self.engine()
        h = _lib.BcBranched()
        h.n_branches, h.n_out, h.batch, h.loss_kind = self.n_branches, self.n_actions, bufs.batch, LOSS_KINDS[self.branch_loss]
        h.feat, h.command = bufs.act[3].data_ptr(), command.data_ptr()
        if target is not None:
            if self.branch_loss == "ce":
                h.labels = target.data_ptr()
            else:
                h.targets = target.data_ptr()
        h.params, h.grads = self._barena.data_ptr(), hb["grads"].data_ptr()
        h.out, h.dout, h.loss = hb["out"].data_ptr(), hb["dout"].data_ptr(), hb["loss"].data_ptr()
        h.gfeat = bufs.ghead.data_ptr() if bufs.ghead is not None else None
        h.partials, h.err_flag = hb["partials"].data_ptr(), eng.err_flag.data_ptr()
        if hb.get("grads_epoch") is not None:     # data parallel: the branch gradients go to the peer half of this step
            h.grads_epoch, h.grads_stride = hb["grads_epoch"].data_ptr(), hb["grads_stride"]
        n = max(bufs.batch, 1) * (1 if self.branch_loss == "ce" else self.n_actions)
        h.loss_scale = 1.0 / n
        with torch.cuda.device(eng.device):
            _lib.check(eng.lib.bc_head_branched(C.byref(h), mode, _stream_ptr()), "bc_head_branched")

    def _check(self, x, command, target):
        eng = self.engine()
        x = eng.check_input(self._to_device(x))
        B = x.shape[0]
        command = self._to_device(command)
        if command.dtype != torch.int64 or tuple(command.shape) != (B,):
            raise ValueError("command must be a (B,) int64 tensor of branch ids")
        if target is not None:
            target = self._to_device(target)
            if self.branch_loss == "ce":
                if target.dtype != torch.int64 or tuple(target.shape) != (B,):
                    raise ValueError("CE targets are (B,) int64 class ids")
            elif target.dtype != torch.float32 or tuple(target.shape) != (B, self.n_actions):
                raise ValueError(f"{self.branch_loss} targets are (B, {self.n_actions}) float32")
            target = target.contiguous()
        return x, command.contiguous(), target

    def _trunk_forward(self, x, backward: bool):
        eng = self.engine()
        bufs = eng.alloc(x.shape[0], x, None, backward)
        with torch.cuda.device(eng.device):
            eng.enqueue_trunk_forward(bufs)
        return bufs

    @torch.no_grad()
    def forward(self, x, command):
        """(B, obs, 256, 256), (B,) branch ids -> (B, n_out) outputs of the commanded branch (inference; train with loss())."""
        x, command, _ = self._check(x, command, None)
        bufs = self._trunk_forward(x, False)
        hb = self._bbufs(x.shape[0])
        self._head(bufs, hb, command, None, 0)
        return hb["out"]

    def _serve(self, bufs, out, actions, command, tail: bool) -> None:
        """Enqueue the serving forward on the current stream (bc_forward_branched_act): conv1..conv4 and the branched head
        kernel, or with `tail` conv1, conv2 and the one-launch tail. out (B, n_out) f32 and actions (B,) int64 or None are
        written; command (B,) int64 is read on the device when the kernels run (a captured graph follows its contents)."""
        eng = self.engine()
        c = eng.ctx(bufs)
        h = _lib.BcBranched()
        h.n_branches, h.n_out, h.batch, h.loss_kind = self.n_branches, self.n_actions, bufs.batch, LOSS_KINDS[self.branch_loss]
        h.command, h.params, h.out = command.data_ptr(), self._barena.data_ptr(), out.data_ptr()
        h.err_flag = eng.err_flag.data_ptr()
        with on_device(eng.device):
            _lib.check(eng.lib.bc_forward_branched_act(C.byref(c), C.byref(h), actions.data_ptr() if actions is not None else None,
                                                       int(bool(tail)), _stream_ptr()), "bc_forward_branched_act")

    @torch.no_grad()
    def act(self, x, command):
        """What a conditional-imitation agent sends per tick: for branch_loss 'ce' the (B,) int64 greedy actions of the
        commanded branches (torch.argmax's rule), for 'l1' / 'mse' their (B, n_out) f32 outputs (steer, throttle, brake).
        Batches up to `tail_batch` take the one-launch tail. A command outside [0, n_branches)
        gives a zero row / action 0 and raises at engine().check_device_errors(). For a fixed-shape serving loop use
        trainer.BranchedActStep (persistent buffers, one CUDA graph per input slot)."""
        x, command, _ = self._check(x, command, None)
        eng = self.engine()
        B = x.shape[0]
        bufs = eng.alloc(B, x, None, False)
        out = torch.empty((B, self.n_actions), dtype=torch.float32, device=eng.device)
        actions = torch.empty(B, dtype=torch.int64, device=eng.device) if self.branch_loss == "ce" else None
        if B:
            self._serve(bufs, out, actions, command, B <= self.tail_batch)
        return actions if actions is not None else out

    def loss(self, x, command, target):
        x, command, target = self._check(x, command, target)
        return _BranchedLoss.apply(x, command, target, self, *self.trunk_parameters(), *self._branch_params)


class _BranchedLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, command, target, net, *params):
        bufs = net._trunk_forward(x, True)
        hb = net._bbufs(x.shape[0])
        net._head(bufs, hb, command, target, 1)
        ctx.net, ctx.bufs, ctx.hb, ctx.command = net, bufs, hb, command
        return hb["loss"]

    @staticmethod
    def backward(ctx, gloss):
        net, bufs, hb = ctx.net, ctx.bufs, ctx.hb
        eng = net.engine()
        hb["dout"].mul_(gloss)
        net._head(bufs, hb, ctx.command, None, 2)
        with torch.cuda.device(eng.device):
            eng.enqueue_trunk_backward(bufs)
        flat = eng._last_flat = eng.grad_view().clone()
        bflat = hb["grads"].clone()
        tg = [flat[p._bc_offset:p._bc_offset + p.numel()].view(p.shape) for p in net.trunk_parameters()]
        bg = [bflat[p._bc_offset:p._bc_offset + p.numel()].view(p.shape) for p in net._branch_params]
        return (None, None, None, None, *tg, *bg)


class MultiArenaAdam(torch.optim.Optimizer):
    """One torch.optim.Optimizer over several flat arenas: a FusedAdam (one fused launch) per arena; the learning rate of
    param_groups[0] -- what MultiStepLR drives -- is handed to all of them.

    The moments and step counts live in the children. self.state exposes their per-parameter views, and state_dict() /
    load_state_dict() use one parameter index space over all arenas: the layout torch.optim.Adam(list(net.parameters()))
    writes, so a checkpoint of either optimiser restores into the other."""

    def __init__(self, param_lists, lr: float = 1e-3):
        params = [p for ps in param_lists for p in ps]
        super().__init__(params, dict(lr=lr, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, amsgrad=False))
        self.children_ = [FusedAdam(list(ps), lr=lr) for ps in param_lists]
        self._linked = [None] * len(self.children_)
        self.exchange = None          # parallel.BranchedPeerExchange when the module path trains data-parallel

    def _link_state(self) -> None:
        """self.state[p] = the child's torch.optim.Adam-compatible views (FusedAdam._bind), refreshed when a child rebinds."""
        for i, c in enumerate(self.children_):
            if c._bound is not None and self._linked[i] is not c._bound:
                for p in c._params:
                    self.state[p] = c.state[p]
                self._linked[i] = c._bound

    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        if self.exchange is not None:          # data parallel: both arenas' gradients -> one exchange launch
            grads = []
            for c in self.children_:
                c.param_groups[0]["lr"] = self.param_groups[0]["lr"]
                arena, _m, _v, _st, flat_g = c._bind()
                grads.append(c._flat_grads(arena, flat_g))
            self.exchange.step_from(*grads)
        else:
            for c in self.children_:
                c.param_groups[0]["lr"] = self.param_groups[0]["lr"]
                c.step()
        self._link_state()
        return loss

    def prepare(self) -> None:
        """Push param_groups[0]['lr'] into every child's device scalar (allocating their state on the first call). Call
        before capturing a CUDA graph that holds the Adam launches and before every replay, so a MultiStepLR milestone
        reaches the captured kernels."""
        for c in self.children_:
            c.param_groups[0]["lr"] = self.param_groups[0]["lr"]
            c.prepare()
        self._link_state()

    def zero_grad(self, set_to_none: bool = True) -> None:
        for c in self.children_:
            c.zero_grad(set_to_none)

    # ------------------------------------------------------------------ checkpoints
    def state_dict(self):
        """torch.optim.Adam's layout: state[i] = {step, exp_avg, exp_avg_sq} of param_groups[0]['params'][i]."""
        self._link_state()
        return super().state_dict()

    def load_state_dict(self, state_dict) -> None:
        """Accepts what state_dict() writes and a torch.optim.Adam state_dict over the same parameter list (its groups'
        indices, in order, are matched to param_groups[0]['params']). Each child gets its parameters' moments and the step
        count (FusedAdam.load_state_dict); the restored learning rate reaches every child's device scalar."""
        groups = state_dict["param_groups"]
        ids = [pid for g in groups for pid in g["params"]]
        own = self.param_groups[0]["params"]
        if len(ids) != len(own):
            raise ValueError(f"the optimiser state holds {len(ids)} parameters, this optimiser has {len(own)}")
        gid = {id(p): pid for p, pid in zip(own, ids)}
        for c in self.children_:
            c.load_state_dict({"state": state_dict["state"],
                               "param_groups": [{"params": [gid[id(p)] for p in c._params], "lr": groups[0]["lr"]}]})
        self.param_groups[0]["lr"] = groups[0]["lr"]
        self.prepare()
