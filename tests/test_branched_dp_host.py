"""Host side of training the branched policy data-parallel, on CPU: the argument checks of the two-arena exchange entry point
(it rejects before any CUDA call, so fake device addresses are enough), the ctypes mirror of bc_branched against the C
header, and the module path refusing the NCCL exchange for the branched policy."""
import ctypes as C
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _peer(rank=0, world=2, null=None):
    from carla_imitation_learning_b200 import _lib
    f = dict(peer_grads_dev=0x1000, peer_signals_dev=0x2000, sync_state=0x3000, err_flag=0x4000)
    if null:
        f[null] = None
    return _lib.BcPeer(f["peer_grads_dev"], f["peer_signals_dev"], f["sync_state"], f["err_flag"], rank, world)


def _call(n=1024, split=512, peer=None, ptrs=None):
    from carla_imitation_learning_b200 import _lib
    _lib.build()
    lib = _lib.lib()
    p = ptrs or [0x10000 * (i + 1) for i in range(8)]
    rc = lib.bc_adam_step_exchange_arenas(*p, n, split, C.byref(peer or _peer()), None, 4, 9, None)
    return rc, lib.bc_last_error_string().decode()


def test_two_arena_exchange_arguments_are_rejected_before_any_launch():
    for i in range(8):                                           # every parameter / moment / state pointer of both arenas
        ptrs = [0x10000 * (k + 1) for k in range(8)]
        ptrs[i] = None
        rc, msg = _call(ptrs=ptrs)
        assert rc == -1 and "null pointer" in msg, i
    for field in ("peer_grads_dev", "peer_signals_dev", "sync_state", "err_flag"):
        rc, msg = _call(peer=_peer(null=field))
        assert rc == -1 and "bc_peer" in msg, field
    for n in (0, -4, 1022):
        rc, msg = _call(n=n, split=256)
        assert rc == -1 and "multiple of 4" in msg, n
    for split in (0, 1024, 2048, -4, 510):
        rc, msg = _call(split=split)
        assert rc == -1 and "split" in msg, split
    for rank, world in ((2, 2), (-1, 2), (0, 0), (0, 65)):
        rc, msg = _call(peer=_peer(rank, world))
        assert rc == -1 and "rank" in msg, (rank, world)
    ptrs = [0x10000 * (k + 1) for k in range(8)]
    ptrs[4] += 4
    rc, msg = _call(ptrs=ptrs)
    assert rc == -1 and "16 B" in msg
    # the operand images follow arena 0: with w_packed, split must be the trunk arena of (obs_size, n_actions)
    from carla_imitation_learning_b200 import _lib
    lib = _lib.lib()
    rc = lib.bc_adam_step_exchange_arenas(*[0x10000 * (k + 1) for k in range(8)], 1024, 512, C.byref(_peer()), 0x90000, 4, 9, None)
    assert rc == -1 and "arena" in lib.bc_last_error_string().decode()


def test_bc_branched_mirror_matches_the_header():
    """sizeof(bc_branched) and every field offset, compiled from include/bc_b200.h, == the ctypes mirror's."""
    from carla_imitation_learning_b200 import _lib
    cc = shutil.which("cc") or shutil.which("gcc")
    if cc is None:
        pytest.skip("no C compiler on this machine")
    fields = [f for f, _ in _lib.BcBranched._fields_]
    src = "#include <stdio.h>\n#include <stddef.h>\n#include \"bc_b200.h\"\nint main(void) {\n"
    src += '    printf("%zu\\n", sizeof(bc_branched));\n'
    src += "".join(f'    printf("%zu\\n", offsetof(bc_branched, {f}));\n' for f in fields) + "    return 0;\n}\n"
    tmp = os.path.join(os.environ.get("TMPDIR", "/tmp"), f"bc_branched_layout_{os.getpid()}")
    with open(tmp + ".c", "w") as fh:
        fh.write(src)
    try:
        subprocess.run([cc, "-I", os.path.join(ROOT, "include"), "-o", tmp, tmp + ".c"], check=True, capture_output=True)
        got = [int(v) for v in subprocess.run([tmp], check=True, capture_output=True, text=True).stdout.split()]
    finally:
        for f in (tmp, tmp + ".c"):
            if os.path.exists(f):
                os.remove(f)
    assert got[0] == C.sizeof(_lib.BcBranched)
    assert got[1:] == [getattr(_lib.BcBranched, f).offset for f in fields]
    assert fields[-2:] == ["grads_epoch", "grads_stride"]


def test_trainer_refuses_the_nccl_exchange_for_the_branched_policy(monkeypatch):
    """Trainer.fit with ddp_exchange 'nccl' on a world of several ranks and an ImitationBranched: refused before any step,
    naming 'peer' as the exchange the branched policy trains with."""
    import torch.distributed as dist
    from carla_imitation_learning_b200.trainer import Trainer
    from src.architectures.branched import ConvNet1Branched
    from src.models.imitation_branched import ImitationBranched
    hp = {"obs_size": 4, "n_actions": 3, "n_branches": 4, "branch_loss": "l1"}
    model = ImitationBranched(dict(hp), ConvNet1Branched(dict(hp)), {})
    monkeypatch.setattr(dist, "is_initialized", lambda: True)
    monkeypatch.setattr(dist, "get_world_size", lambda group=None: 2)
    with pytest.raises(RuntimeError, match="'peer' only"):
        Trainer(max_epochs=1, ddp_exchange="nccl").fit(model)
