"""ctypes binding of libbc_b200.so (the C ABI declared in include/bc_b200.h).

There is no CPU fallback and no alternative backend: if the shared library is missing or
the device is not sm_100, the calls below raise.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_PATH = os.environ.get("BC_LIB_PATH") or os.path.join(HERE, "libbc_b200.so")     # BC_LIB_PATH: A/B runs of two builds on one box
SOURCES = ("stage.cu", "conv_fwd.cu", "conv1_tc.cu", "conv1_fwd4.cu", "conv1_wgrad3.cu", "conv_tc.cu", "conv_sw.cu", "conv4_sw.cu", "head.cu", "policy_tail.cu", "head_branched.cu", "conv_bwd.cu", "abi.cu", "tc_selftest.cu")
# -cudart shared: the library reuses the libcudart.so.12 torch has already loaded (one CUDA runtime per process)
NVCC_FLAGS = ("-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared", "-cudart", os.environ.get("BC_CUDART", "shared"))

BC_F32, BC_BF16, BC_BF16_TP = 0, 1, 2
POLICY_TAIL_MAX_BATCH = 64      # BC_POLICY_TAIL_MAX_BATCH (include/bc_b200.h)
TP_PLANE_ELEMS = 86688


class BcCtx(C.Structure):
    """Mirror of `bc_ctx` (include/bc_b200.h)."""
    _fields_ = [
        ("obs_size", C.c_int32), ("n_actions", C.c_int32), ("batch", C.c_int32), ("x_dtype", C.c_int32),
        ("x_stride_n", C.c_int64), ("x_stride_c", C.c_int64),
        ("x", C.c_void_p), ("y", C.c_void_p), ("params", C.c_void_p), ("grads", C.c_void_p),
        ("act", C.c_void_p * 4), ("amax", C.c_void_p * 4), ("gact", C.c_void_p * 3),
        ("ghead", C.c_void_p), ("hid1", C.c_void_p), ("hid2", C.c_void_p),
        ("logits", C.c_void_p), ("dlogits", C.c_void_p), ("loss", C.c_void_p), ("partials", C.c_void_p),
        ("loss_scale", C.c_float), ("conv_mode", C.c_int32),
        ("w_packed", C.c_void_p), ("err_flag", C.c_void_p), ("act_bf16", C.c_void_p * 3),
        ("c1_acc", C.c_void_p),
        ("x_tp", C.c_void_p), ("x_tp_stride_n", C.c_int64), ("x_tp_stride_c", C.c_int64),
        ("grads_epoch", C.c_void_p), ("grads_stride", C.c_int64),
        ("gact0_p8", C.c_void_p), ("amax0_p8", C.c_void_p),
    ]


class BcPeer(C.Structure):
    """Mirror of `bc_peer` (include/bc_b200.h)."""
    _fields_ = [("peer_grads_dev", C.c_void_p), ("peer_signals_dev", C.c_void_p), ("sync_state", C.c_void_p),
                ("err_flag", C.c_void_p), ("rank", C.c_int32), ("world", C.c_int32)]


class BcBranched(C.Structure):
    """Mirror of `bc_branched` (include/bc_b200.h): the branched-head extension."""
    _fields_ = [("n_branches", C.c_int32), ("n_out", C.c_int32), ("batch", C.c_int32), ("loss_kind", C.c_int32),
                ("feat", C.c_void_p), ("command", C.c_void_p), ("labels", C.c_void_p), ("targets", C.c_void_p),
                ("params", C.c_void_p), ("grads", C.c_void_p), ("out", C.c_void_p), ("dout", C.c_void_p),
                ("gfeat", C.c_void_p), ("loss", C.c_void_p), ("partials", C.c_void_p), ("err_flag", C.c_void_p),
                ("loss_scale", C.c_float)]


EXPORTS = {
    # name: (restype, argtypes)
    "bc_arena_layout": (C.c_int64, [C.c_int, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "bc_partials_floats": (C.c_size_t, [C.c_int, C.c_int]),
    "bc_stage_gray": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
    "bc_pack_weights": (C.c_int, [C.POINTER(BcCtx), C.c_void_p]),
    "bc_packed_weight_bytes": (C.c_size_t, []),
    "bc_stage_gray_tp": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "bc_stage_augment": (C.c_int, [C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "bc_planes_to_tp": (C.c_int, [C.c_void_p, C.c_int, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p]),
    "bc_forward": (C.c_int, [C.POINTER(BcCtx), C.c_void_p]),
    "bc_conv_relu_pool_fwd": (C.c_int, [C.POINTER(BcCtx), C.c_int, C.c_void_p]),
    "bc_head": (C.c_int, [C.POINTER(BcCtx), C.c_int, C.c_void_p]),
    "bc_backward": (C.c_int, [C.POINTER(BcCtx), C.c_int, C.c_void_p]),
    "bc_conv_bwd_dgrad": (C.c_int, [C.POINTER(BcCtx), C.c_int, C.c_void_p]),
    "bc_conv_bwd_wgrad": (C.c_int, [C.POINTER(BcCtx), C.c_int, C.c_void_p]),
    "bc_reduce_partials": (C.c_int, [C.POINTER(BcCtx), C.c_int, C.c_void_p]),
    "bc_reduce_partials_range": (C.c_int, [C.POINTER(BcCtx), C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "bc_loss_reduce": (C.c_int, [C.POINTER(BcCtx), C.c_void_p]),
    "bc_adam_tick": (C.c_int, [C.c_void_p, C.c_void_p]),
    "bc_adam_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "bc_adam_tick_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                    C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "bc_adam_step_exchange": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(BcPeer),
                                        C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "bc_backward_overlap": (C.c_int, [C.POINTER(BcCtx), C.c_int, C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p), C.c_int]),
    "bc_argmax": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "bc_forward_act": (C.c_int, [C.POINTER(BcCtx), C.c_void_p, C.c_int, C.c_void_p]),
    "bc_policy_tail": (C.c_int, [C.POINTER(BcCtx), C.c_void_p, C.c_void_p]),
    "bc_head_branched": (C.c_int, [C.POINTER(BcBranched), C.c_int, C.c_void_p]),
    "bc_head_branched_partials_floats": (C.c_size_t, [C.c_int, C.c_int]),
    "bc_head_branched_layout": (C.c_int64, [C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "bc_forward_branched_act": (C.c_int, [C.POINTER(BcCtx), C.POINTER(BcBranched), C.c_void_p, C.c_int, C.c_void_p]),
    "bc_policy_tail_branched": (C.c_int, [C.POINTER(BcCtx), C.POINTER(BcBranched), C.c_void_p, C.c_void_p]),
    "bc_scale_inplace": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "bc_tc_gemm_selftest": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "bc_tc_mma_bench": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bc_last_error_string": (C.c_char_p, []),
    "bc_device_check": (C.c_int, []),
    "bc_abi_version": (C.c_int, []),
}

_lib = None


def build(verbose: bool = False) -> str:
    """Compile csrc/*.cu for sm_100a into libbc_b200.so (nvcc cross-compiles without a GPU)."""
    srcs = [os.path.join(CSRC, s) for s in SOURCES]
    deps = srcs + [os.path.join(CSRC, h) for h in ("bc_common.cuh", "tc05.cuh", "pack.cuh", "trace.cuh")] + [os.path.join(os.path.dirname(HERE), "include", "bc_b200.h")]
    if os.path.exists(LIB_PATH) and all(os.path.getmtime(LIB_PATH) >= os.path.getmtime(d) for d in deps):
        return LIB_PATH
    nvcc = os.environ.get("NVCC", "nvcc")
    cmd = [nvcc, *NVCC_FLAGS, *os.environ.get("BC_NVCC_EXTRA", "").split(), "-o", LIB_PATH, *srcs]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
    if verbose:
        sys.stderr.write(r.stderr)
    return LIB_PATH


def lib():
    """The loaded library; raises (never falls back) when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -c \"import __graft_entry__ as g; g.build()\"`. "
                "There is no CPU or PyTorch fallback for the BC hot path.")
        import torch  # noqa: F401  (loads libcudart.so.12, which the library links dynamically)
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in EXPORTS.items():
            fn = getattr(l, name)   # AttributeError here = header/library mismatch
            fn.restype, fn.argtypes = res, args
        _lib = l
    return _lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib().bc_last_error_string()
        raise RuntimeError(f"{what or 'bc_b200'} failed (status {rc}): {msg.decode() if msg else ''}")


def arena_layout(obs_size: int, n_actions: int):
    off = (C.c_int64 * 14)()
    siz = (C.c_int64 * 14)()
    total = lib().bc_arena_layout(obs_size, n_actions, off, siz)
    return int(total), [int(v) for v in off], [int(v) for v in siz]
