"""ctypes binding of libdiff3d_b200.so (the C ABI declared in include/diff3d_b200.h).

There is no CPU fallback: if the shared library is missing or cannot be loaded, importing a symbol from it
raises immediately with the build command to run.
"""
from __future__ import annotations

import ctypes as C
import os
import threading
from pathlib import Path

_PKG = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ.get("D3D_LIB", _PKG / "libdiff3d_b200.so"))

GEMM_TC_SPLIT3, GEMM_TC_FP16, GEMM_SIMT_FP32, GEMM_TC_F8C, GEMM_SIMT_F8C, GEMM_TC_F4C, GEMM_SIMT_F4C = 0, 1, 2, 3, 4, 5, 6
GEMM_DEFAULT = GEMM_TC_F4C      # shipped precision mode of the drop-in modules (DESIGN.md section 2)
ATTN_DEFAULT, ATTN_SIMT, ATTN_MMA_SYNC = 0, 1, 2
ROWWISE_LIFT, ROWWISE_POSTNORM, ROWWISE_NORM2, ROWWISE_HEAD = 0, 1, 2, 3     # d3d_debug_rowwise
PROF_CLASSES = ("gemm", "attn_spatial", "attn_temporal", "ln", "lift", "head_ddim")


class Config(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "num_frame", "num_joints", "embed_dim", "depth", "num_heads", "mlp_hidden", "with_time_emb", "max_clips",
        "gemm_mode", "attn_mode", "device", "use_graph")]


class TensorDesc(C.Structure):
    _fields_ = [("name", C.c_char_p), ("data", C.c_void_p), ("numel", C.c_int64), ("on_device", C.c_int32)]


# name -> (restype, argtypes): exactly the prototypes of include/diff3d_b200.h
PROTOTYPES = {
    "d3d_abi_version": (C.c_int, []),
    "d3d_create": (C.c_int, [C.POINTER(Config), C.POINTER(C.c_void_p)]),
    "d3d_destroy": (None, [C.c_void_p]),
    "d3d_last_error": (C.c_char_p, [C.c_void_p]),
    "d3d_load_weights": (C.c_int, [C.c_void_p, C.POINTER(TensorDesc), C.c_int32]),
    "d3d_set_schedule": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_float),
                                   C.POINTER(C.c_float), C.c_int32, C.c_float, C.c_int32]),
    "d3d_forward_denoise": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "d3d_ddim_sample": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_int32, C.c_void_p]),
    "d3d_ddim_sample_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                       C.c_void_p]),
    "d3d_tta_merge": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                C.c_int32, C.c_float, C.c_void_p, C.c_int64, C.c_void_p]),
    "d3d_window_gather": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_int32),
                                    C.POINTER(C.c_int32), C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "d3d_window_scatter": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "d3d_mpjpe_accumulate": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p,
                                       C.c_void_p]),
    "d3d_pose_metrics_accumulate": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p,
                                              C.c_void_p]),
    "d3d_launch_count": (C.c_int64, [C.c_void_p]),
    "d3d_workspace_bytes": (C.c_int64, [C.c_void_p]),
    "d3d_profile_begin": (C.c_int, [C.c_void_p]),
    "d3d_profile_end": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "d3d_op_linear": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "d3d_op_linear_ln": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_float, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p]),
    "d3d_op_linear_dln_linear": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_int64, C.c_int32, C.c_void_p]),
    "d3d_op_linear_bench": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                      C.POINTER(C.c_float)]),
    "d3d_op_layernorm": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.c_int64,
                                   C.c_void_p]),
    "d3d_op_attention": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "d3d_op_time_table": (C.c_int, [C.c_void_p, C.POINTER(C.c_float), C.c_int32, C.c_void_p, C.c_void_p]),
    "d3d_debug_attention_operand": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                              C.c_int32, C.c_void_p]),
    "d3d_debug_forward_blocks": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p,
                                           C.c_void_p]),
    "d3d_debug_rowwise": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
}

_lib = None
_load_lock = threading.Lock()     # nn.DataParallel creates its engines from one thread per device


def load():
    """Load (once, also when several threads ask at the same time) and return the ctypes library with prototypes
    applied."""
    global _lib
    if _lib is not None:
        return _lib
    with _load_lock:
        if _lib is None:
            _lib = _load()
    return _lib


def _load():
    if not LIB_PATH.exists():
        raise RuntimeError(
            f"{LIB_PATH} not found: build it with `python -m diff3dhpe_b200.build` "
            "(diff3dhpe_b200 has no CPU or PyTorch fallback)")
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)          # AttributeError here = header/library mismatch
        fn.restype = res
        fn.argtypes = args
    if lib.d3d_abi_version() != 1:
        raise RuntimeError("libdiff3d_b200.so ABI version mismatch")
    return lib


def last_error(handle) -> str:
    msg = load().d3d_last_error(handle)
    return msg.decode() if msg else ""


def check(rc: int, handle=None, what: str = ""):
    if rc != 0:
        raise RuntimeError(f"{what or 'libdiff3d_b200'} failed (code {rc}): {last_error(handle)}")
