"""ctypes binding of the C-ABI library (`include/smt_b200.h`).

This is the ONLY way the Python host reaches the GPU kernels: there is no CPU fallback and no eager
PyTorch substitute.  If the library is missing or fails to load, every op raises.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SMT_B200_LIB") or os.path.join(_HERE, "_C", "libsmt_b200.so")   # (override: kernel experiments)

F32, BF16, F16 = 0, 1, 2
MEAN_ABS, ABS_MEAN, L1, L2 = 0, 1, 2, 3
STRATEGY_IDS = {"mean_abs": MEAN_ABS, "abs_mean": ABS_MEAN, "L1": L1, "L2": L2}

_DTYPE_IDS = {torch.float32: F32, torch.bfloat16: BF16, torch.float16: F16}


class BlockRef(C.Structure):
    """Mirror of `smt_block_ref`."""
    _fields_ = [("w_ptr", C.c_uint64), ("ldw", C.c_int64), ("row", C.c_int32), ("col", C.c_int32)]


class GemmItem(C.Structure):
    """Mirror of `smt_gemm_item`."""
    _fields_ = [("map_dy", C.c_uint32), ("map_x", C.c_uint32), ("row", C.c_int32), ("col", C.c_int32),
                ("out_off", C.c_int64), ("flags", C.c_uint32), ("sq_slot", C.c_int32)]


ITEM_OVERWRITE = 1   # SMT_ITEM_OVERWRITE


class GemmRun(C.Structure):
    """Mirror of `smt_gemm_run`."""
    _fields_ = [("row", C.c_int32), ("half", C.c_int32), ("ncols", C.c_int32), ("cols", C.c_int32 * 4),
                ("out_blk", C.c_int32 * 4), ("pad_", C.c_int32)]


class SMTLibraryError(RuntimeError):
    pass


_P = C.c_void_p
_SIGNATURES = {
    "smt_last_error": (C.c_char_p, []),
    "smt_version": (C.c_int, []),
    "smt_last_launch_count": (C.c_int, []),
    "smt_device_info": (C.c_int, [C.POINTER(C.c_int)] * 3),
    "smt_score_accumulate": (C.c_int, [_P, _P, C.c_int, C.c_int64, _P]),
    "smt_block_sum_accumulate": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_int64, C.c_int, _P]),
    "smt_block_sum_finalize": (C.c_int, [_P, _P, C.c_int64, C.c_int, _P]),
    "smt_block_score_reduce": (C.c_int, [_P, C.c_int, C.c_int, C.c_int64, C.c_int, C.c_int, _P, _P]),
    "smt_token_block_sums": (C.c_int, [_P, C.c_int, C.c_int64, C.c_int, C.c_int64, C.c_int, _P, _P]),
    "smt_block_outer_accumulate_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int, C.c_int]),
    "smt_block_outer_accumulate": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int, C.c_int, _P, C.c_size_t, _P]),
    "smt_act_score_accumulate": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    "smt_channel_score_reduce": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, _P, _P]),
    "smt_topk_workspace_bytes": (C.c_size_t, [C.c_int64]),
    "smt_topk_blocks": (C.c_int, [_P, _P, _P, C.c_int64, _P, _P, _P, C.c_int, _P, _P, C.c_size_t, _P]),
    "smt_block_gather": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, _P, _P]),
    "smt_block_scatter": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, _P, _P]),
    "smt_channel_gather": (C.c_int, [_P, C.c_int64, C.c_int64, _P, C.c_int, C.c_int, _P, _P]),
    "smt_column_gather": (C.c_int, [_P, C.c_int64, C.c_int, C.c_int, _P, C.c_int, C.c_int, _P, _P]),
    "smt_column_scatter": (C.c_int, [_P, C.c_int64, C.c_int, C.c_int, _P, C.c_int, C.c_int, _P, _P]),
    "smt_block_grad_gemm_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int64, C.c_int]),
    "smt_block_grad_gemm": (C.c_int, [_P, C.c_int64, C.c_int, _P, C.c_int64, C.c_int, C.c_int64, C.c_int,
                                      _P, C.c_int, C.c_int, _P, C.c_int, C.c_int, _P, C.c_size_t, _P]),
    "smt_block_grad_gemm_run_width": (C.c_int, [C.c_int]),
    "smt_block_grad_gemm_runs_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int64]),
    "smt_block_grad_gemm_runs": (C.c_int, [_P, C.c_int64, C.c_int, _P, C.c_int64, C.c_int, C.c_int64, C.c_int,
                                           _P, C.c_int, C.c_int, _P, C.c_int, C.c_int, _P, C.c_size_t, _P]),
    "smt_debug_set_gemm_trace": (C.c_int, [_P, C.c_int]),
    "smt_encode_operand_map": (C.c_int, [_P, _P, C.c_int64, C.c_int64, C.c_int64, C.c_int, C.c_int]),
    "smt_block_grad_gemm_grouped_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int64]),
    "smt_block_grad_gemm_grouped_uses_2sm": (C.c_int, [C.c_int, C.c_int, C.c_int64]),
    "smt_block_grad_gemm_grouped_emits_sq": (C.c_int, [C.c_int, C.c_int, C.c_int64]),
    "smt_block_grad_gemm_grouped": (C.c_int, [_P, _P, C.c_int, C.c_int64, C.c_int, C.c_int, _P, C.c_int,
                                              C.c_int, C.c_int64, _P, _P, C.c_size_t, _P]),
    "smt_block_grad_gemm_plan": (C.c_int, [C.c_int, C.c_int, C.c_int64, C.c_int, C.POINTER(C.c_int),
                                           C.POINTER(C.c_int)]),
    "smt_fused_linear_supported": (C.c_int, [C.c_int, _P, C.c_int, C.c_int, C.c_int]),
    "smt_fused_linear_forward": (C.c_int, [_P, C.c_int64, C.c_int64, C.c_int, C.c_int, _P, _P, _P, _P, _P, C.c_int, _P]),
    "smt_fused_linear_dgrad": (C.c_int, [_P, _P, C.c_int64, C.c_int, C.c_int, _P, _P, _P, _P, C.c_int64, C.c_int, _P]),
    "smt_rmsnorm_forward": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int, C.c_float, _P, _P, _P, _P]),
    "smt_rmsnorm_backward": (C.c_int, [_P, _P, _P, _P, _P, C.c_int64, C.c_int, _P, _P]),
    "smt_rope_forward": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int64, _P, _P, _P]),
    "smt_rope_backward": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int64, _P, _P, _P]),
    "smt_swiglu_forward": (C.c_int, [_P, _P, C.c_int64, _P, _P]),
    "smt_swiglu_backward": (C.c_int, [_P, _P, _P, C.c_int64, _P, _P, _P]),
    "smt_cross_entropy_rows": (C.c_int, [_P, C.c_int64, C.c_int64, C.c_int, _P, C.c_int64, _P, _P, _P]),
    "smt_grad_sqnorm_workspace_bytes": (C.c_size_t, []),
    "smt_grad_sqnorm": (C.c_int, [_P, C.c_int, C.c_int64, _P, _P, C.c_size_t, _P]),
    "smt_compact_adam": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_int64,
                                   C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float,
                                   C.c_float, _P, C.c_int, C.c_float, _P, C.c_int, _P, C.c_int, C.c_int, C.c_int, _P]),
}
EXPORTS = tuple(_SIGNATURES)

_lib = None
_lock = threading.Lock()


def load():
    """Load libsmt_b200.so (once) and attach argument types. Raises if it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise SMTLibraryError(
                f"{LIB_PATH} not found: build it with `python -m sparse_matrix_tuning_b200.build` "
                "(or __graft_entry__.build()). There is no CPU fallback.")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError here = header/library mismatch
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().smt_last_error().decode("utf-8", "replace")
        raise SMTLibraryError(f"{what} failed (code {rc}): {msg}")


def dtype_id(dt: torch.dtype) -> int:
    try:
        return _DTYPE_IDS[dt]
    except KeyError:
        raise SMTLibraryError(f"unsupported dtype {dt} (float32 / bfloat16 / float16 only)") from None


def stream_ptr(device=None) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def require_cuda(*tensors: torch.Tensor) -> None:
    current = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise SMTLibraryError("SMT kernels need CUDA tensors; there is no CPU path "
                                  f"(got a tensor on {t.device})")
        if current is None:
            current = torch.cuda.current_device()
        if t.device.index != current:
            # the library launches on the calling thread's current device (one process per GPU)
            raise SMTLibraryError(f"tensor on {t.device} but the current CUDA device is cuda:{current}; "
                                  "call torch.cuda.set_device / use torch.cuda.device(...) around the op")


def ptr(t) -> int:
    return 0 if t is None else t.data_ptr()


def device_info():
    lib = load()
    a, b, c = C.c_int(), C.c_int(), C.c_int()
    check(lib.smt_device_info(C.byref(a), C.byref(b), C.byref(c)), "smt_device_info")
    return a.value, b.value, c.value
