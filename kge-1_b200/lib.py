"""ctypes binding of the C-ABI library (include/kgeb200.h -> libkgeb200.so).

PyTorch is used only for device memory and streams: every call passes raw device pointers, sizes
and the current CUDA stream.  There is no CPU path and no fallback: a missing library or a
non-CUDA tensor is an error.
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libkgeb200.so")

OK, ERR_ARG, ERR_CUDA, ERR_UNSUPPORTED = 0, 1, 2, 3
MODELS = {"distmult": 0, "complex": 1, "cp": 2, "simple": 3, "rescal": 4, "transe": 5, "rotate": 6}
SP_, _PO = 0, 1
DOT, NEG_L1, NEG_L2, ROT_L1, ROT_L2 = 0, 1, 2, 3, 4
LOSS_KL, LOSS_BCE = 0, 1
MATH_FP32, MATH_TF32, MATH_BF16 = 0, 1, 2
BWD_OVERWRITE_TABLE = 1

_c = ctypes
_p, _i, _l, _f, _u = _c.c_void_p, _c.c_int, _c.c_int64, _c.c_float, _c.c_uint64

# name -> argtypes, exactly the declarations of include/kgeb200.h (checked by tests/test_abi.py)
SIGNATURES = {
    "kgeb_gather_rows": [_p, _l, _i, _p, _i, _l, _p, _p],
    "kgeb_gather_rows_shard": [_p, _l, _l, _i, _p, _i, _l, _p, _p, _p],
    "kgeb_score_spo": [_i, _i, _p, _p, _p, _p, _p, _p, _i, _l, _i, _p, _p],
    "kgeb_score_spo_bwd": [_i, _i, _p, _p, _p, _p, _p, _p, _i, _l, _i, _p, _p, _p, _p, _p],
    "kgeb_query_build": [_i, _i, _p, _p, _p, _p, _p, _i, _l, _i, _p, _p],
    "kgeb_query_bwd": [_i, _i, _p, _p, _p, _p, _p, _i, _l, _i, _p, _p, _p, _p],
    "kgeb_pairs_score": [_i, _p, _p, _p, _i, _l, _l, _i, _p, _p],
    "kgeb_pairs_bwd": [_i, _p, _p, _p, _i, _l, _l, _i, _p, _p, _p, _p, _p],
    "kgeb_ns_candidates": [_p, _p, _l, _l, _p, _p],
    "kgeb_ns_loss": [_i, _p, _l, _l, _f, _f, _p, _p, _p],
    "kgeb_score_all": [_i, _i, _p, _l, _i, _p, _p, _i, _l, _p, _l, _l, _p],
    "kgeb_score_all_bwd": [_i, _p, _l, _i, _p, _p, _i, _l, _p, _p, _l, _l, _p, _p, _p],
    "kgeb_fused_fwd": [_i, _i, _p, _l, _i, _p, _l, _l, _l, _p, _p, _l, _f, _f, _p, _p, _p, _l, _p],
    "kgeb_fused_bwd": [_i, _i, _p, _l, _i, _p, _l, _l, _l, _p, _p, _l, _p, _f, _f, _p, _f, _p, _p, _p, _p, _p, _i, _p, _l, _p],
    "kgeb_fused_flash_fwd": [_p, _l, _i, _p, _l, _l, _l, _p, _p, _l, _p, _p, _p, _p, _p, _l, _p],
    "kgeb_fused_flash_dq": [_p, _l, _i, _p, _l, _l, _p, _p, _l, _p, _p, _f, _p, _p, _p, _p, _l, _p],
    "kgeb_fused_label_rows": [_i, _p, _l, _i, _p, _l, _l, _p, _p, _l, _p, _f, _f, _p, _p, _p, _l, _p],
    "kgeb_fused_label_rows_to": [_i, _p, _l, _i, _p, _l, _l, _p, _p, _l, _p, _f, _f, _p, _p, _l, _p, _p, _l, _p],
    "kgeb_touched_capacity": [],
    "kgeb_touched_build": [_p, _l, _p, _l, _p, _l, _l, _p, _p, _p, _p, _p, _p],
    "kgeb_fused_bwd_update": [_i, _p, _l, _i, _p, _l, _l, _l, _p, _f, _f, _p, _f, _p, _p, _p, _f, _f, _p, _p, _p, _p, _l, _p],
    "kgeb_touched_update": [_p, _p, _p, _p, _p, _p, _l, _p, _p, _i, _f, _f, _p, _p],
    "kgeb_fused_bwd_update_sched": [_i, _p, _l, _i, _p, _l, _l, _l, _p, _f, _f, _p, _f, _p, _p, _p, _p, _f, _p, _p, _p, _p, _l,
                                    _p],
    "kgeb_touched_update_sched": [_p, _p, _p, _p, _p, _p, _l, _p, _p, _i, _p, _f, _p, _p],
    "kgeb_onevsall_batch_build": [_p, _l, _l, _l, _p, _p, _p, _p, _p, _p, _p, _p, _p],
    "kgeb_onevsall_batch_build_inv": [_p, _l, _l, _l, _p, _p, _p, _p, _p, _p, _p, _p, _l, _p],
    "kgeb_fused_bwd_wait_tiles": [_p],
    "kgeb_to_bf16": [_p, _p, _l, _p],
    "kgeb_loss_from_rowstat": [_i, _p, _p, _l, _f, _l, _f, _p, _p, _p, _p],
    "kgeb_zero_if": [_p, _p, _l, _p],
    "kgeb_loss_report": [_p, _p, _l, _p, _p],
    "kgeb_loss_report_inv": [_p, _p, _p, _l, _l, _p, _p],
    "kgeb_rank_count": [_i, _i, _p, _l, _i, _p, _l, _l, _p, _p, _i, _p, _p, _p, _p, _p, _p],
    "kgeb_scatter_add_rows": [_p, _i, _p, _l, _i, _p, _l, _p, _l, _p],
    "kgeb_scatter_add_rows_perm": [_p, _i, _p, _p, _l, _i, _p, _l, _p, _l, _p],
    "kgeb_segment_reduce_rows": [_p, _i, _p, _l, _i, _p, _p, _p, _p, _l, _p],
    "kgeb_adagrad_dense": [_p, _p, _p, _p, _l, _f, _f, _f, _p, _p],
    "kgeb_adagrad_dense_sched": [_p, _p, _p, _p, _l, _p, _f, _f, _p, _p],
    "kgeb_adagrad_rows": [_p, _p, _p, _p, _p, _l, _i, _f, _f, _p],
    "kgeb_adam_dense": [_p, _p, _p, _p, _l, _f, _f, _f, _f, _f, _f, _f, _p],
    "kgeb_csr_lookup": [_p, _l, _p, _l, _p, _p],
    "kgeb_filter_csr_count": [_p, _p, _i, _p, _p, _p, _i, _l, _p, _p, _p],
    "kgeb_filter_csr_fill": [_p, _p, _i, _l, _p, _p, _p, _p, _p],
    "kgeb_kvsall_batch_count": [_p, _p, _p, _l, _p, _p, _p, _p, _p],
    "kgeb_kvsall_batch_fill": [_p, _p, _p, _l, _p, _l, _p, _p, _p],
    "kgeb_kvsall_batch_build": [_p, _p, _p, _l, _l, _l, _l, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _l, _p],
    "kgeb_kvsall_batch_build_inv": [_p, _p, _p, _l, _l, _l, _l, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _l, _l, _p],
    "kgeb_philox_words": [_u, _u, _u, _l, _p, _p],
    "kgeb_philox_advance": [_p, _u, _p],
    "kgeb_sample_uniform": [_p, _l, _l, _p, _p],
    "kgeb_sample_filter": [_p, _l, _p, _p, _p, _l, _l, _p, _p, _p],
    "kgeb_sample_shared": [_p, _l, _p, _l, _l, _i, _p, _p, _p, _l, _p],
    "kgeb_lp_penalty_dense": [_p, _l, _i, _f, _p, _p, _p, _l, _p],
    "kgeb_lp_penalty_rows": [_p, _l, _i, _p, _i, _l, _i, _f, _p, _p, _p, _l, _p],
    "kgeb_adagrad_dense_lp": [_p, _p, _p, _p, _l, _f, _f, _f, _i, _f, _p, _p, _p, _l, _p],
    "kgeb_adagrad_dense_lp_sched": [_p, _p, _p, _p, _l, _p, _f, _f, _i, _f, _p, _p, _p, _l, _p],
    "kgeb_rank_hist": [_p, _p, _l, _l, _p, _p, _p],
    "kgeb_isin_sorted": [_p, _i, _l, _p, _l, _p, _p],
    "kgeb_rank_metrics": [_p, _l, _p, _i, _p, _p, _l, _p],
    "kgeb_ns_fused": [_i, _i, _p, _p, _p, _l, _l, _i, _f, _f, _p, _p, _p, _p, _p],
    "kgeb_ns_bwd_q": [_i, _p, _p, _p, _l, _l, _i, _p, _p, _p, _p],
    "kgeb_ns_cand_grad": [_i, _p, _p, _p, _l, _l, _i, _p, _p, _l, _p, _p, _l, _p],
    "kgeb_p2p_exchange": [_p, _p, _p, _i, _i, _p, _p, _p, _p, _p, _l, _p, _p, _l, _p, _f, _f, _p],
    "kgeb_p2p_exchange_sched": [_p, _p, _p, _i, _i, _p, _p, _p, _p, _p, _l, _p, _p, _l, _p, _p, _f, _p],
    "kgeb_p2p_allreduce": [_p, _p, _i, _i, _p, _p, _l, _i, _p, _p],
    "kgeb_p2p_apply": [_p, _p, _i, _i, _p, _p, _p, _p, _p, _l, _p, _l, _p],
}


class IndexDesc(ctypes.Structure):
    """kgeb_index_t of include/kgeb200.h: one KvsAllIndex resident on the device."""
    _fields_ = [("keys", _c.c_void_p), ("num_keys", _c.c_int64), ("offsets", _c.c_void_p), ("values", _c.c_void_p)]


def ptr_array(ptrs) -> "ctypes.Array":
    """Host array of device pointers (the `const void* const*` arguments of the kgeb_p2p_* entry points)."""
    return (ctypes.c_void_p * len(ptrs))(*[int(p) for p in ptrs])


def index_descs(arrays) -> "ctypes.Array":
    """Host array of kgeb_index_t from [(keys [K,2], offsets [K+1], values)] int64 CUDA tensors."""
    out = (IndexDesc * len(arrays))()
    for d, (keys, offsets, values) in zip(out, arrays):
        for t in (keys, offsets, values):
            if not t.is_cuda or t.dtype != torch.int64 or not t.is_contiguous():
                raise ValueError("index arrays must be contiguous int64 CUDA tensors")
        d.keys, d.num_keys, d.offsets, d.values = keys.data_ptr(), keys.shape[0], offsets.data_ptr(), values.data_ptr()
    return out
_INT64_RESULT = {"kgeb_fused_workspace_bytes": [_l, _i, _l, _l], "kgeb_scatter_workspace_bytes": [_l, _i],
                 "kgeb_kvsall_build_workspace_bytes": [_l, _l], "kgeb_sample_shared_workspace_bytes": [_l],
                 "kgeb_penalty_workspace_bytes": [_l, _l], "kgeb_rank_metrics_workspace_bytes": [],
                 "kgeb_ns_segment_workspace_bytes": [_l]}

_lib: Optional[ctypes.CDLL] = None


def load() -> ctypes.CDLL:
    """Loads libkgeb200.so (built in-tree by __graft_entry__.build()); raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("KGEB200_LIB", LIB_PATH)   # tuning builds (tools/build_variant.sh); default = in-tree library
    if not os.path.exists(path):
        raise ImportError(
            f"{path} not found: the CUDA extension is not built (run `python -c 'import __graft_entry__ as g; "
            "g.build()'` or kge-1_b200/csrc/build.sh).  There is no CPU fallback.")
    lib = ctypes.CDLL(path)
    for name, args in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = _i
    for name, args in _INT64_RESULT.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = _l
    lib.kgeb_last_error.restype = _c.c_char_p
    lib.kgeb_version.argtypes = [_c.c_char_p, _i]
    lib.kgeb_version.restype = _i
    _lib = lib
    return lib


def version() -> str:
    buf = ctypes.create_string_buffer(128)
    load().kgeb_version(buf, 128)
    return buf.value.decode()


def check(status: int) -> None:
    if status == OK:
        return
    msg = load().kgeb_last_error().decode()
    if status == ERR_ARG:
        raise ValueError(msg)
    if status == ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    raise RuntimeError(msg)


def call(name: str, *args) -> None:
    check(getattr(load(), name)(*args))


# ---------------------------------------------------------------------------------------------
# tensor helpers
# ---------------------------------------------------------------------------------------------
def stream_ptr(t: torch.Tensor) -> int:
    return torch.cuda.current_stream(t.device).cuda_stream


def f32(t: torch.Tensor, name: str = "tensor") -> int:
    """Device pointer of a contiguous fp32 CUDA tensor (ValueError otherwise, like the reference's checks)."""
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise ValueError(f"{name} must be a CUDA tensor (no CPU path exists)")
    if t.dtype != torch.float32:
        raise ValueError(f"{name} must be float32 (got {t.dtype})")
    if not t.is_contiguous():
        raise ValueError(f"{name} must be contiguous")
    return t.data_ptr()


def idx(t: Optional[torch.Tensor], name: str = "indexes"):
    """(device pointer, is64) of a 1-D/2-D contiguous int32/int64 CUDA index tensor; (None, 0) for None."""
    if t is None:
        return None, 0
    if not t.is_cuda:
        raise ValueError(f"{name} must be a CUDA tensor")
    if t.dtype not in (torch.int32, torch.int64):
        raise ValueError(f"{name} must be int32 or int64 (got {t.dtype})")
    if not t.is_contiguous():
        raise ValueError(f"{name} must be contiguous")
    return t.data_ptr(), int(t.dtype == torch.int64)


def i64(t: Optional[torch.Tensor], name: str = "tensor"):
    if t is None:
        return None
    if not t.is_cuda or t.dtype != torch.int64 or not t.is_contiguous():
        raise ValueError(f"{name} must be a contiguous int64 CUDA tensor")
    return t.data_ptr()


def same_index_width(*tensors):
    """The C-ABI takes one idx64 flag per call: cast all index tensors to the widest dtype present."""
    present = [t for t in tensors if t is not None]
    wide = any(t.dtype == torch.int64 for t in present)
    out = []
    for t in tensors:
        if t is None:
            out.append(None)
        else:
            if t.dtype not in (torch.int32, torch.int64):
                raise ValueError(f"indexes must be int32 or int64 (got {t.dtype})")
            out.append(t.contiguous() if (t.dtype == torch.int64) == wide else t.long().contiguous())
    return out
