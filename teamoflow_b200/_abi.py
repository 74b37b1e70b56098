"""ctypes binding of ``libtmf.so`` (the C ABI declared in ``include/tmf.h``).

The library is built in-tree (``teamoflow_b200/csrc/libtmf.so``) by ``__graft_entry__.build()``
or ``make -C teamoflow_b200/csrc``.  There is NO fallback: if the library is missing, or a
compute entry point is called without a CUDA device, this module raises.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libtmf.so")

_i32, _i64, _u64, _f32 = C.c_int32, C.c_int64, C.c_uint64, C.c_float
_p, _sz = C.c_void_p, C.c_size_t

# name -> (restype, argtypes); must list every symbol of include/tmf.h (tests/test_abi.py checks it)
SIGNATURES = {
    "tmf_abi_version": (_i32, []),
    "tmf_last_error": (C.c_char_p, []),
    "tmf_rowptr_from_sorted": (_i32, [_p, _i64, _i32, _p, _p]),
    "tmf_coo_split": (_i32, [_p, _i32, _i64, _i64, _i64, _p, _p, _p, _p]),
    "tmf_transpose_ws_bytes": (_sz, [_i64]),
    "tmf_transpose_build": (_i32, [_p, _i64, _i32, _p, _p, _p, _sz, _p]),
    "tmf_tlist_users": (_i32, [_p, _i64, _i64, _p, _i32, _p, _p]),
    "tmf_sample_items": (_i32, [_i32, _i32, _i32, _u64, _p, _p]),
    "tmf_reduce_ws_bytes": (_sz, []),
    "tmf_fill_normal": (_i32, [_p, _i64, _i32, _i32, _u64, _p]),
    "tmf_fill_uniform": (_i32, [_p, _i64, _i32, _i32, _u64, _p]),
    "tmf_l2_normalize_global": (_i32, [_p, _i64, _p, _p]),
    "tmf_spmm_ws_bytes": (_sz, [_i64, _i32]),
    "tmf_spmm_seg": (_i32, [_i32, _p, _i64, _p, _p, _p, _p, _i32, _p, _i32, _i32, _p, _sz, _p]),
    "tmf_user_pass": (_i32, [_i32, _i32, _i32, _i64, _p, _p, _p, _p, _p, _i32, _i32, _p, _i32, _i32, _p, _p, _p, _p, _p, _p, _p,
                             _p, _p, _p, _p, _p]),
    "tmf_user_pass_fixup": (_i32, [_i32, _i32, _p, _p, _p, _p, _i32, _p, _i32, _i64, _p, _p, _p, _p, _p, _p]),
    "tmf_pair_dots": (_i32, [_i64, _p, _p, _p, _p, _i32, _p, _p]),
    "tmf_kl_moments": (_i32, [_i64, _p, _p, _p, _p, _p]),
    "tmf_kl_coef_from_moments": (_i32, [_i64, _p, _p, _p, _p, _p, _p, _p]),
    "tmf_adam1": (_i32, [_p, _p, _i64, _f32, _p]),
    "tmf_adam": (_i32, [_p, _p, _p, _p, _i64, _f32, _i32, _p]),
    "tmf_reduce_sum": (_i32, [_p, _i64, _p, _p, _p]),
    "tmf_bias_add": (_i32, [_p, _i64, _i32, _i32, _p, _i32, _p]),
    "tmf_col_sum": (_i32, [_p, _i64, _i32, _i32, _p, _p, _sz, _p]),
    "tmf_relu_mask": (_i32, [_p, _p, _i64, _p]),
    "tmf_gemm_f32": (_i32, [_i32, _i32, _i32, _i32, _i32, _p, _i32, _p, _i32, _p, _i32, _p]),
    "tmf_gemm_tc_ws_bytes": (_sz, [_i64, _i64, _i64]),
    "tmf_gemm_tc": (_i32, [_i32, _i32, _i64, _i64, _i64, _p, _i64, _p, _i64, _p, _i64, _p, _sz, _p]),
    "tmf_gather_rows2d": (_i32, [_p, _i32, _i64, _p, _i32, _p, _p]),
    "tmf_gather_nd2": (_i32, [_p, _i64, _p, _i64, _p, _p]),
    "tmf_wmrb_forward": (_i32, [_i64, _p, _p, _p, _i32, _f32, _p, _p]),
    "tmf_score_topk_ws_bytes": (_sz, [_i64, _i64, _i32, _i32]),
    "tmf_score_topk": (_i32, [_p, _i64, _p, _i64, _i32, _i32, _i32, _i32, _i32, _p, _p, _p, _sz, _p]),
    "tmf_score_topk_bounded": (_i32, [_p, _i64, _p, _i64, _i32, _i32, _i32, _i32, _i32, _p, _p, _p, _p, _sz, _p]),
    "tmf_score_topk_masked": (_i32, [_p, _i64, _p, _i64, _i32, _i32, _i32, _i32, _i32, _p, _p, _p, _p, _p, _sz, _p]),
    "tmf_score_dense_tc": (_i32, [_p, _i64, _p, _i64, _i32, _i32, _i32, _p, _p, _sz, _p]),
    "tmf_topk_merge": (_i32, [_p, _p, _i32, _i64, _i32, _p, _p, _p]),
    "tmf_predict_dense": (_i32, [_p, _i64, _p, _i64, _i32, _i32, _p, _p]),
    "tmf_rank_rows_ws_bytes": (_sz, [_i64, _i64]),
    "tmf_rank_rows": (_i32, [_p, _i64, _i64, _i32, _p, _p, _sz, _p]),
    "tmf_gather_unobserved": (_i32, [_p, _i64, _i64, _p, _p, _p, _p]),
    "tmf_gather_rate": (_i32, [_p, _i64, _i32, _p, _i64, _p, _i64, _p]),
    "tmf_metrics_hits": (_i32, [_p, _i64, _i32, _p, _p, _p, _p, _p, _p]),
    "tmf_dcg": (_i32, [_p, _i64, _i32, _p, _p, _p, _p, _p]),
    "tmf_idcg": (_i32, [_i64, _i64, _i32, _p, _p, _p, _p, _p]),
    "tmf_peer_alloc": (_i32, [_sz, _p]),
    "tmf_peer_free": (_i32, [_p]),
    "tmf_ipc_export": (_i32, [_p, _p]),
    "tmf_ipc_open": (_i32, [_p, _p]),
    "tmf_ipc_close": (_i32, [_p]),
    "tmf_peer_barrier": (_i32, [_p, _i32, _i32, C.c_uint32, C.c_uint32, _p]),
    "tmf_topk_merge_peer": (_i32, [_p, _p, _i32, _i64, _i64, _i32, _p, _p, _i32, _p]),
    "tmf_peer_reduce_push": (_i32, [_p, _p, _i32, _i32, _i64, _i64, _f32, _p]),
}

_lib = None
# libtmf calls / kernels launched so far (bench.py's "gpu_launches" claim is derived from these)
call_count = 0
launch_count = 0
# kernels per ABI call where it is not 1 (memsets are not counted)
KERNELS_PER_CALL = {"tmf_spmm_seg": 2, "tmf_transpose_build": 3, "tmf_l2_normalize_global": 3, "tmf_kl_moments": 2, "tmf_kl_coef_from_moments": 2,
                    "tmf_reduce_sum": 2, "tmf_gemm_tc": 4, "tmf_col_sum": 2, "tmf_rank_rows": 2, "tmf_score_topk": 8, "tmf_score_topk_bounded": 8,
                    "tmf_score_topk_masked": 8}


class TmfError(RuntimeError):
    pass


def lib():
    """Load (once) and return the ctypes handle.  Raises if the library has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "or `make -C teamoflow_b200/csrc`. teamoflow_b200 has no CPU/PyTorch fallback.")
        h = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(h, name)
            fn.restype = res
            fn.argtypes = args
        if h.tmf_abi_version() != 1:
            raise ImportError("libtmf.so ABI version mismatch; rebuild it")
        _lib = h
    return _lib


def require_cuda():
    if not torch.cuda.is_available():
        raise TmfError("teamoflow_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")


def stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    """Device pointer of a torch tensor (None -> NULL)."""
    if t is None:
        return None
    return C.c_void_p(t.data_ptr())


def call(name, *args):
    """Invoke ``tmf_<name>`` on the current torch stream and raise on a non-zero return code."""
    global call_count, launch_count
    require_cuda()
    h = lib()
    rc = getattr(h, name)(*args, stream())
    call_count += 1
    launch_count += KERNELS_PER_CALL.get(name, 1)
    if rc != 0:
        raise TmfError(f"{name} failed ({rc}): {h.tmf_last_error().decode()}")


def call_nostream(name, *args):
    """Entry points that take no stream (peer-memory allocation / IPC mapping); raises on a non-zero return code."""
    require_cuda()
    h = lib()
    rc = getattr(h, name)(*args)
    if rc != 0:
        raise TmfError(f"{name} failed ({rc}): {h.tmf_last_error().decode()}")


def query(name, *args):
    """Size queries (no stream, no device needed)."""
    return getattr(lib(), name)(*args)
