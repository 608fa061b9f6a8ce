"""ctypes binding of libpipegcn_b200.so (include/pipegcn_b200.h).

The hot path has no Python/torch fall-back: if the shared object is missing the
import of any op raises.  `PG_LIB` may point at an alternative build.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

PG_F32, PG_BF16 = 0, 1
PG_OK, PG_ERR_INVALID, PG_ERR_CUDA, PG_ERR_UNSUPPORTED, PG_ERR_TIMEOUT = 0, -1, -2, -3, -4
IPC_HANDLE_BYTES = 64

_LIB_PATH = Path(os.environ.get("PG_LIB", Path(__file__).resolve().parent / "libpipegcn_b200.so"))


class PgError(RuntimeError):
    pass


class pg_csr(C.Structure):
    _fields_ = [("indptr", C.c_void_p), ("indices", C.c_void_p), ("n_rows", C.c_int32), ("seg_len", C.c_int32),
                ("n_long", C.c_int32), ("n_seg", C.c_int32), ("long_row", C.c_void_p), ("long_seg_ptr", C.c_void_p),
                ("seg_long", C.c_void_p), ("row_order", C.c_void_p), ("nnz", C.c_int64),
                ("chunks", C.c_void_p), ("n_chunks", C.c_int32), ("n_chunks_long", C.c_int32),
                ("pidx", C.c_void_p), ("prow", C.c_void_p)]


class pg_gemm_src(C.Structure):
    _fields_ = [("a", C.c_void_p), ("lda", C.c_int64), ("b", C.c_void_p), ("ldb", C.c_int64), ("k", C.c_int32)]


class pg_msg(C.Structure):
    _fields_ = [("idx", C.c_void_p), ("src_row0", C.c_int64), ("n_rows", C.c_int32), ("cta_begin", C.c_int32),
                ("dst", C.c_void_p), ("ld_dst", C.c_int64), ("ema", C.c_void_p), ("ld_ema", C.c_int64),
                ("flag", C.c_void_p), ("counter", C.c_void_p), ("dst_row0", C.c_int64)]


class pg_drop(C.Structure):
    _fields_ = [("p", C.c_float), ("seed", C.c_uint64), ("step_dev", C.c_void_p), ("step_off", C.c_int32)]


def _load():
    if not _LIB_PATH.exists():
        raise PgError(f"{_LIB_PATH} is missing: build it with `python -m pipegcn_b200.build` "
                      f"(the hot path has no fall-back)")
    lib = C.CDLL(str(_LIB_PATH))
    vp, i32, i64, u32, f32 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint32, C.c_float
    sig = {
        "pg_abi_version": (C.c_int, []),
        "pg_last_error": (C.c_char_p, []),
        "pg_device_info": (C.c_int, [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(i64)]),
        "pg_set_option": (C.c_int, [C.c_char_p, C.c_int]),
        "pg_aggregate": (C.c_int, [C.POINTER(pg_csr), vp, i64, vp, i64, i32, C.c_int, vp, i32, vp, vp]),
        "pg_aggregate_drop": (C.c_int, [C.POINTER(pg_csr), vp, i64, vp, i64, i32, C.c_int, vp, i32, vp,
                                        C.POINTER(pg_drop), vp]),
        "pg_row_div": (C.c_int, [vp, i64, vp, i64, i32, i32, C.c_int, vp, vp]),
        "pg_linear": (C.c_int, [C.c_int, C.c_int, C.POINTER(pg_gemm_src), i32, vp, vp, vp, i64, i32, i32, vp]),
        "pg_linear_drop": (C.c_int, [C.c_int, C.c_int, C.POINTER(pg_gemm_src), i32, vp, vp, vp, i64, i32, i32,
                                     C.POINTER(pg_drop), i64, vp]),
        "pg_wgrad_workspace": (i64, [i32, i32, i32, C.c_int]),
        "pg_wgrad": (C.c_int, [C.c_int, C.POINTER(pg_gemm_src), i32, vp, i64, i32, i32, i32, vp, i64, vp]),
        "pg_split_tf32": (C.c_int, [vp, i64, vp, vp, i64, i32, i32, vp]),
        "pg_row_grid": (C.c_int, [i32]),
        "pg_dropout": (C.c_int, [vp, i64, vp, i64, i32, i32, C.c_int, f32, C.c_uint64, vp, vp]),
        "pg_dropout_rows": (C.c_int, [vp, i64, vp, i64, i64, i32, i32, C.c_int, C.POINTER(pg_drop), vp]),
        "pg_ln_relu_drop_fwd": (C.c_int, [vp, i64, vp, vp, f32, C.c_int, vp, i64, vp, i64, vp, vp, i32, i32, C.c_int,
                                          C.POINTER(pg_drop), vp]),
        "pg_ln_relu_fwd": (C.c_int, [vp, i64, vp, vp, f32, C.c_int, vp, i64, vp, vp, i32, i32, C.c_int, vp]),
        "pg_ln_relu_bwd": (C.c_int, [vp, i64, vp, i64, vp, i64, vp, vp, vp, C.c_int, vp, i64, vp, vp, vp, vp, i32, i32,
                                     C.c_int, vp]),
        "pg_ln_relu_bwd2": (C.c_int, [vp, i64, vp, i64, vp, i64, vp, vp, vp, vp, C.c_int, vp, i64, vp, vp, vp, vp, i32, i32,
                                      C.c_int, vp]),
        "pg_ce_fwd": (C.c_int, [vp, i64, vp, i32, i32, C.c_int, vp, vp, vp, vp]),
        "pg_ce_bwd": (C.c_int, [vp, i64, vp, vp, vp, i32, i32, i32, C.c_int, vp, i64, vp, vp, vp]),
        "pg_bce_fwd": (C.c_int, [vp, i64, vp, i32, i32, i32, C.c_int, vp, vp, vp]),
        "pg_bce_bwd": (C.c_int, [vp, i64, vp, i32, vp, i32, i32, i32, C.c_int, vp, i64, vp, vp, vp]),
        "pg_f1_counts": (C.c_int, [vp, i64, vp, i32, vp, i32, i32, C.c_int, vp, vp]),
        "pg_push_rows_per_cta":(C.c_int, []),
        "pg_halo_push": (C.c_int, [vp, i32, i32, vp, i64, i32, C.c_int, f32, f32, u32, vp, vp]),
        "pg_halo_push_drop": (C.c_int, [vp, i32, i32, vp, i64, i32, C.c_int, f32, f32, u32, vp, C.POINTER(pg_drop), vp]),
        "pg_halo_wait": (C.c_int, [vp, i32, u32, vp, i32, vp, vp, vp]),
        "pg_scale_rows": (C.c_int, [vp, i64, vp, i64, i32, i32, C.c_int, f32, C.c_int, i32, vp, vp]),
        "pg_boundary_add": (C.c_int, [vp, i64, vp, i64, i32, C.c_int, vp, vp, vp, i32, vp]),
        "pg_heap_alloc": (C.c_int, [C.c_size_t, C.POINTER(vp)]),
        "pg_heap_free": (C.c_int, [vp]),
        "pg_ipc_export": (C.c_int, [vp, C.c_char_p]),
        "pg_ipc_import": (C.c_int, [C.c_char_p, C.POINTER(vp)]),
        "pg_ipc_close": (C.c_int, [vp]),
        "pg_enable_peer_access": (C.c_int, [C.c_int]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    if lib.pg_abi_version() != 2:
        raise PgError(f"ABI version mismatch: library {lib.pg_abi_version()}, binding 2")
    return lib, tuple(sig)


lib, EXPORTS = _load()
for _k, _v in (("agg_unroll", os.environ.get("PG_AGG_UNROLL")), ("agg_pack_short", os.environ.get("PG_AGG_PACK")),
               ("agg_impl", os.environ.get("PG_AGG_IMPL")), ("agg_l2_hint", os.environ.get("PG_AGG_L2_HINT")),
               ("agg_occ", os.environ.get("PG_AGG_OCC")), ("agg_overlap", os.environ.get("PG_AGG_OVERLAP")),
               ("agg_narrow", os.environ.get("PG_AGG_NARROW")), ("ln_stage", os.environ.get("PG_LN_STAGE")),
               ("ce_subwarp", os.environ.get("PG_CE_SUBWARP")),
               ("gemm_epi_batch", os.environ.get("PG_GEMM_EPI_BATCH")),
               ("gemm_epi_slabs", os.environ.get("PG_GEMM_EPI_SLABS"))):
    if _v:
        lib.pg_set_option(_k.encode(), int(_v))


def check(rc: int, what: str = ""):
    if rc != PG_OK:
        msg = lib.pg_last_error().decode(errors="replace")
        raise PgError(f"{what or 'libpipegcn_b200'} failed ({rc}): {msg}")


def dtype_code(dtype) -> int:
    import torch
    if dtype == torch.float32:
        return PG_F32
    if dtype == torch.bfloat16:
        return PG_BF16
    raise PgError(f"unsupported activation dtype {dtype}; the hot path runs in float32 or bfloat16")


def stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


# number of kernels launched through this binding (bench.py reports it as `gpu_launches`)
LAUNCHES = 0


def count(n: int = 1):
    global LAUNCHES
    LAUNCHES += n
