"""ctypes binding of the C ABI in ``include/hicgat.h`` (libhicgat_sm100.so).

The library is loaded lazily on first use and there is NO fallback: if it is missing the
call raises, it never routes to a CPU or PyTorch implementation.
"""
from __future__ import annotations

import ctypes as C
import os
import re

_PKG = os.path.dirname(os.path.abspath(__file__))
# HICGAT_LIB: A/B another build of the same ABI (kernel experiments); default = the in-tree library
LIB_PATH = os.environ.get("HICGAT_LIB") or os.path.join(_PKG, "libhicgat_sm100.so")
HEADER = os.path.join(os.path.dirname(_PKG), "include", "hicgat.h")

_p, _i64, _i32, _u32, _u64, _f32, _f64, _sz = C.c_void_p, C.c_int64, C.c_int, C.c_uint32, C.c_uint64, C.c_float, C.c_double, C.c_size_t

# name -> (restype, argtypes); mirrors include/hicgat.h one to one
SIGNATURES = {
    "hicgat_version": (C.c_int, []),
    "hicgat_last_error": (C.c_char_p, []),
    "hicgat_launch_count": (C.c_uint64, []),
    "hicgat_memcpy2d_h2d_async": (C.c_int, [_p, _sz, _p, _sz, _sz, _sz, _p]),
    "hicgat_pairloss_workspace_bytes": (_sz, [_i64, _i64, _i64]),
    "hicgat_pairloss_estimate_cost": (_f64, [_i64, _i64, _i64, _u32]),
    "hicgat_pairloss_workspace_bytes_mode": (_sz, [_i64, _i64, _i64, _u32]),
    "hicgat_pairloss_fwd_bwd": (C.c_int, [_p, _p, _i64, _i64, _i64, _i64, _u32, _f32, _f32, _p, _p, _p, _sz, _p]),
    "hicgat_pairloss_fwd_bwd_packed": (C.c_int, [_p, _p, _i64, _i64, _i64, _i64, _u32, _f32, _f32, _p, _p, _sz, _p]),
    "hicgat_pairloss_set_tuning": (C.c_int, [_i32, _i32]),
    "hicgat_pairloss_set_combine": (C.c_int, [_i32, _i32]),
    "hicgat_pairloss_set_schedule": (C.c_int, [_i32, _i32]),
    "hicgat_pairloss_describe_schedule": (C.c_int, [_i64, _i64, _i64, _p, _i32]),
    "hicgat_pairloss_describe_schedule_mode": (C.c_int, [_i64, _i64, _i64, _u32, _p, _i32]),
    "hicgat_pairloss_sparse_workspace_bytes": (_sz, [_i64, _i64, _i64]),
    "hicgat_pairloss_sparse_fwd_bwd": (C.c_int, [_p, _p, _p, _p, _f32, _i64, _i64, _i64, _u32, _f32, _f32, _p, _p, _p, _sz, _p]),
    "hicgat_pairloss_pearson_grad": (C.c_int, [_p, _p, _i64, _i64, _i64, _i64, _u32, _p, _f32, _i32, _p, _p, _sz, _p]),
    "hicgat_pairloss_sparse_pearson_grad": (C.c_int, [_p, _p, _p, _p, _f32, _i64, _i64, _i64, _u32, _p, _f32, _i32, _p, _p, _sz, _p]),
    "hicgat_asymmetry_f32": (C.c_int, [_p, _i64, _i64, _i64, _i64, _p, _p]),
    "hicgat_asymmetry_f64": (C.c_int, [_p, _i64, _i64, _i64, _i64, _p, _p]),
    "hicgat_pairloss_rowside_add": (C.c_int, [_p, _p, _i64, _i64, _i64, _i64, _f32, _p, _p]),
    "hicgat_allreduce_partials_p2p": (C.c_int, [_p, _p, _i32, _i32, _i64, _i64, _i32, _u32, _p, _p, _p, _p]),
    "hicgat_allreduce_partials_twoshot": (C.c_int, [_p, _p, _p, _i32, _i32, _i64, _i32, _p, _p, _p, _p]),
    "hicgat_rank_histograms": (C.c_int, [_p, _p, _i64, _i64, _i64, _i64, _f32, _f32, _i32, _p, _p, _p]),
    "hicgat_rank_cross_sum": (C.c_int, [_p, _p, _i64, _i64, _i64, _i64, _f32, _f32, _i32, _p, _p, _p, _p]),
    "hicgat_dist_histogram": (C.c_int, [_p, _i64, _i64, _i64, _f32, _i32, _p, _p]),
    "hicgat_edge_dist_bins": (C.c_int, [_p, _p, _p, _i64, _i64, _i64, _f32, _i32, _p, _p]),
    "hicgat_dscc_workspace_bytes": (_sz, [_i64, _i32]),
    "hicgat_dscc_target_ranks": (C.c_int, [_p, _i64, _i64, _f32, _i32, _p, _p, _p, _sz, _p]),
    "hicgat_dscc_dense": (C.c_int, [_p, _p, _i64, _i64, _f32, _i32, _p, _p, _p, _p, _sz, _p]),
    "hicgat_dscc_implicit": (C.c_int, [_p, _p, _p, _p, _i64, _p, _p, _i32, _p, _p, _sz, _p]),
    "hicgat_pairdist_fwd": (C.c_int, [_p, _i64, _p, _i64, _p]),
    "hicgat_pairdist_bwd": (C.c_int, [_p, _i64, _p, _i64, _p, _p]),
    "hicgat_cont2dist_max_f64": (C.c_int, [_p, _i64, _i64, _i64, _i64, _f64, _p, _p, _sz, _p]),
    "hicgat_cont2dist_apply_f64": (C.c_int, [_p, _i64, _i64, _i64, _i64, _f64, _p, _p, _i64, _p, _i64, _p]),
    "hicgat_cont2dist_workspace_bytes": (_sz, [_i64, _i64, _i64]),
    "hicgat_csr_count_f64": (C.c_int, [_p, _i64, _i64, _i32, _p, _p]),
    "hicgat_csr_scan_i64": (C.c_int, [_p, _i64, _p, _p]),
    "hicgat_csr_fill_f64": (C.c_int, [_p, _i64, _i64, _i32, _p, _p, _p, _p]),
    "hicgat_csr_pack_i32": (C.c_int, [_p, _p, _i64, _i64, _p, _p, _p]),
    "hicgat_csr_add_self_loops_i32": (C.c_int, [_p, _p, _i64, _p, _p, _p]),
    "hicgat_sage_norm_values": (C.c_int, [_p, _p, _p, _i64, _p, _p, _p]),
    "hicgat_spmm_csr_f32": (C.c_int, [_p, _p, _p, _p, _i64, _i64, _p, _p]),
    "hicgat_csr_transpose_perm": (C.c_int, [_p, _p, _i64, _p, _p]),
    "hicgat_gat_set_tuning": (C.c_int, [_i32, _i32]),
    "hicgat_gat_fwd": (C.c_int, [_p, _p, _i64, _i32, _i32, _p, _p, _p, _p, _f32, _p, _p, _p, _p, _p]),
    "hicgat_gat_bwd_workspace_bytes": (_sz, [_i64, _i64, _i32, _i32]),
    "hicgat_gat_logits": (C.c_int, [_i64, _i32, _i32, _p, _p, _p, _p, _p, _p]),
    "hicgat_gat_dense_mask_words": (_sz, [_i64]),
    "hicgat_gat_dense_build_mask": (C.c_int, [_p, _p, _i64, _p, _p]),
    "hicgat_gat_dense_workspace_bytes": (_sz, [_i64, _i32, _i32]),
    "hicgat_gat_dense_fwd": (C.c_int, [_p, _p, _p, _i64, _i32, _i32, _p, _p, _p, _p, _f32, _p, _p, _sz, _p]),
    "hicgat_gat_dense_bwd": (C.c_int, [_p, _i64, _i32, _i32, _p, _p, _p, _p, _p, _p, _f32, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "hicgat_gat_param_grads_workspace_bytes": (_sz, [_i64, _i32, _i32]),
    "hicgat_gat_param_grads": (C.c_int, [_i64, _i32, _i32, _p, _p, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "hicgat_split_tf32": (C.c_int, [_p, _i64, _i64, _i64, _p, _i32, _i32, _p]),
    "hicgat_gemm_tf32_workspace_bytes": (_sz, [_i64, _i64, _i64, _i32]),
    "hicgat_gemm_tf32_tn": (C.c_int, [_p, _i64, _p, _i64, _i64, _i64, _i64, _i32, _p, _p, _i64, _p, _sz, _p]),
    "hicgat_ln_relu_add_fwd": (C.c_int, [_p, _p, _p, _p, _f32, _i64, _i32, _p, _p, _p, _p]),
    "hicgat_ln_relu_add_bwd_workspace_bytes": (_sz, [_i64, _i32]),
    "hicgat_ln_relu_add_bwd": (C.c_int, [_p, _p, _p, _p, _p, _p, _i64, _i32, _p, _p, _p, _p, _sz, _p]),
    "hicgat_gemv_f64": (C.c_int, [_p, _i64, _i64, _p, _p, _p]),
    "hicgat_spmv_csr_f64": (C.c_int, [_p, _p, _p, _i64, _p, _p, _p]),
    "hicgat_kr_scale_round_f64": (C.c_int, [_p, _i64, _i64, _p, _p, _i64, _i32, _p]),
    "hicgat_gat_bwd_fused": (C.c_int, [_p, _p, _p, _i64, _i64, _i32, _i32, _p, _p, _p, _p, _f32, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "hicgat_gat_bwd": (C.c_int, [_p, _p, _p, _i64, _i64, _i32, _i32, _p, _p, _p, _f32, _p, _p, _p, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "hicgat_node2vec_walks": (C.c_int, [_p, _p, _p, _p, _i64, _i64, _i32, _f32, _f32, _u64, _p, _p]),
    "hicgat_sgns_epoch": (C.c_int, [_p, _p, _i64, _i32, _p, _p, _i64, _i32, _i32, _i32, _f64, _f64, _i32, _i32, _u64, _i64, _p, _p, _p]),
}

PAIR_GRAD_MSE, PAIR_GRAD_L1, PAIR_MOMENTS, PAIR_MOMENTS_D, PAIR_WS_CLEAN, PAIR_SYMMETRIC, PAIR_NMOM = 1, 2, 4, 8, 16, 32, 8

_lib = None


def declared_symbols() -> list[str]:
    """Every function name ``include/hicgat.h`` declares (used by the export test)."""
    text = open(HEADER).read()
    return sorted(set(re.findall(r"HICGAT_API\s+[\w\s\*]+?\b(hicgat_\w+)\s*\(", text)))


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m hic_gnn_b200.build` "
                "(there is no CPU / PyTorch fallback for the hot path)"
            )
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype, fn.argtypes = res, args
        _lib = handle
    return _lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib().hicgat_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"{what or 'hicgat'} failed (code {rc}): {msg}")


def launch_count() -> int:
    return int(lib().hicgat_launch_count())


_tuning_epoch = 0


def tuning_epoch() -> int:
    return _tuning_epoch


def set_pairloss_schedule(tail_depth: int = -1, tail_min_rows: int = 256) -> None:
    """``hicgat_pairloss_set_schedule`` + invalidation of the cached workspaces."""
    global _tuning_epoch
    check(lib().hicgat_pairloss_set_schedule(tail_depth, tail_min_rows), "hicgat_pairloss_set_schedule")
    _tuning_epoch += 1


def set_pairloss_combine(rowside_groups_max: int = 4, rowside_min_strips: int = 96) -> None:
    """``hicgat_pairloss_set_combine`` + invalidation of the cached workspaces (their size depends on it)."""
    global _tuning_epoch
    check(lib().hicgat_pairloss_set_combine(rowside_groups_max, rowside_min_strips), "hicgat_pairloss_set_combine")
    _tuning_epoch += 1


def set_pairloss_tuning(rows_per_cta: int = 0, variant: int = 0) -> None:
    """``hicgat_pairloss_set_tuning`` + invalidation of the cached workspaces (their size depends
    on the row-chunk length).  ``variant`` 0 = TMA tile ring, 1 = per-lane streaming loads."""
    global _tuning_epoch
    check(lib().hicgat_pairloss_set_tuning(rows_per_cta, variant), "hicgat_pairloss_set_tuning")
    _tuning_epoch += 1
