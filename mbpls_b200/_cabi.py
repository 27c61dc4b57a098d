"""ctypes binding of ``libmbpls_b200.so`` (the C ABI declared in ``include/mbpls_b200.h``).

The library is the product's only compute path: if it is missing, or a call returns a non-zero
status, this module raises -- there is no CPU / PyTorch fallback.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libmbpls_b200.so")

ABI_VERSION = 16

# indices shared with the header
SCAL_UU, SCAL_DIFF, SCAL_TT, SCAL_VV, SCAL_COUNT = 0, 1, 2, 3, 8
CTRL_DONE, CTRL_TRIPS, CTRL_ERROR, CTRL_COUNT = 0, 1, 2, 4
NORM_L2, NORM_L1, NORM_MAX, NORM_MIN = 0, 1, 2, 3

_p = C.c_void_p
_i = C.c_int
_l = C.c_long
_d = C.c_double


class EpilogueArgs(C.Structure):
    _fields_ = [
        ("n", _i), ("B", _i), ("q", _i), ("nanmode", _i), ("norm_kind", _i),
        ("ldt", _l), ("ldf", _l),
        ("max_tol", _d),
        ("red", _p), ("Yt", _p), ("row_flag", _p), ("ycol_flag", _p),
        ("T", _p), ("u", _p), ("ts", _p), ("ts_old", _p), ("a", _p), ("v", _p),
        ("scal", _p), ("ctrl", _p), ("diff_trace", _p), ("diff_trace_len", _i),
    ]


class XchgArgs(C.Structure):
    _fields_ = [
        ("epi", EpilogueArgs),
        ("Tnum", _p), ("Tden", _p), ("ldp", _l), ("block_split_off", _p), ("norm_part", _p), ("n_norm_parts", _i),
        ("world", _i), ("rank", _i),
        ("peer_bufs", _p), ("slot_elems", _l), ("flags_off", _l), ("seq", C.c_ulonglong), ("counters", _p), ("work", _p),
        ("epoch", C.c_ulonglong), ("tpi", _i), ("ch", _i),
    ]


class SmallFitArgs(C.Structure):
    _fields_ = [
        ("n_src", _i), ("p", _i), ("B", _i), ("q", _i), ("K", _i), ("nfits", _i),
        ("ldx", _l), ("Xsrc", _p), ("Ysrc", _p), ("block_off", _p),
        ("standardize", _i), ("norm_kind", _i), ("max_iter", _i), ("max_tol", _d),
        ("train_idx", _p), ("train_cnt", _p), ("ld_idx", _l),
        ("test_idx", _p), ("test_cnt", _p), ("ld_tidx", _l),
        ("ldw", _l),
        ("Xw", _p), ("Yw", _p), ("stats", _p), ("Wt", _p), ("W", _p), ("P", _p), ("Ts", _p), ("U", _p), ("Tb", _p),
        ("small", _p), ("R", _p), ("beta", _p), ("preds", _p), ("scratch", _p), ("scratch_stride", _l),
        ("ytrain_idx", _p), ("fit_preds", _p), ("nslots", _i), ("ticket", _p),
    ]


class RecordArgs(C.Structure):
    _fields_ = [
        ("n", _i), ("p", _i), ("B", _i), ("q", _i), ("nanmode", _i),
        ("ldt", _l), ("T_block_stride", _l),
        ("block_off", _p),
        ("w", _p), ("red", _p), ("T", _p), ("ts", _p), ("u", _p), ("v", _p), ("a", _p),
        ("Wt_k", _p), ("W_k", _p), ("Ts_k", _p), ("U_k", _p), ("T_k", _p), ("V_k", _p), ("A_k", _p),
        ("only_if_done", _p),
    ]


# name -> argtypes; every function returns int.  Keep in sync with include/mbpls_b200.h
# (tests/test_cabi.py parses the header and checks that every declared symbol is exported and listed here).
SIGNATURES = {
    "mbpls_abi_version": [],
    "mbpls_transpose_in_f64": [_p, _l, _i, _i, _p, _l, _i, _p],
    "mbpls_transpose_in_f32": [_p, _l, _i, _i, _p, _l, _i, _p],
    "mbpls_transpose_out_f64": [_p, _l, _i, _i, _p, _l, _i, _p],
    "mbpls_nan_census_f64": [_p, _l, _i, _i, _p, _i, _p, _p, _l, _p, _p],
    "mbpls_standardize_fit_f64": [_p, _l, _i, _i, _p, _p, _p, _p, _p, _i, _p],
    "mbpls_standardize_apply_f64": [_p, _l, _i, _i, _p, _p, _p],
    "mbpls_scaler_inverse_f64": [_p, _l, _i, _i, _p, _p, _p],
    "mbpls_feature_sumsq_f64": [_p, _l, _i, _i, _p, _p],
    "mbpls_scaler_finish_f64": [_p, _p, _p, _d, _p, _p, _i, _p],
    "mbpls_segsum_f64": [_p, _p, _i, _p, _p],
    "mbpls_xtu_feats_per_cta": [_i],
    "mbpls_xtu_num_ctas": [_i],
    "mbpls_xw_ctas_per_sm": [],
    "mbpls_nipals_xtu_f64": [_p, _l, _i, _i, _p, _p, _p, _i, _p, _p, _i, _p, _p],
    "mbpls_block_sumsq_parts_f64": [_p, _i, _p, _i, _p, _p, _p],
    "mbpls_nipals_xw_f64": [_p, _l, _i, _p, _p, _p, _i, _p, _p, _l, _i, _p, _p],
    "mbpls_nipals_reduce_partials_f64": [_p, _p, _l, _i, _i, _p, _p, _i, _p, _i, _p, _p],
    "mbpls_nipals_begin_component_f64": [_p, _i, _p, _p, _p, _p],
    "mbpls_nipals_epilogue_f64": [C.POINTER(EpilogueArgs), _p],
    "mbpls_nipals_xchg_epilogue_f64": [C.POINTER(XchgArgs), _i, _p],
    "mbpls_nipals_record_component_f64": [C.POINTER(RecordArgs), _p],
    "mbpls_smallfit_scratch_doubles": [_i, _i, _l],
    "mbpls_smallfit_nipals_f64": [C.POINTER(SmallFitArgs), _p],
    "mbpls_loadings_deflate_f64": [_p, _l, _i, _i, _p, _p, _p, _p, _p, _p, _i, _i, _p],
    "mbpls_fused_workers_per_sm_pair": [_l],
    "mbpls_fused_total_workers": [_l],
    "mbpls_fused_uses_clusters": [_l],
    "mbpls_nipals_fused_trip_f64": [_p, _l, _i, _p, _p, _p, _p, _p, _p, _i, _i, _p, _p, _p, _l, _p, _p],
    "mbpls_fused_standardize_f64": [_p, _l, _i, _p, _p, _p, _p, _p, _i, _i, _p, _p, _p, _p, _p, _p, _p, _p, _l, _p],
    "mbpls_fused_deflate_f64": [_p, _l, _i, _p, _p, _p, _p, _p, _p, _p, _p, _i, _i, _p, _p, _p, _p, _p, _l, _p, _p],
    "mbpls_vec_dot_f64": [_p, _p, _i, _p, _p],
    "mbpls_nan_bitmask_ldw": [_i],
    "mbpls_nan_bitmask_f64": [_p, _l, _i, _i, _p, _l, _p],
    "mbpls_masked_colden_f64": [_p, _l, _i, _i, _p, _p, _p, _p, _i, _p, _p, _p],
    "mbpls_masked_rowden_f64": [_p, _l, _i, _p, _p, _p, _i, _p, _l, _p, _p],
    "mbpls_gram_num_chunks": [_i],
    "mbpls_gram_partial_f64": [_p, _l, _i, _p, _l, _i, _i, _p, _p],
    "mbpls_reduce_chunks_f64": [_p, _i, _i, _p, _p],
    "mbpls_right_multiply_f64": [_p, _l, _i, _i, _p, _p, _i, _p, _l, _p],
    "mbpls_skinny_gemm_f64": [_p, _l, _i, _p, _l, _i, _p, _p, _i, _p, _l, _p, _p, _p, _p],
    "mbpls_skinny_gemm_tall_f64": [_p, _l, _i, _i, _p, _i, _p, _l, _p, _p],
    "mbpls_rank1_update_f64": [_p, _l, _i, _i, _p, _p, _p],
    "mbpls_rows_sumsq_f64": [_p, _l, _i, _i, _p, _p],
    "mbpls_rows_scale_f64": [_p, _l, _i, _i, _p, _i, _p],
    "mbpls_xt_multi_f64": [_p, _l, _i, _i, _p, _l, _i, _p, _l, _p],
    "mbpls_xt_multi_chunks": [_i, _i],
    "mbpls_xt_multi_split_f64": [_p, _l, _i, _i, _p, _l, _i, _p, _l, _i, _p],
    "mbpls_lincomb_sub_f64": [_p, _p, _p, _l, _i, _p, _i, _p],
    "mbpls_center_normalize_f64": [_p, _i, _i, _i, _p, _p],
    "mbpls_block_sumsq_f64": [_p, _p, _i, _p, _p],
    "mbpls_scale_by_block_f64": [_p, _p, _i, _p, _p, _i, _p],
    "mbpls_crossprod_splits": [_i, _i, _l],
    "mbpls_crossprod_splits_syrk": [_i, _l],
    "mbpls_crossprod_f64": [_p, _l, _p, _l, _i, _i, _l, _i, _i, _p, _l, _i, _p],
    "mbpls_symmetrize_f64": [_p, _l, _i, _p],
    "mbpls_small_top_eigvec_f64": [_p, _l, _i, _p, _p],
    "mbpls_small_pinv_f64": [_p, _l, _i, _d, _p, _l, _p],
    "mbpls_small_top_sv_product_f64": [_p, _l, _p, _l, _i, _p, _p],
    "mbpls_dense_gemv_f64": [_p, _l, _i, _i, _p, _p, _p],
    "mbpls_dense_rank2_f64": [_p, _l, _i, _i, _p, _p, _p, _d, _d, _d, _i, _i, _p],
}

# functions whose int return value is a plain number, not a status
_PLAIN = {"mbpls_abi_version", "mbpls_smallfit_scratch_doubles", "mbpls_fused_workers_per_sm_pair", "mbpls_fused_total_workers", "mbpls_fused_uses_clusters", "mbpls_nan_bitmask_ldw", "mbpls_xtu_feats_per_cta", "mbpls_xtu_num_ctas", "mbpls_gram_num_chunks",
          "mbpls_xw_ctas_per_sm", "mbpls_crossprod_splits", "mbpls_crossprod_splits_syrk", "mbpls_xt_multi_chunks"}


class MbplsCudaError(RuntimeError):
    pass


_lib = None
launch_count = 0  # kernel-launching entry-point calls since import (bench.py reports the delta as gpu_launches)


def load():
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise MbplsCudaError(
            f"{LIB_PATH} not found: the CUDA library has not been built "
            "(run `python -c 'import __graft_entry__ as g; g.build()'`). mbpls_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = C.c_int
    if lib.mbpls_abi_version() != ABI_VERSION:
        raise MbplsCudaError("ABI version mismatch between _cabi.py and libmbpls_b200.so; rebuild")
    _lib = lib
    return lib


def call(name: str, *args) -> int:
    """Invoke an entry point; status-returning functions raise on failure."""
    global launch_count
    lib = load()
    rc = getattr(lib, name)(*args)
    if name in _PLAIN:
        return rc
    launch_count += 1
    if rc != 0:
        if rc >= 1000:
            raise MbplsCudaError(f"{name}: CUDA error {rc - 1000}")
        raise MbplsCudaError(f"{name}: invalid argument (status {rc})")
    return 0
