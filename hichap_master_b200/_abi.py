"""ctypes binding of ``libhichap_b200.so`` (the C ABI declared in ``include/hichap_b200.h``).

There is no CPU fallback: if the shared library is missing the import of any
compute entry point raises, and every non-zero return code becomes a Python
exception carrying ``hc_last_error()``.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libhichap_b200.so")

HC_BIN_SYM_ALL, HC_BIN_SYM_BOTH, HC_BIN_ONESIDED = 0, 1, 2
HC_GAP_PERCENTILE, HC_GAP_FIXED = 0, 1


class HcError(RuntimeError):
    pass


class IceParams(C.Structure):
    """``hc_ice_params``; defaults are cooler's CLI defaults + HiCHap's ``--ignore-diags 1``."""
    _fields_ = [("tol", C.c_double), ("mad_max", C.c_double), ("min_nnz", C.c_int32),
                ("min_count", C.c_int32), ("ignore_diags", C.c_int32), ("max_iters", C.c_int32),
                ("rescale_marginals", C.c_int32), ("poll_every", C.c_int32)]


class IceResult(C.Structure):
    _fields_ = [("scale", C.c_double), ("var", C.c_double), ("iters", C.c_int32),
                ("converged", C.c_int32)]


class IceRunInfo(C.Structure):
    _fields_ = [("launches", C.c_int32), ("loop_ms", C.c_float), ("packed", C.c_int32), ("pack_ms", C.c_float),
                ("overflow_cells", C.c_int64), ("stream_full_ms", C.c_float), ("stream_full_launches", C.c_int32)]


_P, _I32, _I64 = C.c_void_p, C.c_int32, C.c_int64

# name -> (restype, argtypes); mirrors include/hichap_b200.h one to one
SIGNATURES = {
    "hc_version": (C.c_int, []),
    "hc_init": (C.c_int, []),
    "hc_mempool_free_bytes": (C.c_int64, []),
    "hc_last_error": (C.c_char_p, []),
    "hc_launch_count": (C.c_int64, []),
    "hc_bin_pairs_local": (C.c_int, [_P, _P, _P, _P, _P, _I64, _I32, _I32, _P, _P, _P, _P, _I32, _P, _P]),
    "hc_bin_band_work_bytes": (C.c_int64, [_I64, _I32]),
    "hc_bin_pairs_local_banded": (C.c_int, [_P, _P, _P, _P, _P, _I64, _I32, _I32, _P, _P, _P, _P, _P, _I32,
                                            C.POINTER(_I32), _I32, _P, _P, _P]),
    "hc_bin_band_begin": (C.c_int, [_P, _I64, _I32, _P]),
    "hc_bin_band_accumulate": (C.c_int, [_P, _P, _P, _P, _P, _I64, _I32, _I32, _I32, _P, _P, _P, _P, _P, _I32, _I32, _P, _P, _P]),
    "hc_bin_band_finish": (C.c_int, [_P, _P, _P, _P, _P, _I32, C.POINTER(_I32), _I32, _P, _P]),
    "hc_impute_inter": (C.c_int, [_P, _P, _P, _P, _P, _I64, _I32, _P, _P, _I32, _I32, _P, _P, _I32, _I64, _I32, _P, _P, _I32,
                                  _I64, C.c_double, _I32, _I64, _P, _P, _P]),
    "hc_widen_u8_i32": (C.c_int, [_P, _P, _I64, _P]),
    "hc_add_i32": (C.c_int, [_P, _P, _I64, _P]),
    "hc_bin_pairs_whole": (C.c_int, [_P, _P, _P, _P, _P, _I64, _I32, _I32, _P, _P, _I32, _P, _I32, _I64, _P, _P]),
    "hc_dense_nonzero_count": (C.c_int, [_P, _I64, _I32, _I32, _I32, _I32, _P, _P]),
    "hc_dense_nonzero_extract": (C.c_int, [_P, _I64, _I32, _I32, _I32, _I32, _P, _P, _P, _P, _P]),
    "hc_dense_batch_triu_count": (C.c_int, [_P, _P, _P, _P, _P, _I32, _I64, _P, _P]),
    "hc_dense_batch_triu_records": (C.c_int, [_P, _P, _P, _P, _P, _I32, _I64, _P, _P, _P]),
    "hc_ice_dense_marginals": (C.c_int, [_P, _P, _P, _P, _P, _I32, _I32, _P, _P, _P]),
    "hc_ice_filter_bins": (C.c_int, [_P, _P, _I64, _P, _I32, C.POINTER(IceParams), _P, _P, _P]),
    "hc_ice_dense_balance": (C.c_int, [_P, _P, _P, _P, _P, _I32, C.POINTER(_I32), C.POINTER(IceParams),
                                       _P, _P, C.POINTER(IceRunInfo), _P]),
    "hc_rowstats_i32": (C.c_int, [_P, _I64, _I32, _I32, _P, _P, _P]),
    "hc_twostep_alpha": (C.c_int, [_P, _P, _P, _P, _P, _I32, _I32, _I32, _P, _P, _P, _P, _P, _P, _P, _P]),
    "hc_twostep_work_bytes": (C.c_int64, [_I32]),
    "hc_twostep_correct": (C.c_int, [_P, _I64, _I32, _P, _P, _I32, _P, _P, _I64, _P, _P]),
    "hc_twostep_batch_work_bytes": (C.c_int64, [_I64, _I64, _I32]),
    "hc_twostep_batch": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I32, C.POINTER(_I32), C.POINTER(_I64),
                                   C.POINTER(_I32), C.POINTER(_I64), C.POINTER(_I64), _P, C.POINTER(_I64), _P, _P, _P, _P,
                                   _P, _P]),
    "hc_twostep_csr_batch_work_bytes": (C.c_int64, [_I64, _I64, _I32]),
    "hc_twostep_csr_batch": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I32, _I64, _I64, _P, _P, _P, _P, _P, _P,
                                       C.POINTER(_I64), _P, _P]),
    "hc_rownnz_f64": (C.c_int, [_P, _I64, _I32, _I32, _P, _P]),
    "hc_gap_rows": (C.c_int, [_P, _I32, _I32, _I32, _P, _P, _P, _P, _P]),
    "hc_trans2symmetry_f64": (C.c_int, [_P, _I64, _I32, _P, _P, _I64, _P]),
    "hc_correct_vc_work_bytes": (C.c_int64, [_I32, _I32]),
    "hc_correct_vc_f64": (C.c_int, [_P, _I64, _I32, _I32, C.c_double, _P, _I64, _P, _P]),
    "hc_balance_apply_i32": (C.c_int, [_P, _I64, _I32, _P, _P, _I64, _P]),
    "hc_colnnz_f64": (C.c_int, [_P, _I64, _I32, _P, _P]),
    "hc_distance_sums_f64": (C.c_int, [_P, _I64, _I32, _P, _P, _P]),
    "hc_observed_expected_f64": (C.c_int, [_P, _I64, _I32, _P, _P, _I64, _P]),
    "hc_directionality_index_f64": (C.c_int, [_P, _I64, _I32, _P, _P, _I32, _P, _P]),
    "hc_balance_apply_csr_i32": (C.c_int, [_P, _P, _P, _I32, _P, _P, _P]),
    "hc_colnnz_csr": (C.c_int, [_P, _I64, _I32, _P, _P]),
    "hc_distance_sums_csr_work_bytes": (C.c_int64, [_I64]),
    "hc_distance_sums_csr_f64": (C.c_int, [_P, _P, _P, _I64, _I32, _P, _P, _P, _P]),
    "hc_observed_expected_csr_f64": (C.c_int, [_P, _P, _P, _I32, _P, _P, _P]),
    "hc_directionality_index_csc_f64": (C.c_int, [_P, _P, _P, _I32, _P, _P, _I32, _P, _P]),
    "hc_pairs_to_keys": (C.c_int, [_P, _P, _P, _P, _I64, _I32, _P, _P, _I32, _I32, _I32, _P, _P, _P, _P]),
    "hc_sort_work_bytes": (C.c_int64, [_I64]),
    "hc_sort_keys_u64": (C.c_int, [_P, _P, _I64, _I32, _I32, _P, C.POINTER(_I32), _P]),
    "hc_csr_work_bytes": (C.c_int64, [_I64]),
    "hc_csr_count": (C.c_int, [_P, _I64, _P, _P, C.POINTER(_I64), _P]),
    "hc_csr_emit": (C.c_int, [_P, _I64, _P, _P, _I64, _I32, _I64, _I64, _P, _P, _P, _P, _P, _P]),
    "hc_pairs_to_entries": (C.c_int, [_P, _P, _P, _P, _I64, _I32, _P, _P, _I32, _I32, _I32, _I32, _P, _P, _P, _P]),
    "hc_pairs_to_directed_entries": (C.c_int, [_P, _P, _P, _P, _P, _I64, _I32, _P, _P, _I32, _I32, _I32, _I32, _P, _P, _P, _P]),
    "hc_entries_count": (C.c_int, [_P, _I64, _P, _I32, _P, C.POINTER(_I64), _P]),
    "hc_entries_reduce": (C.c_int, [_P, _I64, _P, _P, _I64, _I32, _I32, _P, _P, _P, C.POINTER(_I32), _P]),
    "hc_entries_emit": (C.c_int, [_P, _I64, _P, _P, _I64, _I32, _I32, _I32, _P, _P, _P, _P, C.POINTER(_I32), _P]),
    "hc_entries_transpose": (C.c_int, [_P, _I64, _I32, _I32, _P, _P, _P]),
    "hc_entries_csr_work_bytes": (C.c_int64, [_I64]),
    "hc_entries_to_csr": (C.c_int, [_P, _I64, _P, _P, _I32, _I32, _I64, _I64, _P, _P, _P, _P, _P]),
    "hc_csr_upper_count": (C.c_int, [_P, _P, _I64, _I64, _P, _P]),
    "hc_csr_upper_emit": (C.c_int, [_P, _P, _P, _I64, _I64, _P, _P, _P, _P, _P]),
    "hc_ice_csr_marginals": (C.c_int, [_P, _P, _P, _I64, _I64, _I32, _P, _P, _P]),
    "hc_ice_csr_work_bytes": (C.c_int64, [_I64, _I32]),
    "hc_ice_csr_balance": (C.c_int, [_P, _P, _P, _I64, _I64, _P, _I32, C.POINTER(_I64), C.POINTER(IceParams),
                                     _P, _P, _P, C.POINTER(IceRunInfo), _P, _P]),
    "hc_ingest_parse": (C.c_int, [C.POINTER(C.c_char_p), _I32, _I32, C.POINTER(C.c_char_p), _I32,
                                  C.POINTER(C.c_char_p), _I32, _I32, C.POINTER(_I64)]),
    "hc_ingest_fetch": (C.c_int, [_P, _P, _P, _P, _P]),
    "hc_nccl_available": (C.c_int, []),
    "hc_nccl_unique_id": (C.c_int, [_P]),
    "hc_nccl_comm_init": (C.c_int, [_P, _I32, _I32, C.POINTER(C.c_void_p)]),
    "hc_nccl_comm_destroy": (C.c_int, [_P]),
    "hc_nccl_allreduce_sum_f64": (C.c_int, [_P, _P, _I64, _P]),
}

_lib = None


def lib():
    """Load the shared library (once) and attach the signatures."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise HcError(
            "libhichap_b200.so is not built (%s). Run `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C hichap_master_b200/csrc`. There is no CPU fallback." % LIB_PATH)
    handle = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(handle, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype, fn.argtypes = res, args
    _lib = handle
    return handle


def check(rc: int, what: str):
    if rc != 0:
        msg = lib().hc_last_error().decode("utf-8", "replace")
        raise HcError("%s failed (code %d): %s" % (what, rc, msg))


def launch_count() -> int:
    return int(lib().hc_launch_count())
