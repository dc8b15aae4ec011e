"""ctypes binding of libeaglegpu.so (C ABI declared in include/eagle_gpu.h).

The shared library is built in-tree by `__graft_entry__.build()` / `make -C eagleeverything_b200/csrc`.
There is no fallback of any kind: if the library is missing, or no B200 is visible when a compute
entry point is called, the call raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libeaglegpu.so")

EG_OK, EG_ERR_CUDA, EG_ERR_OPEN, EG_ERR_FORMAT, EG_ERR_ARG, EG_ERR_ALLOC = range(6)


class EagleGpuError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(msg)
        self.code = code


MESSAGE_FN = C.CFUNCTYPE(None, C.c_void_p, C.c_char_p)

_i64 = C.c_int64
_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)
_lp = C.POINTER(C.c_int64)
_vp = C.c_void_p

# name -> (restype, argtypes); every symbol include/eagle_gpu.h declares
SIGNATURES = {
    "eg_init": (C.c_int, [C.c_int]),
    "eg_init_multi": (C.c_int, [C.c_int, C.POINTER(C.c_int)]),
    "eg_gpu_count": (C.c_int, []),
    "eg_shutdown": (C.c_int, []),
    "eg_last_error": (C.c_char_p, []),
    "eg_abi_version": (C.c_int, []),
    "eg_device_count": (C.c_int, []),
    "eg_cache_clear": (None, []),
    "eg_ReadBlock": (C.c_int, [C.c_char_p, _i64, _i64, _i64, _dp]),
    "eg_calculateMMt_rcpp": (C.c_int, [C.c_char_p, C.c_double, C.c_int, _dp, _i64, _lp, C.c_int, MESSAGE_FN, _vp, _dp]),
    "eg_calculate_a_and_vara_rcpp": (C.c_int, [C.c_char_p, _dp, _i64, _dp, _dp, C.c_double, _lp, _dp, C.c_int,
                                               MESSAGE_FN, _vp, _dp, _dp]),
    "eg_calculate_reduced_a_rcpp": (C.c_int, [C.c_char_p, C.c_double, _dp, _dp, C.c_double, _lp, _dp, _i64, C.c_int,
                                              MESSAGE_FN, _vp, _dp]),
    "eg_extract_geno_rcpp": (C.c_int, [C.c_char_p, C.c_double, _i64, _lp, _ip]),
    "eg_createM_ASCII_rcpp": (C.c_int, [C.c_char_p] * 6 + [C.c_double, _lp, C.c_int, MESSAGE_FN, _vp, C.c_char_p,
                                        C.POINTER(C.c_int)]),
    "eg_createMt_ASCII_rcpp": (C.c_int, [C.c_char_p] * 3 + [C.c_double, _lp, C.c_int, MESSAGE_FN, _vp]),
    "eg_ReshapeM_rcpp": (C.c_int, [C.c_char_p, C.c_char_p, _lp, _i64, _lp, _lp]),
    "eg_getRowColumn": (C.c_int, [C.c_char_p, _lp]),
    "eg_tokenise_chunks": (_i64, [_i64]),
    "eg_tokenise_chunk_bytes": (_i64, []),
    "eg_dev_tokenise_scan": (C.c_int, [_vp, _i64, _vp, _vp, _vp]),
    "eg_dev_tokenise_emit": (C.c_int, [_vp, _i64, _vp, _i64, C.c_char_p, C.c_char_p, C.c_char_p, C.c_char_p, _vp, _i64,
                                       _vp, _vp]),
    "eg_dev_ped_alleles": (C.c_int, [_vp, _i64, _vp, _i64, _vp, _i64, _vp, _vp]),
    "eg_dev_ped_genotypes": (C.c_int, [_vp, _i64, _i64, C.c_int, _i64, _vp, _vp, _vp, _vp]),
    "eg_dev_encode_ascii": (C.c_int, [_vp, _i64, _i64, _i64, _i64, _vp, _vp]),
    "eg_store_from_host_ascii": (C.c_int, [_vp, _i64, _i64, _i64, _i64, C.POINTER(_vp)]),
    "eg_store_from_host_ascii_rows": (C.c_int, [_vp, _i64, _i64, _i64, _i64, C.POINTER(_vp)]),
    "eg_store_from_file": (C.c_int, [C.c_char_p, _i64, _i64, _i64, _i64, C.POINTER(_vp)]),
    "eg_store_drop_individuals": (C.c_int, [_vp, _lp, _i64, C.c_int, C.POINTER(_vp)]),
    "eg_dev_gather_rows": (C.c_int, [_vp, _i64, _i64, _i64, _vp, _i64, _vp, _i64, _vp]),
    "eg_dev_gather_cols": (C.c_int, [_vp, _i64, _i64, _vp, _i64, _vp, _i64, _vp]),
    "eg_packed_words_per_row": (C.c_int64, [_i64]),
    "eg_store_from_host_packed": (C.c_int, [_vp, _i64, _i64, C.c_int, C.POINTER(_vp)]),
    "eg_store_to_host_packed": (C.c_int, [_vp, _vp]),
    "eg_dev_pack_2bit": (C.c_int, [_vp, _i64, _i64, _i64, _vp, _vp]),
    "eg_dev_unpack_2bit": (C.c_int, [_vp, _i64, _i64, _vp, _i64, _vp, _vp]),
    "eg_store_from_bed": (C.c_int, [C.c_char_p, _i64, _i64, _i64, _i64, C.c_int, _lp, C.POINTER(_vp)]),
    "eg_store_from_host_bed": (C.c_int, [_vp, _i64, _i64, _i64, _i64, C.c_int, _lp, C.POINTER(_vp)]),
    "eg_bed_to_ascii": (C.c_int, [C.c_char_p, _i64, _i64, C.c_char_p, C.c_char_p]),
    "eg_store_stream_file": (C.c_int, [C.c_char_p, _i64, _i64, C.c_int, C.POINTER(_vp)]),
    "eg_store_stream_bed": (C.c_int, [C.c_char_p, _i64, _i64, _i64, _i64, C.c_int, C.POINTER(_vp)]),
    "eg_store_stream_host_bed": (C.c_int, [_vp, _i64, _i64, _i64, _i64, C.c_int, C.POINTER(_vp)]),
    "eg_store_transpose": (C.c_int, [_vp, C.POINTER(_vp)]),
    "eg_store_free": (C.c_int, [_vp]),
    "eg_store_info": (C.c_int, [_vp, _lp, _lp, _lp, C.POINTER(_vp)]),
    "eg_store_mmt": (C.c_int, [_vp, _lp, _i64, _dp]),
    "eg_store_a_and_vara": (C.c_int, [_vp, _lp, _i64, _dp, _dp, _dp, _dp, _dp]),
    "eg_store_extract_col": (C.c_int, [_vp, _i64, _ip]),
    "eg_dev_decode": (C.c_int, [_vp, _i64, _i64, _i64, _i64, _vp, _i64, _vp, _vp]),
    "eg_dev_decode_kb": (C.c_int, [_vp, _i64, _i64, _i64, _i64, _vp, _i64, _i64, _vp, _vp]),
    "eg_dev_decode_bed": (C.c_int, [_vp, _i64, _i64, _vp, _i64, _i64, _i64, _vp, _vp]),
    "eg_dev_transpose_kb_i8": (C.c_int, [_vp, _i64, _i64, _vp, _i64, _vp]),
    "eg_dev_syrk_i8_kb": (C.c_int, [_vp, _i64, _i64, _vp, _i64, _vp]),
    "eg_dev_transpose_i8": (C.c_int, [_vp, _i64, _i64, _i64, _vp, _i64, _vp]),
    "eg_dev_syrk_i8": (C.c_int, [_vp, _i64, _i64, _i64, _vp, _i64, _vp]),
    "eg_dev_syrk_zero_cols": (C.c_int, [_vp, _i64, _i64, _lp, _i64, _vp, _i64, _vp]),
    "eg_dev_mmt_finalize": (C.c_int, [_vp, _i64, _i64, _vp, _vp]),
    "eg_scan_wp_elems": (_i64, [_i64]),
    "eg_dev_scan_prepare": (C.c_int, [_vp, _vp, _vp, _i64, _vp, _vp, _vp]),
    "eg_prep_uses_i8": (C.c_int, [_i64]),
    "eg_dev_symmetry": (C.c_int, [_vp, _i64, _dp, _dp, _vp]),
    "eg_dev_inputs_symmetric": (C.c_int, [_vp, _vp, _i64, C.POINTER(C.c_int), _vp]),
    "eg_dev_scan_prepare_cols": (C.c_int, [_vp, _vp, _i64, _i64, _i64, C.c_int, _vp, _vp, _vp]),
    "eg_dev_scan_fold": (C.c_int, [_vp, _vp, _i64, C.c_int, _vp, _vp]),
    "eg_dev_scan": (C.c_int, [_vp, _i64, _i64, _i64, _vp, _lp, _i64, _vp, _vp, _vp]),
    "eg_dev_argmax_tsq": (C.c_int, [_vp, _vp, _i64, _vp, _vp, _vp]),
    "eg_dev_gemv_i8": (C.c_int, [_vp, _i64, _i64, _i64, _vp, C.c_double, _vp, _vp]),
    "eg_dev_extract_col": (C.c_int, [_vp, _i64, _i64, _i64, _vp, _vp]),
    "eg_dev_synth_ascii": (C.c_int, [_vp, _i64, _i64, _i64, _i64, _i64, C.c_uint64, _vp]),
    "eg_set_scan_mode": (C.c_int, [C.c_int]),
    "eg_get_scan_mode": (C.c_int, []),
    "eg_set_scan_digits": (C.c_int, [C.c_int]),
    "eg_get_scan_digits": (C.c_int, []),
    "eg_calculateMMt_sqrt_and_sqrtinv": (C.c_int, [_dp, _i64, C.c_int, MESSAGE_FN, _vp, _dp, _dp, C.POINTER(C.c_int)]),
    "eg_calculateH": (C.c_int, [_dp, _i64, C.c_double, C.c_double, MESSAGE_FN, _vp, _dp, C.POINTER(C.c_int)]),
    "eg_calculateP": (C.c_int, [_dp, _dp, _i64, C.c_int, _dp]),
    "eg_calculate_reduced_a": (C.c_int, [C.c_double, _dp, _dp, _dp, _i64, _dp]),
    "eg_calculate_reduced_vara": (C.c_int, [_dp, _i64, C.c_int, C.c_double, C.c_double, _dp, _dp]),
    "eg_emma_eigen_L_wo_Z": (C.c_int, [_dp, _i64, _dp, _dp]),
    "eg_emma_eigen_R_wo_Z": (C.c_int, [_dp, _dp, _i64, C.c_int, _dp, _dp]),
    "eg_dev_eigen_sym": (C.c_int, [_vp, _i64, _vp, _vp]),
    "eg_dev_emma_SKS": (C.c_int, [_vp, _vp, _i64, C.c_int, _vp, _vp, _vp, _vp]),
    "eg_dev_emma_eigen_R_wo_Z": (C.c_int, [_vp, _vp, _vp, _i64, C.c_int, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "eg_dev_sqrt_and_sqrtinv": (C.c_int, [_vp, _i64, _vp, _vp, _vp, C.POINTER(C.c_int), _dp, _vp]),
    "eg_dev_calculateH": (C.c_int, [_vp, _i64, C.c_double, C.c_double, _vp, _vp]),
    "eg_dev_calculateP": (C.c_int, [_vp, _vp, _i64, C.c_int, _vp, _vp, _vp]),
    "eg_dev_calculate_reduced_a": (C.c_int, [C.c_double, _vp, _vp, _vp, _i64, _vp, _vp, _vp]),
    "eg_dev_calculate_reduced_vara": (C.c_int, [_vp, C.c_int, C.c_double, C.c_double, _vp, _i64, _vp, _vp, _vp, _vp]),
    "eg_emma_eigen_R_wo_Z_eigbasis": (C.c_int, [_dp, _dp, _dp, _i64, C.c_int, _dp, _dp, _lp]),
    "eg_dev_project_i8": (C.c_int, [_vp, _i64, _i64, _i64, _vp, _vp, _i64, _vp]),
    "eg_dev_bscan": (C.c_int, [_vp, _i64, _i64, _i64, _vp, _vp, C.c_int, _vp, _vp, _vp]),
    "eg_last_secular_times": (C.c_int, [_dp]),
    "eg_dev_transpose_f64": (C.c_int, [_vp, _i64, _vp, _vp]),
    "eg_dev_eigbasis_apply": (C.c_int, [_vp, _i64, _vp, C.c_int, C.c_int, _vp, _vp]),
    "eg_dev_scan_prepare_eig": (C.c_int, [_vp, _vp, _i64, _vp, _vp, C.c_int, _vp, _vp, _vp, _vp, _vp]),
    "eg_last_scan_kernel": (C.c_int, [_dp, _dp]),
    "eg_last_prep_kernels": (C.c_int, [_dp, _dp]),
    "eg_launch_count": (C.c_longlong, []),
    "eg_last_timing": (C.c_int, [_dp, C.c_int]),
}

_lib = None


def load():
    """dlopen libeaglegpu.so and attach signatures.  Raises if the library has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise ImportError(
                f"{SO_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or `make -C eagleeverything_b200/csrc`).  There is no CPU fallback.")
        lib = C.CDLL(SO_PATH, mode=C.RTLD_GLOBAL)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc):
    if rc != EG_OK:
        msg = load().eg_last_error()
        raise EagleGpuError(rc, (msg or b"").decode("utf-8", "replace") or f"libeaglegpu error {rc}")


def require_gpu():
    """Fail loudly when the CUDA path cannot run (no silent fallback anywhere in this package)."""
    lib = load()
    if lib.eg_device_count() <= 0:
        raise EagleGpuError(EG_ERR_CUDA, "no CUDA device visible: the Eagle hot path has no CPU fallback")
    return lib
