"""ctypes binding of libbsgpu.so -- the C ABI declared in include/bsgpu.h.

The library is loaded from the package directory (built in-tree by ``bigsnpr_b200.build``).  There
is no fallback: if the shared object is missing, or no CUDA device is visible, calls raise.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libbsgpu.so")

c_int_p = C.POINTER(C.c_int)
c_dbl_p = C.POINTER(C.c_double)
c_u8_p = C.POINTER(C.c_uint8)
c_i64_p = C.POINTER(C.c_int64)
vp = C.c_void_p

# name -> (restype, argtypes); every symbol of include/bsgpu.h
SIGNATURES = {
    "bsg_last_error": (C.c_char_p, []),
    "bsg_version": (C.c_int, []),
    "bsg_device_count": (C.c_int, []),
    "bsg_open_bed": (C.c_int, [C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(vp)]),
    "bsg_open_packed": (C.c_int, [c_u8_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(vp)]),
    "bsg_open_synth": (C.c_int, [C.c_int, C.c_int, C.c_uint64, C.c_double, C.c_int64, C.c_int, C.c_int, C.POINTER(vp)]),
    "bsg_open_synth_ld": (C.c_int, [C.c_int, C.c_int, C.c_uint64, C.c_double, C.c_int64, C.c_double, C.c_int, C.c_int, C.c_int,
                                    C.POINTER(vp)]),
    "bsg_open_fbm256": (C.c_int, [c_u8_p, C.c_int, C.c_int, c_dbl_p, C.c_int, C.c_int, C.POINTER(vp)]),
    "bsg_close": (None, [vp]),
    "bsg_nrow": (C.c_int, [vp]),
    "bsg_ncol": (C.c_int, [vp]),
    "bsg_layouts": (C.c_int, [vp]),
    "bsg_has_na": (C.c_int, [vp]),
    "bsg_packed_bytes": (C.c_int64, [vp]),
    "bsg_export_packed": (C.c_int, [vp, c_u8_p]),
    "bsg_prodvec": (C.c_int, [vp, c_int_p, C.c_int, c_int_p, C.c_int, c_dbl_p, c_dbl_p, c_dbl_p, c_dbl_p]),
    "bsg_cprodvec": (C.c_int, [vp, c_int_p, C.c_int, c_int_p, C.c_int, c_dbl_p, c_dbl_p, c_dbl_p, c_dbl_p]),
    "bsg_view_create": (C.c_int, [vp, c_int_p, C.c_int, c_int_p, C.c_int, c_dbl_p, c_dbl_p, C.POINTER(vp)]),
    "bsg_view_destroy": (None, [vp]),
    "bsg_view_prodvec": (C.c_int, [vp, c_dbl_p, c_dbl_p]),
    "bsg_view_cprodvec": (C.c_int, [vp, c_dbl_p, c_dbl_p]),
    "bsg_view_prodvec_dev": (C.c_int, [vp, vp, vp, vp]),
    "bsg_view_cprodvec_dev": (C.c_int, [vp, vp, vp, vp]),
    "bsg_colstats": (C.c_int, [vp, c_int_p, C.c_int, c_int_p, C.c_int, c_dbl_p, c_dbl_p, c_int_p, c_int_p]),
    "bsg_col_counts": (C.c_int, [vp, c_int_p, C.c_int, c_int_p, C.c_int, c_int_p]),
    "bsg_row_counts": (C.c_int, [vp, c_int_p, C.c_int, c_int_p, C.c_int, c_int_p]),
    "bsg_snp_colstats": (C.c_int, [vp, c_int_p, C.c_int, c_int_p, C.c_int, c_dbl_p, c_dbl_p]),
    "bsg_read_bed": (C.c_int, [vp, c_int_p, C.c_int, c_int_p, C.c_int, C.c_int, c_int_p]),
    "bsg_read_bed_scaled": (C.c_int, [vp, c_int_p, C.c_int, c_int_p, C.c_int, c_dbl_p, c_dbl_p, c_dbl_p]),
    "bsg_cor": (C.c_int, [vp, c_int_p, C.c_int, c_int_p, C.c_int, C.c_double, c_dbl_p, c_dbl_p, C.c_int,
                          c_i64_p, C.POINTER(c_int_p), C.POINTER(c_dbl_p)]),
    "bsg_ld_scores": (C.c_int, [vp, c_int_p, C.c_int, c_int_p, C.c_int, C.c_double, c_dbl_p, c_dbl_p]),
    "bsg_free": (None, [vp]),
    "bsg_clumping_chr": (C.c_int, [vp, c_int_p, C.c_int, c_int_p, C.c_int, c_dbl_p, c_dbl_p, c_int_p, c_dbl_p, C.c_double,
                                   C.c_double, c_int_p]),
    "bsg_clumping_chr_fbm": (C.c_int, [vp, c_int_p, C.c_int, c_int_p, C.c_int, c_dbl_p, c_dbl_p, c_int_p, c_dbl_p, C.c_double,
                                   C.c_double, c_int_p]),
    "bsg_readbina2": (C.c_int, [vp, c_int_p, C.c_int, c_int_p, C.c_int, C.POINTER(C.c_uint8)]),
    "bsg_writebina": (C.c_int, [vp, C.c_char_p, c_int_p, C.c_int, c_int_p, C.c_int]),
    "bsg_set_prodvec_path": (C.c_int, [C.c_int]),
    "bsg_set_scaling_reuse": (C.c_int, [C.c_int]),
    "bsg_prod_and_rowsumssq": (C.c_int, [vp, c_int_p, C.c_int, c_int_p, C.c_int, c_dbl_p, c_dbl_p, c_dbl_p, C.c_int,
                                         c_dbl_p, c_dbl_p]),
    "bsg_multlinreg": (C.c_int, [vp, c_int_p, C.c_int, c_int_p, C.c_int, c_dbl_p, C.c_int, c_dbl_p]),
    "bsg_code256_kind": (C.c_int, [c_dbl_p]),
    "bsg_impute": (C.c_int, [c_u8_p, C.c_int, C.c_int, C.c_int, C.c_uint64, C.c_int, c_int_p]),
    "bsg_tcrossprod": (C.c_int, [vp, c_int_p, C.c_int, c_int_p, C.c_int, c_dbl_p, c_dbl_p, c_dbl_p]),
    "bsg_tcrossprod_dev": (C.c_int, [vp, c_int_p, C.c_int, c_int_p, C.c_int, c_dbl_p, c_dbl_p, vp]),
    "bsg_randomsvd": (C.c_int, [vp, c_int_p, C.c_int, c_int_p, C.c_int, c_dbl_p, c_dbl_p, C.c_int, C.c_double,
                                C.c_int, c_dbl_p, c_dbl_p, c_dbl_p, c_dbl_p, c_dbl_p, c_int_p, c_int_p]),
    "bsg_randomsvd_ex": (C.c_int, [vp, c_int_p, C.c_int, c_int_p, C.c_int, c_dbl_p, c_dbl_p, C.c_int, C.c_double,
                                   C.c_int, c_dbl_p, c_dbl_p, c_dbl_p, c_dbl_p, c_dbl_p, c_int_p, c_int_p, vp, vp, vp,
                                   C.c_int]),
    "bsg_randomsvd_nconv": (C.c_int, []),
    "bsg_group_open_bed": (C.c_int, [C.c_char_p, C.c_int, C.c_int, c_int_p, C.c_int, C.c_int, C.POINTER(vp)]),
    "bsg_group_open_synth": (C.c_int, [C.c_int, C.c_int, C.c_uint64, C.c_double, C.c_double, C.c_int, c_int_p, C.c_int, C.c_int,
                                       C.POINTER(vp)]),
    "bsg_group_close": (None, [vp]),
    "bsg_group_ndev": (C.c_int, [vp]),
    "bsg_group_nrow": (C.c_int, [vp]),
    "bsg_group_ncol": (C.c_int, [vp]),
    "bsg_group_shard": (vp, [vp, C.c_int]),
    "bsg_group_shard_begin": (C.c_int, [vp, C.c_int]),
    "bsg_group_prodvec": (C.c_int, [vp, c_int_p, C.c_int, c_int_p, C.c_int, c_dbl_p, c_dbl_p, c_dbl_p, c_dbl_p]),
    "bsg_group_cprodvec": (C.c_int, [vp, c_int_p, C.c_int, c_int_p, C.c_int, c_dbl_p, c_dbl_p, c_dbl_p, c_dbl_p]),
    "bsg_group_randomsvd": (C.c_int, [vp, c_int_p, C.c_int, c_int_p, C.c_int, c_dbl_p, c_dbl_p, C.c_int, C.c_double, C.c_int,
                                      c_dbl_p, c_dbl_p, c_dbl_p, c_dbl_p, c_dbl_p, c_int_p, c_int_p]),
    "bsg_group_tcrossprod": (C.c_int, [vp, c_int_p, C.c_int, c_int_p, C.c_int, c_dbl_p, c_dbl_p, c_dbl_p]),
    "bsg_comm_create": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int64, C.POINTER(vp), c_u8_p]),
    "bsg_comm_connect": (C.c_int, [vp, c_u8_p]),
    "bsg_comm_destroy": (None, [vp]),
    "bsg_comm_rank": (C.c_int, [vp]),
    "bsg_comm_world": (C.c_int, [vp]),
    "bsg_comm_check": (C.c_int, [vp]),
    "bsg_comm_allreduce_dev": (C.c_int, [vp, vp, C.c_int64, vp]),
    "bsg_view_prodvec_allreduce_dev": (C.c_int, [vp, vp, vp, vp, vp]),
    "bsg_randomsvd_comm": (C.c_int, [vp, vp, c_int_p, C.c_int, c_int_p, C.c_int, c_dbl_p, c_dbl_p, C.c_int, C.c_int, C.c_double,
                                     C.c_int, c_dbl_p, c_dbl_p, c_dbl_p, c_dbl_p, c_dbl_p, c_int_p, c_int_p]),
    "bsg_launch_count": (C.c_int64, []),
    "bsg_last_kernel_ms": (C.c_double, []),
    "bsg_set_kernel_timing": (C.c_int, [C.c_int]),
    "bsg_kernel_time_stats": (C.c_int, [c_int_p, c_dbl_p]),
}


class BsgError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(msg)
        self.code = code


_lib = None


def lib():
    """Load libbsgpu.so (once).  Raises if the CUDA extension has not been built -- no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise ImportError(
                f"{SO_PATH} is missing: build the CUDA extension first (python -m bigsnpr_b200.build). "
                "bigsnpr_b200 has no CPU fallback.")
        L = C.CDLL(SO_PATH)
        for name, (res, args) in SIGNATURES.items():
            f = getattr(L, name)
            f.restype = res
            f.argtypes = args
        _lib = L
    return _lib


def check(rc: int):
    if rc:
        raise BsgError(rc, lib().bsg_last_error().decode("utf-8", "replace"))
