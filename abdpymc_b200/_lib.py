"""ctypes binding of libabd_b200.so (C ABI in include/abd_b200.h).

The library is built in-tree by ``__graft_entry__.build()`` (or ``python -m abdpymc_b200.build``).
There is no CPU fallback: if the shared library is missing, or no CUDA device is present,
every entry point fails loudly.
"""

from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

PKG = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ.get("ABD_B200_LIB", PKG / "libabd_b200.so"))  # override: developer builds only

N_THETA, N_Q, N_SUMS, MAX_GAPS = 13, 17, 16, 127
GIBBS_METROPOLIS, GIBBS_HEATBATH, GIBBS_BLOCKED = 0, 1, 2

c_double_p = C.POINTER(C.c_double)
c_int8_p = C.POINTER(C.c_int8)
c_uint8_p = C.POINTER(C.c_uint8)
c_int32_p = C.POINTER(C.c_int32)
c_int64_p = C.POINTER(C.c_int64)
c_uint64_p = C.POINTER(C.c_uint64)


class AbdCohort(C.Structure):
    """struct abd_cohort (include/abd_b200.h)."""

    _fields_ = [
        ("n_gaps", C.c_int32), ("n_inds", C.c_int32), ("n_splits", C.c_int32), ("splits", C.c_int32 * 2),
        ("pcrpos", c_uint8_p), ("vacs", c_uint8_p),
        ("n_rows_s", C.c_int64), ("x_s", c_double_p), ("od_s", c_double_p), ("gap_s", c_int32_p), ("ind_s", c_int32_p),
        ("n_rows_n", C.c_int64), ("x_n", c_double_p), ("od_n", c_double_p), ("gap_n", c_int32_p), ("ind_n", c_int32_p),
        ("total_inds", C.c_int64), ("total_rows_s", C.c_int64), ("total_rows_n", C.c_int64),
        ("ind_offset", C.c_int64),
    ]  # fmt: skip


class AbdError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"libabd_b200 error {code}: {message}")
        self.code = code


#: every symbol include/abd_b200.h declares: name -> (restype, argtypes)
H = C.c_void_p
SIGNATURES = {
    "abd_last_error": (C.c_char_p, []),
    "abd_version": (C.c_int, []),
    "abd_create": (C.c_int, [C.POINTER(H), C.POINTER(AbdCohort), C.c_int]),
    "abd_destroy": (C.c_int, [H]),
    "abd_save_cache": (C.c_int, [H, C.c_char_p]),
    "abd_create_from_cache": (C.c_int, [C.POINTER(H), C.c_char_p, C.c_int]),
    "abd_cohort_info": (C.c_int, [H, c_int32_p, c_int32_p, c_int32_p]),
    "abd_sizes": (C.c_int, [H, c_int32_p, c_int32_p, c_int64_p, c_int64_p]),
    "abd_algorithmic_bytes_logp": (C.c_int64, [H, C.c_int]),
    "abd_algorithmic_bytes_gibbs": (C.c_int64, [H, C.c_int]),
    "abd_launch_count": (C.c_int64, [H]),
    "abd_upload_state": (C.c_int, [H, C.c_int, C.c_void_p, C.c_void_p]),
    "abd_download_state": (C.c_int, [H, C.c_int, C.c_void_p, C.c_void_p]),
    "abd_loglik_grad": (C.c_int, [H, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "abd_logp_dlogp": (C.c_int, [H, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "abd_cond_logodds": (C.c_int, [H, C.c_int] + [C.c_void_p] * 7),
    "abd_gibbs_sweep": (C.c_int, [H, C.c_int] + [C.c_void_p] * 5 + [C.c_uint64, C.c_uint64, C.c_int, C.c_double, C.c_void_p]),
    "abd_deterministics": (C.c_int, [H, C.c_int] + [C.c_void_p] * 6),
    "abd_loglik_rows": (C.c_int, [H, C.c_int] + [C.c_void_p] * 5),
    "abd_loglik_rows_dev": (C.c_int, [H, C.c_int] + [C.c_void_p] * 6),
    "abd_sums_dev": (C.c_int, [H, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "abd_finalize_loglik_dev": (C.c_int, [H, C.c_int] + [C.c_void_p] * 5),
    "abd_finalize_logp_dev": (C.c_int, [H, C.c_int] + [C.c_void_p] * 5),
    "abd_loglik_grad_dev": (C.c_int, [H, C.c_int] + [C.c_void_p] * 6),
    "abd_logp_dlogp_dev": (C.c_int, [H, C.c_int] + [C.c_void_p] * 6),
    "abd_gibbs_sweep_dev": (C.c_int, [H, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_uint64, C.c_uint64, C.c_int, C.c_double, C.c_void_p, C.c_void_p]),
    "abd_deterministics_dev": (C.c_int, [H, C.c_int] + [C.c_void_p] * 7),
    "abd_deterministics_accum_dev": (C.c_int, [H, C.c_int, C.c_void_p, C.c_int] + [C.c_void_p] * 6),
    "abd_leapfrog_dev": (C.c_int, [H, C.c_int, C.c_int] + [C.c_void_p] * 9),
    "abd_leapfrog_status": (C.c_int, [H, C.c_int]),
    "abd_hmc_begin_dev": (C.c_int, [H, C.c_int] + [C.c_void_p] * 4 + [C.c_uint64, C.c_uint64] + [C.c_void_p] * 5),
    "abd_hmc_end_dev": (C.c_int, [H, C.c_int] + [C.c_void_p] * 9 + [C.c_uint64, C.c_uint64] + [C.c_void_p] * 3
                        + [C.c_int, C.c_double, C.c_void_p]),
    "abd_nuts_state_doubles": (C.c_int64, [C.c_int]),
    "abd_nuts_begin_dev": (C.c_int, [H, C.c_int, C.c_int] + [C.c_void_p] * 5 + [C.c_uint64, C.c_uint64] + [C.c_void_p] * 7),
    "abd_nuts_leaf_dev": (C.c_int, [H, C.c_int, C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 6 + [C.c_uint64, C.c_uint64]
                          + [C.c_void_p] * 4),
    "abd_nuts_extend_dev": (C.c_int, [H, C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 6 + [C.c_uint64, C.c_uint64]
                            + [C.c_void_p] * 6),
    "abd_nuts_end_dev": (C.c_int, [H, C.c_int, C.c_int] + [C.c_void_p] * 9 + [C.c_int, C.c_double, C.c_void_p]),
    "abd_xch_alloc": (C.c_int, [H, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "abd_xch_connect": (C.c_int, [H, C.c_void_p]),
    "abd_logp_dlogp_sharded_dev": (C.c_int, [H, C.c_int] + [C.c_void_p] * 6),
    "abd_xch_status": (C.c_int, [H]),
    "abd_leapfrog_sharded_dev": (C.c_int, [H, C.c_int] + [C.c_void_p] * 9),
    "abd_xch_stats": (C.c_int, [H, C.c_void_p, C.c_int]),
    "abd_state_dev": (C.c_int, [H, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]),
    "abd_state_touch": (C.c_int, [H]),
    "abd_set_chain_offset": (C.c_int, [H, C.c_int64]),
    "abd_set_tuning": (C.c_int, [H, C.c_int, C.c_int]),
    "abd_last_plan": (C.c_int, [H, C.c_void_p]),
    "abd_debug_fast_math": (C.c_int, [C.c_int, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
}  # fmt: skip

_lib = None


def load(path: Path | None = None) -> C.CDLL:
    """Load the shared library and bind every declared symbol (no CUDA call is made)."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = Path(path) if path else LIB_PATH
    if not p.exists():
        raise AbdError(-100, f"{p} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                             "(there is no CPU fallback)")
    lib = C.CDLL(str(p))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    if path is None:
        _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        raise AbdError(rc, load().abd_last_error().decode())
