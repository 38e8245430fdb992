"""ctypes binding of libgpexp_b200.so (the C ABI declared in include/gpexp_b200.h).

There is no CPU fallback: if the shared library has not been built, importing this module
raises ImportError, and creating a handle without a CUDA device raises GpxError.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GPX_LIB") or os.path.join(HERE, "lib", "libgpexp_b200.so")  # GPX_LIB: A/B builds only

GPX_VERSION = 200
GPX_MAX_DIM = 16
GPX_KROWS = 16
GPX_I8_MAX_N = 16384  # largest design size the INT8 IVAR core runs
GPX_PIVOT_HDR = 3 + GPX_MAX_DIM
GPX_COMM_ID_BYTES = 128
SE, MATERN32, MEHLER, MATERN12, MATERN52 = 0, 1, 2, 3, 4
SIDE_A, SIDE_B = 0, 1
ROW_KERNEL, ROW_MATRIX = 0, 1
PRO_EXPANDED, PRO_DIFF = 1, 2
MEASURE_BOX, MEASURE_GAUSS = 1, 2


class GpxError(RuntimeError):
    """A C-ABI call returned non-zero (message from gpx_last_error)."""


if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
        "or `make -C gpexp_b200/csrc`.  gpexp_b200 has no CPU fallback.")

lib = C.CDLL(LIB_PATH)

_p = C.c_void_p
_i64 = C.c_int64
_int = C.c_int
_dbl = C.c_double



class IvarState(C.Structure):
    """gpx_ivar_state (include/gpexp_b200.h): device pointers and sizes of one greedy-IVAR engine."""
    _fields_ = [("Xm", _p), ("M", _i64), ("ldm", _i64), ("Wm", _p), ("varM", _p), ("Ma_rows", _p),
                ("Xc", _p), ("C", _i64), ("ldc", _i64), ("Wc", _p), ("varC", _p), ("Cb_rows", _p),
                ("ncap", _i64), ("index_offset", _i64), ("prologue", _int), ("nseg", _int),
                ("noise", _dbl), ("zero_tol", _dbl),
                ("workspace", _p), ("scores", _p), ("best", _p), ("idx", _p),
                ("rec", _p), ("rec_all", _p), ("rec_win", _p),
                ("U", _p), ("ldu", _i64), ("picks", _p), ("pick_scores", _p), ("pick_pivots", _p),
                ("cov", _p), ("ldcov", _i64), ("ldp", _i64), ("wM", _p)]


class VarState(C.Structure):
    """gpx_var_state: device pointers and sizes of one greedy max-variance engine."""
    _fields_ = [("X", _p), ("C", _i64), ("ld", _i64), ("W", _p), ("var", _p), ("weights", _p),
                ("ncap", _i64), ("index_offset", _i64), ("noise", _dbl),
                ("best", _p), ("idx", _p), ("rec", _p), ("rec_all", _p), ("rec_win", _p),
                ("picks", _p), ("pick_scores", _p), ("pick_pivots", _p)]


# name -> argtypes (restype int unless listed in _RESTYPES); mirrors include/gpexp_b200.h one to one
SIGNATURES = {
    "gpx_version": [],
    "gpx_last_error": [],
    "gpx_launch_count": [],
    "gpx_create": [_int, C.POINTER(_p)],
    "gpx_destroy": [_p],
    "gpx_set_kernel": [_p, _int, _int, C.POINTER(_dbl), _int],
    "gpx_kernel_pairwise": [_p, _p, _i64, _i64, _p, _i64, _i64, _p, _p],
    "gpx_prior_diag": [_p, _p, _i64, _i64, _p, _p],
    "gpx_gram": [_p, _p, _i64, _i64, _p, _i64, _i64, _p, _i64, _int, _p, _dbl, _p],
    "gpx_potrf": [_p, _p, _i64, _i64, _p, _p],
    "gpx_chol_append": [_p, _p, _i64, _i64, _p, _dbl, _p, _p],
    "gpx_set_center": [_p, C.POINTER(_dbl)],
    "gpx_prep_side": [_p, _int, _p, _i64, _i64, _p, _i64, _p, _p],
    "gpx_trsm_gram": [_p, _p, _i64, _i64, _p, _i64, _p, _i64, _i64, _p, _i64, _p, _p],
    "gpx_trsm": [_p, _p, _i64, _i64, _p, _i64, _i64, _p],
    "gpx_trsm_back": [_p, _p, _i64, _i64, _p, _i64, _i64, _p],
    "gpx_trtri_t": [_p, _p, _i64, _i64, _p, _i64, _p],
    "gpx_dgemm_tn_sub": [_p, _p, _i64, _p, _i64, _p, _i64, _i64, _i64, _i64, _int, _p],
    "gpx_dgemm_tn_sub_padded": [_p, _p, _i64, _p, _i64, _p, _i64, _i64, _i64, _i64, _int, _p],
    "gpx_gather_pivot": [_p, _p, _i64, _i64, _p, _p, _i64, _p, _p, _i64, _p, _dbl, _p, _p],
    "gpx_gather_pivot_nu": [_p, _p, _i64, _i64, _p, _p, _i64, _p, _p, _i64, _p, _p, _dbl, _p, _p],
    "gpx_select_pivot": [_p, _p, _int, _i64, _i64, _int, _p, _p],
    "gpx_append_row": [_p, _int, _p, _p, _p, _i64, _i64, _p, _i64, _i64, _p, _p],
    "gpx_argreduce": [_p, _p, _p, _p, _i64, _int, _p, _p, _p],
    "gpx_sum": [_p, _p, _i64, _p, _p],
    "gpx_sum_w": [_p, _p, _p, _i64, _p, _p],
    "gpx_set_ivar_ring": [_p, _int],
    "gpx_set_ivar_core": [_p, _int],
    "gpx_ivar_scratch_bytes": [_p, _i64, _i64, _i64],
    "gpx_set_ivar_scratch": [_p, _p, _i64],
    "gpx_score_ivar_workspace": [_p, _i64, _i64],
    "gpx_score_ivar": [_p, _int, _p, _i64, _p, _p, _i64, _p, _i64, _p, _p, _i64, _i64, _dbl, _dbl, _p, _p, _p, _p, _p, _p],
    "gpx_score_ivar_w": [_p, _int, _p, _i64, _p, _p, _i64, _p, _i64, _p, _p, _i64, _i64, _dbl, _dbl, _p, _p, _p, _p, _p, _p,
                         _p],
    "gpx_set_measure": [_p, _int, _int, C.POINTER(_dbl), C.POINTER(_dbl)],
    "gpx_phi_gram": [_p, _p, _i64, _i64, _p, _i64, _i64, _p, _i64, _p],
    "gpx_phi_diag": [_p, _p, _i64, _i64, _p, _p],
    "gpx_phi_append_row": [_p, _p, _p, _i64, _i64, _p, _i64, _i64, _p],
    "gpx_psi_row": [_p, _p, _i64, _p, _i64, _p, _i64, _i64, _p, _i64, _p],
    "gpx_ivar_measure_score": [_p, _p, _p, _p, _i64, _p, _p, _i64, _i64, _int, _p, _i64, _dbl, _dbl, _p, _p, _p, _p, _p],
    "gpx_cov_segments": [_i64, _i64],
    "gpx_cov_update": [_p, _p, _i64, _i64, _i64, _p, _p, _p, _i64, _p],
    "gpx_cov_update_w": [_p, _p, _i64, _i64, _i64, _p, _p, _p, _p, _i64, _p],
    "gpx_cov_from_factors": [_p, _int, _p, _i64, _p, _i64, _p, _i64, _p, _i64, _i64, _p, _i64, _p],
    "gpx_score_ivar_partials": [_p, _p, _int, _i64, _p, _i64, _p, _i64, _dbl, _dbl, _p, _p, _p, _p, _p],
    "gpx_score_ivar_partials_w": [_p, _p, _int, _i64, _p, _i64, _p, _i64, _dbl, _dbl, _p, _p, _p, _p, _p, _p],
    "gpx_score_mi": [_p, _p, _p, _dbl, _p, _i64, _p, _p, _p, _p],
    "gpx_score_mi_nu": [_p, _p, _p, _p, _dbl, _p, _i64, _p, _p, _p, _p],
    "gpx_mi_prec_column_workspace": [_i64, _i64],
    "gpx_mi_prec_column": [_p, _p, _i64, _i64, _i64, _i64, _i64, _i64, _p, _p, _p, _p, _p],
    "gpx_gather_column": [_p, _p, _i64, _i64, _p, _p, _p, _p],
    "gpx_local_index": [_p, _p, _i64, _i64, _p, _p],
    "gpx_local_index_cyclic": [_p, _p, _i64, _i64, _i64, _i64, _p, _p],
    "gpx_add_at_rows": [_p, _p, _i64, _p, _i64, _dbl, _p],
    "gpx_add_at_rows_vec": [_p, _p, _i64, _p, _i64, _p, _dbl, _p],
    "gpx_dgemm_tn_sub_lower": [_p, _p, _i64, _p, _i64, _p, _i64, _i64, _i64, _i64, _int, _int, _int, _p],
    "gpx_colsumsq": [_p, _p, _i64, _i64, _i64, _p, _p, _p],
    "gpx_transpose": [_p, _p, _i64, _i64, _i64, _p, _i64, _p],
    "gpx_set_mask": [_p, _p, _p, C.c_uint8, _p],
    "gpx_store_pivot": [_p, _p, _i64, _p, _i64, _p, _p, _p, _p],
    "gpx_design_delete_factor": [_p, _p, _i64, _i64, _i64, _p, _p, _p, _p, _p],
    "gpx_design_delete_rows": [_p, _p, _i64, _i64, _p, _i64, _i64, _p, _p],
    "gpx_exchange_keep": [_p, _p, _i64, _i64, _p, _dbl, _p, _p, _p, _p],
    "gpx_design_delete_factors": [_p, _i64, _i64, _p, _i64, _p, _p, _p, _p, _p, _i64, _p, _p],
    "gpx_exchange_keep_max": [_p, _p, _i64, _i64, _i64, _i64, _i64, _p, _p, _dbl, _p, _p, _p, _p],
    "gpx_exchange_unmask": [_p, _p, _i64, _i64, _i64, _i64, _i64, _p, _p],
    "gpx_exchange_record": [_p, _p, _p, _i64, _p, _p, _p, _p, _p],
    "gpx_comm_unique_id": [_p, _int],
    "gpx_comm_init": [_p, _p, _int, _int],
    "gpx_comm_destroy": [_p],
    "gpx_comm_size": [_p],
    "gpx_comm_allgather": [_p, _p, _p, _i64, _p],
    "gpx_comm_bcast": [_p, _p, _i64, _int, _p],
    "gpx_comm_allreduce_sum": [_p, _p, _i64, _p],
    "gpx_ivar_greedy_run": [_p, C.POINTER(IvarState), _i64, _i64, _p],
    "gpx_ivar_greedy_small": [_p, C.POINTER(IvarState), _i64, _i64, _p],
    "gpx_var_greedy_run": [_p, C.POINTER(VarState), _i64, _i64, _p],
    "gpx_state_bytes": [_int],
    "gpx_se_dgram": [_p, _p, _i64, _i64, _p, _i64, _i64, _p, _i64, _p],
    "gpx_se_var_grad": [_p, _p, _i64, _i64, _p, _i64, _i64, _p, _p, _p, _p, _p],
    "gpx_se_loglike_grad_workspace": [_i64, _int],
    "gpx_se_loglike_grad": [_p, _p, _i64, _i64, _p, _i64, _p, _p, _p, _p],
    "gpx_gram_matvec_workspace": [_i64],
    "gpx_gram_matvec": [_p, _p, _i64, _i64, _p, _i64, _i64, _p, _p, _p, _p],
    "gpx_scale_rows_cols": [_p, _p, _i64, _i64, _i64, _p, _p, _dbl, _p, _i64, _p],
    "gpx_diag_update": [_p, _p, _i64, _i64, _dbl, _p, _dbl, _p],
    "gpx_axpby": [_p, _i64, _dbl, _p, _dbl, _p, _p],
    "gpx_coldot": [_p, _p, _p, _i64, _i64, _i64, _p, _p, _p],
    "gpx_rowsum": [_p, _p, _i64, _i64, _i64, _dbl, _p, _p],
    "gpx_rowsum_w": [_p, _p, _i64, _i64, _i64, _p, _p, _p],
    "gpx_logdet_chol": [_p, _p, _i64, _i64, _p, _p],
    "gpx_bench_dmma": [_p, _i64, _p, _p],
    "gpx_bench_dfma": [_p, _i64, _p, _p],
}
_RESTYPES = {"gpx_last_error": C.c_char_p, "gpx_score_ivar_workspace": _i64, "gpx_ivar_scratch_bytes": _i64, "gpx_mi_prec_column_workspace": _i64,
             "gpx_state_bytes": _i64, "gpx_launch_count": _i64, "gpx_se_loglike_grad_workspace": _i64,
             "gpx_gram_matvec_workspace": _i64}

for _name, _args in SIGNATURES.items():
    _fn = getattr(lib, _name)  # AttributeError here == the .so does not export a declared symbol
    _fn.argtypes = _args
    _fn.restype = _RESTYPES.get(_name, _int)


if lib.gpx_state_bytes(0) != C.sizeof(IvarState) or lib.gpx_state_bytes(1) != C.sizeof(VarState):
    raise ImportError("gpexp_b200: the state structs of libgpexp_b200.so do not match this binding; rebuild the library")


def last_error() -> str:
    msg = lib.gpx_last_error()
    return msg.decode() if msg else ""


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        raise GpxError(f"{what or 'gpexp_b200'} failed with code {rc}: {last_error()}")
