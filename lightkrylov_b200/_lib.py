"""ctypes loader of liblkb.so.  Fails loudly when the CUDA extension is missing -- there is no
CPU fallback anywhere in this package."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# LKB_SO: an alternative build of the SAME library for kernel A/B experiments (profiles/*.sh); never a different backend
SO_PATH = os.environ.get("LKB_SO") or os.path.join(_HERE, "csrc", "liblkb.so")
_lib = None


class LkbError(RuntimeError):
    pass


class GmresIO(C.Structure):
    _fields_ = [("kdim", C.c_int32), ("maxiter", C.c_int32), ("n_iter", C.c_int32), ("n_inner", C.c_int32),
                ("n_outer", C.c_int32), ("converged", C.c_int32), ("info", C.c_int32),
                ("res", C.POINTER(C.c_double)), ("res_cap", C.c_int32), ("res_len", C.c_int32)]


class CgIO(C.Structure):
    _fields_ = [("maxiter", C.c_int32), ("n_iter", C.c_int32), ("converged", C.c_int32), ("info", C.c_int32),
                ("res", C.POINTER(C.c_double)), ("res_cap", C.c_int32), ("res_len", C.c_int32)]


MATVEC_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p)
PRECOND_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_double, C.c_double, C.c_void_p)

_vp, _i, _i32, _i64, _u64, _d = C.c_void_p, C.c_int, C.c_int32, C.c_int64, C.c_uint64, C.c_double
_P = C.POINTER

# name -> (restype, argtypes); mirrors include/lkb.h one to one
SIGNATURES = {
    "lkb_init": (_i, [_i, _P(_vp)]),
    "lkb_nccl_unique_id": (_i, [_vp]),
    "lkb_init_dist": (_i, [_i, _i, _i, _vp, _P(_vp)]),
    "lkb_finalize": (_i, [_vp]),
    "lkb_sync": (_i, [_vp]),
    "lkb_stream": (_vp, [_vp]),
    "lkb_last_error": (C.c_char_p, []),
    "lkb_set_seed": (_i, [_vp, _u64]),
    "lkb_set_graphs": (_i, [_vp, _i]),
    "lkb_set_option": (_i, [_vp, C.c_char_p, _i]),
    "lkb_p2p_export": (_i, [_vp, _vp]),
    "lkb_p2p_attach": (_i, [_vp, _vp]),
    "lkb_rank": (_i, [_vp]),
    "lkb_world": (_i, [_vp]),
    "lkb_vec_create": (_i, [_vp, _i, _i64, _i64, _i64, _P(_vp)]),
    "lkb_vec_wrap": (_i, [_vp, _i, _i64, _i64, _i64, _vp, _P(_vp)]),
    "lkb_vec_clone": (_i, [_vp, _P(_vp)]),
    "lkb_vec_destroy": (_i, [_vp]),
    "lkb_vec_zero": (_i, [_vp]),
    "lkb_vec_rand": (_i, [_vp, _i32]),
    "lkb_vec_fill_random": (_i, [_vp, _i, _u64]),
    "lkb_vec_scal": (_i, [_vp, _vp]),
    "lkb_vec_axpby": (_i, [_vp, _vp, _vp, _vp]),
    "lkb_vec_dot": (_i, [_vp, _vp, _vp]),
    "lkb_vec_norm": (_i, [_vp, _P(_d)]),
    "lkb_vec_size": (_i64, [_vp]),
    "lkb_vec_local_size": (_i64, [_vp]),
    "lkb_vec_ptr": (_vp, [_vp]),
    "lkb_vec_put": (_i, [_vp, _vp]),
    "lkb_vec_get": (_i, [_vp, _vp]),
    "lkb_basis_create": (_i, [_vp, _i, _i64, _i64, _i64, _i, _P(_vp)]),
    "lkb_basis_destroy": (_i, [_vp]),
    "lkb_basis_col": (_i, [_vp, _i, _P(_vp)]),
    "lkb_basis_zero": (_i, [_vp, _i, _i]),
    "lkb_basis_view": (_i, [_vp, _i, _i, _P(_vp)]),
    "lkb_basis_axpby": (_i, [_vp, _vp, _i, _vp, _vp, _i, _i]),
    "lkb_basis_rand": (_i, [_vp, _i, _i, _i32]),
    "lkb_orthonormalize_basis": (_i, [_vp, _i, _i, _P(_i32)]),
    "lkb_initialize_krylov_subspace": (_i, [_vp, _vp, _i, _i]),
    "lkb_initialize_random_orthonormal_basis": (_i, [_vp, _i, _i]),
    "lkb_basis_put": (_i, [_vp, _i, _i, _vp, _i64]),
    "lkb_basis_get": (_i, [_vp, _i, _i, _vp, _i64]),
    "lkb_basis_ncols": (_i, [_vp]),
    "lkb_basis_ld": (_i64, [_vp]),
    "lkb_basis_innerprod": (_i, [_vp, _i, _vp, _i, _i, _vp, _i]),
    "lkb_basis_lincomb_sub": (_i, [_vp, _i, _vp, _i, _vp, _i, _i]),
    "lkb_basis_lincomb": (_i, [_vp, _i, _vp, _vp]),
    "lkb_dgs_step": (_i, [_vp, _i, _vp, _i, _i, _i32, _vp, _i, _P(_i32)]),
    "lkb_orthogonalize_against_basis": (_i, [_vp, _i, _vp, _i, _i, _i32, _vp, _i, _P(_i32)]),
    "lkb_qr": (_i, [_vp, _i, _i, _vp, _i, _d, _P(_i32)]),
    "lkb_qr_pivoting": (_i, [_vp, _i, _i, _vp, _i, _P(_i32), _d, _P(_i32)]),
    "lkb_op_stencil5_create": (_i, [_vp, _i, _i64, _i64, _vp, _i64, _i64, _P(_vp)]),
    "lkb_op_stencil7_create": (_i, [_vp, _i, _i64, _i64, _i64, _vp, _i64, _i64, _P(_vp)]),
    "lkb_op_csr_create": (_i, [_vp, _i, _i64, _i64, _vp, _vp, _vp, _P(_vp)]),
    "lkb_op_csr_create_device": (_i, [_vp, _i, _i64, _i64, _vp, _vp, _vp, _i32, _P(_vp)]),
    "lkb_csr_random_device": (_i, [_vp, _i, _i64, _i64, _i64, _i32, _u64, _P(_vp), _P(_vp), _P(_vp)]),
    "lkb_dev_free": (_i, [_vp]),
    "lkb_op_csr_create_dist": (_i, [_vp, _i, _i64, _i64, _i64, _i64, _i64, _i64, _vp, _vp, _vp, _P(_vp)]),
    "lkb_op_csr_create_dist_device": (_i, [_vp, _i, _i64, _i64, _i64, _i64, _i64, _i64, _vp, _vp, _vp, _i32, _P(_vp)]),
    "lkb_op_dense_create": (_i, [_vp, _i, _i64, _i64, _vp, _P(_vp)]),
    "lkb_op_callback_create": (_i, [_vp, _i, _i64, _i64, MATVEC_FN, _vp, _i32, _P(_vp)]),
    "lkb_op_diag_create": (_i, [_vp, _P(_vp)]),
    "lkb_op_jacobi_create": (_i, [_vp, _P(_vp)]),
    "lkb_op_chebyshev_create": (_i, [_vp, _i32, _d, _d, _P(_vp)]),
    "lkb_op_poly_create": (_i, [_vp, _i32, _P(_d), _P(_vp)]),
    "lkb_op_gmres_poly_create": (_i, [_vp, _i32, _u64, _P(_vp)]),
    "lkb_op_multigrid_create": (_i, [_vp, _i32, _P(_vp)]),
    "lkb_op_poly_roots": (_i, [_vp, _i32, _P(_i32), _P(_d)]),
    "lkb_op_destroy": (_i, [_vp]),
    "lkb_op_matvec": (_i, [_vp, _vp, _vp]),
    "lkb_op_rmatvec": (_i, [_vp, _vp, _vp]),
    "lkb_op_counters": (_i, [_vp, _P(_i64), _P(_i64)]),
    "lkb_op_reset_counters": (_i, [_vp]),
    "lkb_arnoldi": (_i, [_vp, _vp, _vp, _i, _P(_i32), _i32, _i32, _d, _i32, _i32]),
    "lkb_lanczos": (_i, [_vp, _vp, _vp, _i, _P(_i32), _i32, _i32, _d]),
    "lkb_bidiag": (_i, [_vp, _vp, _vp, _vp, _i, _P(_i32), _i32, _i32, _d]),
    "lkb_krylov_schur": (_i, [_vp, _vp, _i, _i, _P(_i32)]),
    "lkb_gmres": (_i, [_vp, _vp, _vp, _P(_i32), _d, _d, _i32, _P(GmresIO)]),
    "lkb_cg": (_i, [_vp, _vp, _vp, _P(_i32), _d, _d, _P(CgIO)]),
    "lkb_gmres_precond": (_i, [_vp, _vp, _vp, _P(_i32), _d, _d, _i32, _P(GmresIO), PRECOND_FN, _vp]),
    "lkb_fgmres": (_i, [_vp, _vp, _vp, _P(_i32), _d, _d, _i32, _P(GmresIO), PRECOND_FN, _vp]),
    "lkb_cg_precond": (_i, [_vp, _vp, _vp, _P(_i32), _d, _d, _P(CgIO), PRECOND_FN, _vp]),
    "lkb_gmres_precond_op": (_i, [_vp, _vp, _vp, _P(_i32), _d, _d, _i32, _P(GmresIO), _vp]),
    "lkb_cg_precond_op": (_i, [_vp, _vp, _vp, _P(_i32), _d, _d, _P(CgIO), _vp]),
    "lkb_eigs": (_i, [_vp, _vp, _i, _P(_d), _P(_d), _P(_i32), _vp, _i32, _d, _i32]),
    "lkb_eighs": (_i, [_vp, _vp, _i, _P(_d), _P(_d), _P(_i32), _vp, _i32, _d]),
    "lkb_svds": (_i, [_vp, _vp, _P(_d), _vp, _i, _P(_d), _P(_i32), _vp, _i32, _d]),
    "lkb_kexpm_vec": (_i, [_vp, _vp, _vp, _d, _d, _P(_i32), _i32, _i32]),
    "lkb_kexpm_mat": (_i, [_vp, _vp, _vp, _i, _d, _d, _P(_i32), _i32, _i32]),
    "lkb_krylov_expta": (_i, [_vp, _vp, _vp, _d, _P(_i32), _i32]),
    "lkb_write_results": (_i, [C.c_char_p, _i32, _P(_d), _P(_d), _i32, _d]),
    "lkb_save_eigenspectrum": (_i, [C.c_char_p, _i32, _i32, _P(_d), _P(_d), _i32]),
    "lkb_set_lapack": (_i, [C.c_char_p, C.c_char_p, C.c_char_p]),
    "lkb_set_profile": (_i, [_vp, _i]),
    "lkb_get_profile": (_i, [_vp, _P(_d), _P(_i64)]),
    "lkb_kernel_launches": (_i64, [_vp]),
    "lkb_debug_ktime": (_i, [_vp, _i]),
    "lkb_debug_ktime_read": (_i, [_vp, _P(_u64), _i]),
}


def load():
    """Load liblkb.so and bind every entry point of include/lkb.h."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise LkbError(f"{SO_PATH} is missing: run `python -m lightkrylov_b200.build` "
                       "(nvcc, sm_100a).  There is no CPU fallback.")
    lib = C.CDLL(SO_PATH, mode=C.RTLD_GLOBAL)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)           # AttributeError = header / library mismatch: fail loudly
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().lkb_last_error().decode(errors="replace")
        raise LkbError(f"{what} failed with code {rc}: {msg}")
