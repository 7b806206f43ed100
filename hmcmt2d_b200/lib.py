"""ctypes binding of libhmcmt_b200.so (include/hmcmt_b200.h).  No fallback: if the CUDA library
is missing or cannot be loaded every entry point raises."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libhmcmt_b200.so")

_i64p = C.POINTER(C.c_int64)
_i32p = C.POINTER(C.c_int32)
_f64p = C.POINTER(C.c_double)


class HmcmtError(RuntimeError):
    """Raised for negative status codes (MUMPS convention, MUMPSfuncs.jl:59-73)."""

    MESSAGES = {-10: "numerically singular matrix", -13: "memory allocation error", -40: "matrix is not positive definite",
                -3: "bad argument", -21: "a parameter bound could not be met within 500 reflections", -98: "no CUDA device (there is no CPU fallback)", -99: "CUDA error"}

    def __init__(self, code: int, where: str):
        self.code = code
        super().__init__(f"hmcmt_b200: {where} failed with status {code}: {self.MESSAGES.get(code, 'error')}")


class Problem(C.Structure):
    """`hmcmt_problem` (include/hmcmt_b200.h)."""
    _fields_ = [
        ("ny", C.c_int32), ("nz", C.c_int32), ("yLen", _f64p), ("zLen", _f64p), ("origin", C.c_double * 2),
        ("nFreq", C.c_int32), ("freqs", _f64p), ("nRx", C.c_int32), ("rxLoc", _f64p),
        ("nComp", C.c_int32), ("compMode", _i32p), ("nData", C.c_int32),
        ("freqID", _i64p), ("rxID", _i64p), ("dtID", _i64p),
        ("obsData", _f64p), ("dataErr", _f64p), ("nAC", C.c_int32), ("activeIdx", _i32p), ("bgModel", _f64p),
        ("wmRowPtr", _i32p), ("wmColIdx", _i32p), ("wmVal", _f64p),
        ("regParam", C.c_double), ("sigBounds", C.c_double * 2), ("nChains", C.c_int32), ("device", C.c_int32),
    ]


_lib = None


def load() -> C.CDLL:
    """Load the CUDA library; raises (never falls back) when it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: build it with `python -m hmcmt2d_b200.build` "
                          "(nvcc, sm_100a). hmcmt2d_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    vp = C.c_void_p
    lib.hmcmt_version.restype = C.c_char_p
    lib.hmcmt_plan_create.argtypes = [C.POINTER(Problem), C.POINTER(vp)]
    lib.hmcmt_plan_create_rho_phase.argtypes = [C.POINTER(Problem), C.POINTER(vp)]
    lib.hmcmt_destroy.argtypes = [vp]
    lib.hmcmt_destroy.restype = None
    lib.hmcmt_plan_info.argtypes = [vp, C.c_int]
    lib.hmcmt_plan_info.restype = C.c_int64
    lib.hmcmt_forward.argtypes = [vp, _f64p, _f64p, _f64p, _f64p]
    lib.hmcmt_forward_sigma.argtypes = [vp, _f64p, _f64p, _f64p, _f64p]
    lib.hmcmt_jtvec.argtypes = [vp, _f64p, _f64p]
    lib.hmcmt_jacobian.argtypes = [vp, _f64p]
    lib.hmcmt_jvec.argtypes = [vp, _f64p, _f64p]
    lib.hmcmt_gn_hessvec.argtypes = [vp, _f64p, C.c_int32, _f64p]
    lib.hmcmt_gauss_newton.argtypes = [vp, _f64p, C.c_int32, C.c_int32, C.c_double, C.c_int32, C.c_double, C.c_double, _f64p,
                                       _f64p, _i32p]
    lib.hmcmt_status.argtypes = [vp]
    lib.hmcmt_set_mass_matrix.argtypes = [vp, C.c_int32]
    lib.hmcmt_set_response_kind.argtypes = [vp, C.c_int32]
    lib.hmcmt_get_responses.argtypes = [vp, _f64p]
    lib.hmcmt_forward_gradient.argtypes = [vp, _f64p, _f64p, _f64p, _f64p]
    lib.hmcmt_forward_gradient_total.argtypes = [vp, _f64p, _f64p, _f64p, _f64p]
    lib.hmcmt_set_state.argtypes = [vp, _f64p, _f64p, _f64p]
    lib.hmcmt_get_state.argtypes = [vp, _f64p, _f64p]
    lib.hmcmt_leapfrog_trajectory.argtypes = [vp, C.c_double, _i32p, _f64p, _f64p]
    lib.hmcmt_leapfrog_steps_device.argtypes = [vp, C.c_double, C.c_int32]
    lib.hmcmt_step_partial.argtypes = [vp, C.c_double]
    lib.hmcmt_exchange_buffer.argtypes = [vp, C.POINTER(vp), _i64p]
    lib.hmcmt_step_finish.argtypes = [vp, C.c_double]
    lib.hmcmt_sync.argtypes = [vp]
    lib.hmcmt_nccl_unique_id.argtypes = [C.c_char_p]
    lib.hmcmt_nccl_init.argtypes = [vp, C.c_char_p, C.c_int32, C.c_int32]
    lib.hmcmt_leapfrog_steps_sharded.argtypes = [vp, C.c_double, C.c_int32]
    lib.hmcmt_timer_start.argtypes = [vp]
    lib.hmcmt_timer_stop.argtypes = [vp, C.POINTER(C.c_float)]
    lib.hmcmt_kernel_time.argtypes = [vp, C.c_int, C.POINTER(C.c_float), _i64p]
    lib.hmcmt_kernel_time_split.argtypes = [vp, C.POINTER(C.c_float), C.POINTER(C.c_float)]
    lib.hmcmt_run_chain.argtypes = [vp, C.c_double, C.c_int32, C.c_double, _f64p, _f64p, _i32p, _f64p, _f64p, C.c_int32,
                                    _f64p, _f64p, _i32p, _f64p]
    lib.hmcmt_export_system.argtypes = [vp, C.c_int32, C.c_int32, C.c_int32, _i64p, _i64p, _f64p, _f64p, _f64p]
    for name in ("factor_mumps_cmplx_", "factor_mumps_"):
        fn = getattr(lib, name)
        fn.argtypes = [_i64p, _i64p, _i64p, _f64p, _i64p, _i64p, _i64p]
        fn.restype = C.c_int64
    for name in ("solve_mumps_cmplx_", "solve_mumps_"):
        fn = getattr(lib, name)
        fn.argtypes = [_i64p, _i64p, _f64p, _f64p, _i64p]
        fn.restype = C.c_int64
    for name in ("solve_mumps_sparse_rhs_", "solve_mumps_cmplx_sparse_rhs_"):
        fn = getattr(lib, name)
        fn.argtypes = [_i64p, _i64p, _i64p, _f64p, _i64p, _i64p, _f64p, _i64p]
        fn.restype = None
    for name in ("destroy_mumps_", "destroy_mumps_cmplx_"):
        fn = getattr(lib, name)
        fn.argtypes = [_i64p]
        fn.restype = C.c_int64
    _lib = lib
    return lib


EXPORTED_SYMBOLS = [
    "factor_mumps_cmplx_", "factor_mumps_", "solve_mumps_cmplx_", "solve_mumps_", "solve_mumps_sparse_rhs_",
    "solve_mumps_cmplx_sparse_rhs_", "destroy_mumps_", "destroy_mumps_cmplx_",
    "hmcmt_plan_create", "hmcmt_plan_create_rho_phase", "hmcmt_destroy", "hmcmt_plan_info", "hmcmt_forward", "hmcmt_forward_sigma", "hmcmt_jtvec",
    "hmcmt_forward_gradient", "hmcmt_forward_gradient_total", "hmcmt_jacobian", "hmcmt_jvec", "hmcmt_gn_hessvec", "hmcmt_gauss_newton", "hmcmt_status", "hmcmt_set_mass_matrix", "hmcmt_set_response_kind", "hmcmt_get_responses",
    "hmcmt_set_state", "hmcmt_get_state", "hmcmt_leapfrog_trajectory", "hmcmt_leapfrog_steps_device", "hmcmt_sync",
    "hmcmt_step_partial", "hmcmt_exchange_buffer", "hmcmt_step_finish", "hmcmt_nccl_unique_id", "hmcmt_nccl_init",
    "hmcmt_leapfrog_steps_sharded",
    "hmcmt_timer_start", "hmcmt_timer_stop", "hmcmt_kernel_time", "hmcmt_kernel_time_split", "hmcmt_run_chain", "hmcmt_export_system", "hmcmt_version",
]


def f64(a):
    return a.ctypes.data_as(_f64p)


def i64(a):
    return a.ctypes.data_as(_i64p)


def i32(a):
    return a.ctypes.data_as(_i32p)


def check(code: int, where: str):
    if code < 0:
        raise HmcmtError(int(code), where)
    return code


# ---- MUMPS-wrapper mirror (MUMPS/src/MUMPSfuncs.jl): factorMUMPS / applyMUMPS / destroyMUMPS --------------------

class MUMPSfactorization:
    """`MUMPSfactorization` MUMPS.jl:7-13."""

    def __init__(self, ptr, n, is_complex):
        self.ptr, self.n, self.is_complex = ptr, n, is_complex


def factorMUMPS(A, sym: int = 0, ooc: int = 0) -> MUMPSfactorization:
    """`factorMUMPS` MUMPSfuncs.jl:24-56.  A: scipy.sparse matrix (converted to full 1-based CSC)."""
    lib = load()
    A = A.tocsc()
    A.sort_indices()
    if A.shape[0] != A.shape[1]:
        raise ValueError("factorMUMPS: Matrix must be square!")
    n = C.c_int64(A.shape[0])
    s, o, st = C.c_int64(sym), C.c_int64(ooc), C.c_int64(0)
    rowval = (A.indices.astype(np.int64) + 1)
    colptr = (A.indptr.astype(np.int64) + 1)
    is_c = np.iscomplexobj(A.data)
    vals = np.ascontiguousarray(A.data.astype(np.complex128 if is_c else np.float64))
    fn = lib.factor_mumps_cmplx_ if is_c else lib.factor_mumps_
    ptr = fn(C.byref(n), C.byref(s), C.byref(o), vals.ctypes.data_as(_f64p), i64(rowval), i64(colptr), C.byref(st))
    check(st.value, "factorMUMPS")
    return MUMPSfactorization(ptr, A.shape[0], is_c)


def applyMUMPS(factor: MUMPSfactorization, rhs, tr: int = 0):
    """`applyMUMPS` MUMPSfuncs.jl:75-132.  rhs: (n,) or (n, nrhs)."""
    lib = load()
    rhs = np.asarray(rhs)
    if rhs.shape[0] != factor.n:
        raise ValueError(f"applyMUMPS: wrong size of rhs, size(A)={factor.n}, size(rhs)={rhs.shape}")
    nrhs = 1 if rhs.ndim == 1 else rhs.shape[1]
    cplx_io = factor.is_complex or np.iscomplexobj(rhs)
    dt = np.complex128 if cplx_io else np.float64
    b = np.asfortranarray(rhs.astype(dt).reshape(factor.n, nrhs))
    x = np.zeros_like(b, order="F")
    h, nr, t = C.c_int64(factor.ptr), C.c_int64(nrhs), C.c_int64(tr)
    fn = lib.solve_mumps_cmplx_ if cplx_io else lib.solve_mumps_
    rc = fn(C.byref(h), C.byref(nr), b.ctypes.data_as(_f64p), x.ctypes.data_as(_f64p), C.byref(t))
    check(rc, "applyMUMPS")
    return x[:, 0].copy() if rhs.ndim == 1 else np.ascontiguousarray(x)


def destroyMUMPS(factor: MUMPSfactorization):
    """`destroyMUMPS` MUMPSfuncs.jl:148-176 (poisons the handle)."""
    lib = load()
    h = C.c_int64(factor.ptr)
    (lib.destroy_mumps_cmplx_ if factor.is_complex else lib.destroy_mumps_)(C.byref(h))
    factor.ptr, factor.n = -1, -1


def solveMUMPS(A, rhs, sym: int = 0, ooc: int = 0, tr: int = 0):
    """`solveMUMPS` MUMPSfuncs.jl:2-20."""
    f = factorMUMPS(A, sym, ooc)
    try:
        return applyMUMPS(f, rhs, tr)
    finally:
        destroyMUMPS(f)
