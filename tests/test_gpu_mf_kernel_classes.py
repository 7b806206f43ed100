"""Every kernel class of the multifrontal solver against an extended-precision reference, through the Level-1 ABI
(HMCMT_SHIM_SOLVER=mf).  The matrices of tests/mf_class_cases.py reach, together, every single-CTA instantiation (1 ... 16 warps),
both layouts of the single-CTA kernel, the global-memory path entered by size and by child count with 1, 2 and 3 pivot chunks,
every width of the warp solves and both CTA-solve widths; tests/test_mf_classes_cpu.py checks on the CPU that they still do.

On every matrix (complex and its real twin) and every knob setting of mf_class_cases.ROUTINGS:
  * forward error against the reference <= 100 eps kappa_1 (kappa_1 estimated by onenormest on the reference's factor);
  * normwise relative residual < 1e-14;
  * the solutions of the five warp routings are bit-identical: each tile sees the same sequence of operations in every
    instantiation (rolled or unrolled gj_invert8, paired or single Schur tiles, F22 scattered into shared memory or gathered
    from the children in the same child order).
Then the Level-1 edges: right-hand sides beyond the 16 of one solve launch, the sparse right-hand-side entry points, and the scale
equivariance of the factorisation (2^k A is factorised and solved exactly like A for every k whose entries stay normal)."""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

from tests import mf_class_cases as mc

pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps


def reference(A, b):
    """x_ref: splu in complex128 refined three times with residuals b - A x formed in extended precision (plain CSR product);
    kappa_1 estimate of A from the same factor"""
    assert np.finfo(np.longdouble).nmant >= 63, \
        "the reference needs an extended-precision long double (64-bit mantissa); numpy's long double here has " \
        f"{np.finfo(np.longdouble).nmant} mantissa bits"
    A = sp.csc_matrix(A, dtype=np.complex128)
    lu = spla.splu(A)
    R = A.tocsr()
    R.sort_indices()
    assert (np.diff(R.indptr) > 0).all()
    vals, cols, starts = R.data.astype(np.clongdouble), R.indices, R.indptr[:-1]
    bl = b.astype(np.clongdouble)
    x = lu.solve(b.astype(np.complex128)).astype(np.clongdouble)
    for _ in range(3):
        r = bl - np.add.reduceat(vals * x[cols], starts)
        x = x + lu.solve(r.astype(np.complex128)).astype(np.clongdouble)
    n = A.shape[0]
    inv = spla.LinearOperator((n, n), matvec=lambda v: lu.solve(np.asarray(v, dtype=np.complex128).ravel()),
                              rmatvec=lambda v: lu.solve(np.asarray(v, dtype=np.complex128).ravel(), trans="H"), dtype=np.complex128)
    return x.astype(np.complex128), spla.onenormest(A) * spla.onenormest(inv)


def relres(A, x, b):
    return np.linalg.norm(A @ x - b) / np.linalg.norm(b)


@pytest.fixture
def knobs(monkeypatch):
    """sets every knob of the analysis and the schedule (the others at the library's defaults), multifrontal path forced"""
    def apply(env):
        for k in mc.KNOBS:
            monkeypatch.setenv(k, env.get(k, mc.DEFAULTS[k]))
        monkeypatch.setenv("HMCMT_SHIM_SOLVER", "mf")
    return apply


def solve(A, b):
    from hmcmt2d_b200 import lib
    F = lib.factorMUMPS(A, 1)
    try:
        return lib.applyMUMPS(F, b)
    finally:
        lib.destroyMUMPS(F)


@pytest.mark.parametrize("real", [False, True], ids=["complex", "real"])
@pytest.mark.parametrize("name", sorted(mc.CASES))
def test_kernel_classes_against_reference(knobs, name, real):
    A = mc.CASES[name][0](real)
    n = A.shape[0]
    rng = np.random.default_rng(11)
    b = rng.standard_normal(n) if real else rng.standard_normal(n) + 1j * rng.standard_normal(n)
    xref, kappa = reference(A, b)
    bound = 100 * EPS * kappa
    assert bound <= 1e-9, (name, kappa)
    xs, worst = {}, 0.0
    for r, env in mc.ROUTINGS.items():
        knobs(env)
        x = solve(A, b)
        assert x.dtype == (np.float64 if real else np.complex128)
        err = np.abs(x - xref).max() / np.abs(xref).max()
        worst = max(worst, err / bound)
        assert err <= bound, (name, r, err, bound)
        assert relres(A, x, b) < 1e-14, (name, r, relres(A, x, b))
        xs[r] = x
    print(f"\n[mf classes] {name} {'real' if real else 'complex'}: n {n}  kappa_1 ~ {kappa:.2e}  bound {bound:.1e}  "
          f"largest error / bound {worst:.2e}")
    for r in mc.WARP_ROUTINGS[1:]:
        assert np.array_equal(xs[r], xs[mc.WARP_ROUTINGS[0]]), \
            (name, r, np.abs(xs[r] - xs[mc.WARP_ROUTINGS[0]]).max())


# ---- Level-1 edges -----------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("real", [False, True], ids=["complex", "real"])
def test_many_rhs_equal_single_solves(knobs, real):
    """nrhs beyond one solve launch (16) is split into chunks; every vector is solved independently: bit for bit the same as
    the vectors solved one at a time"""
    from hmcmt2d_b200 import lib
    knobs({})
    A = mc.CASES["mt2d_37x53"][0](real)
    n = A.shape[0]
    rng = np.random.default_rng(12)
    B = rng.standard_normal((n, 33)) if real else rng.standard_normal((n, 33)) + 1j * rng.standard_normal((n, 33))
    F = lib.factorMUMPS(A, 1)
    try:
        single = np.stack([lib.applyMUMPS(F, B[:, j]) for j in range(33)], axis=1)
        for nrhs in (15, 16, 17, 33):
            X = lib.applyMUMPS(F, B[:, :nrhs])
            assert np.array_equal(X, single[:, :nrhs]), nrhs
    finally:
        lib.destroyMUMPS(F)
    assert relres(A, single[:, 32], B[:, 32]) < 1e-14


@pytest.mark.parametrize("real", [False, True], ids=["complex", "real"])
def test_sparse_rhs_equals_dense(knobs, real):
    """solve_mumps[_cmplx]_sparse_rhs_ (MUMPSfuncs.jl:115-118, 139-143) with empty columns, 17 columns (two solve launches):
    bit for bit the dense solve of the same right-hand sides"""
    from hmcmt2d_b200 import lib
    knobs({})
    L = lib.load()
    A = mc.CASES["divgrad_9x10x11"][0](real)
    n, nrhs = A.shape[0], 17
    rng = np.random.default_rng(13)
    Bs = sp.random(n, nrhs, density=0.02, format="csc", random_state=rng, dtype=np.float64)
    if not real:
        Bs = (Bs + 1j * sp.random(n, nrhs, density=0.02, format="csc", random_state=rng)).tocsc()
    Bs = Bs.tolil()
    for j in (0, 5, 16):                                  # empty columns, the last one included
        Bs[:, j] = 0
    Bs = sp.csc_matrix(Bs)
    Bs.eliminate_zeros()
    Bs.sort_indices()
    assert np.diff(Bs.indptr)[[0, 5, 16]].sum() == 0 and Bs.nnz > 0
    F = lib.factorMUMPS(A, 1)
    try:
        dense = lib.applyMUMPS(F, Bs.toarray())
        dt = np.float64 if real else np.complex128
        nz = np.ascontiguousarray(Bs.data.astype(dt))
        rowval = Bs.indices.astype(np.int64) + 1
        colptr = Bs.indptr.astype(np.int64) + 1
        x = np.zeros((nrhs, n), dtype=dt)                 # column-major n x nrhs
        fn = L.solve_mumps_sparse_rhs_ if real else L.solve_mumps_cmplx_sparse_rhs_
        h, nzr, nr, tr = C.c_int64(F.ptr), C.c_int64(Bs.nnz), C.c_int64(nrhs), C.c_int64(0)
        fn(C.byref(h), C.byref(nzr), C.byref(nr), nz.ctypes.data_as(lib._f64p), lib.i64(rowval), lib.i64(colptr),
           x.ctypes.data_as(lib._f64p), C.byref(tr))
    finally:
        lib.destroyMUMPS(F)
    assert np.array_equal(x.T, dense)
    assert not x[[0, 5, 16]].any() and x.any()


# ---- scale equivariance ------------------------------------------------------------------------------------------------

SCALES = [s * k for k in (1, 64, 300, 505, 520, 530, 700, 900) for s in (1, -1)]
SCALE_CASES = {      # name -> (matrix, knobs): the band kernel, single-CTA fronts only, global-memory fronts only
    "band_12x30": (lambda real: mc.mt2d(12, 30, 7, real), None),
    "mf_small": (lambda real: mc.CASES["mt2d_21x19"][0](real), {}),
    "mf_global": (lambda real: mc.CASES["mt2d_37x53"][0](real), {"HMCMT_MF_FSMALL": "0"}),
}


@pytest.mark.parametrize("real", [False, True], ids=["complex", "real"])
@pytest.mark.parametrize("case", sorted(SCALE_CASES))
def test_scale_equivariance(knobs, monkeypatch, case, real):
    """A pivot-free elimination whose own scalings are powers of two commutes with A -> 2^k A: the solution is 2^-k x(A) bit
    for bit while every entry of A, of the factors and of x stays a normal number (|k| <= 900 here).  Far below that the
    pivots fall under the singularity threshold (1e-290) and the factorisation must say so (-10), never report success with
    a non-finite solution."""
    from hmcmt2d_b200 import lib
    build, env = SCALE_CASES[case]
    if env is None:
        for k in mc.KNOBS + ("HMCMT_SHIM_SOLVER",):
            monkeypatch.delenv(k, raising=False)
    else:
        knobs(env)
    A = sp.csc_matrix(build(real))
    n = A.shape[0]
    b = np.random.default_rng(14).standard_normal(n)
    x0 = solve(A, b)
    assert relres(A, x0, b) < 1e-14
    failed = []
    for k in SCALES:
        As = A.copy()
        As.data = As.data * np.ldexp(1.0, k)
        try:
            x = solve(As, b)
        except lib.HmcmtError as e:
            failed.append((k, f"status {e.code}"))
            continue
        if not np.array_equal(x, x0 * np.ldexp(1.0, -k)):
            failed.append((k, "finite" if np.isfinite(x).all() else "non-finite", float(np.nanmax(np.abs(x * np.ldexp(1.0, k) - x0)))))
    assert not failed, failed
    As = A.copy()
    As.data = As.data * np.ldexp(1.0, -1000)
    with pytest.raises(lib.HmcmtError) as e:
        x = solve(As, b)
        print(f"2^-1000 A: status 0, finite solution: {np.isfinite(x).all()}")
    assert e.value.code == -10
