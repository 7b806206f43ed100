"""diag(A^-1) by selected inversion of the multifrontal factor (Solver::inverse_diag, mf_selinv.cuh) through the Level-1 entry
hmcmt_factor_inverse_diag / lib.inverse_diag (HMCMT_SHIM_SOLVER=mf).  On every matrix of tests/mf_class_cases.py, complex and its
real twin, under every knob setting of mf_class_cases.ROUTINGS (so every front class: single-CTA fronts of 1 ... 16 warps,
global-memory fronts entered by size and by child count with 1, 2 and 3 pivot chunks):
  * against diag(A^-1) from splu solves of unit vectors, refined once with residuals in extended precision: all i where n <= 3000,
    1024 fixed-seed indices otherwise; bound max|d - d_ref| <= 100 eps kappa_1 max|d_ref|;
  * the five warp routings give bit-identical diagonals (their factors are bit-identical; the sweep reads no routing knob);
  * repeated calls are bit-identical and a solve after the call equals a solve before it, bit for bit.
Then: a complex matrix with zero imaginary part gives an exactly zero imaginary diagonal whose real part is the real handle's, bit
for bit; a band-routed and an unknown handle are refused with -3."""
import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

from tests import mf_class_cases as mc

pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps


def reference_diag(A, idx):
    """diag(A^-1)[idx] from splu solves of the unit vectors e_i, refined once with residuals e_i - A x formed in extended
    precision; kappa_1 estimate from the same factor"""
    assert np.finfo(np.longdouble).nmant >= 63, "the reference needs an extended-precision long double"
    A = sp.csc_matrix(A, dtype=np.complex128)
    n = A.shape[0]
    lu = spla.splu(A)
    R = A.tocsr()
    R.sort_indices()
    vals, cols, starts = R.data.astype(np.clongdouble), R.indices, R.indptr[:-1]
    out = np.empty(len(idx), dtype=np.complex128)
    for b0 in range(0, len(idx), 64):
        blk = idx[b0:b0 + 64]
        E = np.zeros((n, len(blk)), dtype=np.complex128)
        E[blk, np.arange(len(blk))] = 1.0
        X = lu.solve(E).astype(np.clongdouble)
        res = E.astype(np.clongdouble) - np.add.reduceat(vals[:, None] * X[cols, :], starts, axis=0)
        X = X + lu.solve(res.astype(np.complex128)).astype(np.clongdouble)
        out[b0:b0 + len(blk)] = X[blk, np.arange(len(blk))].astype(np.complex128)
    inv = spla.LinearOperator((n, n), matvec=lambda v: lu.solve(np.asarray(v, dtype=np.complex128).ravel()),
                              rmatvec=lambda v: lu.solve(np.asarray(v, dtype=np.complex128).ravel(), trans="H"), dtype=np.complex128)
    return out, spla.onenormest(A) * spla.onenormest(inv)


@pytest.fixture
def knobs(monkeypatch):
    """sets every knob of the analysis and the schedule (the others at the library's defaults), multifrontal path forced"""
    def apply(env):
        for k in mc.KNOBS:
            monkeypatch.setenv(k, env.get(k, mc.DEFAULTS[k]))
        monkeypatch.setenv("HMCMT_SHIM_SOLVER", "mf")
    return apply


def _indices(n):
    return np.arange(n) if n <= 3000 else np.sort(np.random.default_rng(5).choice(n, 1024, replace=False))


@pytest.mark.parametrize("real", [False, True], ids=["complex", "real"])
@pytest.mark.parametrize("name", sorted(mc.CASES))
def test_inverse_diag_against_reference(knobs, name, real):
    from hmcmt2d_b200 import lib
    A = mc.CASES[name][0](real)
    n = A.shape[0]
    idx = _indices(n)
    dref, kappa = reference_diag(A, idx)
    bound = 100 * EPS * kappa * np.abs(dref).max()
    b = np.random.default_rng(2).standard_normal(n)
    ds, worst = {}, 0.0
    for r, env in mc.ROUTINGS.items():
        knobs(env)
        F = lib.factorMUMPS(A, 1)
        try:
            x0 = lib.applyMUMPS(F, b)
            d = lib.inverse_diag(F)
            assert d.dtype == (np.float64 if real else np.complex128)
            assert np.array_equal(lib.inverse_diag(F), d), (name, r, "repeat")
            assert np.array_equal(lib.applyMUMPS(F, b), x0), (name, r, "solve after the call")
        finally:
            lib.destroyMUMPS(F)
        err = np.abs(d[idx] - dref).max()
        worst = max(worst, err / bound)
        assert err <= bound, (name, r, err, bound)
        ds[r] = d
    print(f"\n[selinv] {name} {'real' if real else 'complex'}: n {n}  kappa_1 ~ {kappa:.2e}  largest error / bound {worst:.2e}")
    for r in mc.WARP_ROUTINGS[1:]:
        assert np.array_equal(ds[r], ds[mc.WARP_ROUTINGS[0]]), (name, r)


def test_zero_imaginary_part_equals_real_handle(knobs):
    from hmcmt2d_b200 import lib
    knobs({})
    A = mc.CASES["divgrad_9x10x11"][0](True)
    Fr = lib.factorMUMPS(A, 1)
    Fc = lib.factorMUMPS(sp.csc_matrix(A, dtype=np.complex128), 1)
    try:
        dr, dc = lib.inverse_diag(Fr), lib.inverse_diag(Fc)
    finally:
        lib.destroyMUMPS(Fr)
        lib.destroyMUMPS(Fc)
    assert np.all(dc.imag == 0.0)
    assert np.array_equal(dc.real, dr)


def test_band_and_unknown_handles_refused(monkeypatch):
    from hmcmt2d_b200 import lib
    monkeypatch.delenv("HMCMT_SHIM_SOLVER", raising=False)
    n = 200
    A = sp.diags([np.full(n, 4.0), -np.ones(n - 1), -np.ones(n - 1)], [0, 1, -1], format="csc")
    F = lib.factorMUMPS(A, 1)
    try:
        with pytest.raises(lib.HmcmtError) as e:
            lib.inverse_diag(F)
        assert e.value.code == -3
    finally:
        lib.destroyMUMPS(F)
    with pytest.raises(lib.HmcmtError) as e:
        lib.inverse_diag(lib.MUMPSfactorization(123456789, n, False))
    assert e.value.code == -3
