"""Projected Gauss-Newton-CG on the device (Plan.gauss_newton / hmcmt_gauss_newton): against the CPU reference
(tests/gn_reference.py) for impedance, rho / phase and tipper plans; the exact first step on both solvers; the bounds; chains
independent of each other; determinism across calls and launch modes; the resident state it leaves; descent on a synthetic
problem on the multifrontal path; argument errors."""
import numpy as np
import pytest

from tests import gn_reference as gnr
from tests.helpers import tiny_problem
from tests.test_gpu_jvec import _model, _plan, _problem

pytestmark = pytest.mark.gpu
CMP = dict(max_cg=5, cg_tol=0.0)


def _compare(pl, prob, m0, iters=3, **kw):
    """m_k after k = 1..iters iterations (a run of k iterations each), history and info against the reference.  The plan gets
    the reference's m_ref first: a new plan's m_ref is zero, and U (hence every step) depends on it."""
    pl.set_state(mref=prob.mref)
    _, _, ref_info, _ = gnr.gauss_newton(prob, m0, max_iter=iters, **kw)
    for k in range(1, iters + 1):
        m, h, info = pl.gauss_newton(m0, max_iter=k, **kw)
        rm, rh, rinfo, _ = gnr.gauss_newton(prob, m0, max_iter=k, **kw)
        scale = max(np.abs(rm - np.clip(m0, prob.lo, prob.hi)).max(), 1e-300)
        assert np.abs(m[0] - rm).max() <= 1e-8 * scale, (k, np.abs(m[0] - rm).max() / scale)
        assert tuple(info[0]) == rinfo, (k, info[0], rinfo)
        n = rinfo[0] + 1
        for col in (0, 1):
            assert np.abs(h[0, :n, col] - rh[:n, col]).max() <= 1e-9 * np.abs(rh[:n, col]).max(), (k, col)
        assert np.array_equal(h[0, :, 3], rh[:, 3]) and np.array_equal(h[0, :, 5], rh[:, 5]) and np.array_equal(h[0, :, 4], rh[:, 4])
        assert np.all(h[0, n:] == 0.0)
    return m[0], ref_info


@pytest.mark.parametrize("kind", ["impedance", "rho_phase", "tipper"])
def test_against_cpu_reference(kind):
    mesh, data, inv, prior, _ = _problem(kind)
    pl, _ = _plan(mesh, data, inv, prior)
    _, info = _compare(pl, gnr.Problem(mesh, data, inv, prior), _model(inv), **CMP)
    assert info[0] >= 1
    pl.close()


@pytest.mark.parametrize("solver", ["band", "mf"])
def test_exact_first_step(solver, monkeypatch):
    """A full CG (beta = 100: cond(H) ~ 200, see test_gn_reference_cpu.py) with the bounds far away: (m_1 - m_0) / alpha is the
    dense Newton step from the plan's own jacobian()."""
    monkeypatch.setenv("HMCMT_SOLVER", solver)
    mesh, data, inv, prior = tiny_problem(seed=19)
    prior.regParam = 100.0
    prior.sigBounds = [1e-12, 1e6]
    pl, (pm, pd, pi, pp) = _plan(mesh, data, inv, prior)
    m0 = _model(inv)
    _, _, g = pl.forward_gradient(m0, total=True)
    J = pl.jacobian()[0]
    D = np.exp(m0)
    H = D[:, None] * np.real(np.conj(J).T @ (np.abs(pi.dataW)[:, None] ** 2 * J)) * D[None, :] + 100.0 * pi.Wm.toarray()
    want = np.linalg.solve(H, -g[0])
    m1, h, info = pl.gauss_newton(m0, max_iter=1, max_cg=pl.nAC, cg_tol=1e-12, max_step=1e3)
    assert info[0, 0] == 1
    step = (m1[0] - m0) / h[0, 1, 4]
    assert np.abs(step - want).max() <= 1e-8 * np.abs(want).max()
    pl.close()


def test_bounds():
    """A narrow box the unconstrained step leaves: iterates inside, the active cells kept, the reference's iterates."""
    mesh, data, inv, prior = tiny_problem(seed=19)
    prior.sigBounds = [float(np.exp(inv.strModel.min() + 0.3)), float(np.exp(inv.strModel.max() - 0.3))]
    pl, _ = _plan(mesh, data, inv, prior)
    prob = gnr.Problem(mesh, data, inv, prior)
    m0 = _model(inv)
    _compare(pl, prob, m0, iters=3, **CMP)
    _, _, (nacc, _), steps = gnr.gauss_newton(prob, m0, max_iter=3, **CMP)
    prev = None
    for k in range(nacc + 1):
        m = pl.gauss_newton(m0, max_iter=k, **CMP)[0][0]
        assert np.all(m >= prob.lo) and np.all(m <= prob.hi)
        if k >= 1:
            mk, act, _, _, _ = steps[k - 1]
            assert np.array_equal(m[act], prev[act])
        prev = m
    assert any(a.any() for _, a, _, _, _ in steps)          # some cell was active
    pl.close()


def test_chains_independent():
    """A 2-chain plan against two 1-chain plans, bit for bit; also with one chain that stops at iteration 0 (its start is the
    end of a run whose line search failed) while the other keeps going."""
    mesh, data, inv, prior = tiny_problem(seed=7)
    ma, mb = _model(inv), _model(inv, seed=21)
    one = []
    for m0 in (ma, mb):
        p1, _ = _plan(mesh, data, inv, prior)
        one.append(p1.gauss_newton(m0, max_iter=4))
        p1.close()
    p2, _ = _plan(mesh, data, inv, prior, nChains=2)
    two = p2.gauss_newton(np.stack([ma, mb]), max_iter=4)
    for c in range(2):
        for x, y in zip(two, one[c]):
            assert np.array_equal(x[c], y[0]), c
    # the end of a run that stops on a failed line search
    p1, _ = _plan(mesh, data, inv, prior)
    mend, _, info = p1.gauss_newton(ma, max_iter=40, max_cg=40, cg_tol=1e-10, tol_rel=0.0)
    assert info[0, 1] == 2, info
    again = p1.gauss_newton(mend, max_iter=5, max_cg=40, cg_tol=1e-10, tol_rel=0.0)
    assert tuple(again[2][0]) == (0, 2) and np.array_equal(again[0][0], mend[0])
    other = p1.gauss_newton(mb, max_iter=5, max_cg=40, cg_tol=1e-10, tol_rel=0.0)
    assert other[2][0, 0] >= 2
    p1.close()
    two = p2.gauss_newton(np.stack([mend[0], mb]), max_iter=5, max_cg=40, cg_tol=1e-10, tol_rel=0.0)
    for c, ref in enumerate((again, other)):
        for x, y in zip(two, ref):
            assert np.array_equal(x[c], y[0]), c
    p2.close()


def test_determinism_and_issue_order(monkeypatch):
    """Two calls are bit-identical; so are plans without the CUDA graph and with one stream group."""
    monkeypatch.setenv("HMCMT_SOLVER", "mf")
    mesh, data, inv, prior = tiny_problem(seed=7)
    m0 = _model(inv)
    pl, _ = _plan(mesh, data, inv, prior)
    a = pl.gauss_newton(m0, max_iter=3)
    b = pl.gauss_newton(m0, max_iter=3)
    pl.close()
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    for env in ("HMCMT_GRAPH", "HMCMT_GROUPS"):
        monkeypatch.setenv(env, "0" if env == "HMCMT_GRAPH" else "1")
        p, _ = _plan(mesh, data, inv, prior)
        c = p.gauss_newton(m0, max_iter=3)
        p.close()
        monkeypatch.delenv(env)
        for x, y in zip(a, c):
            assert np.array_equal(x, y), env


def test_resident_state():
    """After the call the plan is evaluated at m_out: forward_gradient(m_out, total=True) reproduces the last history row's phi_d
    and its jvec is the one of the resident state; momentum and m_ref are those set before."""
    mesh, data, inv, prior = tiny_problem(seed=7)
    m0 = _model(inv)
    rng = np.random.default_rng(3)
    p0, mref = rng.standard_normal(len(m0)), inv.strModel + 0.1
    dsig = rng.standard_normal(len(m0)) * np.exp(m0)
    pl, _ = _plan(mesh, data, inv, prior)
    pl.set_state(m0, p0, mref)
    m, h, info = pl.gauss_newton(max_iter=3)
    assert info[0, 0] >= 1
    jv = pl.jvec(dsig)
    mm, pp = pl.get_state()
    assert np.array_equal(mm, m) and np.array_equal(pp[0], p0)
    _, phi, g = pl.forward_gradient(m, total=True)
    assert phi[0] == h[0, info[0, 0], 0]
    assert np.array_equal(pl.jvec(dsig), jv)
    ref, _ = _plan(mesh, data, inv, prior)
    ref.set_state(mref=mref)
    assert np.array_equal(ref.forward_gradient(m, total=True)[2], g)          # m_ref unchanged
    ref.close()
    pl.close()


def test_synthetic_descent_multifrontal(monkeypatch):
    """synthetic.make_problem (40 x 30 cells: 1271 unknowns per system, multifrontal), noise-free data of true_model: U does not
    increase over any iteration and the final |P g| is below the initial one."""
    from hmcmt2d_b200 import api, synthetic
    monkeypatch.setenv("HMCMT_SOLVER", "mf")
    mesh, data, inv, prior = synthetic.make_problem(40, 30, 4, nRx=10)
    fw = api.Plan(mesh, data, inv, prior)
    pred = fw.forward(sigma=synthetic.true_model(mesh), fields=False)[0][0]
    fw.close()
    mesh2, data2, inv2, prior2 = synthetic.make_problem(40, 30, 4, nRx=10, obs=pred, err=0.05 * np.abs(pred))
    pl = api.Plan(mesh2, data2, inv2, prior2)
    assert pl.info(0) >= 1000 and pl.info(11) == 1
    m, h, info = pl.gauss_newton(max_iter=5)
    n = info[0, 0]
    assert n >= 2
    U = h[0, : n + 1, 0] + h[0, : n + 1, 1]
    assert np.all(np.diff(U) <= 0.0), U
    assert h[0, n, 2] < h[0, 0, 2]
    pl.close()


def test_argument_errors():
    from hmcmt2d_b200 import lib as _lib
    mesh, data, inv, prior = tiny_problem(seed=7)
    pl, _ = _plan(mesh, data, inv, prior)
    n = pl.nAC
    m, hist, info = np.zeros(n), np.zeros((4, 6)), np.zeros(2, dtype=np.int32)
    f = lambda **kw: pl.L.hmcmt_gauss_newton(pl.h, None, kw.get("it", 3), kw.get("cg", 5), kw.get("cgt", 1e-2), kw.get("ls", 4),
                                             kw.get("st", 3.0), kw.get("tol", 1e-4), kw.get("m", _lib.f64(m)),
                                             kw.get("h", _lib.f64(hist)), kw.get("i", _lib.i32(info)))
    assert f(it=1) == 0
    for bad in (dict(m=None), dict(h=None), dict(i=None), dict(it=-1), dict(cg=0), dict(ls=0), dict(st=0.0), dict(st=-1.0),
                dict(st=float("nan")), dict(cgt=-1e-3), dict(cgt=float("inf")), dict(cgt=float("nan")), dict(tol=-1.0),
                dict(tol=float("inf"))):
        assert f(**bad) == -3, bad
    assert pl.L.hmcmt_gauss_newton(None, None, 1, 1, 0.0, 1, 1.0, 0.0, _lib.f64(m), _lib.f64(hist), _lib.i32(info)) == -3
    pl.close()
