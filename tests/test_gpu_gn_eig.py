"""The low-rank Gauss-Newton Hessian on the device (Plan.gn_eig / hmcmt_gn_eig), the mass matrix kind 2 it gives and the Laplace
draws (Plan.laplace_sample / hmcmt_laplace_sample): the exact regime against scipy.linalg.eigh(H, beta Wm) with H from the plan's
own jacobian() for impedance, rho / phase and tipper plans on both solvers; the randomized regime against the numpy restatement
(tests/gn_eig_reference.py); Rayleigh quotients at a real multifrontal tree; the sampler's drift and momentum draws with M = beta Wm
+ H_k; determinism, chain independence and the resident state; argument errors."""
import numpy as np
import pytest
import scipy.linalg as sla

from tests import gn_eig_reference as ger
from tests.helpers import tiny_problem
from tests.test_gpu_jvec import _model, _plan, _problem

pytestmark = pytest.mark.gpu


def _dense_H(pl, pi, m):
    """D Re(J^H Wd^2 J) D at m from the plan's own explicit Jacobian (the plan is left evaluated at m)."""
    pl.forward(m=m, fields=False)
    J = pl.jacobian()[0]
    D = np.exp(m)
    return D[:, None] * np.real(np.conj(J).T @ (np.abs(pi.dataW)[:, None] ** 2 * J)) * D[None, :]


@pytest.mark.parametrize("solver", ["band", "mf"])
@pytest.mark.parametrize("kind", ["impedance", "rho_phase", "tipper"])
def test_exact_regime_against_eigh(kind, solver, monkeypatch):
    """r = nAC = 40: the k' pairs against the top k' of eigh(H, beta Wm); the 1e-12 cut on G = Y^T B Y drops only directions
    below 1e-5 lambda_max; V^T beta Wm V = I."""
    monkeypatch.setenv("HMCMT_SOLVER", solver)
    mesh, data, inv, prior, _ = _problem(kind)
    pl, (pm, pd, pi, pp) = _plan(mesh, data, inv, prior)
    n, beta = pl.nAC, float(pp.regParam)
    m = _model(inv)
    H = _dense_H(pl, pi, m)
    lam, V, info = pl.gn_eig(n, r=n, seed=1)
    rk, kk = info[0]
    want = sla.eigh(H, beta * pi.Wm.toarray(), eigvals_only=True)[::-1]
    lmax = want[0]
    assert kk >= np.count_nonzero(want > 1e-5 * lmax) and rk >= kk, (rk, kk)
    err = np.abs(lam[0, :kk] - want[:kk])
    assert err[want[:kk] > 1e-4 * lmax].max() <= 1e-8 * lmax, err.max() / lmax
    assert err.max() <= 1e-6 * lmax, err.max() / lmax
    Vk = V[0, :kk].T
    assert np.abs(Vk.T @ (beta * pi.Wm @ Vk) - np.eye(kk)).max() <= 1e-10
    assert np.all(lam[0, kk:] == 0.0) and np.all(V[0, kk:] == 0.0)
    pl.close()


def test_randomized_regime_against_reference():
    """r = 12 < nAC: lambda, V and (r', k') against the numpy restatement fed the same Omega and the dense H."""
    mesh, data, inv, prior = tiny_problem(seed=19)
    pl, (pm, pd, pi, pp) = _plan(mesh, data, inv, prior)
    m = _model(inv)
    H = _dense_H(pl, pi, m)
    om = np.random.default_rng(4).standard_normal((1, 12, pl.nAC))
    lam, V, info = pl.gn_eig(6, 12, omega=om)
    rl, rV, rinfo = ger.gn_eig(H, pi.Wm, float(pp.regParam), om[0], 6)
    assert tuple(info[0]) == rinfo
    assert np.abs(lam[0] - rl).max() <= 1e-10 * rl[0]
    assert np.abs(V[0].T - rV).max() <= 1e-6 * np.abs(rV).max()
    pl.close()


def _tree_problem(ny=50, nz=87):
    from tests.test_gpu_hmc_shapes import _problem as shapes_problem
    return shapes_problem(ny, nz)


def test_rayleigh_quotients_at_a_real_tree():
    """nAC = 4000 on the multifrontal path, r = 64: v_i^T H v_j = lambda_i delta_ij through gn_hessvec, V^T beta Wm V = I.  The
    survey has 8 complex data, so H has rank <= 16 and the sketch keeps at most 16 columns."""
    from hmcmt2d_b200 import api
    mesh, data, inv, prior = _tree_problem()
    pl = api.Plan(mesh, data, inv, prior)
    assert pl.nAC == 4000 and pl.info(11) == 1
    pl.forward(m=inv.strModel, fields=False)
    lam, V, info = pl.gn_eig(8, 64, seed=3)
    rk, kk = info[0]
    assert 8 <= rk <= 16 and kk == 8, (rk, kk)
    Vk = V[0, :kk]
    HV = np.stack([pl.gn_hessvec(v)[0] for v in Vk])
    R = Vk @ HV.T
    assert np.abs(np.diag(R) - lam[0]).max() <= 1e-8 * lam[0, 0]
    assert np.abs(R - np.diag(np.diag(R))).max() <= 1e-8 * lam[0, 0]
    assert np.abs(Vk @ (prior.regParam * inv.Wm @ Vk.T) - np.eye(kk)).max() <= 1e-10
    pl.close()


def _kind2_plan(nChains=3, seed=5):
    from hmcmt2d_b200 import api
    from tests.test_gpu_hmc_shapes import _start
    mesh, data, inv, prior = _tree_problem(25, 48)
    pl = api.Plan(mesh, data, inv, prior, nChains=nChains)
    m, _, _ = _start(inv, prior, nChains, np.random.default_rng(seed), margin=3.5)
    pl.forward(m=m, fields=False)
    lam, V, info = pl.gn_eig(8, 16, seed=seed)
    assert np.all(info[:, 1] == 8)
    mass = [ger.LowRankMass(inv.Wm, float(prior.regParam), V[c].T, lam[c]) for c in range(nChains)]
    return pl, (mesh, data, inv, prior), m, mass


def test_mass_kind2_drift_and_momentum():
    """One device step with M = beta Wm + H_k: the drift is dt M^{-1} p; 2 -> 0 -> 2 switches; after run_chain the momentum is
    S clip(z) of the last draw."""
    from tests.test_gpu_hmc_shapes import NS, _chain_setup, _run
    pl, prob, m, mass = _kind2_plan()
    n = pl.nAC
    rng = np.random.default_rng(8)
    p0 = rng.standard_normal((3, n))
    x = np.stack([mass[c].inv(p0[c]) for c in range(3)])
    dt = 2.5 / np.abs(x).max()

    def step():
        pl.set_state(m, p0, m)
        pl.leapfrog_steps_device(dt, 1)
        assert pl.status() == 0
        return pl.get_state()[0]

    pl.set_mass_matrix(2)
    m1 = step()
    for c in range(3):
        got = (m1[c] - m[c]) / dt
        assert np.abs(got - x[c]).max() <= 1e-9 * np.abs(x[c]).max(), c
    pl.set_mass_matrix(0)
    m0 = step()
    assert np.abs((m0 - m) / dt - p0).max() <= 1e-12 * np.abs(p0).max()
    pl.set_mass_matrix(2)
    assert np.array_equal(step(), m1)
    st = _chain_setup(prob, 3, 31)
    _run(pl, st, 0.05, True)
    _, p = pl.get_state()
    for c in range(3):
        want = mass[c].sqrt(np.clip(st["z_mom"][NS - 1, c], -2.5, 2.5))
        assert np.abs(p[c] - want).max() <= 1e-10 * np.abs(want).max(), c
    pl.close()
    # set_mass_matrix(2) before any decomposition
    from hmcmt2d_b200 import api
    fresh = api.Plan(*prob)
    assert fresh.L.hmcmt_set_mass_matrix(fresh.h, 2) == -3
    assert fresh.L.hmcmt_set_mass_matrix(fresh.h, 3) == -3
    fresh.close()


def test_laplace_draws():
    """m_lin + M^{-1} S z for 3 chains and 4 draws; the chain state stays."""
    pl, _, m, mass = _kind2_plan()
    pl.set_state(p=np.full((3, pl.nAC), 0.25))
    z = np.random.default_rng(9).standard_normal((3, 4, pl.nAC))
    out = pl.laplace_sample(z)
    for c in range(3):
        want = mass[c].laplace(m[c][:, None], z[c].T).T
        assert np.abs(out[c] - want).max() <= 1e-10 * np.abs(want - m[c]).max(), c
    mm, pp = pl.get_state()
    assert np.array_equal(mm, m) and np.all(pp == 0.25)
    pl.close()


def test_determinism_chains_and_resident_state():
    """Repeated calls bit-identical; chain j of a 3-chain plan equals a 1-chain plan given Omega_j; m, p and every product of the
    resident fields and factors are unchanged by gn_eig and laplace_sample."""
    mesh, data, inv, prior = tiny_problem(seed=7)
    n = len(inv.strModel)
    rng = np.random.default_rng(12)
    m = inv.strModel[None, :] + 0.2 * rng.standard_normal((3, n))
    om = rng.standard_normal((3, 20, n))
    pl, _ = _plan(mesh, data, inv, prior, nChains=3)
    pl.forward(m=m, fields=False)
    pl.set_state(p=np.full((3, n), -0.5))
    dsig = rng.standard_normal((3, n))
    jv, hv = pl.jvec(dsig), pl.gn_hessvec(dsig)
    a = pl.gn_eig(10, 20, omega=om)
    b = pl.gn_eig(10, 20, omega=om)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    pl.set_mass_matrix(2)
    pl.laplace_sample(ns=2)
    mm, pp = pl.get_state()
    assert np.array_equal(mm, m) and np.all(pp == -0.5)
    assert np.array_equal(pl.jvec(dsig), jv) and np.array_equal(pl.gn_hessvec(dsig), hv)
    pl.close()
    one, _ = _plan(mesh, data, inv, prior)
    for c in range(3):
        one.forward(m=m[c], fields=False)
        s = one.gn_eig(10, 20, omega=om[c:c + 1])
        for x, y in zip(a, s):
            assert np.array_equal(x[c], y[0]), c
    one.close()


def test_argument_errors():
    from hmcmt2d_b200 import lib as _lib
    mesh, data, inv, prior = tiny_problem(seed=7)
    pl, _ = _plan(mesh, data, inv, prior)
    n = pl.nAC
    om, lam, V, info = np.zeros(n * n), np.zeros(n), np.zeros(n * n), np.zeros(2, dtype=np.int32)
    f = lambda k=4, r=8, o=True, l=True, i=True: pl.L.hmcmt_gn_eig(pl.h, k, r, _lib.f64(om) if o else None, _lib.f64(lam) if l else None,
                                                                  None, _lib.i32(info) if i else None)
    assert f() == -3                                           # no forward evaluation yet
    z = np.zeros(n)
    assert pl.L.hmcmt_laplace_sample(pl.h, 1, _lib.f64(z), _lib.f64(z)) == -3
    pl.forward(m=_model(inv), fields=False)
    om[:] = np.random.default_rng(1).standard_normal(n * n)
    assert f() == 0
    for bad in (dict(k=0), dict(k=9, r=8), dict(r=n + 1), dict(k=1, r=97), dict(o=False), dict(l=False), dict(i=False)):
        assert f(**bad) == -3, bad
    assert pl.L.hmcmt_gn_eig(None, 1, 1, _lib.f64(om), _lib.f64(lam), None, _lib.i32(info)) == -3
    assert pl.L.hmcmt_laplace_sample(pl.h, 0, _lib.f64(z), _lib.f64(z)) == -3
    assert pl.L.hmcmt_laplace_sample(pl.h, 1, None, _lib.f64(z)) == -3
    assert pl.L.hmcmt_laplace_sample(pl.h, 1, _lib.f64(z), None) == -3
    assert pl.L.hmcmt_laplace_sample(pl.h, 1, _lib.f64(z), _lib.f64(z)) == 0
    assert np.isfinite(z).all()
    pl.close()
