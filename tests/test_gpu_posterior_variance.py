"""Prior and Laplace posterior variances and the resolution diagonal of a plan (Plan.posterior_variance /
hmcmt_posterior_variance), diag(Wm^-1) from a selected inversion of the plan's resident Wm factor, and the model files of
api.getLaplacePosteriorModel.
  * Exact regime (tiny problem, k = r = nAC) for impedance, rho / phase and tipper plans on both solvers, H from the plan's own
    jacobian(): prior_var against diag(inv(beta Wm)); post_var and resolution against the dense Woodbury formulas from the
    (lambda, V) gn_eig returned (1e-10); and against the full answers diag(inv(H + beta Wm)) and diag(inv(H + beta Wm) H), within
    a bound computed from E = H - H_k (H_k = beta Wm V Lambda V^T beta Wm, what gn_eig delivers): with M = beta Wm + H_k and
    Mf = beta Wm + H, Mf^-1 - M^-1 = -M^-1 E Mf^-1, so |d_i| <= |M^-1 e_i| |E|_2 |Mf^-1 e_i| for post_var, and
    Mf^-1 H - M^-1 H_k = Mf^-1 E - M^-1 E Mf^-1 H_k for the resolution.  |E|_2 / lambda_max is printed: the accuracy of the
    decomposition near gn_eig's cut, which is what limits post_var as delivered.
  * The multifrontal tree of Wm (nAC = 4 000, gathers and global fronts): prior_var against a dense inverse of beta Wm,
    post_var / resolution against the dense Woodbury formulas from gn_eig's (lambda, V).
  * A cfg2-size active grid (nAC = 18 600, two frequencies): prior_var on 64 fixed-seed cells against splu solves.
  * The sample variance of 4 000 laplace_sample draws lies within a 5 sigma chi^2 band of post_var on every cell.
  * 3 chains equal three 1-chain plans bit for bit; the chain state and a following leapfrog_steps_device step (mass kind 2)
    are bit-identical with and without the call; repeated calls are bit-identical.
  * Argument errors: beta <= 0, all outputs NULL, post_var / resolution without a decomposition.
  * getLaplacePosteriorModel's files read back (the repository's model reader) to the returned values."""
import os

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

from tests.helpers import tiny_problem
from tests.test_gpu_gn_eig import _dense_H
from tests.test_gpu_jvec import _model, _plan, _problem

pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps


def _rel(a, b):
    return np.abs(a - b).max() / np.abs(b).max()


def _woodbury(Binv_diag, B, V, lam):
    """diag(M^-1) = diag(B^-1) - sum_j d_j V_ij^2 and diag(V D V^T B) from (lam, V [k, n])"""
    d = lam / (1 + lam)
    return Binv_diag - np.einsum("ji,j->i", V ** 2, d), np.einsum("ji,j,ji->i", V, d, V @ B)


@pytest.mark.parametrize("solver", ["band", "mf"])
@pytest.mark.parametrize("kind", ["impedance", "rho_phase", "tipper"])
def test_exact_regime_against_dense(kind, solver, monkeypatch):
    monkeypatch.setenv("HMCMT_SOLVER", solver)
    mesh, data, inv, prior, _ = _problem(kind)
    pl, (pm, pd, pi, pp) = _plan(mesh, data, inv, prior)
    n, beta = pl.nAC, float(pp.regParam)
    m = _model(inv)
    H = _dense_H(pl, pi, m)
    B = beta * pi.Wm.toarray()
    lam, V, info = pl.gn_eig(n, r=n, seed=1)
    kk = int(info[0][1])
    pv, qv, rv = pl.posterior_variance()
    Binv = np.linalg.inv(B)
    assert _rel(pv, np.diag(Binv)) <= 1e-10
    Vk, lk = V[0, :kk].T, lam[0, :kk]
    BV = B @ Vk
    Hk = BV @ np.diag(lk) @ BV.T
    Minv = np.linalg.inv(B + Hk)
    assert _rel(qv[0], np.diag(Minv)) <= 1e-10, _rel(qv[0], np.diag(Minv))
    want_r = np.einsum("ij,j,ij->i", Vk, lk / (1 + lk), BV)
    assert _rel(rv[0], want_r) <= 1e-10, _rel(rv[0], want_r)
    # the full answers, within the bound from E = H - H_k
    E = H - Hk
    e2 = np.linalg.norm(E, 2)
    Mf = np.linalg.inv(B + H)
    full_q, full_r = np.diag(Mf), np.diag(Mf @ H)
    nM, nMf = np.linalg.norm(Minv, axis=0), np.linalg.norm(Mf, axis=0)
    bound_q = nM * e2 * nMf + 1e-10 * np.abs(full_q).max()
    bound_r = nMf * e2 + nM * e2 * np.linalg.norm(Mf @ Hk, axis=0) + 1e-10 * np.abs(full_r).max()
    err_q, err_r = np.abs(qv[0] - full_q), np.abs(rv[0] - full_r)
    print(f"\n[posterior variance] {kind} {solver}: k' {kk}  |H - H_k|_2 / lambda_max {e2 / lk[0]:.2e}  "
          f"post_var max rel error {err_q.max() / np.abs(full_q).max():.2e} (bound use {(err_q / bound_q).max():.2f})  "
          f"resolution max error {err_r.max():.2e} (bound use {(err_r / bound_r).max():.2f})")
    assert np.all(err_q <= bound_q) and np.all(err_r <= bound_r)
    pl.close()


def test_multifrontal_tree_of_wm():
    """nAC = 4 000 (50 x 87 cells): Wm's multifrontal tree has several levels, gathers and global fronts"""
    from hmcmt2d_b200 import api
    from tests.test_gpu_gn_eig import _tree_problem
    mesh, data, inv, prior = _tree_problem()
    pl = api.Plan(mesh, data, inv, prior)
    assert pl.nAC == 4000
    pl.forward(m=inv.strModel, fields=False)
    lam, V, info = pl.gn_eig(8, 64, seed=3)
    kk = int(info[0][1])
    pv, qv, rv = pl.posterior_variance()
    B = float(prior.regParam) * inv.Wm.toarray()
    kappa = np.linalg.cond(B)
    Binv = np.linalg.inv(B)
    tol = max(1e-10, 100 * EPS * kappa)
    assert _rel(pv, np.diag(Binv)) <= tol, (_rel(pv, np.diag(Binv)), kappa)
    want_q, want_r = _woodbury(np.diag(Binv), B, V[0, :kk], lam[0, :kk])
    assert _rel(qv[0], want_q) <= tol, _rel(qv[0], want_q)
    assert _rel(rv[0], want_r) <= tol, _rel(rv[0], want_r)
    print(f"\n[posterior variance] nAC 4000: kappa(beta Wm) {kappa:.2e}  prior {_rel(pv, np.diag(Binv)):.1e}  "
          f"post {_rel(qv[0], want_q):.1e}  resolution {_rel(rv[0], want_r):.1e}")
    pl.close()


def test_prior_variance_at_cfg2_size():
    from hmcmt2d_b200 import api, synthetic
    mesh, data, inv, prior = synthetic.make_problem(200, 100, 2)
    pl = api.Plan(mesh, data, inv, prior)
    n = pl.nAC
    assert n == 18600
    pv, _, _ = pl.posterior_variance(prior=True, posterior=False, resolution=False)
    B = sp.csc_matrix(float(prior.regParam) * inv.Wm)
    lu = spla.splu(B)
    idx = np.sort(np.random.default_rng(6).choice(n, 64, replace=False))
    E = np.zeros((n, len(idx)))
    E[idx, np.arange(len(idx))] = 1.0
    ref = lu.solve(E)[idx, np.arange(len(idx))]
    inv_op = spla.LinearOperator((n, n), matvec=lambda v: lu.solve(np.asarray(v).ravel()),
                                 rmatvec=lambda v: lu.solve(np.asarray(v).ravel(), trans="T"), dtype=np.float64)
    kappa = spla.onenormest(B) * spla.onenormest(inv_op)
    assert _rel(pv[idx], ref) <= max(1e-10, 100 * EPS * kappa), (_rel(pv[idx], ref), kappa)
    pl.close()


def test_laplace_draws_match_post_var():
    """4 000 draws: sum_s (x_s - m_lin)^2 / (N post_var) ~ chi^2_N / N, mean 1, standard deviation sqrt(2 / N)"""
    from tests.test_gpu_gn_eig import _kind2_plan
    pl, _, m, _ = _kind2_plan(nChains=1)
    _, qv, _ = pl.posterior_variance(prior=False, posterior=True, resolution=False)
    N = 4000
    x = pl.laplace_sample(ns=N, seed=17)[0]
    ratio = ((x - m[0]) ** 2).mean(axis=0) / qv[0]
    assert np.all(np.abs(ratio - 1) <= 5 * np.sqrt(2.0 / N)), np.abs(ratio - 1).max()
    pl.close()


def test_chains_equal_single_chain_plans():
    mesh, data, inv, prior = tiny_problem(seed=7)
    n = len(inv.strModel)
    rng = np.random.default_rng(12)
    m = inv.strModel[None, :] + 0.2 * rng.standard_normal((3, n))
    om = rng.standard_normal((3, 20, n))
    pl, _ = _plan(mesh, data, inv, prior, nChains=3)
    pl.forward(m=m, fields=False)
    pl.gn_eig(10, 20, omega=om)
    a = pl.posterior_variance()
    pl.close()
    one, _ = _plan(mesh, data, inv, prior)
    for c in range(3):
        one.forward(m=m[c], fields=False)
        one.gn_eig(10, 20, omega=om[c:c + 1])
        s = one.posterior_variance()
        assert np.array_equal(a[0], s[0])
        assert np.array_equal(a[1][c], s[1][0]) and np.array_equal(a[2][c], s[2][0]), c
    one.close()


def test_resident_state_step_and_repeats(monkeypatch):
    """the chain state, the mass kind and a following leapfrog_steps_device step are the same with and without the call"""
    monkeypatch.setenv("HMCMT_SOLVER", "mf")
    mesh, data, inv, prior, _ = _problem("impedance")
    m = _model(inv)
    p0 = np.random.default_rng(3).standard_normal(len(m))
    res = []
    for call in (False, True):
        pl, _ = _plan(mesh, data, inv, prior)
        pl.forward(m=m, fields=False)
        pl.gn_eig(8, r=16, seed=2)
        pl.set_mass_matrix(2)
        pl.set_state(m, p0, m)
        s0 = pl.get_state()
        if call:
            a, b = pl.posterior_variance(), pl.posterior_variance()
            for x, y in zip(a, b):
                assert np.array_equal(x, y)
            for x, y in zip(s0, pl.get_state()):
                assert np.array_equal(x, y)
        pl.leapfrog_steps_device(1e-3, 1)
        assert pl.status() == 0
        res.append(pl.get_state())
        pl.close()
    for x, y in zip(*res):
        assert np.array_equal(x, y)


def test_argument_errors(monkeypatch):
    from hmcmt2d_b200 import api, lib
    monkeypatch.setenv("HMCMT_SOLVER", "mf")
    mesh, data, inv, prior, _ = _problem("impedance")
    pl, (pm, pd, pi, pp) = _plan(mesh, data, inv, prior)
    pl.forward(m=_model(inv), fields=False)
    pl.posterior_variance(posterior=False, resolution=False)         # the prior needs no decomposition
    for post, res in ((True, False), (False, True)):
        with pytest.raises(lib.HmcmtError) as e:
            pl.posterior_variance(prior=False, posterior=post, resolution=res)
        assert e.value.code == -3
    with pytest.raises(lib.HmcmtError) as e:
        pl.posterior_variance(False, False, False)
    assert e.value.code == -3
    assert pl.L.hmcmt_posterior_variance(None, lib.f64(np.zeros(pl.nAC)), None, None) == -3
    pl.close()
    for beta in (0.0, -1.0):
        pp.regParam = beta
        zb = api.Plan(pm, pd, pi, pp)
        with pytest.raises(lib.HmcmtError) as e:
            zb.posterior_variance(posterior=False, resolution=False)
        assert e.value.code == -3
        zb.close()


def test_laplace_model_files_read_back(tmp_path):
    from hmcmt2d_b200 import api
    from hmcmt2d_b200.fileio import readEMModel2D
    mesh, data, inv, prior, _ = _problem("impedance")
    pl, (pm, pd, pi, pp) = _plan(mesh, data, inv, prior)
    m = _model(inv)
    pl.forward(m=m, fields=False)
    pl.gn_eig(8, r=16, seed=2)
    mean, std = api.getLaplacePosteriorModel(pl, m, pm, pi, str(tmp_path))
    _, qv, _ = pl.posterior_variance(prior=False, posterior=True, resolution=False)
    assert np.array_equal(mean, m) and np.array_equal(std, np.sqrt(qv[0]))
    off = len(pm.yLen) * len(pm.airLayer)                      # the files hold the earth cells (air rows are not written)
    for name, want in (("laplaceMeanModel.model", np.exp(m)), ("laplaceStdModel.model", std)):
        f = readEMModel2D(os.path.join(str(tmp_path), name))
        full = (pi.activeCell @ want + pi.bgModel)[off:]
        got = np.asarray(f.sigma)[off:]
        assert got.shape == full.shape
        assert np.all(np.abs(got - full) <= 5.01e-3 * np.abs(full)), name       # the files carry three digits (%4.2e)
    pl.close()
