"""The CPU reference of the projected Gauss-Newton-CG solver (tests/gn_reference.py) pinned on the tiny problem: a full CG is
the dense Newton solve, g is the gradient of U, and the iterates stay in the box while U never increases."""
import numpy as np

from tests import gn_reference as gnr
from tests.helpers import tiny_problem


def _start(inv, seed=20):
    return inv.strModel + 0.2 * np.random.default_rng(seed).standard_normal(len(inv.strModel))


def test_full_cg_is_the_dense_solve():
    """beta = 100 keeps cond(H) near 200, so that nAC CG iterations reach the dense solve in floating point (at beta = 1,
    cond(H) ~ 1e4 and CG needs about 70)."""
    mesh, data, inv, prior = tiny_problem(seed=19)
    prior.regParam = 100.0
    prob = gnr.Problem(mesh, data, inv, prior)
    m = _start(inv)
    _, _, g = prob.evaluate(m)
    H = prob.hessian(m)
    free = np.zeros(len(m), dtype=bool)
    delta, it = gnr.cg(H, g, free, len(m), 1e-14)
    want = np.linalg.solve(H, -g)
    assert it >= 1
    assert np.abs(delta - want).max() <= 1e-10 * np.abs(want).max()


def test_gradient_matches_central_differences():
    """g against central differences of U along directions on the interior cells.  The oracle's data gradient carries the
    reference's boundary-condition approximations, which show on the tiny mesh's bottom cell row and edge columns (up to 2 % of
    max |g| there), so those cells are left out and the bound is 1e-3; the model-norm part is exact."""
    mesh, data, inv, prior = tiny_problem(seed=19)
    prob = gnr.Problem(mesh, data, inv, prior)
    m = _start(inv)
    _, _, g = prob.evaluate(m)
    ny = mesh.gridSize[0]
    interior = np.array([k * ny + j for k in range(3) for j in range(2, ny - 2)])
    rng = np.random.default_rng(3)
    h = 1e-6
    for _ in range(3):
        v = np.zeros(len(m))
        v[interior] = rng.standard_normal(len(interior))
        fd = (prob.U(m + h * v) - prob.U(m - h * v)) / (2 * h)
        assert abs(fd - g @ v) <= 1e-3 * np.abs(g[interior]).max() * np.abs(v).sum(), (fd, g @ v)
    # the model-norm part alone, on every cell
    dm = m - prob.mref
    v = rng.standard_normal(len(m))
    pm = lambda x: 0.5 * float((x - prob.mref) @ (prob.Wm @ (x - prob.mref))) * prob.beta
    fd = (pm(m + h * v) - pm(m - h * v)) / (2 * h)
    assert abs(fd - prob.beta * (prob.Wm @ dm) @ v) <= 1e-7 * abs(fd)


def test_iterates_in_bounds_and_descending():
    mesh, data, inv, prior = tiny_problem(seed=19)
    m0 = _start(inv)
    prior.sigBounds = [float(np.exp(inv.strModel.min() + 0.3)), float(np.exp(inv.strModel.max() - 0.3))]
    prob = gnr.Problem(mesh, data, inv, prior)
    m, hist, (nacc, reason), steps = gnr.gauss_newton(prob, m0, max_iter=4, max_cg=5, cg_tol=0.0)
    assert nacc >= 2 and len(steps) == nacc
    hits = 0
    for mk, act, delta, Uk, Un in steps:
        assert np.all(mk >= prob.lo) and np.all(mk <= prob.hi)
        assert Un <= Uk
        assert np.all(delta[act] == 0.0)
        hits += int(np.any((mk == prob.lo) | (mk == prob.hi)))
    assert hits >= 1                                  # the box is reached: the projection is exercised
    assert np.all(m >= prob.lo) and np.all(m <= prob.hi)
    U = hist[: nacc + 1, 0] + hist[: nacc + 1, 1]
    assert np.all(np.diff(U) <= 0.0)
