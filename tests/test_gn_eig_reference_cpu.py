"""The numpy restatement of hmcmt_gn_eig (tests/gn_eig_reference.py) on random PSD H and SPD Wm: its Jacobi against LAPACK, the exact
regime against scipy.linalg.eigh(H, beta Wm), V^T B V = I, the mass matrix kind 2 identities (S S^T = M, Woodbury = dense inverse,
M^{-1} S = S^{-T}) and a sketch wider than the rank of H."""
import numpy as np
import pytest
import scipy.linalg as sla

from tests import gn_eig_reference as ger


def _spd(n, rng):
    """A banded SPD matrix shaped like Wm: a 2-D Laplacian-like stencil plus a small diagonal shift."""
    ny = max(2, int(np.sqrt(n)))
    W = np.zeros((n, n))
    for i in range(n):
        W[i, i] = 4.0 + 0.1 + rng.uniform(0.0, 0.5)
        for j in (i + 1, i + ny):
            if j < n:
                W[i, j] = W[j, i] = -1.0 + rng.uniform(-0.2, 0.2)
    return W


def _psd(n, rank, rng, decay=0.7):
    X = rng.standard_normal((n, rank)) * decay ** np.arange(rank)[None, :]
    return X @ X.T * 50.0


@pytest.mark.parametrize("r", [1, 2, 7, 16, 33, 96])
def test_jacobi_matches_lapack(r):
    rng = np.random.default_rng(r)
    G = rng.standard_normal((r, r))
    G = G @ G.T + np.diag(rng.uniform(0.0, 1.0, r))
    lam, U = ger.jacobi_eig(G)
    want = np.linalg.eigvalsh(G)[::-1]
    assert np.all(np.diff(lam) <= 0.0)
    assert np.abs(lam - want).max() <= 1e-13 * np.abs(want).max()
    assert np.abs(U.T @ U - np.eye(r)).max() <= 1e-13
    assert np.abs(G @ U - U * lam[None, :]).max() <= 1e-12 * np.abs(want).max()
    at = np.argmax(np.abs(U), axis=0)
    assert np.all(U[at, np.arange(r)] > 0.0)


@pytest.mark.parametrize("n,rank,beta", [(40, 20, 1.0), (40, 12, 0.3), (64, 30, 10.0)])
def test_exact_regime_against_eigh(n, rank, beta):
    """r = n: the k' pairs kept are the top k' of eigh(H, beta Wm) to 1e-10 lambda_max, V^T B V = I, H V = B V diag(lambda)."""
    rng = np.random.default_rng(n + rank)
    Wm, H = _spd(n, rng), _psd(n, rank, rng, decay=0.97)
    B = beta * Wm
    k = n
    lam, V, (rk, kk) = ger.gn_eig(H, Wm, beta, rng.standard_normal((n, n)), k)
    want = sla.eigh(H, B, eigvals_only=True)[::-1]
    lmax = want[0]
    assert kk >= np.count_nonzero(want > 1e-5 * lmax) and rk >= kk
    assert np.abs(lam[:kk] - want[:kk]).max() <= 1e-10 * lmax
    assert np.all(lam[kk:] == 0.0) and np.all(V[:, kk:] == 0.0)
    Vk = V[:, :kk]
    assert np.abs(Vk.T @ B @ Vk - np.eye(kk)).max() <= 1e-10
    big = lam[:kk] > 1e-3 * lmax
    assert np.abs(H @ Vk[:, big] - B @ Vk[:, big] * lam[:kk][big]).max() <= 1e-9 * lmax * np.abs(B @ Vk[:, big]).max()


def test_steep_spectrum_cut():
    """A spectrum over 15 decades: the 1e-12 cut on G = Y^T B Y (whose eigenvalues go as lambda^2) drops the directions below
    about 1e-6 lambda_max, never one above 1e-5 lambda_max, and the pairs kept stay accurate."""
    rng = np.random.default_rng(8)
    n, beta = 40, 1.0
    Wm, H = _spd(n, rng), _psd(n, n, rng, decay=0.7)
    lam, V, (rk, kk) = ger.gn_eig(H, Wm, beta, rng.standard_normal((n, n)), n)
    want = sla.eigh(H, beta * Wm, eigvals_only=True)[::-1]
    assert np.count_nonzero(want > 1e-5 * want[0]) <= kk < n
    assert np.abs(lam[:kk] - want[:kk]).max() <= 1e-6 * want[0]
    assert np.abs(V[:, :kk].T @ (beta * Wm) @ V[:, :kk] - np.eye(kk)).max() <= 1e-10


def test_randomized_regime_captures_the_top_pairs():
    """r < n on a decaying spectrum: the leading pairs to a small relative error."""
    rng = np.random.default_rng(3)
    n, beta = 120, 2.0
    Wm, H = _spd(n, rng), _psd(n, 60, rng, decay=0.8)
    lam, V, (rk, kk) = ger.gn_eig(H, Wm, beta, rng.standard_normal((20, n)), 8)
    want = sla.eigh(H, beta * Wm, eigvals_only=True)[::-1]
    assert rk == 20 and kk == 8
    assert np.abs(lam - want[:8]).max() <= 1e-4 * want[0]


def test_sketch_wider_than_rank():
    """rank(H) = 5 < r = 20: r' = 5, k' <= 5, and nothing fails."""
    rng = np.random.default_rng(11)
    n = 50
    Wm, H = _spd(n, rng), _psd(n, 5, rng, decay=1.0)
    lam, V, (rk, kk) = ger.gn_eig(H, Wm, 1.5, rng.standard_normal((20, n)), 10)
    assert rk == 5 and kk == 5
    want = sla.eigh(H, 1.5 * Wm, eigvals_only=True)[::-1]
    assert np.abs(lam[:5] - want[:5]).max() <= 1e-10 * want[0]
    assert np.all(lam[5:] == 0.0) and np.all(V[:, 5:] == 0.0)


def test_zero_hessian_keeps_nothing():
    rng = np.random.default_rng(2)
    n = 30
    lam, V, (rk, kk) = ger.gn_eig(np.zeros((n, n)), _spd(n, rng), 1.0, rng.standard_normal((6, n)), 3)
    assert (rk, kk) == (0, 0) and np.all(lam == 0.0) and np.all(V == 0.0)


@pytest.mark.parametrize("beta", [0.5, 4.0])
def test_mass_matrix_identities(beta):
    """S S^T = M, the Woodbury M^{-1} = dense inverse, M^{-1} S = S^{-T}, Laplace draws m_lin + S^{-T} z."""
    rng = np.random.default_rng(int(beta * 10))
    n = 48
    Wm, H = _spd(n, rng), _psd(n, 20, rng, decay=0.9)
    lam, V, (_, kk) = ger.gn_eig(H, Wm, beta, rng.standard_normal((16, n)), 10)
    assert kk == 10
    mm = ger.LowRankMass(Wm, beta, V, lam)
    M = mm.dense()
    S = mm.S()
    sc = np.abs(M).max()
    assert np.abs(S @ S.T - M).max() <= 1e-12 * sc
    P = rng.standard_normal((n, 5))
    Minv = np.linalg.inv(M)
    assert np.abs(mm.inv(P) - Minv @ P).max() <= 1e-10 * np.abs(Minv @ P).max()
    assert np.abs(mm.inv(S) - np.linalg.inv(S).T).max() <= 1e-10 * np.abs(np.linalg.inv(S)).max()
    z = rng.standard_normal((n, 3))
    assert np.abs(mm.sqrt(z) - S @ z).max() <= 1e-12 * np.abs(S @ z).max()
    m_lin = rng.standard_normal(n)
    draw = mm.laplace(m_lin[:, None], z)
    assert np.abs(draw - (m_lin[:, None] + np.linalg.solve(S.T, z))).max() <= 1e-10 * np.abs(draw - m_lin[:, None]).max()
    # with H_k = B V Lambda V^T B the mass matrix is the generalized eigendecomposition's low-rank part plus the prior
    Hk = (beta * Wm @ V) @ np.diag(lam) @ (beta * Wm @ V).T
    assert np.abs(M - beta * Wm - Hk).max() <= 1e-12 * sc
