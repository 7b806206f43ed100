"""The randomized generalized eigensolver of hmcmt_gn_eig and the mass matrix kind 2 / Laplace draws built on it, in numpy, step for
step (include/hmcmt_b200.h, DESIGN.md 4.9), for one chain given dense H, Wm, beta and Omega: the CPU reference of the device code.
The small eigendecompositions restate k_jacobi_eig (cyclic Jacobi in the round-robin order, the same stop test, sort and signs)."""
import numpy as np
import scipy.linalg as sla

SWEEPS = 30          # kJacobiSweeps
TOL = 1e-14          # kJacobiTol: stop when |offdiag(A)|_F <= TOL |A|_F
KEEP = 1e-12         # B-orthonormalisation keeps sigma_i > KEEP sigma_max


def _sign(U):
    """Each column with its largest-magnitude entry (lowest index on ties) positive."""
    U = np.array(U, dtype=np.float64)
    if U.shape[0] == 0:
        return U
    at = np.argmax(np.abs(U), axis=0)                    # the first maximum: lowest index on ties
    s = np.where(U[at, np.arange(U.shape[1])] < 0.0, -1.0, 1.0)
    return U * s[None, :]


def jacobi_eig(G):
    """k_jacobi_eig: A = (G + G^T) / 2 = U diag(lam) U^T, lam descending (ties by index), U's columns signed by _sign."""
    A = 0.5 * (np.asarray(G, dtype=np.float64) + np.asarray(G, dtype=np.float64).T)
    r = A.shape[0]
    m = r + (r & 1)
    V = np.eye(r)
    tol2 = TOL * TOL * np.sum(A * A)
    for _ in range(SWEEPS):
        off2 = np.sum((A - np.diag(np.diag(A))) ** 2)
        if not off2 > tol2:
            break
        for rd in range(m - 1):
            P, Q, C, S = [], [], [], []
            for k in range(m // 2):
                a = m - 1 if k == 0 else (rd + k) % (m - 1)
                b = rd if k == 0 else (rd - k + m - 1) % (m - 1)
                p, q = min(a, b), max(a, b)
                if q >= r or A[p, q] == 0.0:
                    continue
                tau = (A[q, q] - A[p, p]) / (2.0 * A[p, q])
                t = (1.0 if tau >= 0.0 else -1.0) / (abs(tau) + np.hypot(1.0, tau))
                c = 1.0 / np.sqrt(1.0 + t * t)
                P.append(p), Q.append(q), C.append(c), S.append(t * c)
            if not P:
                continue
            P, Q, C, S = np.array(P), np.array(Q), np.array(C), np.array(S)
            ap, aq, vp, vq = A[:, P].copy(), A[:, Q].copy(), V[:, P].copy(), V[:, Q].copy()
            A[:, P], A[:, Q] = C * ap - S * aq, S * ap + C * aq
            V[:, P], V[:, Q] = C * vp - S * vq, S * vp + C * vq
            ap, aq = A[P, :].copy(), A[Q, :].copy()
            A[P, :], A[Q, :] = C[:, None] * ap - S[:, None] * aq, S[:, None] * ap + C[:, None] * aq
            A[P, Q] = 0.0
            A[Q, P] = 0.0
    d = np.diag(A).copy()
    order = np.argsort(-d, kind="stable")
    return d[order], _sign(V[:, order])


def _leading(x, n, test):
    k = 0
    while k < n and test(x[k]):
        k += 1
    return k


def gn_eig(H, Wm, beta, Omega, k):
    """One chain of hmcmt_gn_eig.  H [n, n] (PSD), Wm [n, n] (SPD, dense or sparse), Omega [r, n].
    -> (lam [k], V [n, k], (r', k')), zero beyond k'."""
    Wm = Wm.toarray() if hasattr(Wm, "toarray") else np.asarray(Wm, dtype=np.float64)
    Omega = np.asarray(Omega, dtype=np.float64)
    r, n = Omega.shape
    B = beta * Wm
    # (1)-(2) Y = B^{-1} H Omega: one product and one Wm solve per column, divided by beta
    Y = sla.cho_solve(sla.cho_factor(Wm, lower=True), H @ Omega.T) / beta
    # (3) B-orthonormalise twice; the columns past r' are zero
    for _ in range(2):
        sig, P = jacobi_eig(Y.T @ (B @ Y))
        rk = _leading(sig, r, lambda s: s > KEEP * sig[0])
        C = np.zeros((r, r))
        C[:, :rk] = P[:, :rk] / np.sqrt(sig[:rk])
        Y = Y @ C
    # (4) T = Q^T H Q; (5) the k' leading pairs with lambda > 0, V = Q U, signs
    lamT, U = jacobi_eig(Y.T @ (H @ Y))
    kk = _leading(lamT, min(k, rk), lambda x: x > 0.0)
    C = np.zeros((r, k))
    C[:, :kk] = U[:, :kk]
    V = _sign(Y @ C)
    lam = np.zeros(k)
    lam[:kk] = lamT[:kk]
    return lam, V, (rk, kk)


class LowRankMass:
    """M = beta Wm + B V diag(lam) V^T B (mass matrix kind 2) from the decomposition of gn_eig."""

    def __init__(self, Wm, beta, V, lam):
        self.Wm = Wm.toarray() if hasattr(Wm, "toarray") else np.asarray(Wm, dtype=np.float64)
        self.beta, self.V, self.lam = float(beta), np.asarray(V), np.asarray(lam)
        self.L = np.linalg.cholesky(self.Wm)
        self.W = np.sqrt(self.beta) * self.L.T @ self.V
        self.d = self.lam / (1.0 + self.lam)
        self.a = self.lam / (1.0 + np.sqrt(1.0 + self.lam))        # sqrt(1 + lambda) - 1 without cancellation

    def dense(self):
        BV = self.beta * self.Wm @ self.V
        return self.beta * self.Wm + BV @ np.diag(self.lam) @ BV.T

    def inv(self, p):
        """M^{-1} p = Wm^{-1} p / beta - V (d .* V^T p)."""
        d = self.d if np.ndim(p) == 1 else self.d[:, None]
        return np.linalg.solve(self.Wm, p) / self.beta - self.V @ (d * (self.V.T @ p))

    def sqrt(self, z):
        """S z = sqrt(beta) L (z + W (a .* W^T z)), S S^T = M."""
        a = self.a if np.ndim(z) == 1 else self.a[:, None]
        return np.sqrt(self.beta) * self.L @ (z + self.W @ (a * (self.W.T @ z)))

    def S(self):
        return np.sqrt(self.beta) * self.L @ (np.eye(len(self.L)) + self.W @ np.diag(self.a) @ self.W.T)

    def laplace(self, m_lin, z):
        """m_lin + M^{-1} S z: a draw of N(m_lin, M^{-1})."""
        return m_lin + self.inv(self.sqrt(z))
