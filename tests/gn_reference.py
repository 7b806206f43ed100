"""Projected Gauss-Newton-CG in numpy, step for step as hmcmt_gauss_newton (include/hmcmt_b200.h): the CPU reference of the
device solver.  H = D Re(J^H Wd^2 J) D + beta Wm with J the oracle's explicit Jacobian (compJacMat, or its Rho_Pha / tipper
twins); U and g from the oracle's gradient path (compDataGradient) plus the model-norm term."""
import copy

import numpy as np

from oracle import forward as ofwd
from oracle import jacobian as ojac
from oracle import sampler as osamp
from tests import rho_phase_oracle as rpo
from tests import tipper_oracle as tpo

ARMIJO = 1e-4
TIE = 1e-6          # an Armijo test this close (relative) to its threshold is a test-setup error, not a comparison


class NearTie(AssertionError):
    pass


class Problem:
    """U, g and the Gauss-Newton Hessian of one oracle problem (impedance, Rho_Pha or tipper data)."""

    def __init__(self, mesh, data, inv, prior):
        self.mesh, self.data, self.prior = copy.deepcopy(mesh), data, prior
        self.inv = copy.copy(inv)
        self.lo, self.hi = np.log(prior.sigBounds[0]), np.log(prior.sigBounds[1])
        self.beta = float(prior.regParam)
        self.mref = np.array(inv.refModel, dtype=np.float64)
        self.Wm = inv.Wm.tocsr()
        rho, tip = "Rho_Pha" in data.dataType, "TZY" in data.dataComp
        self.fwd = tpo if tip else ofwd
        self.jac = rpo if rho else tpo if tip else ojac
        self.grad = rpo if rho else tpo if tip else osamp

    def evaluate(self, m):
        """(phi_d, phi_m, g) at m: the sampler's potential energy in two parts and its gradient in ln sigma."""
        self.inv.strModel = np.array(m, dtype=np.float64)
        _, phid, gd = self.grad.compDataGradient(self.mesh, self.data, self.inv, self.prior)
        dm = m - self.mref
        wdm = self.Wm @ dm
        return float(phid), 0.5 * float(dm @ wdm) * self.beta, gd + self.beta * wdm

    def U(self, m):
        phid, phim, _ = self.evaluate(m)
        return phid + phim

    def hessian(self, m):
        inv = self.inv
        self.mesh.sigma = inv.activeCell @ np.exp(m) + inv.bgModel
        _, fw = self.fwd.MT2DFwdSolver(self.mesh, self.data)
        J = self.jac.compJacMat(fw.exTE, fw.hxTM, self.mesh, self.data, inv.activeCell, fw.AinvTE, fw.AinvTM)
        D = np.exp(m)
        w2 = np.abs(np.asarray(inv.dataW)) ** 2
        H = D[:, None] * np.real(np.conj(J).T @ (w2[:, None] * J)) * D[None, :]
        return H + self.beta * self.Wm.toarray()


def active_set(m, g, lo, hi):
    return ((m <= lo) & (g > 0.0)) | ((m >= hi) & (g < 0.0))


def cg(H, g, act, max_cg, cg_tol):
    """CG from 0 on P H P delta = -P g -> (delta, iterations).  p^T q <= 0 stops it (delta = r_0 at its first iteration)."""
    r = np.where(act, 0.0, -g)
    p = r.copy()
    delta = np.zeros_like(g)
    rr = rr0 = float(r @ r)
    it = 0
    for _ in range(max_cg):
        q = np.where(act, 0.0, H @ p)
        pq = float(p @ q)
        if not pq > 0.0:
            if it == 0:
                delta = r.copy()
            break
        alpha = rr / pq
        delta = delta + alpha * p
        r = r - alpha * q
        rn = float(r @ r)
        it += 1
        if np.sqrt(rn) <= cg_tol * np.sqrt(rr0):
            break
        p = r + (rn / rr) * p
        rr = rn
    return delta, it


def gauss_newton(prob, m0, max_iter=10, max_cg=10, cg_tol=1e-2, max_ls=8, max_step=3.0, tol_rel=1e-4):
    """-> (m, history [max_iter + 1, 6], (accepted steps, stop reason), steps): the layout of hmcmt_gauss_newton; steps lists
    (m_k, active set, delta, U_k, U_{k+1}) of every accepted iteration."""
    lo, hi = prob.lo, prob.hi
    m = np.clip(np.asarray(m0, dtype=np.float64), lo, hi)
    phid, phim, g = prob.evaluate(m)
    U = phid + phim
    act = active_set(m, g, lo, hi)
    gn = np.sqrt(float(np.where(act, 0.0, g) @ np.where(act, 0.0, g)))
    hist = np.zeros((max_iter + 1, 6))
    hist[0, :3] = phid, phim, gn
    nacc, reason, steps = 0, 0, []
    if gn == 0.0:
        return m, hist, (0, 1), steps
    for _ in range(max_iter):
        delta, ncg = cg(prob.hessian(m), g, act, max_cg, cg_tol)
        mx = np.abs(delta).max()
        if mx > max_step:
            delta = delta / mx * max_step
        for t in range(max_ls):
            al = 2.0 ** -t
            mt = np.clip(m + al * delta, lo, hi)
            gtd = float(g @ (mt - m))
            pdt, pmt, gt = prob.evaluate(mt)
            thr = U + ARMIJO * gtd
            if abs((pdt + pmt) - thr) <= TIE * max(abs(pdt + pmt), abs(thr)):
                raise NearTie(f"Armijo test within {TIE} of its threshold: {pdt + pmt} vs {thr}")
            if pdt + pmt <= thr:
                break
        else:
            reason = 2
            break
        nacc += 1
        steps.append((m, act, delta, U, pdt + pmt))
        Uold = U
        m, g, phid, phim, U = mt, gt, pdt, pmt, pdt + pmt
        act = active_set(m, g, lo, hi)
        gn = np.sqrt(float(np.where(act, 0.0, g) @ np.where(act, 0.0, g)))
        hist[nacc] = phid, phim, gn, ncg, al, t + 1
        if Uold - U <= tol_rel * Uold or gn == 0.0:
            reason = 1
            break
    return m, hist, (nacc, reason), steps
