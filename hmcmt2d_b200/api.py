"""Host-side mirror of the reference's solver / sampler interface for the hot path, above the C ABI.

Same names, argument meaning and error behaviour as the Julia functions they replace:

    readstartupFile            HMCSampler/readstartupFile.jl:4-103
    setupInverseDataModel      HMCStruct/HMCStruct.jl:99-125
    MT2DFwdSolver              MTFwdSolver/MT2DFwdSolver.jl:74-216
    compJacTMatVec             MTSensitivity/compJacTMatVec.jl:8-329
    compDataGradient           HMCSampler/HMCSampler.jl:277-330
    proposeLeapfrog            HMCSampler/HMCSampler.jl:206-269
    getHamiltonian             HMCSampler/HMCSampler.jl:358-397
    runHMCSampler              HMCSampler/HMCSampler.jl:72-196
    parallelHMCSampler         HMCSampler/parallelHMC.jl:10-49
    outputHMCSamples           HMCSampler/HMCSampler.jl:785-828
    getPosteriorModel          HMCSampler/HMCSampler.jl:605-642

Everything numerical runs in libhmcmt_b200.so on the GPU; this module only marshals arrays.  There is
no CPU path: without the library (or without a CUDA device) every call raises.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass, field
from typing import List, Optional

import numpy as np
import scipy.sparse as sp

from . import lib as _lib
from .fileio import (HMCPrior, MTData, TensorMesh2D, parseStartup, readEMModel2D, readMT2DData, writeEMModel2D)

MU0 = 4 * np.pi * 1e-7


@dataclass
class InvDataModel:
    """Mirror of `InvDataModel` (HMCStruct.jl:75-91).  activeCell is the selector matrix (nCell x nAC);
    dataW holds the diagonal of Wd."""
    obsData: np.ndarray
    dataW: np.ndarray
    strModel: np.ndarray
    refModel: np.ndarray
    activeCell: sp.csr_matrix
    bgModel: np.ndarray
    Wm: sp.csr_matrix
    dataErr: np.ndarray = None


@dataclass
class HMCParameter:
    """Mirror of `HMCParameter` (HMCStruct.jl:42-52) for the identity mass matrix."""
    nparam: int
    rhomodel: np.ndarray
    momentum: np.ndarray


@dataclass
class HMCStatus:
    """Mirror of `HMCStatus` (HMCStruct.jl:60-70)."""
    nAccept: int
    nReject: int
    acceptstats: np.ndarray
    hmstats: np.ndarray          # 4 x (nsamples+1): dataMisfit, mnorm, ke, he


@dataclass
class MT2DFwdData:
    """Mirror of `MT2DFwdData` (MT2DFwdSolver.jl:44-53): fields are nNode x nFreq; the factor
    handles AinvTE/AinvTM are the device-resident plan that owns the factors."""
    exTE: np.ndarray
    hxTM: np.ndarray
    AinvTE: object
    AinvTM: object
    linearSolver: str = "b200"
    generation: int = -1        # evaluation counter of the plan when these fields / factors were produced


def setActiveElement(sigma, sigFix, fixIndex=None):
    """`setActiveElement` (HMCUtility.jl:217-258)."""
    sigma = np.asarray(sigma, dtype=np.float64)
    frozen = np.zeros(len(sigma), dtype=bool)
    bg = np.zeros(len(sigma))
    for s in sigFix:
        hit = sigma == s                      # exact compare, as the reference
        bg[hit] += s
        frozen |= hit
    if fixIndex is not None and len(fixIndex):
        frozen[fixIndex] = True
        bg[fixIndex] = sigma[fixIndex]
    act = np.nonzero(~frozen)[0]
    P = sp.csr_matrix((np.ones(len(act)), (act, np.arange(len(act)))), shape=(len(sigma), len(act)))
    return P, bg


def _cell_gradient(ny, nz):
    """`getCellGradient2D` (MT2DOperators.jl:52-63): unscaled +-1 differences."""
    def d(n):
        return sp.diags([-np.ones(n), np.ones(n)], [0, 1], shape=(n, n + 1))
    return sp.vstack([sp.kron(sp.identity(nz), d(ny - 1)), sp.kron(d(nz - 1), sp.identity(ny))], format="csr")


def setupInverseDataModel(mtMesh: TensorMesh2D, sigFix, sigLB, sigUB, obsData, dataErr, fixIndex=None) -> InvDataModel:
    """`setupInverseDataModel` (HMCStruct.jl:99-125)."""
    P, bg = setActiveElement(mtMesh.sigma, sigFix, fixIndex)
    dataW = 1.0 / np.abs(np.asarray(dataErr, dtype=np.float64))       # compDataWeightMat HMCUtility.jl:168-190
    m0 = np.log(P.T @ np.asarray(mtMesh.sigma))
    G = _cell_gradient(*mtMesh.gridSize) @ P
    Wm = (G.T @ G).tocsr()
    Wm.sort_indices()
    return InvDataModel(np.asarray(obsData), dataW, m0, m0.copy(), P, bg, Wm, np.asarray(dataErr, dtype=np.float64))


def readstartupFile(startupfile: str):
    """`readstartupFile` (readstartupFile.jl:4-103) -> (mtMesh, mtData, invParam, hmcprior)."""
    if not os.path.isfile(startupfile):
        raise FileNotFoundError(f"{startupfile} does not exist, please try again.")
    base = os.path.dirname(os.path.abspath(startupfile))
    datafile, modelfile, sigmin, sigmax, sigfix, prior = parseStartup(startupfile)
    mtData, obs, err = readMT2DData(os.path.join(base, datafile))
    mtMesh = readEMModel2D(os.path.join(base, modelfile))
    invParam = setupInverseDataModel(mtMesh, sigfix, sigmin, sigmax, obs, err)
    return mtMesh, mtData, invParam, prior


# ---------------------------------------------------------------------------------------------------
# plan management


# DataComp of "Rho_Pha" surveys, in the row order of MT2DFwdSolver.jl:191-205, and the modes they select
_RHO_PHA_COMPS = {("RhoXY", "PhsXY"): [0], ("RhoYX", "PhsYX"): [1], ("RhoXY", "PhsXY", "RhoYX", "PhsYX"): [0, 1]}
# DataComp entries of "Impedance" surveys and their hmcmt_problem.compMode: the impedances (MT2DFwdSolver.jl:183-187) and the TE
# tipper TZY = Hz/Hy (include/hmcmt_b200.h), any of them in this order
_IMPEDANCE_COMPS = {"ZXY": 0, "ZYX": 1, "TZY": 2}


def _comp_mode(comp: str) -> int:
    """System a DataComp entry is computed in: 0 TE (ZXY, TZY, RhoXY, PhsXY), 1 TM (ZYX, RhoYX, PhsYX)."""
    return 0 if ("XY" in comp or comp == "TZY") else 1


class Plan:
    """Owns one `hmcmt_plan` (device-resident problem: mesh, survey, weights, factors, chain state).
    DataType "Impedance": packed data arrays are complex; DataComp is ZXY, ZYX and the tipper TZY, or any of them in that order.  DataType "Rho_Pha": one real apparent resistivity or phase per row
    (dtID = 2 mode + 1 / 2), and every packed data array (predictions, J^T v input, Jacobian rows, chain samples) is real."""

    def __init__(self, mtMesh: TensorMesh2D, mtData: MTData, invParam: InvDataModel, hmcprior: HMCPrior,
                 nChains: int = 1, device: int = 0):
        self.rho_phase = "Rho_Pha" in mtData.dataType
        if not self.rho_phase and "Impedance" not in mtData.dataType:
            raise NotImplementedError(f"DataType {mtData.dataType}")
        self.L = _lib.load()
        self.generation = 0
        ny, nz = mtMesh.gridSize
        self.ny, self.nz = int(ny), int(nz)
        self.nChains = int(nChains)
        self.dtype = np.float64 if self.rho_phase else np.complex128
        if self.rho_phase:
            comp_mode = _RHO_PHA_COMPS.get(tuple(mtData.dataComp))
            if comp_mode is None:
                raise ValueError("DataComp must be [RhoXY, PhsXY, RhoYX, PhsYX] in that order, or the two of one mode "
                                 "(MT2DFwdSolver.jl:191-205)")
        else:
            comp_mode = []
            for c in mtData.dataComp:
                if c not in _IMPEDANCE_COMPS:
                    raise NotImplementedError(f"data component {c}")
                comp_mode.append(_IMPEDANCE_COMPS[c])
            if comp_mode != sorted(set(comp_mode)):
                raise ValueError("DataComp must be [ZXY, ZYX, TZY] or a part of it, in that order (MT2DFwdSolver.jl:183-187)")
        act = np.asarray(invParam.activeCell.tocsc().indices, dtype=np.int32)      # one row index per column
        Wm = invParam.Wm.tocsr()
        Wm.sort_indices()
        self._keep = dict(
            yLen=np.ascontiguousarray(mtMesh.yLen, dtype=np.float64), zLen=np.ascontiguousarray(mtMesh.zLen, dtype=np.float64),
            freqs=np.ascontiguousarray(mtData.freqs, dtype=np.float64), rx=np.ascontiguousarray(mtData.rxLoc, dtype=np.float64),
            comp=np.asarray(comp_mode, dtype=np.int32), fid=np.ascontiguousarray(mtData.freqID, dtype=np.int64),
            rid=np.ascontiguousarray(mtData.rxID, dtype=np.int64), did=np.ascontiguousarray(mtData.dtID, dtype=np.int64),
            obs=np.ascontiguousarray(invParam.obsData, dtype=self.dtype),
            err=np.ascontiguousarray(1.0 / invParam.dataW, dtype=np.float64), act=act,
            bg=np.ascontiguousarray(invParam.bgModel, dtype=np.float64),
            wp=np.ascontiguousarray(Wm.indptr, dtype=np.int32), wi=np.ascontiguousarray(Wm.indices, dtype=np.int32),
            wv=np.ascontiguousarray(Wm.data, dtype=np.float64))
        k = self._keep
        pr = _lib.Problem()
        pr.ny, pr.nz = self.ny, self.nz
        pr.yLen, pr.zLen = _lib.f64(k["yLen"]), _lib.f64(k["zLen"])
        pr.origin[0], pr.origin[1] = float(mtMesh.origin[0]), float(mtMesh.origin[1])
        pr.nFreq, pr.freqs = len(k["freqs"]), _lib.f64(k["freqs"])
        pr.nRx, pr.rxLoc = k["rx"].shape[0], _lib.f64(k["rx"])
        pr.nComp, pr.compMode = len(comp_mode), _lib.i32(k["comp"])
        pr.nData = len(k["obs"])
        pr.freqID, pr.rxID, pr.dtID = _lib.i64(k["fid"]), _lib.i64(k["rid"]), _lib.i64(k["did"])
        pr.obsData = k["obs"].ctypes.data_as(C.POINTER(C.c_double))
        pr.dataErr = _lib.f64(k["err"])
        pr.nAC, pr.activeIdx, pr.bgModel = len(act), _lib.i32(k["act"]), _lib.f64(k["bg"])
        pr.wmRowPtr, pr.wmColIdx, pr.wmVal = _lib.i32(k["wp"]), _lib.i32(k["wi"]), _lib.f64(k["wv"])
        pr.regParam = float(hmcprior.regParam)
        pr.sigBounds[0], pr.sigBounds[1] = float(hmcprior.sigBounds[0]), float(hmcprior.sigBounds[1])
        pr.nChains, pr.device = self.nChains, int(device)
        h = C.c_void_p()
        create = self.L.hmcmt_plan_create_rho_phase if self.rho_phase else self.L.hmcmt_plan_create
        _lib.check(create(C.byref(pr), C.byref(h)), "hmcmt_plan_create")
        self.h = h
        self.nAC, self.nData, self.nFreq = len(act), pr.nData, pr.nFreq
        self.nNode = (self.ny + 1) * (self.nz + 1)
        self.nCell = self.ny * self.nz
        self.compTE, self.compTM = 0 in comp_mode or 2 in comp_mode, 1 in comp_mode

    def info(self, what: int) -> int:
        return int(self.L.hmcmt_plan_info(self.h, what))

    def close(self):
        if getattr(self, "h", None):
            self.L.hmcmt_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- array helpers --
    def _m(self, m):
        m = np.ascontiguousarray(m, dtype=np.float64).reshape(self.nChains, self.nAC)
        return m

    def forward(self, m=None, sigma=None, fields=True):
        self.generation = getattr(self, "generation", 0) + 1       # MT2DFwdData handles of earlier evaluations become stale
        pred = np.zeros((self.nChains, self.nData), dtype=self.dtype)
        ex = np.zeros((self.nChains, self.nFreq, self.nNode), dtype=np.complex128) if (fields and self.compTE) else None
        hx = np.zeros((self.nChains, self.nFreq, self.nNode), dtype=np.complex128) if (fields and self.compTM) else None
        cp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double)) if a is not None else None
        if sigma is not None:
            s = np.ascontiguousarray(sigma, dtype=np.float64).reshape(self.nChains, self.nCell)
            _lib.check(self.L.hmcmt_forward_sigma(self.h, _lib.f64(s), cp(pred), cp(ex), cp(hx)), "hmcmt_forward_sigma")
        else:
            mm = self._m(m)
            _lib.check(self.L.hmcmt_forward(self.h, _lib.f64(mm), cp(pred), cp(ex), cp(hx)), "hmcmt_forward")
        return pred, ex, hx

    def jtvec(self, v):
        """real(J^T conj(v)) w.r.t. the active-cell conductivities for the last forward evaluation (real v, J^T v, for Rho_Pha)."""
        v = np.ascontiguousarray(v, dtype=self.dtype).reshape(self.nChains, self.nData)
        g = np.zeros((self.nChains, self.nAC))
        _lib.check(self.L.hmcmt_jtvec(self.h, v.ctypes.data_as(C.POINTER(C.c_double)), _lib.f64(g)), "hmcmt_jtvec")
        return g

    def jacobian(self):
        """Explicit Jacobian d pred / d sigma_active of the last forward evaluation: [nChains, nData, nAC], complex dZ/dsigma
        (Impedance) or real d rho_a / d sigma, d phase / d sigma rows (Rho_Pha)."""
        J = np.zeros((self.nChains, self.nData, self.nAC), dtype=self.dtype)
        _lib.check(self.L.hmcmt_jacobian(self.h, J.ctypes.data_as(C.POINTER(C.c_double))), "hmcmt_jacobian")
        return J

    def jvec(self, dsig):
        """J dsig for the last forward evaluation, J being what `jacobian` returns: dsig [nChains, nAC] conductivity perturbation
        of the active cells -> [nChains, nData] (complex, or real rows for Rho_Pha), without forming J."""
        d = np.ascontiguousarray(dsig, dtype=np.float64).reshape(self.nChains, self.nAC)
        jv = np.zeros((self.nChains, self.nData), dtype=self.dtype)
        _lib.check(self.L.hmcmt_jvec(self.h, _lib.f64(d), jv.ctypes.data_as(C.POINTER(C.c_double))), "hmcmt_jvec")
        return jv

    def gn_hessvec(self, v, total=False):
        """Gauss-Newton Hessian of the data misfit in ln(sigma) times v: D Re(J^H Wd^2 J) D v, D = diag(sigma_active), for the
        last forward evaluation; total=True adds the model-norm part beta Wm v."""
        vv = self._m(v)
        hv = np.zeros((self.nChains, self.nAC))
        _lib.check(self.L.hmcmt_gn_hessvec(self.h, _lib.f64(vv), 1 if total else 0, _lib.f64(hv)), "hmcmt_gn_hessvec")
        return hv

    def gauss_newton(self, m0=None, mref=None, max_iter=10, max_cg=10, cg_tol=1e-2, max_ls=8, max_step=3.0, tol_rel=1e-4):
        """Posterior mode of every chain by projected Gauss-Newton-CG (hmcmt_gauss_newton): minimises phi_d(m) + 1/2 beta
        (m - m_ref)^T Wm (m - m_ref) within the plan's bounds, every CG product from the resident factors.  m0: start model
        (default: the plan's current model); mref: sets the reference model first (set_state).  Returns (m [nChains, nAC],
        history [nChains, max_iter + 1, 6] = (phi_d, phi_m, |P g|, CG iterations, alpha, line-search trials) per accepted step,
        info [nChains, 2] = (accepted steps, stop reason: 0 max_iter, 1 tolerance, 2 line search failed)).  The plan is left
        evaluated at m: forward_gradient(m, total=True) would reproduce its state, and jvec / gn_hessvec / jacobian work there."""
        if mref is not None:
            self.set_state(mref=mref)
        self.generation = getattr(self, "generation", 0) + 1
        m = np.zeros((self.nChains, self.nAC))
        hist = np.zeros((self.nChains, max(int(max_iter), 0) + 1, 6))
        info = np.zeros((self.nChains, 2), dtype=np.int32)
        mm = None if m0 is None else self._m(m0)
        _lib.check(self.L.hmcmt_gauss_newton(self.h, None if mm is None else _lib.f64(mm), int(max_iter), int(max_cg), float(cg_tol), int(max_ls), float(max_step),
                                             float(tol_rel), _lib.f64(m), _lib.f64(hist), _lib.i32(info)), "hmcmt_gauss_newton")
        return m, hist, info

    def gn_eig(self, k, r=None, omega=None, seed=0):
        """Low-rank Gauss-Newton Hessian at the last forward evaluation (after gauss_newton: the mode), hmcmt_gn_eig: the k dominant
        pairs of H v = lambda beta Wm v, H = D Re(J^H Wd^2 J) D, by a randomized eigensolver with r test vectors (default min(nAC,
        96, k + 10)).  omega [nChains, r, nAC] standard normal, drawn with numpy from seed when not given.  The plan keeps the
        decomposition for set_mass_matrix(2) and laplace_sample.  Returns (lam [nChains, k] descending, V [nChains, k, nAC] with
        V^T beta Wm V = I, info [nChains, 2] = (columns kept after B-orthonormalisation, pairs kept)); entries beyond the pairs
        kept are zero."""
        k = int(k)
        if r is None:
            r = min(self.nAC, 96, k + 10)
        r = int(r)
        if omega is None:
            omega = np.random.default_rng(seed).standard_normal((self.nChains, r, self.nAC))
        om = np.ascontiguousarray(omega, dtype=np.float64).reshape(self.nChains, r, self.nAC)
        lam = np.zeros((self.nChains, k))
        V = np.zeros((self.nChains, k, self.nAC))
        info = np.zeros((self.nChains, 2), dtype=np.int32)
        _lib.check(self.L.hmcmt_gn_eig(self.h, k, r, _lib.f64(om), _lib.f64(lam), _lib.f64(V), _lib.i32(info)), "hmcmt_gn_eig")
        return lam, V, info

    def set_mass_matrix(self, kind):
        """Mass matrix of the sampler: 0 identity, 1 Wm, 2 beta Wm + H_k (the low-rank Gauss-Newton Hessian of gn_eig)."""
        _lib.check(self.L.hmcmt_set_mass_matrix(self.h, int(kind)), "hmcmt_set_mass_matrix")

    def laplace_sample(self, z=None, ns=1, seed=0):
        """Draws of the Laplace approximation N(m_lin, M^-1), M = beta Wm + H_k of gn_eig at its linearisation point m_lin
        (hmcmt_laplace_sample): m_lin + M^-1 S z, S S^T = M.  z [nChains, ns, nAC] standard normal, drawn with numpy from seed
        when not given.  The bounds are not applied.  Returns [nChains, ns, nAC]."""
        if z is None:
            z = np.random.default_rng(seed).standard_normal((self.nChains, int(ns), self.nAC))
        zz = np.ascontiguousarray(z, dtype=np.float64)
        ns = zz.size // (self.nChains * self.nAC)
        zz = zz.reshape(self.nChains, ns, self.nAC)
        out = np.zeros_like(zz)
        _lib.check(self.L.hmcmt_laplace_sample(self.h, ns, _lib.f64(zz), _lib.f64(out)), "hmcmt_laplace_sample")
        return out

    def posterior_variance(self, prior=True, posterior=True, resolution=True):
        """Per-cell variances in ln sigma (hmcmt_posterior_variance): (prior_var [nAC] = diag((beta Wm)^-1), post_var [nChains, nAC]
        = diag(M^-1) of the Laplace approximation with M = beta Wm + H_k of gn_eig, resolution [nChains, nAC] = diag(V D V^T beta Wm)).
        An output not asked for is None; post_var and resolution need gn_eig first.  The bounds are not applied."""
        pv = np.zeros(self.nAC) if prior else None
        qv = np.zeros((self.nChains, self.nAC)) if posterior else None
        rv = np.zeros((self.nChains, self.nAC)) if resolution else None
        ptr = lambda a: _lib.f64(a) if a is not None else None  # noqa: E731
        _lib.check(self.L.hmcmt_posterior_variance(self.h, ptr(pv), ptr(qv), ptr(rv)), "hmcmt_posterior_variance")
        return pv, qv, rv

    def forward_gradient(self, m, total=False):
        """compDataGradient (HMCSampler.jl:277-330): predicted data, data misfit, gradient w.r.t. ln(sigma).  total=True adds the
        model-norm part beta Wm (m - m_ref) on the device (m_ref from set_state), as proposeLeapfrog does right afterwards."""
        self.generation = getattr(self, "generation", 0) + 1
        mm = self._m(m)
        pred = np.zeros((self.nChains, self.nData), dtype=self.dtype)
        phi = np.zeros(self.nChains)
        g = np.zeros((self.nChains, self.nAC))
        fn = self.L.hmcmt_forward_gradient_total if total else self.L.hmcmt_forward_gradient
        _lib.check(fn(self.h, _lib.f64(mm), pred.ctypes.data_as(C.POINTER(C.c_double)), _lib.f64(phi), _lib.f64(g)),
                   "hmcmt_forward_gradient")
        return pred, phi, g

    def set_state(self, m=None, p=None, mref=None):
        a = [None if x is None else self._m(x) for x in (m, p, mref)]
        _lib.check(self.L.hmcmt_set_state(self.h, *[None if x is None else _lib.f64(x) for x in a]), "hmcmt_set_state")

    def get_state(self):
        m = np.zeros((self.nChains, self.nAC))
        p = np.zeros((self.nChains, self.nAC))
        _lib.check(self.L.hmcmt_get_state(self.h, _lib.f64(m), _lib.f64(p)), "hmcmt_get_state")
        return m, p

    def leapfrog_trajectory(self, dt, intstep, want_pred=True):
        L = np.ascontiguousarray(np.broadcast_to(np.asarray(intstep, dtype=np.int32), (self.nChains,)))
        stats = np.zeros((self.nChains, 4))
        pred = np.zeros((self.nChains, self.nData), dtype=self.dtype) if want_pred else None
        _lib.check(self.L.hmcmt_leapfrog_trajectory(self.h, float(dt), _lib.i32(L), _lib.f64(stats),
                                                    None if pred is None else pred.ctypes.data_as(C.POINTER(C.c_double))),
                   "hmcmt_leapfrog_trajectory")
        return stats, pred

    def leapfrog_steps_device(self, dt, nsteps):
        _lib.check(self.L.hmcmt_leapfrog_steps_device(self.h, float(dt), int(nsteps)), "hmcmt_leapfrog_steps_device")

    def sync(self):
        _lib.check(self.L.hmcmt_sync(self.h), "hmcmt_sync")

    def timer_start(self):
        _lib.check(self.L.hmcmt_timer_start(self.h), "hmcmt_timer_start")

    def timer_stop(self) -> float:
        ms = C.c_float(0)
        _lib.check(self.L.hmcmt_timer_stop(self.h, C.byref(ms)), "hmcmt_timer_stop")
        return float(ms.value)

    def kernel_time(self, reset=True):
        ms, n = C.c_float(0), C.c_int64(0)
        _lib.check(self.L.hmcmt_kernel_time(self.h, int(reset), C.byref(ms), C.byref(n)), "hmcmt_kernel_time")
        return float(ms.value), int(n.value)

    def kernel_time_split(self):
        """(factorisation alone, forward solve alone) of the evaluations timed since the last reset, ms."""
        a, b = C.c_float(0), C.c_float(0)
        _lib.check(self.L.hmcmt_kernel_time_split(self.h, C.byref(a), C.byref(b)), "hmcmt_kernel_time_split")
        return float(a.value), float(b.value)

    def status(self) -> int:
        """Device error flags of everything queued so far (synchronises, clears): 0, -10 singular pivot, -21 bounds."""
        return int(self.L.hmcmt_status(self.h))

    def run_chain(self, dt, nsamples, rhoref, z_init, intsteps, u_accept, z_mom, reuse_last_forward=True, m_start=None):
        nc = self.nChains
        z_init = np.ascontiguousarray(z_init, dtype=np.float64).reshape(nc, self.nAC)
        intsteps = np.ascontiguousarray(intsteps, dtype=np.int32).reshape(nsamples)
        u_accept = np.ascontiguousarray(u_accept, dtype=np.float64).reshape(nc, nsamples)
        z_mom = np.ascontiguousarray(z_mom, dtype=np.float64).reshape(nsamples, nc, self.nAC)
        model = np.zeros((nc, nsamples, self.nAC))
        stats = np.zeros((nc, nsamples + 1, 4))
        acc = np.zeros((nc, nsamples), dtype=np.int32)
        data = np.zeros((nc, nsamples + 1, self.nData), dtype=self.dtype)
        ms = None if m_start is None else np.ascontiguousarray(m_start, dtype=np.float64).reshape(nc, self.nAC)
        _lib.check(self.L.hmcmt_run_chain(self.h, float(dt), int(nsamples), float(rhoref), None if ms is None else _lib.f64(ms),
                                          _lib.f64(z_init), _lib.i32(intsteps),
                                          _lib.f64(u_accept), _lib.f64(z_mom), int(bool(reuse_last_forward)), _lib.f64(model),
                                          _lib.f64(stats), _lib.i32(acc), data.ctypes.data_as(C.POINTER(C.c_double))),
                   "hmcmt_run_chain")
        return model, stats, acc, data

    def export_system(self, mode, freq, chain=0):
        """Aii (scipy CSC rebuilt from the reference-numbered 1-based CSC), rhs, bc of one system."""
        N = self.info(0)
        nnz = 5 * N - 2 * (self.ny - 1) - 2 * (self.nz - 1)
        colptr = np.zeros(N + 1, dtype=np.int64)
        rowval = np.zeros(nnz, dtype=np.int64)
        nzval = np.zeros(nnz, dtype=np.complex128)
        rhs = np.zeros(N, dtype=np.complex128)
        bc = np.zeros(2 * (self.ny + self.nz), dtype=np.complex128)
        cp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
        _lib.check(self.L.hmcmt_export_system(self.h, chain, mode, freq, _lib.i64(colptr), _lib.i64(rowval), cp(nzval), cp(rhs), cp(bc)),
                   "hmcmt_export_system")
        return colptr, rowval, nzval, rhs, bc


    # -- frequency-sharded step (include/hmcmt_b200.h) --
    def step_partial(self, dt):
        _lib.check(self.L.hmcmt_step_partial(self.h, float(dt)), "hmcmt_step_partial")

    def step_finish(self, dt):
        _lib.check(self.L.hmcmt_step_finish(self.h, float(dt)), "hmcmt_step_finish")

    def exchange_buffer(self):
        """(device pointer, number of doubles) of the per-step exchange buffer [gdata(nAC) | phi_d] x nChains."""
        ptr, n = C.c_void_p(), C.c_int64(0)
        _lib.check(self.L.hmcmt_exchange_buffer(self.h, C.byref(ptr), C.byref(n)), "hmcmt_exchange_buffer")
        return int(ptr.value), int(n.value)


# ---------------------------------------------------------------------------------------------------
# frequency sharding (SURVEY.md 8e, BASELINE.json configs[3]): the (frequency, mode) systems are independent given sigma


def shard_frequencies(mtData: MTData, invParam: InvDataModel, rank: int, world: int):
    """Frequencies rank, rank+world, ... (round-robin: every frequency costs the same, identical sparsity pattern).
    -> (MTData restricted to those frequencies with freqID renumbered 1..n, InvDataModel with the matching observation
    rows, `rows` = positions of those observations in the full data vector)."""
    nF = len(mtData.freqs)
    mine = np.arange(rank, nF, world)
    if len(mine) == 0:
        raise ValueError(f"rank {rank} of {world} owns no frequency (nFreq = {nF})")
    newid = np.zeros(nF + 1, dtype=np.int64)
    newid[mine + 1] = np.arange(1, len(mine) + 1)
    fid = np.asarray(mtData.freqID)
    rows = np.nonzero(newid[fid] > 0)[0]
    # dataID is the (comp, rx, freq) presence mask of readMT2DData.jl:165-172: keep the frequency planes this rank owns
    nRx, nDt = np.asarray(mtData.rxLoc).shape[0], len(mtData.dataComp)
    mask = np.asarray(mtData.dataID, dtype=bool).reshape(nF, nRx, nDt)[mine].reshape(-1)
    sub = MTData(np.array(mtData.rxLoc), np.array(mtData.freqs)[mine], mtData.dataType, list(mtData.dataComp),
                 np.asarray(mtData.rxID)[rows], newid[fid[rows]], np.asarray(mtData.dtID)[rows], mask, mtData.compTE, mtData.compTM)
    dataW = np.asarray(invParam.dataW)[rows]
    inv = InvDataModel(np.asarray(invParam.obsData)[rows], dataW, np.array(invParam.strModel), np.array(invParam.refModel),
                       invParam.activeCell, np.array(invParam.bgModel), invParam.Wm, 1.0 / dataW)
    return sub, inv, rows


def shard_systems(mtData: MTData, invParam: InvDataModel, rank: int, world: int):
    """Balanced partition of the (frequency, mode) SYSTEMS: with an even number of ranks and a TE + TM survey the first half of
    the ranks takes the TE systems and the second half the TM systems, frequencies round-robin inside each half (120 systems
    over 8 ranks = 15 each at cfg4, instead of 8 / 7 frequencies x 2 modes).  Otherwise falls back to `shard_frequencies`.
    A rank takes every DataComp entry its mode computes: ZXY and TZY, or ZYX, or the rho_a and phase rows of one mode.
    -> (MTData of this rank, InvDataModel with its observation rows, `rows` = their positions in the full data vector)."""
    comp_modes = np.array([_comp_mode(c) for c in mtData.dataComp])
    two_modes = bool(mtData.compTE and mtData.compTM) and set(comp_modes.tolist()) == {0, 1}
    if world < 2 or world % 2 or not two_modes:
        return shard_frequencies(mtData, invParam, rank, world)
    half = world // 2
    mode = 0 if rank < half else 1                              # 0: ZXY (TE), 1: ZYX (TM)
    nF = len(mtData.freqs)
    mine = np.arange(rank % half, nF, half)
    if len(mine) == 0:
        raise ValueError(f"rank {rank} of {world} owns no system (nFreq = {nF})")
    newid = np.zeros(nF + 1, dtype=np.int64)
    newid[mine + 1] = np.arange(1, len(mine) + 1)
    fid, did = np.asarray(mtData.freqID), np.asarray(mtData.dtID)
    comps = np.nonzero(comp_modes == mode)[0]                   # DataComp entries of this mode, in order
    newdid = np.zeros(len(comp_modes) + 1, dtype=np.int64)
    newdid[comps + 1] = np.arange(1, len(comps) + 1)
    rows = np.nonzero((newid[fid] > 0) & (newdid[did] > 0))[0]
    nRx, nDt = np.asarray(mtData.rxLoc).shape[0], len(mtData.dataComp)
    mask = np.asarray(mtData.dataID, dtype=bool).reshape(nF, nRx, nDt)[mine][:, :, comps].reshape(-1)
    sub = MTData(np.array(mtData.rxLoc), np.array(mtData.freqs)[mine], mtData.dataType, [mtData.dataComp[k] for k in comps],
                 np.asarray(mtData.rxID)[rows], newid[fid[rows]], newdid[did[rows]], mask, mode == 0, mode == 1)
    dataW = np.asarray(invParam.dataW)[rows]
    inv = InvDataModel(np.asarray(invParam.obsData)[rows], dataW, np.array(invParam.strModel), np.array(invParam.refModel),
                       invParam.activeCell, np.array(invParam.bgModel), invParam.Wm, 1.0 / dataW)
    return sub, inv, rows


class FreqShardedPlan:
    """One rank's share of a system-sharded problem (SURVEY.md 8e).  `group` is a torch.distributed process group used for the
    plumbing (rendezvous, host-buffer evaluations); the data-path collective of the device-resident leapfrog steps — one
    sum-all-reduce of [gdata | phi_d] per step — is issued by the library itself through NCCL on the plan's stream when the
    group's backend is NCCL (`in_library_nccl`), else by torch.distributed on the exchange buffer."""

    def __init__(self, mtMesh, mtData, invParam, hmcprior, rank: int, world: int, device: int = 0, group=None, balance="systems"):
        self.rank, self.world, self.group = int(rank), int(world), group
        self.nDataFull = len(np.asarray(invParam.obsData))
        self.rho_phase = "Rho_Pha" in mtData.dataType              # real predictions
        shard = shard_systems if balance == "systems" else shard_frequencies
        sub, inv, self.rows = shard(mtData, invParam, rank, world)
        self.plan = Plan(mtMesh, sub, inv, hmcprior, nChains=1, device=device)
        self.nAC, self.device = self.plan.nAC, int(device)
        self._xt = None
        self.in_library_nccl = False
        if self.world > 1:
            import torch.distributed as dist
            if dist.is_initialized() and dist.get_backend(group) == "nccl":
                uid = C.create_string_buffer(128)
                if self.rank == 0:
                    _lib.check(self.plan.L.hmcmt_nccl_unique_id(uid), "hmcmt_nccl_unique_id")
                box = [uid.raw]
                dist.broadcast_object_list(box, src=0, group=group)
                _lib.check(self.plan.L.hmcmt_nccl_init(self.plan.h, box[0], self.rank, self.world), "hmcmt_nccl_init")
                self.in_library_nccl = True

    # host-buffer evaluation: compDataGradient over all frequencies
    def forward_gradient(self, m):
        import torch
        import torch.distributed as dist
        pred, phi, g = self.plan.forward_gradient(m)
        full = np.zeros(self.nDataFull, dtype=np.float64 if self.rho_phase else np.complex128)
        full[self.rows] = pred[0]
        packed = np.concatenate([g[0], phi, full.view(np.float64)])
        if self.world > 1:
            t = torch.from_numpy(packed)
            if dist.get_backend(self.group) == "nccl":
                t = t.cuda(self.device)
            dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group)
            packed = t.cpu().numpy()
        nAC = self.nAC
        data = packed[nAC + 1:]
        return (data if self.rho_phase else data.view(np.complex128)), float(packed[nAC]), packed[:nAC]

    # device-resident leapfrog steps with one all-reduce per step
    def _exchange_tensor(self):
        import torch
        if self._xt is None:
            ptr, n = self.plan.exchange_buffer()

            class _View:
                __cuda_array_interface__ = dict(shape=(n,), typestr="<f8", data=(ptr, False), version=2)
            self._xt = torch.as_tensor(_View(), device=f"cuda:{self.device}")
        return self._xt

    def leapfrog_steps_device(self, dt, nsteps):
        if self.world == 1:
            self.plan.leapfrog_steps_device(dt, nsteps)
            return
        if self.in_library_nccl:
            _lib.check(self.plan.L.hmcmt_leapfrog_steps_sharded(self.plan.h, float(dt), int(nsteps)), "hmcmt_leapfrog_steps_sharded")
            return
        import torch
        import torch.distributed as dist
        xt = self._exchange_tensor()
        for _ in range(int(nsteps)):
            self.plan.step_partial(dt)
            self.plan.sync()                                   # the plan's stream is not torch's
            dist.all_reduce(xt, op=dist.ReduceOp.SUM, group=self.group)
            torch.cuda.current_stream(self.device).synchronize()
            self.plan.step_finish(dt)

    def set_state(self, m=None, p=None, mref=None):
        self.plan.set_state(m, p, mref)

    def get_state(self):
        return self.plan.get_state()

    def sync(self):
        self.plan.sync()

    def close(self):
        self.plan.close()


def _plan_for(mtMesh, mtData, invParam, hmcprior, nChains=1, device=0) -> Plan:
    """One plan per (invParam, nChains, device), cached on the invParam object like the reference caches
    operators on the mesh (`mtMesh.setup`)."""
    cache = invParam.__dict__.setdefault("_plans", {})
    key = (id(mtMesh), id(mtData), nChains, device, float(hmcprior.regParam), tuple(hmcprior.sigBounds))
    if key not in cache:
        cache[key] = Plan(mtMesh, mtData, invParam, hmcprior, nChains, device)
    # hmcprior.massType: "diagonal" (identity) or non-diagonal M = Wm (setMassMatrix HMCSampler.jl:463-489)
    _lib.check(cache[key].L.hmcmt_set_mass_matrix(cache[key].h, 0 if hmcprior.massType == "diagonal" else 1), "hmcmt_set_mass_matrix")
    return cache[key]


def _forward_only_plan(mtMesh, mtData, device=0) -> Plan:
    """Plan without observations for `MT2DFwdSolver(mtMesh, mtData)`.  For "Rho_Pha" data the plan is built on the impedance
    bookkeeping of the modes present (one component per mode, every (freq, rx) pair) and switched to apparent resistivity /
    phase responses; the reference's interleaving and dataID mask are applied by the caller."""
    cache = mtData.__dict__.setdefault("_fwd_plans", {})
    key = (id(mtMesh), device)
    if key not in cache:
        md = mtData
        if "Rho_Pha" in mtData.dataType:
            comps = (["ZXY"] if mtData.compTE else []) + (["ZYX"] if mtData.compTM else [])
            nF, nRx, nC = len(mtData.freqs), np.asarray(mtData.rxLoc).shape[0], len(comps)
            f, r, c = np.meshgrid(np.arange(1, nF + 1), np.arange(1, nRx + 1), np.arange(1, nC + 1), indexing="ij")
            md = MTData(np.asarray(mtData.rxLoc), np.asarray(mtData.freqs), "Impedance", comps, r.reshape(-1).astype(np.int64),
                        f.reshape(-1).astype(np.int64), c.reshape(-1).astype(np.int64), np.ones(nF * nRx * nC, dtype=bool),
                        mtData.compTE, mtData.compTM)
        nData = int(np.count_nonzero(md.dataID))
        inv = setupInverseDataModel(mtMesh, [1e-8], 0.0, 0.0, np.zeros(nData, dtype=np.complex128), np.ones(nData))
        pl = Plan(mtMesh, md, inv, HMCPrior(), 1, device)
        if "Rho_Pha" in mtData.dataType:
            _lib.check(pl.L.hmcmt_set_response_kind(pl.h, 1), "hmcmt_set_response_kind")
        cache[key] = pl
    return cache[key]


class FactorHandle:
    """What `MT2DFwdData.AinvTE / AinvTM` carry here: the device-resident plan that owns the factors, and the evaluation they
    belong to (the reference stores one MUMPS handle per frequency, MT2DFwdSolver.jl:119-120)."""

    def __init__(self, plan: Plan, generation: int):
        self.plan, self.generation = plan, generation


# ---------------------------------------------------------------------------------------------------
# reference-named entry points


def MT2DFwdSolver(mtMesh: TensorMesh2D, mtData: MTData, linearSolver: str = "b200", plan: Optional[Plan] = None):
    """`MT2DFwdSolver(mtMesh, mtData; linearSolver)` (MT2DFwdSolver.jl:74-216) -> (predData, MT2DFwdData).
    DataType "Impedance": complex predData; "Rho_Pha": real [rho_a, phase] pairs interleaved per (freq, rx) as
    MT2DFwdSolver.jl:191-205 does, masked by dataID."""
    pl = plan or _forward_only_plan(mtMesh, mtData)
    pred, ex, hx = pl.forward(sigma=np.asarray(mtMesh.sigma))
    nNode, nF = pl.nNode, pl.nFreq
    exte = ex[0].T.copy() if ex is not None else np.zeros((nNode, nF), dtype=np.complex128)
    hxtm = hx[0].T.copy() if hx is not None else np.zeros((nNode, nF), dtype=np.complex128)
    h = FactorHandle(pl, pl.generation)
    if "Rho_Pha" in mtData.dataType:
        nC = int(pl.compTE) + int(pl.compTM)
        out = np.zeros((pl.nChains, pl.nFreq, np.asarray(mtData.rxLoc).shape[0], nC, 2))
        _lib.check(pl.L.hmcmt_get_responses(pl.h, _lib.f64(out)), "hmcmt_get_responses")
        # per (freq, rx): [rhoTE, phsTE, rhoTM, phsTM]  (vec of vcat(transpose(respTE), transpose(respTM)), :199-203)
        predData = out[0].reshape(-1)[np.asarray(mtData.dataID, dtype=bool)]
        return predData, MT2DFwdData(exte, hxtm, h, h, "b200", pl.generation)
    return pred[0], MT2DFwdData(exte, hxtm, h, h, "b200", pl.generation)


def compJacTMatVec(exTE, hxTM, datVec, mt2dMesh, mtData, activeCell=None, AinvTE=None, AinvTM=None, linSolver: str = "b200"):
    """`compJacTMatVec` (compJacTMatVec.jl:8-329): real(J^T v) over the active cells.  The fields and factors live on the
    device inside the plan carried by AinvTE/AinvTM (as returned by MT2DFwdSolver) and are reused for the adjoint solves
    (compJacTMatVec.jl:220-224); a handle of an earlier evaluation of the same plan is refused instead of silently returning
    the gradient at another model."""
    h = AinvTE if isinstance(AinvTE, FactorHandle) else AinvTM
    if not isinstance(h, FactorHandle):
        raise ValueError("compJacTMatVec needs the factor handle returned by MT2DFwdSolver (AinvTE/AinvTM)")
    pl = h.plan
    if h.generation != pl.generation:
        raise RuntimeError("compJacTMatVec: the factors of this MT2DFwdData were overwritten by a later evaluation on the same "
                           "mesh / survey; call MT2DFwdSolver again (one set of factors is kept resident per plan)")
    if "Rho_Pha" in mtData.dataType:
        raise NotImplementedError("the reference never forms sVec for 'Rho_Pha' data ('Rho_Phs', compJacTMatVec.jl:104,189,260)")
    g = pl.jtvec(datVec)[0]
    if activeCell is not None:
        # map by cell index, whatever the caller's selector looks like (the plan's active set is 'all non-air cells')
        full = np.zeros(pl.nCell)
        full[pl._keep["act"]] = g
        return np.asarray(activeCell.T @ full).reshape(-1)
    return g


def compJacMatVec(exTE, hxTM, dsig, mt2dMesh, mtData, activeCell=None, AinvTE=None, AinvTM=None):
    """J dsig, the forward-mode twin of `compJacTMatVec`: the predicted impedances' derivative along the conductivity
    perturbation dsig of the active cells (the columns of activeCell, or the plan's own active set), for the fields / factors of
    the MT2DFwdData the handles belong to.  Equals compJacMat(...) @ dsig without forming the matrix."""
    h = AinvTE if isinstance(AinvTE, FactorHandle) else AinvTM
    if not isinstance(h, FactorHandle):
        raise ValueError("compJacMatVec needs the factor handle returned by MT2DFwdSolver (AinvTE/AinvTM)")
    pl = h.plan
    if h.generation != pl.generation:
        raise RuntimeError("compJacMatVec: the factors of this MT2DFwdData were overwritten by a later evaluation on the same "
                           "mesh / survey; call MT2DFwdSolver again (one set of factors is kept resident per plan)")
    if "Rho_Pha" in mtData.dataType:
        raise NotImplementedError("explicit Jacobian products: Impedance data only, as compJacMat (Plan.jvec serves Rho_Pha)")
    d = np.asarray(dsig, dtype=np.float64).reshape(-1)
    if activeCell is not None:
        # map by cell index, whatever the caller's selector looks like (the plan's active set is 'all non-air cells')
        d = np.asarray(activeCell @ d).reshape(-1)[pl._keep["act"]]
    return pl.jvec(d)[0]


def compJacMat(exTE, hxTM, mt2dMesh, mtData, activeCell=None, AinvTE=None, AinvTM=None, linSolver: str = "b200"):
    """`compJacMat` (compJacMat.jl:7-381): explicit complex Jacobian (nData x nAC) of the predicted impedances with respect
    to the active-cell conductivities, for the fields / factors of the MT2DFwdData the handles belong to."""
    h = AinvTE if isinstance(AinvTE, FactorHandle) else AinvTM
    if not isinstance(h, FactorHandle):
        raise ValueError("compJacMat needs the factor handle returned by MT2DFwdSolver (AinvTE/AinvTM)")
    pl = h.plan
    if h.generation != pl.generation:
        raise RuntimeError("compJacMat: the factors of this MT2DFwdData were overwritten by a later evaluation")
    if "Rho_Pha" in mtData.dataType:
        raise NotImplementedError("explicit Jacobian: Impedance data only")
    J = pl.jacobian()[0]
    if activeCell is not None:
        full = np.zeros((J.shape[0], pl.nCell), dtype=np.complex128)
        full[:, pl._keep["act"]] = J
        return np.asarray((activeCell.T @ full.T).T)
    return J


def compJacTMat(exTE, hxTM, mt2dMesh, mtData, activeCell=None, AinvTE=None, AinvTM=None, linSolver: str = "b200"):
    """`compJacTMat` (compJacTMat.jl:9-406): the transposed Jacobian (nAC x nData)."""
    return compJacMat(exTE, hxTM, mt2dMesh, mtData, activeCell, AinvTE, AinvTM, linSolver).T.copy()


def compDataGradient(mtMesh, mtData, invParam: InvDataModel, hmcprior: HMCPrior):
    """4-argument `compDataGradient` (HMCSampler.jl:277-330) -> (predData, dataMisfit, dataGrad)."""
    pl = _plan_for(mtMesh, mtData, invParam, hmcprior)
    pred, phi, g = pl.forward_gradient(invParam.strModel)
    mtMesh.sigma = invParam.activeCell @ np.exp(invParam.strModel) + invParam.bgModel
    hmcprior.nfevals += 0
    return pred[0], float(phi[0]), g[0]


def getHamiltonian(mtData, mtMesh, invParam, hmcprior, hmcParam: HMCParameter):
    """`getHamiltonian` (HMCSampler.jl:358-397) -> (dataMisfit, kp, hmp, mnorm, predData)."""
    pl = _plan_for(mtMesh, mtData, invParam, hmcprior)
    pred, _, _ = pl.forward(m=invParam.strModel, fields=False)
    res = invParam.dataW * (pred[0] - invParam.obsData)
    dm = float(np.real(0.5 * np.vdot(res, res)))
    if hmcprior.massType == "diagonal":
        kp = 0.5 * float(hmcParam.momentum @ hmcParam.momentum)
    else:                                                    # invM = Wm^{-1} (setMassMatrix(invParam) HMCSampler.jl:478-489)
        import scipy.sparse.linalg as spla
        kp = 0.5 * float(hmcParam.momentum @ spla.spsolve(invParam.Wm.tocsc(), hmcParam.momentum))
    d = invParam.strModel - invParam.refModel
    mnorm = 0.5 * float(d @ (invParam.Wm @ d)) * hmcprior.regParam
    return dm, kp, dm + kp + mnorm, mnorm, pred[0]


def proposeLeapfrog(hmcParamCurrent: HMCParameter, mtMesh, mtData, invParam, hmcprior, intstep: Optional[int] = None, rng=None):
    """`proposeLeapfrog` (HMCSampler.jl:206-269) -> (propModel, propMomentum); the whole trajectory runs on
    the device.  `intstep` injects the reference's `rand(t1:t2)` draw (:233)."""
    pl = _plan_for(mtMesh, mtData, invParam, hmcprior)
    if intstep is None:
        rng = rng or np.random.default_rng()
        intstep = int(rng.integers(hmcprior.timestep[0], hmcprior.timestep[1] + 1))
    pl.set_state(hmcParamCurrent.rhomodel, hmcParamCurrent.momentum, invParam.refModel)
    pl.leapfrog_trajectory(hmcprior.dt, intstep, want_pred=False)
    m, p = pl.get_state()
    invParam.strModel = m[0].copy()
    hmcprior.nfevals += intstep + 1
    return m[0], p[0]


@dataclass
class RandomStreams:
    """Injected random draws in the reference's order (SURVEY.md A.7)."""
    u_start: float
    z_init: np.ndarray
    intsteps: np.ndarray
    u_accept: np.ndarray
    z_momentum: np.ndarray

    @staticmethod
    def make(seed, nparam, nsamples, timestep):
        rng = np.random.default_rng(seed)
        return RandomStreams(float(rng.random()), rng.standard_normal(nparam),
                             rng.integers(timestep[0], timestep[1] + 1, size=nsamples),
                             rng.random(nsamples), rng.standard_normal((nsamples, nparam)))


def runHMCSampler(mtMesh, mtData, invParam: InvDataModel, hmcprior: HMCPrior, streams: Optional[RandomStreams] = None,
                  nsamples: Optional[int] = None, seed: int = 0, reuse_last_forward: bool = True, device: int = 0):
    """`runHMCSampler` (HMCSampler.jl:72-196) -> (hmcmodel [nparam x nsamples], HMCStatus, hmcdata [ndata x (nsamples+1)])."""
    nparam = len(invParam.strModel)
    nsamples = hmcprior.totalsamples if nsamples is None else nsamples
    streams = streams or RandomStreams.make(seed, nparam, nsamples, hmcprior.timestep)
    pl = _plan_for(mtMesh, mtData, invParam, hmcprior, 1, device)
    rho0 = 1.0 / np.exp(invParam.strModel[0])                      # unique(strModel)[1]  (:100-101)
    rhoref = float(np.round(rho0 * 0.5 + (rho0 * 1.5 - rho0 * 0.5) * streams.u_start))
    print(f"Homogeneous starting model with a resistivity of {rhoref} Ωm is used.")
    start = np.log(np.ones(nparam) / rhoref)
    m_file = np.array(invParam.strModel, dtype=np.float64)        # hmcParamCurrent.rhomodel = copy(invParam.strModel) (:87)
    invParam.strModel = start.copy()
    invParam.refModel = start.copy()
    model, stats, acc, data = pl.run_chain(hmcprior.dt, nsamples, rhoref, streams.z_init, streams.intsteps[:nsamples],
                                           streams.u_accept[:nsamples], streams.z_momentum[:nsamples], reuse_last_forward, m_start=m_file)
    hmcprior.nfevals += int(np.sum(streams.intsteps[:nsamples]) + nsamples)
    st = HMCStatus(int(acc[0].sum()), int(nsamples - acc[0].sum()), acc[0].astype(bool), stats[0].T.copy())
    return model[0].T.copy(), st, data[0].T.copy()


def getPosteriorModel(hmcmodel, mtMesh, invParam, hmcprior, outdir: str = "."):
    """`getPosteriorModel` (HMCSampler.jl:605-642): meanModel.model / stdModel.model after burn-in."""
    burn = hmcprior.burninsamples
    ens = hmcmodel[:, burn:]
    mean = ens.mean(axis=1)
    var = (ens ** 2).mean(axis=1) - mean ** 2
    var[var < 0] = np.finfo(float).eps
    std = np.sqrt(var)
    out = TensorMesh2D(mtMesh.yLen, mtMesh.zLen, mtMesh.airLayer, mtMesh.gridSize, mtMesh.origin, None)
    out.sigma = invParam.activeCell @ np.exp(mean) + invParam.bgModel
    writeEMModel2D(os.path.join(outdir, "meanModel.model"), out)
    out.sigma = invParam.activeCell @ std + invParam.bgModel
    writeEMModel2D(os.path.join(outdir, "stdModel.model"), out)
    return mean, std


def getLaplacePosteriorModel(plan, m_map, mtMesh, invParam, outdir: str = ".", chain: int = 0):
    """The Laplace approximation's counterpart of getPosteriorModel: laplaceMeanModel.model holds exp(m_map) and
    laplaceStdModel.model the posterior standard deviation in ln sigma, sqrt(diag(M^-1)) of Plan.posterior_variance (M = beta Wm
    + H_k of the plan's gn_eig decomposition), in the same format and active-cell / background composition as meanModel.model /
    stdModel.model, so the Laplace and HMC maps compare file to file.  m_map: [nAC] (or [nChains, nAC], row `chain` used);
    `chain` selects the plan's chain.  Returns (m_map, std) of that chain."""
    m = np.asarray(m_map, dtype=np.float64)
    if m.ndim == 2:
        m = m[chain]
    _, post, _ = plan.posterior_variance(prior=False, posterior=True, resolution=False)
    std = np.sqrt(np.maximum(post[chain], 0.0))
    out = TensorMesh2D(mtMesh.yLen, mtMesh.zLen, mtMesh.airLayer, mtMesh.gridSize, mtMesh.origin, None)
    out.sigma = invParam.activeCell @ np.exp(m) + invParam.bgModel
    writeEMModel2D(os.path.join(outdir, "laplaceMeanModel.model"), out)
    out.sigma = invParam.activeCell @ std + invParam.bgModel
    writeEMModel2D(os.path.join(outdir, "laplaceStdModel.model"), out)
    return m, std


def outputHMCSamples(hmcmodel, hmcstats: HMCStatus, hmcdata, ichain: int = 1, cputime: float = 0.0, outdir: str = "."):
    """`outputHMCSamples` (HMCSampler.jl:785-828): hmcsamples_id*.model/.data and hmcstatistics_id*.log."""
    nparam, nsamples = hmcmodel.shape
    with open(os.path.join(outdir, f"hmcsamples_id{ichain}.model"), "w") as fh:
        for k in range(nsamples):
            fh.write("".join("%8.4e " % v for v in hmcmodel[:, k]) + "\n")
    with open(os.path.join(outdir, f"hmcsamples_id{ichain}.data"), "w") as fh:
        for k in range(nsamples + 1):
            fh.write("".join("%12.4e %12.4e" % (v.real, v.imag) for v in hmcdata[:, k]) + "\n")
    hs = hmcstats.hmstats
    with open(os.path.join(outdir, f"hmcstatistics_id{ichain}.log"), "w") as fh:
        fh.write("Total elapsed time (s): %8.2f\n" % cputime)
        fh.write("Totalsamples: %6d, nAccept: %6d, nReject: %6d\n" % (nsamples, hmcstats.nAccept, hmcstats.nReject))
        fh.write("Starting status: dtMisfit=%8.1f,mNorm=%8.1f,KEnergy=%8.1f,HEnergy=%8.1f\n" % tuple(hs[:, 0]))
        fh.write("iterNo   dtMisfit  mNorm   KEnergy  HEnergy  Accept \n")
        for k in range(1, nsamples + 1):
            fh.write("%6d %8.4e %8.4e %8.4e %8.4e %2d\n" % (k, hs[0, k], hs[1, k], hs[2, k], hs[3, k], int(hmcstats.acceptstats[k - 1])))


def parallelHMCSampler(mtMesh, mtData, invParam, hmcprior, pids: List[int], seeds: Optional[List[int]] = None,
                       nsamples: Optional[int] = None, outdir: Optional[str] = "."):
    """`parallelHMCSampler` (parallelHMC.jl:10-49): one independent chain per entry of `pids`; like the reference, the
    hmcsamples_id*/hmcstatistics_id* files of every chain are written (to `outdir`, default the working directory,
    parallelHMC.jl:41-45; None disables).  Under torchrun (one process per GPU) rank r runs chains r, r+world, ... on its
    own device with no data-path communication (replicas only) and rank 0 gathers the samples.  In a single process the
    chains run one after the other and `pids` — Julia worker ids in the reference (workers() starts at 2) — are mapped to
    CUDA devices by POSITION: chain k runs on device k mod (number of visible devices)."""
    import copy
    import time
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1:
        import torch.distributed as dist
        if not dist.is_available() or not dist.is_initialized():
            raise RuntimeError("parallelHMCSampler: WORLD_SIZE > 1 but torch.distributed is not initialised "
                               "(call torch.distributed.init_process_group first, e.g. under torchrun)")
        device = int(os.environ.get("LOCAL_RANK", "0"))
        ndev = 1
    else:
        device = None
        try:
            import torch
            ndev = max(1, torch.cuda.device_count())
        except Exception:
            ndev = 1
    seeds = seeds or list(range(1, len(pids) + 1))
    results = {}
    for k, _pid in enumerate(pids):
        if world > 1 and k % world != rank:
            continue
        inv_k, prior_k = copy.copy(invParam), copy.copy(hmcprior)
        inv_k.__dict__.pop("_plans", None)
        t0 = time.time()
        out = runHMCSampler(mtMesh, mtData, inv_k, prior_k, nsamples=nsamples, seed=seeds[k],
                            device=device if device is not None else k % ndev)
        results[k] = (out, time.time() - t0)
    if world > 1:
        import torch.distributed as dist
        gathered = [None] * world
        dist.all_gather_object(gathered, results)
        results = {k: v for part in gathered for k, v in part.items()}
    if outdir is not None and rank == 0:
        for k, ((model, st, data), cpu) in sorted(results.items()):
            outputHMCSamples(model, st, data, ichain=k + 1, cputime=cpu, outdir=outdir)
    order = sorted(results)
    return [results[k][0][0] for k in order], [results[k][0][1] for k in order], [results[k][0][2] for k in order]
