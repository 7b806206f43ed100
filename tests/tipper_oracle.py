"""CPU reference for the TE tipper TZY = Hz/Hy, built on the unchanged oracle (test infrastructure).

The reference has no tipper; this module applies the repository's definition (include/hmcmt_b200.h) on top of the oracle.  For
frequency f and receiver r of the TE system, with F0 = Ex on the receiver node row,
    Hz0_j = (F0_{j+1} - F0_j)/(yLen_j i omega mu0)       at the cell centres (Bz0/mu0 of getDataFuncSensTE)
    Hzr   = linRxMap2^T Hz0                              (normalised interpolation on the cell centres, sensUtils.jl:17-52)
    Hyr   = linRxMap^T Hy0                               (Hy0 and its normalised node interpolation of getDataFuncSensTE)
    T     = Hzr / Hyr.
Its linearisation gives the rows L_T (nRx x nNode, on the Ex field) and Q_T (nRx x nCell, the direct sigma dependence of Hy0)
in the oracle's own form.  J^T v runs the oracle's compJacTMatVec once per (frequency, TE) system with the receiver functional
extended by these rows: the tipper rows become extra "ZXY" rows with receiver ids nRx + r that select the stacked rows L_T, Q_T,
so s_T = L_T^T conj(v_T) joins the impedance source before the single adjoint solve.  The explicit Jacobian runs the oracle's
compJacMat with L_T, Q_T in place of the impedance rows.  The sampler entry points run the oracle's own with this forward and J^T v.
"""
import contextlib

import numpy as np
import scipy.sparse as sp

from oracle import fileio as ofio
from oracle import forward as ofwd
from oracle import jacobian as ojac
from oracle import operators as ops
from oracle import sampler as osamp
from oracle import sensitivity as osens
from oracle.forward import MU0

COMPS = ["ZXY", "ZYX", "TZY"]


def tipperFuncSensTE(omega, rx: osens.PreRxSens, Ex01):
    """-> (T [nRx], L_T [nRx x nNode], Q_T [nRx x nCell]) of one TE system; Ex01 = (Ex on row zid, Ex on row zid + 1)."""
    dEx0, dEx1 = rx.dFn0, rx.dFn1
    sigma1, dsigma1, yLen, zLen1 = rx.sigma1, rx.dsigma1, rx.yLen, rx.zLen1
    ny = len(yLen)
    # Hy0, dHy0, dHy0_dsig: the expressions of getDataFuncSensTE (oracle/sensitivity.py), which returns only the impedance rows
    dtmp = ops.sdiag(1.0 / yLen / (1j * omega)) @ ops.ddx(ny)
    dHzQ = (0.75 * (dtmp @ dEx0) + 0.25 * (dtmp @ dEx1)) / MU0
    HzQ = (0.75 * (ops.ddx(ny) @ Ex01[:, 0]) + 0.25 * (ops.ddx(ny) @ Ex01[:, 1])) / yLen / (1j * omega) / MU0
    dHyH = -(dEx1[1:-1, :] - dEx0[1:-1, :]) / zLen1 / (1j * omega * MU0)
    HyH = -(Ex01[1:-1, 1] - Ex01[1:-1, 0]) / zLen1 / (1j * omega * MU0)
    ExQ = 0.75 * Ex01[1:-1, 0] + 0.25 * Ex01[1:-1, 1]
    dExQ = 0.75 * dEx0[1:-1, :] + 0.25 * dEx1[1:-1, :]
    avm = ops.avnc(ny - 1)
    ybar = avm @ yLen
    sigma1v = (avm @ (sigma1 * yLen)) / ybar
    dsigma1v = ops.sdiag(1.0 / ybar) @ avm @ ops.sdiag(yLen) @ dsigma1
    ddHzQ = ops.sdiag(1.0 / ybar) @ ops.ddx(ny - 1) @ dHzQ
    Hy0 = np.zeros(ny + 1, dtype=np.complex128)
    Hy0[1:-1] = HyH - ((ops.ddx(ny - 1) @ HzQ) / ybar - sigma1v * ExQ) * (0.5 * zLen1)
    Hy0[0], Hy0[-1] = Hy0[1], Hy0[-2]
    dHy0 = osens._copy_ends(osens._pad_rows(dHyH - (ddHzQ - ops.sdiag(sigma1v) @ dExQ) * (0.5 * zLen1), ny))
    dHy0_dsig = osens._copy_ends(osens._pad_rows(0.5 * zLen1 * (ops.sdiag(ExQ) @ dsigma1v), ny))
    # the tipper
    hz = ops.sdiag(1.0 / (yLen * 1j * omega * MU0)) @ ops.ddx(ny)
    Hzr = rx.linRxMap2.T @ (hz @ Ex01[:, 0])
    Hyr = rx.linRxMap.T @ Hy0
    T = Hzr / Hyr
    L = ops.sdiag(1.0 / Hyr) @ (rx.linRxMap2.T @ hz @ dEx0) - ops.sdiag(T / Hyr) @ (rx.linRxMap.T @ dHy0)
    Q = -ops.sdiag(T / Hyr) @ (rx.linRxMap.T @ dHy0_dsig)
    return T, sp.csr_matrix(L), sp.csr_matrix(Q)


def _rx_sens(mesh, rxLoc):
    yNode = np.concatenate([[0.0], np.cumsum(mesh.yLen)]) - mesh.origin[0]
    zNode = np.concatenate([[0.0], np.cumsum(mesh.zLen)]) - mesh.origin[1]
    return osens.preSetRxFieldSens(rxLoc, yNode, zNode, np.asarray(mesh.sigma))


def _te_rows(mesh, rxLoc, exTE, iF, freq):
    ny = len(mesh.yLen)
    rx = _rx_sens(mesh, rxLoc)
    zid = rx.zid
    Ex01 = np.stack([exTE[zid * (ny + 1):(zid + 1) * (ny + 1), iF], exTE[(zid + 1) * (ny + 1):(zid + 2) * (ny + 1), iF]], axis=1)
    return tipperFuncSensTE(2 * np.pi * freq, rx, Ex01)


def rxTipper(exTE, mesh, rxLoc, freqs):
    """T [nFreq, nRx] from the TE node fields [nNode, nFreq]."""
    return np.array([_te_rows(mesh, rxLoc, exTE, iF, f)[0] for iF, f in enumerate(freqs)])


def _full_impedance(data, comps):
    nF, nRx, nC = len(data.freqs), data.rxLoc.shape[0], len(comps)
    f, r, c = np.meshgrid(np.arange(1, nF + 1), np.arange(1, nRx + 1), np.arange(1, nC + 1), indexing="ij")
    return ofio.MTData(data.rxLoc, data.freqs, "Impedance", comps, r.ravel(), f.ravel(), c.ravel(), np.ones(f.size, dtype=bool),
                       "ZXY" in comps, "ZYX" in comps)


def _impedance_comps(data):
    return [c for c in ("ZXY", "ZYX") if c in data.dataComp or (c == "ZXY" and "TZY" in data.dataComp)]


def MT2DFwdSolver(mesh, data, factor_fn=ofwd.default_factor):
    """The oracle's forward for the impedances of the survey's modes, and T from its TE fields; rows (freq, rx, comp), dataID-masked."""
    comps = _impedance_comps(data)
    pz, fwd = ofwd.MT2DFwdSolver(mesh, _full_impedance(data, comps), factor_fn)
    nF, nRx = len(data.freqs), data.rxLoc.shape[0]
    pz = pz.reshape(nF, nRx, len(comps))
    T = rxTipper(fwd.exTE, mesh, data.rxLoc, data.freqs) if "TZY" in data.dataComp else None
    out = np.stack([T if c == "TZY" else pz[:, :, comps.index(c)] for c in data.dataComp], axis=2)
    return out.reshape(-1)[np.asarray(data.dataID, dtype=bool)], fwd


@contextlib.contextmanager
def _patched(module, name, fn):
    saved = getattr(module, name)
    setattr(module, name, fn)
    try:
        yield
    finally:
        setattr(module, name, saved)


def _with_tipper_rows(omega, rx, Ex01):
    """getDataFuncSensTE with the tipper rows stacked below the impedance rows: [L; L_T], [Q; Q_T]."""
    L, Q = _getDataFuncSensTE(omega, rx, Ex01)
    _, LT, QT = tipperFuncSensTE(omega, rx, Ex01)
    return sp.vstack([L, LT], format="csr"), sp.vstack([Q, QT], format="csr")


_getDataFuncSensTE = osens.getDataFuncSensTE


def compJacTMatVec(exTE, hxTM, datVec, mesh, data, activeCell=None, AinvTE=None, AinvTM=None, **kw):
    """real(J^T v) over the active cells: the oracle's compJacTMatVec, with the tipper rows as "ZXY" rows of receiver id nRx + r."""
    if "TZY" not in data.dataComp:
        return osens.compJacTMatVec(exTE, hxTM, datVec, mesh, data, activeCell, AinvTE, AinvTM, **kw)
    nRx = data.rxLoc.shape[0]
    comp = np.array([data.dataComp[d - 1] for d in data.dtID])
    isT = comp == "TZY"
    imp = ofio.MTData(data.rxLoc, data.freqs, "Impedance", ["ZXY", "ZYX"], np.asarray(data.rxID) + nRx * isT, data.freqID,
                      np.where(comp == "ZYX", 2, 1).astype(np.int64), np.ones(len(comp), dtype=bool), True, "ZYX" in data.dataComp)
    with _patched(osens, "getDataFuncSensTE", _with_tipper_rows):
        return osens.compJacTMatVec(exTE, hxTM, datVec, mesh, imp, activeCell, AinvTE, AinvTM, **kw)


def compJacMat(exTE, hxTM, mesh, data, activeCell, AinvTE, AinvTM):
    """Explicit complex Jacobian (nData x nAC) in the survey's row order: the oracle's compJacMat for the impedance rows, and again
    with L_T, Q_T as the TE receiver functional for the tipper rows."""
    comps = _impedance_comps(data)
    nF, nRx = len(data.freqs), data.rxLoc.shape[0]
    JZ = ojac.compJacMat(exTE, hxTM, mesh, _full_impedance(data, comps), activeCell, AinvTE, AinvTM).reshape(nF, nRx, len(comps), -1)
    JT = None
    if "TZY" in data.dataComp:
        with _patched(ojac, "getDataFuncSensTE", lambda omega, rx, Ex01: tipperFuncSensTE(omega, rx, Ex01)[1:]):
            JT = ojac.compJacMat(exTE, hxTM, mesh, _full_impedance(data, ["ZXY"]), activeCell, AinvTE, AinvTM).reshape(nF, nRx, -1)
    J = np.stack([JT if c == "TZY" else JZ[:, :, comps.index(c)] for c in data.dataComp], axis=2)
    return J.reshape(nF * nRx * len(data.dataComp), -1)[np.asarray(data.dataID, dtype=bool)]


@contextlib.contextmanager
def _sampler():
    """The oracle's sampler with this module's forward and J^T v for the duration of a call."""
    with _patched(osamp, "MT2DFwdSolver", MT2DFwdSolver), _patched(osamp, "compJacTMatVec", compJacTMatVec):
        yield


def compDataGradient(mesh, data, inv, prior, **kw):
    with _sampler():
        return osamp.compDataGradient(mesh, data, inv, prior, **kw)


def getHamiltonian(data, mesh, inv, prior, momentum, **kw):
    with _sampler():
        return osamp.getHamiltonian(data, mesh, inv, prior, momentum, **kw)


def proposeLeapfrog(model, momentum, mesh, data, inv, prior, intstep, **kw):
    with _sampler():
        return osamp.proposeLeapfrog(model, momentum, mesh, data, inv, prior, intstep, **kw)


def runHMCSampler(mesh, data, inv, prior, streams, **kw):
    with _sampler():
        return osamp.runHMCSampler(mesh, data, inv, prior, streams, **kw)
