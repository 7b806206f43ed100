"""CPU reference for apparent resistivity / phase ("Rho_Pha") data, built on the unchanged oracle (test infrastructure).

The reference's sensitivity code never reaches this data type ("Rho_Phs" in compJacTMatVec.jl:104 vs "Rho_Pha" in its reader
and forward), so the oracle restates impedance only.  This module applies the repository's definition on top of it: for rows
rho_a = |Z|^2/(omega mu0) and phase = atan2(Im Z, Re Z) 180/pi,
    d rho_a = 2/(omega mu0) Re(conj(Z) dZ),     d phase = 180/pi Im(dZ/Z),
so a real vector v over the rows becomes, per (frequency, receiver, mode) slot, the complex weight
    V = v_rho 2/(omega mu0) Z + v_phi 180/pi i Z/|Z|^2
and real(J_Z^T conj(V)) (the oracle's impedance compJacTMatVec) is sum_i v_i d pred_i / d sigma.  The explicit Jacobian takes the
other route: the oracle's impedance rows and the chain rule, a second derivation of the same quantity.  The sampler entry points
run the oracle's own (compDataGradient, proposeLeapfrog, runHMCSampler) with this J^T v in place of the impedance one.
"""
import contextlib

import numpy as np

from oracle import fileio as ofio
from oracle import jacobian as ojac
from oracle import sampler as osamp
from oracle import sensitivity as osens
from oracle.forward import MU0, compFieldsAtRxTE, compFieldsAtRxTM, receiver_row


def _is_rho_phase(data):
    return "Rho_Pha" in data.dataType


def rxImpedance(fields, mesh, rxLoc, freq, isTE):
    """Impedances at the receivers of one (frequency, mode) from the node field of that system, as the forward computes them
    (compFieldsAtRxTE mt2DTE.jl:153-210 / compFieldsAtRxTM mt2DTM.jl:152-210)."""
    yLen, zLen = np.asarray(mesh.yLen), np.asarray(mesh.zLen)
    ny = len(yLen)
    yNode = np.concatenate([[0.0], np.cumsum(yLen)]) - mesh.origin[0]
    zid = receiver_row(mesh, rxLoc)
    F01 = np.stack([fields[zid * (ny + 1):(zid + 1) * (ny + 1)], fields[(zid + 1) * (ny + 1):(zid + 2) * (ny + 1)]], axis=1)
    sigma1 = np.asarray(mesh.sigma)[zid * ny:(zid + 1) * ny]
    num, den = (compFieldsAtRxTE if isTE else compFieldsAtRxTM)(2 * np.pi * freq, rxLoc, yNode, zLen[zid], sigma1, F01)
    return num / den


def _mode_of(comp):
    return 1 if "XY" in comp else 2                      # 1: ZXY (TE), 2: ZYX (TM)


def rhoPhaseAdjointWeights(exTE, hxTM, datVec, mesh, data):
    """Real v over the Rho_Pha rows -> (V, Impedance MTData with one row per (freq, rx, mode) slot that has a row)."""
    datVec = np.asarray(datVec, dtype=np.float64)
    slots = {}
    for i in range(len(datVec)):
        comp = data.dataComp[data.dtID[i] - 1]
        key = (int(data.freqID[i]), int(data.rxID[i]), _mode_of(comp))
        slots.setdefault(key, [0.0, 0.0])[0 if comp.startswith("Rho") else 1] += datVec[i]
    keys = sorted(slots)
    Z = {}
    V = np.zeros(len(keys), dtype=np.complex128)
    for k, (f, r, c) in enumerate(keys):
        if (f, c) not in Z:
            Z[(f, c)] = rxImpedance((exTE if c == 1 else hxTM)[:, f - 1], mesh, data.rxLoc, data.freqs[f - 1], c == 1)
        z = Z[(f, c)][r - 1]
        vr, vp = slots[(f, r, c)]
        V[k] = vr * 2.0 / (2 * np.pi * data.freqs[f - 1] * MU0) * z + vp * 180.0 / np.pi * 1j * z / abs(z) ** 2
    arr = np.asarray(keys, dtype=np.int64).reshape(-1, 3)
    imp = ofio.MTData(data.rxLoc, data.freqs, "Impedance", ["ZXY", "ZYX"], arr[:, 1], arr[:, 0], arr[:, 2],
                      np.ones(len(keys), dtype=bool), data.compTE, data.compTM)
    return V, imp


def compJacTMatVec(exTE, hxTM, datVec, mesh, data, activeCell=None, AinvTE=None, AinvTM=None, **kw):
    """real(J^T v) over the active cells: the oracle's own for Impedance data, through the adjoint weights V for Rho_Pha."""
    if _is_rho_phase(data):
        datVec, data = rhoPhaseAdjointWeights(exTE, hxTM, datVec, mesh, data)
    return osens.compJacTMatVec(exTE, hxTM, datVec, mesh, data, activeCell, AinvTE, AinvTM, **kw)


def compJacMat(exTE, hxTM, mesh, data, activeCell, AinvTE, AinvTM):
    """Explicit real Jacobian (nData x nAC) of Rho_Pha rows: the oracle's impedance rows of every (freq, rx, mode) slot, then
    the chain rule, rows [rho, phase] per slot in (freq, rx, comp) order, masked by dataID."""
    modes = ([1] if data.compTE else []) + ([2] if data.compTM else [])
    nF, nRx, nC = len(data.freqs), data.rxLoc.shape[0], len(modes)
    f, r, c = np.meshgrid(np.arange(1, nF + 1), np.arange(1, nRx + 1), np.arange(1, nC + 1), indexing="ij")
    imp = ofio.MTData(data.rxLoc, data.freqs, "Impedance", ["ZXY", "ZYX"][modes[0] - 1:modes[-1]], r.ravel(), f.ravel(),
                      c.ravel(), np.ones(f.size, dtype=bool), data.compTE, data.compTM)
    JZ = ojac.compJacMat(exTE, hxTM, mesh, imp, activeCell, AinvTE, AinvTM).reshape(nF, nRx, nC, -1)
    rows = np.zeros((nF, nRx, nC, 2, JZ.shape[-1]))
    for iF in range(nF):
        omega = 2 * np.pi * data.freqs[iF]
        for k, mode in enumerate(modes):
            z = rxImpedance((exTE if mode == 1 else hxTM)[:, iF], mesh, data.rxLoc, data.freqs[iF], mode == 1)[:, None]
            dZ = JZ[iF, :, k, :]
            rows[iF, :, k, 0] = 2.0 / (omega * MU0) * np.real(np.conj(z) * dZ)
            rows[iF, :, k, 1] = 180.0 / np.pi * np.imag(dZ / z)
    return rows.reshape(nF * nRx * nC * 2, -1)[np.asarray(data.dataID, dtype=bool)]


@contextlib.contextmanager
def _sampler_jtvec():
    """The oracle's sampler with this module's J^T v (which is the oracle's own for Impedance data) for the duration of a call."""
    saved = osamp.compJacTMatVec
    osamp.compJacTMatVec = compJacTMatVec
    try:
        yield
    finally:
        osamp.compJacTMatVec = saved


def compDataGradient(mesh, data, inv, prior, **kw):
    with _sampler_jtvec():
        return osamp.compDataGradient(mesh, data, inv, prior, **kw)


def proposeLeapfrog(model, momentum, mesh, data, inv, prior, intstep, **kw):
    with _sampler_jtvec():
        return osamp.proposeLeapfrog(model, momentum, mesh, data, inv, prior, intstep, **kw)


def runHMCSampler(mesh, data, inv, prior, streams, **kw):
    with _sampler_jtvec():
        return osamp.runHMCSampler(mesh, data, inv, prior, streams, **kw)
