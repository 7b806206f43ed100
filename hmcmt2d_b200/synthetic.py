"""Synthetic problem generator of SURVEY.md section 8(d): mesh pattern copied from the reference's
examples (8 padding cells growing x2 each side of a 200 m core, 7 air layers, 100 m earth layers with the
last 8 growing x2), log-spaced frequencies, receivers on the air/earth interface, 100 Ohm-m background
with a 10 Ohm-m block.  Sizes are totals including padding and air."""
from __future__ import annotations

import dataclasses

import numpy as np

from .api import InvDataModel, setupInverseDataModel
from .fileio import HMCPrior, MTData, TensorMesh2D

AIR = np.array([100.0, 300.0, 1000.0, 3000.0, 1e4, 3e4, 1e5])      # listed bottom-up (dprism2d_G96x49.mod:17-18)


def make_mesh(ny: int, nz: int, core_dy: float = 200.0, earth_dz: float = 100.0, npad: int = 8) -> TensorMesh2D:
    if ny <= 2 * npad or nz <= len(AIR) + npad:
        raise ValueError("mesh too small for the padding / air pattern")
    pad = core_dy * 2.0 ** np.arange(1, npad + 1)
    ylen = np.concatenate([pad[::-1], np.full(ny - 2 * npad, core_dy), pad])
    nearth = nz - len(AIR)
    zearth = np.concatenate([np.full(nearth - npad, earth_dz), earth_dz * 2.0 ** np.arange(1, npad + 1)])
    zlen = np.concatenate([AIR[::-1], zearth])
    origin = np.array([pad.sum(), AIR.sum()])
    sigma = np.concatenate([np.full(ny * len(AIR), 1e-8), np.full(ny * nearth, 0.01)])
    return TensorMesh2D(ylen, zlen, AIR.copy(), (ny, nz), origin, sigma)


def true_model(mesh: TensorMesh2D) -> np.ndarray:
    """100 Ohm-m background with a 10 Ohm-m block (dprism-like)."""
    ny, nz = mesh.gridSize
    nair = len(mesh.airLayer)
    sig = np.asarray(mesh.sigma).copy().reshape(nz, ny)
    j0, j1 = int(ny * 0.42), int(ny * 0.58)
    k0, k1 = nair + max(3, (nz - nair) // 10), nair + max(6, (nz - nair) // 4)
    sig[k0:k1, j0:j1] = 0.1
    return sig.reshape(-1)


def make_survey(mesh: TensorMesh2D, nFreq: int, nRx: int = 40, fmax_exp: float = 2.0, fmin_exp: float = -3.0) -> MTData:
    ny = mesh.gridSize[0]
    npad = 8
    core = mesh.yLen[npad:ny - npad].sum()
    freqs = np.logspace(fmax_exp, fmin_exp, nFreq)
    rx = np.stack([np.linspace(0.0, 0.98 * core, nRx), np.zeros(nRx)], axis=1)
    comps = ["ZXY", "ZYX"]
    f, r, c = np.meshgrid(np.arange(1, nFreq + 1), np.arange(1, nRx + 1), np.arange(1, 3), indexing="ij")
    mask = np.ones(nFreq * nRx * 2, dtype=bool)
    return MTData(rx, freqs, "Impedance", comps, r.reshape(-1).astype(np.int64), f.reshape(-1).astype(np.int64),
                  c.reshape(-1).astype(np.int64), mask, True, True)


def halfspace_data(data: MTData, sigma: float = 0.01, noise: float = 0.05, seed: int = 7):
    """Analytic half-space impedances Z = sqrt(i w mu0 / sigma) (ZXY) and -Z (ZYX) with relative noise —
    a cheap observation set for parity tests and the benchmark (data = f(true)(1+0.05 N), err = 0.05|Z|)."""
    rng = np.random.default_rng(seed)
    mu0 = 4e-7 * np.pi
    om = 2 * np.pi * data.freqs[data.freqID - 1]
    z = np.sqrt(1j * om * mu0 / sigma)
    z = np.where(data.dtID == 1, z, -z)
    obs = z * (1.0 + noise * rng.standard_normal(len(z)))
    return obs, noise * np.abs(z)


def make_problem(ny: int, nz: int, nFreq: int, nRx: int = 40, obs=None, err=None, dt: float = 0.03,
                 timestep=(6, 10), rho_bounds=(1.0, 1e4), beta: float = 1.0, **survey_kw):
    """-> (mtMesh, mtData, invParam, hmcprior) exactly as `readstartupFile` would return them."""
    mesh = make_mesh(ny, nz)
    data = make_survey(mesh, nFreq, nRx, **survey_kw)
    if obs is None:
        obs, err = halfspace_data(data)
    inv = setupInverseDataModel(mesh, [1e-8], 1.0 / rho_bounds[1], 1.0 / rho_bounds[0], obs, err)
    prior = HMCPrior(burninsamples=0, totalsamples=10, sigBounds=[1.0 / rho_bounds[1], 1.0 / rho_bounds[0]], dt=dt,
                     timestep=list(timestep), regParam=beta)
    return mesh, data, inv, prior


def stress_model(inv: InvDataModel, seed: int = 1) -> np.ndarray:
    """Evaluation model for timing: ln sigma = ln 0.01 + 0.7 N(0,1) i.i.d. per earth cell (SURVEY.md 8d)."""
    rng = np.random.default_rng(seed)
    return np.log(0.01) + 0.7 * rng.standard_normal(len(inv.strModel))


def true_model_data(data: MTData, pred_true, noise: float = 0.05, seed: int = 7):
    """Observations of SURVEY.md 8(d): data = forward(true model) (1 + 0.05 N), err = 0.05 |Z|.  `pred_true` is the forward
    response of `true_model(mesh)` in the data ordering, computed by whichever engine the caller runs."""
    rng = np.random.default_rng(seed)
    z = np.asarray(pred_true)
    return z * (1.0 + noise * rng.standard_normal(len(z))), noise * np.abs(z)


def rho_phase_problem(data: MTData, inv: InvDataModel, rho_err: float = 0.05, phase_err: float = 1.5):
    """The same survey as "Rho_Pha" data: every impedance row becomes an apparent resistivity rho_a = |Z|^2/(omega mu0) row and a
    phase atan2(Im Z, Re Z) row in degrees (DataComp RhoXY, PhsXY / RhoYX, PhsYX, the row order of MT2DFwdSolver.jl:191-205),
    converted from the impedance observations; errors rho_err x rho_a and an absolute phase_err degrees.
    -> (MTData, InvDataModel) with the model part of `inv` unchanged."""
    mu0 = 4e-7 * np.pi
    z = np.asarray(inv.obsData, dtype=np.complex128)
    fid, rid, did = (np.asarray(a, dtype=np.int64) for a in (data.freqID, data.rxID, data.dtID))
    rho = np.abs(z) ** 2 / (2 * np.pi * np.asarray(data.freqs)[fid - 1] * mu0)
    obs = np.stack([rho, np.degrees(np.arctan2(z.imag, z.real))], axis=1).reshape(-1)
    err = np.stack([rho_err * rho, np.full(len(z), phase_err)], axis=1).reshape(-1)
    comps = [name + ("XY" if "XY" in c else "YX") for c in data.dataComp for name in ("Rho", "Phs")]
    nF, nRx = len(data.freqs), np.asarray(data.rxLoc).shape[0]
    mask = np.repeat(np.asarray(data.dataID, dtype=bool).reshape(nF, nRx, len(data.dataComp)), 2, axis=2).reshape(-1)
    rp = MTData(np.array(data.rxLoc), np.array(data.freqs), "Rho_Pha", comps, np.repeat(rid, 2), np.repeat(fid, 2),
                np.stack([2 * did - 1, 2 * did], axis=1).reshape(-1), mask, data.compTE, data.compTM)
    return rp, dataclasses.replace(inv, obsData=obs, dataW=1.0 / err, dataErr=err)


def tipper_problem(data: MTData, inv: InvDataModel, tipper_obs, tipper_err: float = 0.02):
    """The impedance survey `data` with tipper rows TZY = Hz/Hy added at every (frequency, receiver): `tipper_obs` [nFreq * nRx]
    complex, frequency-major, and an absolute error `tipper_err` per row (the tipper vanishes over a layered earth, so an error
    relative to |T| would give the rows of laterally uniform ground unbounded weights).  Rows in (freq, rx, comp) order.
    -> (MTData with DataComp + [TZY], InvDataModel with the merged observations) with the model part of `inv` unchanged."""
    if "Impedance" not in data.dataType or "TZY" in data.dataComp:
        raise ValueError("tipper rows are added to an impedance survey without them")
    nF, nRx, nC = len(data.freqs), np.asarray(data.rxLoc).shape[0], len(data.dataComp)
    t = np.asarray(tipper_obs, dtype=np.complex128).reshape(nF * nRx)
    fid = np.concatenate([data.freqID, np.repeat(np.arange(1, nF + 1), nRx)]).astype(np.int64)
    rid = np.concatenate([data.rxID, np.tile(np.arange(1, nRx + 1), nF)]).astype(np.int64)
    did = np.concatenate([data.dtID, np.full(nF * nRx, nC + 1)]).astype(np.int64)
    obs = np.concatenate([np.asarray(inv.obsData, dtype=np.complex128), t])
    err = np.concatenate([1.0 / np.asarray(inv.dataW, dtype=np.float64), np.full(nF * nRx, float(tipper_err))])
    order = np.lexsort((did, rid, fid))
    mask = np.concatenate([np.asarray(data.dataID, dtype=bool).reshape(nF, nRx, nC), np.ones((nF, nRx, 1), dtype=bool)], axis=2)
    td = MTData(np.array(data.rxLoc), np.array(data.freqs), "Impedance", list(data.dataComp) + ["TZY"], rid[order], fid[order],
                did[order], mask.reshape(-1), True, data.compTM)
    return td, dataclasses.replace(inv, obsData=obs[order], dataW=1.0 / err[order], dataErr=err[order])
