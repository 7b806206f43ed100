"""Builders for the apparent resistivity / phase ("Rho_Pha") tests: oracle-side surveys over the receivers and frequencies of an
impedance problem, with observations from the oracle forward plus noise."""
import numpy as np

from oracle import fileio as ofio
from oracle import forward as ofwd
from oracle import sampler as osamp

COMPS = ["RhoXY", "PhsXY", "RhoYX", "PhsYX"]


def rho_phase_data(data, modes=(0, 1), keep=None):
    """Oracle MTData of DataType Rho_Pha over the frequencies / receivers of `data`: rows [Rho, Phs] of each mode in `modes`
    per (freq, rx), sorted; `keep` (optional) masks rows out (dataID)."""
    nF, nRx = len(data.freqs), data.rxLoc.shape[0]
    comps = [c for m in modes for c in COMPS[2 * m:2 * m + 2]]
    f, r, c = np.meshgrid(np.arange(1, nF + 1), np.arange(1, nRx + 1), np.arange(1, len(comps) + 1), indexing="ij")
    mask = np.ones(f.size, dtype=bool) if keep is None else np.asarray(keep, dtype=bool)
    return ofio.MTData(np.array(data.rxLoc), np.array(data.freqs), "Rho_Pha", comps, r.ravel()[mask].astype(np.int64),
                       f.ravel()[mask].astype(np.int64), c.ravel()[mask].astype(np.int64), mask.copy(), 0 in modes, 1 in modes)


def rho_phase_obs(pred, data, seed=7, rho_err=0.05, phase_err=1.5):
    """Noisy observations of `pred`: errors rho_err x rho_a and an absolute phase_err degrees."""
    rng = np.random.default_rng(seed)
    phs = np.array([data.dataComp[d - 1].startswith("Phs") for d in data.dtID])
    err = np.where(phs, phase_err, rho_err * np.abs(pred))
    return pred + err * rng.standard_normal(len(pred)), err


def rho_phase_problem(mesh, data, prior, modes=(0, 1), keep=None, seed=7):
    """Oracle (mesh, Rho_Pha data, inv, prior): observations from the oracle forward at mesh.sigma plus noise."""
    d = rho_phase_data(data, modes, keep)
    pred, _ = ofwd.MT2DFwdSolver(mesh, d)
    obs, err = rho_phase_obs(pred, d, seed)
    return mesh, d, osamp.setupInverseDataModel(mesh, [1e-8], obs, err), prior


def ragged_mask(data, seed=3, drop=0.3):
    """Keep-mask over the full Rho_Pha rows of `data` (both modes) with some slots holding only rho_a or only phase."""
    nF, nRx = len(data.freqs), data.rxLoc.shape[0]
    keep = np.random.default_rng(seed).random(nF * nRx * 4) > drop
    keep[:4] = [True, False, False, True]          # slot (f0, rx0, TE): rho only; (f0, rx0, TM): phase only
    return keep
