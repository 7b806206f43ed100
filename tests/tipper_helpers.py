"""Builders for the tipper (TZY) tests: oracle-side surveys over the receivers and frequencies of an impedance problem, with the
tipper observations from the CPU reference's forward plus noise."""
import dataclasses

import numpy as np

from oracle import fileio as ofio
from tests import tipper_oracle as tpo


def survey(data, comps, keep=None):
    """Oracle MTData of DataType Impedance over the frequencies / receivers of `data` with DataComp `comps` (a part of
    [ZXY, ZYX, TZY], in that order), rows (freq, rx, comp); `keep` (optional) masks rows out (dataID)."""
    nF, nRx = len(data.freqs), data.rxLoc.shape[0]
    f, r, c = np.meshgrid(np.arange(1, nF + 1), np.arange(1, nRx + 1), np.arange(1, len(comps) + 1), indexing="ij")
    mask = np.ones(f.size, dtype=bool) if keep is None else np.asarray(keep, dtype=bool)
    return ofio.MTData(np.array(data.rxLoc), np.array(data.freqs), "Impedance", list(comps), r.ravel()[mask].astype(np.int64),
                       f.ravel()[mask].astype(np.int64), c.ravel()[mask].astype(np.int64), mask.copy(),
                       "ZXY" in comps or "TZY" in comps, "ZYX" in comps)


def tipper_problem(mesh, data, inv, seed=7, err=0.02):
    """Oracle (data + TZY rows at every (freq, rx), inv with the merged observations): the impedance rows keep the observations
    and errors of `inv`, the tipper rows are the CPU reference's T at mesh.sigma plus noise, absolute error `err`."""
    nF, nRx, nC = len(data.freqs), data.rxLoc.shape[0], len(data.dataComp)
    keep = np.concatenate([np.asarray(data.dataID, dtype=bool).reshape(nF, nRx, nC), np.ones((nF, nRx, 1), dtype=bool)], axis=2)
    d = survey(data, list(data.dataComp) + ["TZY"], keep.reshape(-1))
    pred, _ = tpo.MT2DFwdSolver(mesh, d)
    isT = d.dtID == nC + 1
    rng = np.random.default_rng(seed)
    obs = np.array(pred)
    obs[~isT] = inv.obsData
    obs[isT] += err * (rng.standard_normal(isT.sum()) + 1j * rng.standard_normal(isT.sum())) / np.sqrt(2)
    errs = np.where(isT, err, 0.0)
    errs[~isT] = 1.0 / np.asarray(inv.dataW)
    return d, dataclasses.replace(inv, obsData=obs, dataW=1.0 / errs)
