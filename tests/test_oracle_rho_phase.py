"""Apparent resistivity / phase ("Rho_Pha") data on the CPU: the CPU reference's J^T v (tests/rho_phase_oracle.py, built
on the oracle) against its chain-rule Jacobian and against central differences of its misfit, and the sharding of a Rho_Pha survey over ranks (world-size-2 gloo group with a
stub plan, as test_freqshard_gloo.py)."""
import os
import socket

import numpy as np
import torch.distributed as dist
import torch.multiprocessing as mp

from hmcmt2d_b200 import api, synthetic
from tests.helpers import tiny_problem, to_oracle
from tests import rho_phase_oracle as rpo
from tests.rho_phase_helpers import ragged_mask, rho_phase_problem


def _fields(mesh, data):
    from oracle import forward as ofwd
    return ofwd.MT2DFwdSolver(mesh, data)


def test_oracle_jtvec_equals_chain_rule_jacobian():
    """Two derivations of the same quantity: J^T v through the per-slot adjoint weight V on the oracle's impedance J^T v, and the explicit
    real rows (2/(omega mu0)) Re(conj(Z) J_Z), (180/pi) Im(J_Z/Z) on the oracle's impedance Jacobian (tests/rho_phase_oracle.py); both modes with a ragged mask, and one mode."""
    mesh, data, inv, prior = tiny_problem(seed=4)
    rng = np.random.default_rng(5)
    for modes, keep in (((0, 1), ragged_mask(data)), ((0,), None), ((1,), None)):
        _, d, oinv, _ = rho_phase_problem(mesh, data, prior, modes, keep)
        pred, fwd = _fields(mesh, d)
        assert pred.dtype == np.float64
        J = rpo.compJacMat(fwd.exTE, fwd.hxTM, mesh, d, oinv.activeCell, fwd.AinvTE, fwd.AinvTM)
        assert J.shape == (len(pred), oinv.activeCell.shape[1]) and J.dtype == np.float64
        v = rng.standard_normal(len(pred))
        g = rpo.compJacTMatVec(fwd.exTE, fwd.hxTM, v, mesh, d, oinv.activeCell, fwd.AinvTE, fwd.AinvTM)
        assert np.abs(g - J.T @ v).max() <= 1e-12 * np.abs(g).max(), modes


def test_oracle_gradient_central_differences():
    """Central differences h = 1e-5 in ln(sigma) of the oracle's Rho_Pha misfit against its adjoint gradient on 10 probe cells of
    the survey's core columns, away from the bottom 5 cell rows.  The reference's boundary-derivative approximations (SURVEY.md
    A.6) live in the bottom rows and in the padding columns next to the side boundaries: there the impedance misfit of the same
    problem misses its central differences by up to ~1e-3 of max|g| as well, independently of h."""
    mesh, data, inv, prior = synthetic.make_problem(24, 20, 3, nRx=4)
    om, od, oinv, op = to_oracle(mesh, data, inv, prior)
    om.sigma = synthetic.true_model(mesh)
    _, d, rinv, _ = rho_phase_problem(om, od, op)
    rng = np.random.default_rng(5)
    m = np.log(0.01) + 0.5 * rng.standard_normal(len(rinv.strModel))
    rinv.strModel = m.copy()
    _, phi0, g = rpo.compDataGradient(om, d, rinv, op)
    assert phi0 > 0
    ny, nz = mesh.gridSize
    nrows = nz - len(mesh.airLayer)
    assert nrows == 13 and len(m) == ny * nrows
    h = 1e-5
    worst = 0.0
    npad = 8                                             # synthetic.make_mesh: 8 padding columns on each side
    for r, c in zip(rng.integers(0, nrows - 5, size=10), rng.integers(npad + 1, ny - npad - 1, size=10)):
        a = int(r) * ny + int(c)
        phis = []
        for s in (h, -h):
            rinv.strModel = m.copy()
            rinv.strModel[a] += s
            phis.append(rpo.compDataGradient(om, d, rinv, op)[1])
        worst = max(worst, abs((phis[0] - phis[1]) / (2 * h) - g[a]) / np.abs(g).max())
    assert worst <= 1e-5, worst


def _rho_phase_survey(nF=6):
    mesh, data, inv, prior = synthetic.make_problem(24, 20, nF, nRx=3)
    d, rinv = synthetic.rho_phase_problem(data, inv)
    return mesh, d, rinv, prior


def test_rho_phase_conversion():
    mesh, data, inv, prior = synthetic.make_problem(24, 20, 2, nRx=3)
    d, rinv = synthetic.rho_phase_problem(data, inv)
    assert d.dataType == "Rho_Pha" and d.dataComp == ["RhoXY", "PhsXY", "RhoYX", "PhsYX"] and len(d.dtID) == 2 * len(data.dtID)
    z = inv.obsData
    om = 2 * np.pi * data.freqs[data.freqID - 1]
    assert np.allclose(rinv.obsData[0::2], np.abs(z) ** 2 / (om * 4e-7 * np.pi), rtol=1e-14, atol=0)
    assert np.allclose(rinv.obsData[1::2], np.angle(z, deg=True), rtol=1e-14, atol=0)
    assert np.allclose(rinv.dataErr[1::2], 1.5) and np.allclose(rinv.dataErr[0::2], 0.05 * rinv.obsData[0::2])
    assert np.count_nonzero(d.dataID) == len(d.dtID)


def test_rho_phase_system_partition():
    """shard_systems deals the rho / phase rows of a two-mode survey by mode (dtID in {2 mode + 1, 2 mode + 2}); the rows and masks
    of all ranks partition the full data vector, and each rank's rows belong to its mode and frequencies."""
    mesh, data, inv, prior = _rho_phase_survey()
    nF, nRx = len(data.freqs), data.rxLoc.shape[0]
    full_mask = data.dataID.reshape(nF, nRx, 4)
    for shard, worlds in ((api.shard_systems, (2, 4, 6)), (api.shard_frequencies, (1, 2, 3))):
        for world in worlds:
            seen = np.zeros(len(inv.obsData), int)
            mask_seen = np.zeros((nF, nRx, 4), int)
            for rank in range(world):
                sub, sinv, rows = shard(data, inv, rank, world)
                seen[rows] += 1
                assert np.array_equal(sinv.obsData, inv.obsData[rows]) and np.array_equal(sinv.dataW, inv.dataW[rows])
                assert np.array_equal(sub.freqs[sub.freqID - 1], data.freqs[data.freqID[rows] - 1])
                assert [sub.dataComp[k - 1] for k in sub.dtID] == [data.dataComp[k - 1] for k in data.dtID[rows]]
                fidx = np.nonzero(np.isin(data.freqs, sub.freqs))[0]
                cidx = [data.dataComp.index(c) for c in sub.dataComp]
                assert np.count_nonzero(sub.dataID) == len(rows)
                mask_seen[np.ix_(fidx, np.arange(nRx), cidx)] += sub.dataID.reshape(len(fidx), nRx, len(cidx))
                if shard is api.shard_systems:
                    mode = 0 if rank < world // 2 else 1
                    assert np.isin(data.dtID[rows], (2 * mode + 1, 2 * mode + 2)).all()
                    assert sub.dataComp == data.dataComp[2 * mode:2 * mode + 2] and sub.compTE == (mode == 0)
                    assert len(sub.freqs) == nF // (world // 2)
            assert (seen == 1).all() and np.array_equal(mask_seen, full_mask.astype(int))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


class _RealStubPlan:
    """Stands in for api.Plan on a Rho_Pha shard: real predictions, and a misfit / gradient that are sums over the data rows, like
    the real data misfit and its gradient."""

    def __init__(self, mesh, data, inv, prior, nChains=1, device=0):
        self.data, self.inv, self.nAC = data, inv, len(inv.strModel)

    def forward_gradient(self, m):
        d = self.data
        f = d.freqs[d.freqID - 1]
        comp = np.array([{"RhoXY": 1.0, "PhsXY": 2.0, "RhoYX": 3.0, "PhsYX": 4.0}[d.dataComp[k - 1]] for k in d.dtID])
        pred = (f * d.rxID + comp) * np.sum(m)
        r = self.inv.dataW * (pred - self.inv.obsData)
        g = (np.cos(np.outer(f * comp, np.arange(self.nAC))) * (self.inv.dataW * r)[:, None]).sum(axis=0) * m
        return pred[None, :], np.array([0.5 * np.sum(r * r)]), g[None, :]

    def close(self):
        pass


def _worker(rank, world, port):
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    real = api.Plan
    api.Plan = _RealStubPlan
    try:
        mesh, data, inv, prior = _rho_phase_survey(5)
        m = np.linspace(-5.0, -4.0, len(inv.strModel))
        sp = api.FreqShardedPlan(mesh, data, inv, prior, rank, world)            # balanced (frequency, mode) systems
        assert sp.plan.data.dataComp == data.dataComp[2 * rank:2 * rank + 2]
        pred, phi, g = sp.forward_gradient(m)
        fpred, fphi, fg = _RealStubPlan(mesh, data, inv, prior).forward_gradient(m)
        assert pred.dtype == np.float64 and np.allclose(pred, fpred[0], rtol=1e-14, atol=0)
        assert abs(phi - fphi[0]) <= 1e-12 * abs(fphi[0])
        assert np.allclose(g, fg[0], rtol=1e-12, atol=1e-12 * np.abs(fg).max())
    finally:
        api.Plan = real
    dist.barrier()
    dist.destroy_process_group()


def test_rho_phase_system_shards_world2():
    mp.spawn(_worker, args=(2, _free_port()), nprocs=2, join=True)
