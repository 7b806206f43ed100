"""The TE tipper TZY = Hz/Hy on the CPU: known answers of the CPU reference (tests/tipper_oracle.py, built on the oracle) — mirror
antisymmetry and a laterally uniform earth —, its gradient against central differences of its misfit and against the sum of the
impedance and tipper parts, J^T v against its explicit Jacobian, and the sharding of a ZXY / ZYX / TZY survey over ranks
(world-size-2 gloo group with a stub plan, as test_freqshard_gloo.py)."""
import os
import socket

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

from hmcmt2d_b200 import api, synthetic
from tests.helpers import tiny_problem, to_oracle
from tests import tipper_oracle as tpo
from tests.tipper_helpers import survey, tipper_problem


def _mirror_problem(sigma):
    """synthetic.make_mesh(150, 20) (mirror-symmetric about the core centre y0, as true_model is at this width), 3 frequencies,
    receivers at y0 -/+ a, none on a node or a cell centre."""
    mesh, data, inv, prior = synthetic.make_problem(150, 20, 3, nRx=4)
    om, od, _, _ = to_oracle(mesh, data, inv, prior)
    om.sigma = sigma(mesh)
    y0 = 0.5 * (150 - 16) * 200.0
    a = np.array([30.0, 170.0, 290.0, 530.0])
    rx = np.stack([np.concatenate([y0 - a, y0 + a]), np.zeros(2 * len(a))], axis=1)
    od.rxLoc = rx
    d = survey(od, ["ZXY", "ZYX", "TZY"])
    pred, _ = tpo.MT2DFwdSolver(om, d)
    return pred.reshape(3, 2 * len(a), 3)


def test_mirror_antisymmetry():
    """A model and receivers symmetric about the core centre: Ex is even in y - y0, so is Hy, and Hz ~ dEx/dy is odd.  Hence
    ZXY(y0 + a) = ZXY(y0 - a) and T(y0 + a) = -T(y0 - a), to round-off."""
    model = synthetic.true_model(synthetic.make_mesh(150, 20)).reshape(20, 150)
    assert np.array_equal(model, model[:, ::-1])
    p = _mirror_problem(synthetic.true_model)
    Z, Zyx, T = p[:, :, 0], p[:, :, 1], p[:, :, 2]
    n = Z.shape[1] // 2
    assert np.abs(T).max() > 1e-3
    assert np.abs(T[:, n:] + T[:, :n]).max() <= 1e-10 * np.abs(T).max()
    assert np.abs(Z[:, n:] - Z[:, :n]).max() <= 1e-10 * np.abs(Z).max()
    assert np.abs(Zyx[:, n:] - Zyx[:, :n]).max() <= 1e-10 * np.abs(Zyx).max()


def test_laterally_uniform_earth():
    """Uniform 100 Ohm m earth: max |T| at the core receivers is 6.4e-6, against 2.6e-2 over the block of true_model.  It is not
    zero because the side boundary values are the analytic 1-D fields, which the finite-difference interior reproduces only to
    its discretisation error; that mismatch is a lateral gradient of Ex that decays through the padding into the core."""
    Tu = _mirror_problem(lambda mesh: np.array(mesh.sigma))[:, :, 2]
    Tb = _mirror_problem(synthetic.true_model)[:, :, 2]
    assert np.abs(Tu).max() < 1e-5
    assert np.abs(Tu).max() < 1e-3 * np.abs(Tb).max()


@pytest.mark.parametrize("comps", [["ZXY", "ZYX", "TZY"], ["ZXY", "TZY"], ["ZYX", "TZY"], ["TZY"]])
def test_jtvec_equals_explicit_jacobian(comps):
    """Two derivations of the same quantity: J^T v with s_T = L_T^T conj(v_T) added to the impedance source before the oracle's
    adjoint solve, and the oracle's forward-sensitivity Jacobian with L_T, Q_T as the receiver functional; ragged mask."""
    mesh, data, inv, prior = tiny_problem(seed=4)
    keep = np.random.default_rng(1).random(len(data.freqs) * data.rxLoc.shape[0] * len(comps)) > 0.3
    d = survey(data, comps, keep)
    pred, fwd = tpo.MT2DFwdSolver(mesh, d)
    J = tpo.compJacMat(fwd.exTE, fwd.hxTM, mesh, d, inv.activeCell, fwd.AinvTE, fwd.AinvTM)
    assert J.shape == (len(pred), inv.activeCell.shape[1]) == (np.count_nonzero(keep), inv.activeCell.shape[1])
    rng = np.random.default_rng(2)
    v = rng.standard_normal(len(pred)) + 1j * rng.standard_normal(len(pred))
    g = tpo.compJacTMatVec(fwd.exTE, fwd.hxTM, v, mesh, d, inv.activeCell, fwd.AinvTE, fwd.AinvTM)
    assert np.abs(g - np.real(J.T @ np.conj(v))).max() <= 1e-12 * np.abs(g).max()


def test_gradient_central_differences():
    """Central differences h = 1e-5 in ln(sigma) of the misfit of a ZXY / ZYX / TZY survey against its adjoint gradient on 10
    probe cells of the core columns, away from the bottom 5 cell rows (where the reference's boundary-derivative approximations,
    SURVEY.md A.6, live), to 1e-5 of max|g|, the bound the impedance gradient meets there."""
    mesh, data, inv, prior = synthetic.make_problem(24, 20, 3, nRx=4)
    om, od, oinv, op = to_oracle(mesh, data, inv, prior)
    om.sigma = synthetic.true_model(mesh)
    d, tinv = tipper_problem(om, od, oinv)
    rng = np.random.default_rng(5)
    m = np.log(0.01) + 0.5 * rng.standard_normal(len(tinv.strModel))
    tinv.strModel = m.copy()
    _, phi0, g = tpo.compDataGradient(om, d, tinv, op)
    assert phi0 > 0
    ny, nz = mesh.gridSize
    nrows = nz - len(mesh.airLayer)
    h = 1e-5
    worst = 0.0
    npad = 8
    for r, c in zip(rng.integers(0, nrows - 5, size=10), rng.integers(npad + 1, ny - npad - 1, size=10)):
        a = int(r) * ny + int(c)
        phis = []
        for s in (h, -h):
            tinv.strModel = m.copy()
            tinv.strModel[a] += s
            phis.append(tpo.compDataGradient(om, d, tinv, op)[1])
        worst = max(worst, abs((phis[0] - phis[1]) / (2 * h) - g[a]) / np.abs(g).max())
    assert worst <= 1e-5, worst


def test_joint_gradient_is_the_sum_of_its_parts():
    """With identical impedance rows, the misfit and gradient of the Z + T survey are those of the Z-only survey plus those of the
    T-only survey."""
    mesh, data, inv, prior = tiny_problem(seed=6)
    d, tinv = tipper_problem(mesh, data, inv)
    comp = np.array([d.dataComp[k - 1] for k in d.dtID])
    m = tinv.strModel + 0.3 * np.random.default_rng(7).standard_normal(len(tinv.strModel))
    parts = []
    for sel, comps in ((comp != "TZY", ["ZXY", "ZYX"]), (comp == "TZY", ["TZY"])):
        sd = survey(data, comps, d.dataID.reshape(3, 4, 3)[:, :, [d.dataComp.index(c) for c in comps]].reshape(-1))
        si = type(tinv)(tinv.obsData[sel], tinv.dataW[sel], m.copy(), m.copy(), tinv.activeCell, tinv.bgModel, tinv.Wm)
        parts.append(tpo.compDataGradient(mesh, sd, si, prior))
    tinv.strModel = m.copy()
    pred, phi, g = tpo.compDataGradient(mesh, d, tinv, prior)
    assert np.array_equal(pred[comp != "TZY"], parts[0][0]) and np.array_equal(pred[comp == "TZY"], parts[1][0])
    assert abs(phi - parts[0][1] - parts[1][1]) <= 1e-12 * phi
    assert np.abs(g - parts[0][2] - parts[1][2]).max() <= 1e-12 * np.abs(g).max()


def _tipper_survey(nF=6):
    mesh, data, inv, prior = synthetic.make_problem(24, 20, nF, nRx=3)
    nRx = data.rxLoc.shape[0]
    t = 0.01 * (np.arange(nF * nRx) + 1j)
    d, tinv = synthetic.tipper_problem(data, inv, t)
    return mesh, d, tinv, prior


def test_tipper_rows_merge():
    mesh, data, inv, prior = synthetic.make_problem(24, 20, 2, nRx=3)
    t = np.arange(6) * (1 + 2j)
    d, tinv = synthetic.tipper_problem(data, inv, t)
    assert d.dataComp == ["ZXY", "ZYX", "TZY"] and d.compTE and d.compTM
    assert np.array_equal(d.dtID, np.tile([1, 2, 3], 6)) and np.array_equal(d.rxID, np.repeat(np.tile([1, 2, 3], 2), 3))
    assert np.array_equal(tinv.obsData[2::3], t) and np.array_equal(tinv.obsData[d.dtID != 3], inv.obsData)
    assert np.allclose(tinv.dataErr[2::3], 0.02) and np.allclose(tinv.dataW, 1.0 / tinv.dataErr)
    assert np.count_nonzero(d.dataID) == len(d.dtID)
    with pytest.raises(ValueError):
        synthetic.tipper_problem(d, tinv, t)


def test_tipper_system_partition():
    """shard_systems deals a ZXY / ZYX / TZY survey by system: the TE ranks take the ZXY and TZY rows, the TM ranks the ZYX rows;
    the rows and masks of all ranks partition the full data vector."""
    mesh, data, inv, prior = _tipper_survey()
    nF, nRx = len(data.freqs), data.rxLoc.shape[0]
    full_mask = data.dataID.reshape(nF, nRx, 3)
    for shard, worlds in ((api.shard_systems, (2, 4, 6)), (api.shard_frequencies, (1, 2, 3))):
        for world in worlds:
            seen = np.zeros(len(inv.obsData), int)
            mask_seen = np.zeros((nF, nRx, 3), int)
            for rank in range(world):
                sub, sinv, rows = shard(data, inv, rank, world)
                seen[rows] += 1
                assert np.array_equal(sinv.obsData, inv.obsData[rows]) and np.array_equal(sinv.dataW, inv.dataW[rows])
                assert [sub.dataComp[k - 1] for k in sub.dtID] == [data.dataComp[k - 1] for k in data.dtID[rows]]
                fidx = np.nonzero(np.isin(data.freqs, sub.freqs))[0]
                cidx = [data.dataComp.index(c) for c in sub.dataComp]
                assert np.count_nonzero(sub.dataID) == len(rows)
                mask_seen[np.ix_(fidx, np.arange(nRx), cidx)] += sub.dataID.reshape(len(fidx), nRx, len(cidx))
                if shard is api.shard_systems:
                    te = rank < world // 2
                    assert sub.dataComp == (["ZXY", "TZY"] if te else ["ZYX"]) and sub.compTE == te and sub.compTM == (not te)
                    assert len(sub.freqs) == nF // (world // 2)
            assert (seen == 1).all() and np.array_equal(mask_seen, full_mask.astype(int))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


class _StubPlan:
    """Stands in for api.Plan on a shard: complex predictions, and a misfit / gradient that are sums over the data rows, like the
    real data misfit and its gradient."""

    def __init__(self, mesh, data, inv, prior, nChains=1, device=0):
        self.data, self.inv, self.nAC = data, inv, len(inv.strModel)

    def forward_gradient(self, m):
        d = self.data
        f = d.freqs[d.freqID - 1]
        comp = np.array([{"ZXY": 1.0, "ZYX": 2.0, "TZY": 3.0}[d.dataComp[k - 1]] for k in d.dtID])
        pred = (f * d.rxID + comp) * np.sum(m) * (1 + 0.5j)
        r = self.inv.dataW * (pred - self.inv.obsData)
        g = (np.cos(np.outer(f * comp, np.arange(self.nAC))) * np.abs(self.inv.dataW * r)[:, None]).sum(axis=0) * m
        return pred[None, :], np.array([0.5 * np.sum(np.abs(r) ** 2)]), g[None, :]

    def close(self):
        pass


def _worker(rank, world, port):
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    real = api.Plan
    api.Plan = _StubPlan
    try:
        mesh, data, inv, prior = _tipper_survey(5)
        m = np.linspace(-5.0, -4.0, len(inv.strModel))
        sp = api.FreqShardedPlan(mesh, data, inv, prior, rank, world)            # balanced (frequency, mode) systems
        assert sp.plan.data.dataComp == (["ZXY", "TZY"] if rank == 0 else ["ZYX"])
        pred, phi, g = sp.forward_gradient(m)
        fpred, fphi, fg = _StubPlan(mesh, data, inv, prior).forward_gradient(m)
        assert pred.dtype == np.complex128 and np.allclose(pred, fpred[0], rtol=1e-14, atol=0)
        assert abs(phi - fphi[0]) <= 1e-12 * abs(fphi[0])
        assert np.allclose(g, fg[0], rtol=1e-12, atol=1e-12 * np.abs(fg).max())
    finally:
        api.Plan = real
    dist.barrier()
    dist.destroy_process_group()


def test_tipper_system_shards_world2():
    mp.spawn(_worker, args=(2, _free_port()), nprocs=2, join=True)
