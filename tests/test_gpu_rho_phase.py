"""Apparent resistivity / phase ("Rho_Pha") data on the device against the CPU reference on the same inputs (the oracle
with the Rho_Pha adjoint weights of tests/rho_phase_oracle.py): predictions, misfit and
gradient, J^T v and the explicit Jacobian, leapfrog, Hamiltonian and a short chain, the execution modes, and a Rho_Pha startup
file through the reference-named entry points.  Tolerances as in test_gpu_parity.py."""
import copy
import os
import socket

import numpy as np
import pytest

from tests.helpers import GOLDEN, load_example, tiny_problem, to_oracle, to_product
from tests import rho_phase_oracle as rpo
from tests.rho_phase_helpers import ragged_mask, rho_phase_problem

pytestmark = pytest.mark.gpu
TOL = 1e-9


def _rel(a, b):
    return float(np.abs(np.asarray(a) - np.asarray(b)).max() / np.abs(b).max())


def _oracle_grad(mesh, data, inv, prior, m):
    inv.strModel = m.copy()
    return rpo.compDataGradient(mesh, data, inv, prior)


def _self_sensitivity(mesh, data, inv, prior, m, g0, pred0):
    """Oracle vs oracle with the frequencies moved by one ulp (test_gpu_parity.py)."""
    d2 = copy.copy(data)
    d2.freqs = np.nextafter(data.freqs, np.inf)
    pred1, _, g1 = _oracle_grad(mesh, d2, inv, prior, m)
    return _rel(g1, g0), (np.abs(pred1 - pred0) / np.abs(pred0)).max()


def _gpu(mesh, data, inv, prior, m):
    from hmcmt2d_b200 import api
    pm, pd, pi, pp = to_product(mesh, data, inv, prior)
    pi.strModel = m.copy()
    pred, phi, g = api.compDataGradient(pm, pd, pi, pp)
    return pred, phi, g, (pm, pd, pi, pp)


def test_tiny_parity_ragged_and_single_mode():
    """Both modes with a ragged mask (some slots hold only rho_a or only the phase), then a TE-only and a TM-only survey."""
    mesh, data, inv, prior = tiny_problem(seed=3)
    rng = np.random.default_rng(4)
    for modes, keep in (((0, 1), ragged_mask(data)), ((0,), None), ((1,), None)):
        _, d, rinv, _ = rho_phase_problem(mesh, data, prior, modes, keep)
        m = rinv.strModel + 0.3 * rng.standard_normal(len(rinv.strModel))
        opred, ophi, og = _oracle_grad(mesh, d, rinv, prior, m)
        pred, phi, g, _ = _gpu(mesh, d, rinv, prior, m)
        assert pred.dtype == np.float64 and pred.shape == opred.shape == (len(d.dtID),)
        assert (np.abs(pred - opred) / np.abs(opred)).max() < TOL, modes
        assert abs(phi - ophi) / abs(ophi) < TOL, modes
        assert _rel(g, og) < TOL, modes


@pytest.mark.parametrize("solver", ["mf", "band"])
@pytest.mark.parametrize("name", ["dprism3d", "coprod2"])
def test_example_parity(name, solver, monkeypatch):
    """The example geometries with Rho_Pha observations from the oracle forward plus noise, on both solvers."""
    monkeypatch.setenv("HMCMT_SOLVER", solver)
    mesh, data, inv, prior = load_example(name)
    _, d, rinv, _ = rho_phase_problem(mesh, data, prior)
    rng = np.random.default_rng(1)
    m = np.log(0.01) + 0.7 * rng.standard_normal(len(rinv.strModel))
    opred, ophi, og = _oracle_grad(mesh, d, rinv, prior, m)
    sens_g, sens_p = _self_sensitivity(mesh, d, rinv, prior, m, og, opred)
    pred, phi, g, _ = _gpu(mesh, d, rinv, prior, m)
    assert (np.abs(pred - opred) / np.abs(opred)).max() < max(TOL, 20 * sens_p)
    assert abs(phi - ophi) / abs(ophi) < max(TOL, 20 * sens_p)
    assert _rel(g, og) < max(TOL, 20 * sens_g), (_rel(g, og), sens_g)


def test_cfg2_shape_gradient():
    """The mesh and survey tools/dev/t_rho_phase.py times (200 x 100 cells, 30 frequencies, stress model), the Rho_Pha observations
    converted from the impedance observations of synthetic.make_problem."""
    from hmcmt2d_b200 import api, synthetic
    mesh, data, inv, prior = synthetic.make_problem(200, 100, 30)
    d, rinv = synthetic.rho_phase_problem(data, inv)
    m = synthetic.stress_model(rinv)
    pl = api.Plan(mesh, d, rinv, prior)
    pred, phi, g = pl.forward_gradient(m)
    assert pl.status() == 0
    pl.close()
    om, od, oi, op = to_oracle(mesh, d, rinv, prior)
    opred, ophi, og = _oracle_grad(om, od, oi, op, m)
    sens_g, sens_p = _self_sensitivity(om, od, oi, op, m, og, opred)
    assert (np.abs(pred[0] - opred) / np.abs(opred)).max() < max(TOL, 20 * sens_p)
    assert abs(phi[0] - ophi) / abs(ophi) < max(TOL, 20 * sens_p)
    assert _rel(g[0], og) < max(TOL, 20 * sens_g), (_rel(g[0], og), sens_g)


def test_coprod2_finite_difference_check():
    """Central differences h = 1e-5 in ln(sigma) of the device misfit against the device gradient (as
    test_gpu_parity.py::test_cfg5_finite_difference_check), probe cells in the middle half of the columns, away from the bottom 5
    cell rows and from the side boundaries (where the reference's boundary-derivative approximations live, SURVEY.md A.6)."""
    from hmcmt2d_b200 import api
    mesh, data, inv, prior = load_example("coprod2")
    _, d, rinv, _ = rho_phase_problem(mesh, data, prior)
    pm, pd, pi, pp = to_product(mesh, d, rinv, prior)
    rng = np.random.default_rng(5)
    m = np.log(0.01) + 0.7 * rng.standard_normal(len(rinv.strModel))
    pl = api.Plan(pm, pd, pi, pp)
    _, phi0, g = pl.forward_gradient(m)
    g = g[0]
    ny, nz = mesh.gridSize
    nrows = nz - len(mesh.airLayer)
    assert len(m) == ny * nrows
    h = 1e-5
    worst = 0.0
    for r, c in zip(rng.integers(0, nrows - 5, size=10), rng.integers(ny // 4, 3 * ny // 4, size=10)):
        a = int(r) * ny + int(c)
        mp, mm = m.copy(), m.copy()
        mp[a] += h
        mm[a] -= h
        fd = (pl.forward_gradient(mp)[1][0] - pl.forward_gradient(mm)[1][0]) / (2 * h)
        worst = max(worst, abs(fd - g[a]) / np.abs(g).max())
    assert worst < 1e-4, worst
    pl.close()


def test_jtvec_and_jacobian():
    """Plan.jtvec and Plan.jacobian (real rows d rho_a / d sigma, d phase / d sigma) against the oracle, and J^T v == jtvec(v) on the
    device; the predictions of the plan are intact after the adjoint passes."""
    from hmcmt2d_b200 import api
    from oracle import forward as ofwd
    mesh, data, inv, prior = tiny_problem(seed=19)
    _, d, rinv, _ = rho_phase_problem(mesh, data, prior, keep=ragged_mask(data, seed=5))
    pm, pd, pi, pp = to_product(mesh, d, rinv, prior)
    m = rinv.strModel + 0.2 * np.random.default_rng(20).standard_normal(len(rinv.strModel))
    pl = api.Plan(pm, pd, pi, pp)
    pred, _, _ = pl.forward(m=m, fields=False)
    J = pl.jacobian()[0]
    mesh.sigma = rinv.activeCell @ np.exp(m) + rinv.bgModel
    opred, ofw = ofwd.MT2DFwdSolver(mesh, d)
    oJ = rpo.compJacMat(ofw.exTE, ofw.hxTM, mesh, d, rinv.activeCell, ofw.AinvTE, ofw.AinvTM)
    assert pred.dtype == J.dtype == np.float64 and J.shape == oJ.shape == (len(d.dtID), len(m))
    assert _rel(pred[0], opred) < TOL
    assert _rel(J, oJ) < TOL
    v = np.random.default_rng(2).standard_normal(len(d.dtID))
    g = pl.jtvec(v)[0]
    og = rpo.compJacTMatVec(ofw.exTE, ofw.hxTM, v, mesh, d, rinv.activeCell, ofw.AinvTE, ofw.AinvTM)
    assert _rel(g, og) < TOL
    assert _rel(J.T @ v, g) < 1e-11
    pred2, _, _ = pl.forward(m=m, fields=False)
    assert np.array_equal(pred2, pred)
    pl.close()


def test_leapfrog_and_hamiltonian():
    from hmcmt2d_b200 import api
    from oracle import sampler as osamp
    mesh, data, inv, prior = tiny_problem(seed=21)
    _, d, rinv, _ = rho_phase_problem(mesh, data, prior)
    pm, pd, pi, pp = to_product(mesh, d, rinv, prior)
    rng = np.random.default_rng(22)
    m0 = rinv.strModel + 0.2 * rng.standard_normal(len(rinv.strModel))
    p0 = np.clip(rng.standard_normal(len(m0)), -2.5, 2.5)
    om, op = rpo.proposeLeapfrog(m0.copy(), p0.copy(), mesh, d, rinv, prior, 3)
    gm, gp = api.proposeLeapfrog(api.HMCParameter(len(m0), m0.copy(), p0.copy()), pm, pd, pi, pp, intstep=3)
    assert np.abs(gm - om).max() < 1e-9 * max(1.0, np.abs(om).max())
    assert np.abs(gp - op).max() < 1e-8 * max(1.0, np.abs(op).max())
    od, ok, oh, omn, opred = osamp.getHamiltonian(d, mesh, rinv, prior, op)
    gd, gk, gh, gmn, gpred = api.getHamiltonian(pd, pm, pi, pp, api.HMCParameter(len(m0), gm, gp))
    assert abs(gd - od) / od < 1e-8 and abs(gk - ok) / ok < 1e-8 and abs(gh - oh) / abs(oh) < 1e-8
    assert gpred.dtype == np.float64 and _rel(gpred, opred) < 1e-8


def test_short_chain_parity():
    """runHMCSampler with injected draws, 5 samples: accept flags, models, statistics and the real hmcdata."""
    from hmcmt2d_b200 import api
    from oracle import sampler as osamp
    mesh, data, inv, prior = tiny_problem(seed=31)
    prior.dt = 0.02
    _, d, rinv, _ = rho_phase_problem(mesh, data, prior)
    ns, n = 5, len(rinv.strModel)
    st = osamp.make_streams(7, n, ns, prior.timestep)
    pm, pd, pi, pp = to_product(mesh, d, rinv, prior)
    omodel, ostats, odata = rpo.runHMCSampler(mesh, d, copy.copy(rinv), prior, st, nsamples=ns)
    gs = api.RandomStreams(st.u_start, st.z_init, st.intsteps, st.u_accept, st.z_momentum)
    gmodel, gstat, gdata = api.runHMCSampler(pm, pd, pi, pp, gs, nsamples=ns)
    assert gdata.dtype == np.float64 and gdata.shape == odata.shape == (len(d.dtID), ns + 1)
    assert np.array_equal(gstat.acceptstats, ostats["acceptstats"])
    assert np.abs(gmodel - omodel).max() < 1e-7
    assert _rel(gstat.hmstats, ostats["hmstats"]) < 1e-7
    assert _rel(gdata, odata.real) < 1e-7 and not np.iscomplexobj(gdata)


def test_execution_modes_are_bit_identical(monkeypatch):
    """A Rho_Pha plan goes through the captured graph like an impedance plan: one stream vs groups of systems, eager launches vs
    graph replay, device-resident leapfrog steps and host-buffer evaluations give the same bits; so do 3 batched chains and 3
    single-chain plans."""
    from hmcmt2d_b200 import api, synthetic
    mesh, data, inv, prior = synthetic.make_problem(70, 50, 4, nRx=9)
    d, rinv = synthetic.rho_phase_problem(data, inv)
    m0 = synthetic.stress_model(rinv)
    p0 = np.clip(np.random.default_rng(0).standard_normal(len(m0)), -2.5, 2.5)
    results = []
    for groups, graph in [("3", "1"), ("1", "1"), ("3", "0")]:
        monkeypatch.setenv("HMCMT_SOLVER", "mf")
        monkeypatch.setenv("HMCMT_GROUPS", groups)
        monkeypatch.setenv("HMCMT_GRAPH", graph)
        pl = api.Plan(mesh, d, rinv, prior)
        assert pl.info(11) == 1
        pl.set_state(m0, p0, m0)
        pl.leapfrog_steps_device(prior.dt, 4)
        assert pl.status() == 0
        m, p = pl.get_state()
        outs = [pl.forward_gradient(m0) for _ in range(3)]          # eager, captured, replayed
        for o in outs[1:]:
            assert all(np.array_equal(a, b) for a, b in zip(o, outs[0]))
        assert outs[0][0].dtype == np.float64
        results.append((m.copy(), p.copy()) + tuple(np.array(a) for a in outs[0]))
        pl.close()
    for r in results[1:]:
        assert all(np.array_equal(a, b) for a, b in zip(r, results[0]))
    monkeypatch.delenv("HMCMT_GROUPS")
    monkeypatch.delenv("HMCMT_GRAPH")
    ms = m0[None, :] + 0.3 * np.random.default_rng(13).standard_normal((3, len(m0)))
    pl3 = api.Plan(mesh, d, rinv, prior, nChains=3)
    pred3, phi3, g3 = pl3.forward_gradient(ms)
    pl3.close()
    pl1 = api.Plan(mesh, d, rinv, prior, nChains=1)
    for c in range(3):
        pred, phi, g = pl1.forward_gradient(ms[c])
        assert np.array_equal(pred[0], pred3[c]) and phi[0] == phi3[c] and np.array_equal(g[0], g3[c])
    pl1.close()


def test_startup_file_through_the_sampler(tmp_path):
    """A Rho_Pha startup file (the coprod2 example with its data rewritten as apparent resistivity / phase) through readstartupFile,
    runHMCSampler, outputHMCSamples and parallelHMCSampler."""
    import shutil
    from hmcmt2d_b200 import api, fileio, synthetic
    src = os.path.join(GOLDEN, "coprod2")
    data, obs, err = fileio.readMT2DData(os.path.join(src, "coprod2data.dat"))
    inv = api.InvDataModel(obs, 1.0 / np.abs(err), None, None, None, None, None, np.abs(err))
    d, rinv = synthetic.rho_phase_problem(data, inv)
    fileio.writeMT2DData(str(tmp_path / "coprod2rp.dat"), d, rinv.obsData, rinv.dataErr)
    shutil.copy(os.path.join(src, "coprod2.mod"), tmp_path / "coprod2.mod")
    text = open(os.path.join(src, "startupfile")).read().replace("coprod2data.dat", "coprod2rp.dat")
    (tmp_path / "startupfile").write_text(text)
    mesh, mdata, minv, prior = api.readstartupFile(str(tmp_path / "startupfile"))
    assert mdata.dataType == "Rho_Pha" and mdata.dataComp == d.dataComp and minv.obsData.dtype == np.float64
    model, stats, hmcdata = api.runHMCSampler(mesh, mdata, minv, prior, nsamples=2, seed=3)
    assert model.shape == (len(minv.strModel), 2) and hmcdata.shape == (len(minv.obsData), 3)
    assert np.isfinite(stats.hmstats).all() and np.isfinite(hmcdata).all()
    api.outputHMCSamples(model, stats, hmcdata, outdir=str(tmp_path))
    assert (tmp_path / "hmcsamples_id1.data").read_text().count("\n") == 3
    mesh, mdata, minv, prior = api.readstartupFile(str(tmp_path / "startupfile"))
    out = tmp_path / "parallel"
    out.mkdir()
    models, _, _ = api.parallelHMCSampler(mesh, mdata, minv, prior, [2], nsamples=1, outdir=str(out))
    assert models[0].shape == (len(minv.strModel), 1) and (out / "hmcstatistics_id1.log").exists()


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _shard_worker(rank, world, port, out):
    import torch.distributed as dist
    from hmcmt2d_b200 import api, synthetic
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    mesh, data, inv, prior = synthetic.make_problem(48, 40, 4, nRx=8)
    d, rinv = synthetic.rho_phase_problem(data, inv)
    m = synthetic.stress_model(rinv)
    sp = api.FreqShardedPlan(mesh, d, rinv, prior, rank, world, device=rank)
    pred, phi, g = sp.forward_gradient(m)
    sp.close()
    if rank == 0:
        np.savez(out, pred=pred, phi=phi, g=g)
    dist.barrier()
    dist.destroy_process_group()


def test_freq_sharded_plan_two_devices(tmp_path):
    """FreqShardedPlan over 2 devices (one TE and one TM rank) equals the unsharded evaluation."""
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 visible GPUs")
    from hmcmt2d_b200 import api, synthetic
    out = str(tmp_path / "sharded.npz")
    mp.spawn(_shard_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    r = np.load(out)
    mesh, data, inv, prior = synthetic.make_problem(48, 40, 4, nRx=8)
    d, rinv = synthetic.rho_phase_problem(data, inv)
    m = synthetic.stress_model(rinv)
    pl = api.Plan(mesh, d, rinv, prior)
    pred, phi, g = pl.forward_gradient(m)
    pl.close()
    assert r["pred"].dtype == np.float64 and np.array_equal(r["pred"], pred[0])
    assert abs(float(r["phi"]) - phi[0]) <= 1e-12 * phi[0]
    assert _rel(r["g"], g[0]) < 1e-12
