"""The TE tipper TZY = Hz/Hy on the device against the CPU reference on the same inputs (the oracle with the tipper rows of
tests/tipper_oracle.py): predictions, misfit and gradient, J^T v and the explicit Jacobian, leapfrog, Hamiltonian and a short
chain, antisymmetry, unchanged impedance predictions, the execution modes, the plan-creation rules and a TZY data file through
the reference-named entry points.  Tolerances as in test_gpu_parity.py."""
import copy
import ctypes as C
import os
import socket

import numpy as np
import pytest

from tests.helpers import GOLDEN, load_example, tiny_problem, to_oracle, to_product
from tests import tipper_oracle as tpo
from tests.tipper_helpers import survey, tipper_problem

pytestmark = pytest.mark.gpu
TOL = 1e-9


def _rel(a, b):
    return float(np.abs(np.asarray(a) - np.asarray(b)).max() / np.abs(b).max())


def _oracle_grad(mesh, data, inv, prior, m):
    inv.strModel = m.copy()
    return tpo.compDataGradient(mesh, data, inv, prior)


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
    return pred, phi, g


def _subset(d, inv, comps):
    """The rows of the survey `d` (+ TZY) with DataComp `comps`, and their observations."""
    comp = np.array([d.dataComp[k - 1] for k in d.dtID])
    sel = np.isin(comp, comps)
    nF, nRx = len(d.freqs), d.rxLoc.shape[0]
    keep = np.asarray(d.dataID, dtype=bool).reshape(nF, nRx, len(d.dataComp))[:, :, [d.dataComp.index(c) for c in comps]]
    sd = survey(d, comps, keep.reshape(-1))
    return sd, type(inv)(inv.obsData[sel], inv.dataW[sel], inv.strModel.copy(), inv.refModel.copy(), inv.activeCell, inv.bgModel,
                         inv.Wm)


@pytest.mark.parametrize("comps", [["ZXY", "ZYX", "TZY"], ["ZXY", "TZY"], ["ZYX", "TZY"], ["TZY"]])
def test_tiny_parity(comps):
    """Every DataComp with a tipper, the full set also with a ragged mask."""
    mesh, data, inv, prior = tiny_problem(seed=3)
    rng = np.random.default_rng(4)
    d, tinv = tipper_problem(mesh, data, inv)
    cases = [_subset(d, tinv, comps)]
    if len(comps) == 3:
        keep = rng.random(len(d.dtID)) > 0.3
        keep[:3] = [True, False, True]                    # (f0, rx0): ZXY and TZY without ZYX
        rd = survey(data, comps, keep)
        cases.append((rd, type(tinv)(tinv.obsData[keep], tinv.dataW[keep], tinv.strModel, tinv.refModel, tinv.activeCell,
                                     tinv.bgModel, tinv.Wm)))
    for sd, si in cases:
        m = si.strModel + 0.3 * rng.standard_normal(len(si.strModel))
        opred, ophi, og = _oracle_grad(mesh, sd, si, prior, m)
        pred, phi, g = _gpu(mesh, sd, si, prior, m)
        assert pred.dtype == np.complex128 and pred.shape == opred.shape == (len(sd.dtID),)
        assert _rel(pred, opred) < TOL, comps
        assert abs(phi - ophi) / abs(ophi) < TOL, comps
        assert _rel(g, og) < TOL, comps


@pytest.mark.parametrize("solver", ["mf", "band"])
@pytest.mark.parametrize("name", ["dprism3d", "coprod2"])
def test_example_parity(name, solver, monkeypatch):
    """The example geometries with their impedance observations and tipper rows from the CPU reference plus noise, both solvers."""
    monkeypatch.setenv("HMCMT_SOLVER", solver)
    mesh, data, inv, prior = load_example(name)
    d, tinv = tipper_problem(mesh, data, inv)
    rng = np.random.default_rng(1)
    m = np.log(0.01) + 0.7 * rng.standard_normal(len(tinv.strModel))
    opred, ophi, og = _oracle_grad(mesh, d, tinv, prior, m)
    sens_g, sens_p = _self_sensitivity(mesh, d, tinv, prior, m, og, opred)
    pred, phi, g = _gpu(mesh, d, tinv, prior, m)
    assert _rel(pred, opred) < max(TOL, 20 * sens_p)
    assert abs(phi - ophi) / abs(ophi) < max(TOL, 20 * sens_p)
    assert _rel(g, og) < max(TOL, 20 * sens_g), (_rel(g, og), sens_g)


def _cfg2_tipper(nF=30, ny=200, nz=100, nRx=40):
    """synthetic.make_problem with tipper rows observed from the device forward of true_model."""
    from hmcmt2d_b200 import api, synthetic
    mesh, data, inv, prior = synthetic.make_problem(ny, nz, nF, nRx=nRx)
    d0, _ = synthetic.tipper_problem(data, inv, np.zeros(nF * data.rxLoc.shape[0]))
    tm = copy.copy(mesh)
    tm.sigma = synthetic.true_model(mesh)
    pred, _ = api.MT2DFwdSolver(tm, d0)
    d, tinv = synthetic.tipper_problem(data, inv, pred[d0.dtID == 3])
    return mesh, data, inv, prior, d, tinv


def test_cfg2_shape_gradient():
    """The mesh and survey tools/dev/t_tipper.py times (200 x 100 cells, 30 frequencies, 40 receivers, stress model)."""
    from hmcmt2d_b200 import api, synthetic
    mesh, _, _, prior, d, tinv = _cfg2_tipper()
    m = synthetic.stress_model(tinv)
    pl = api.Plan(mesh, d, tinv, prior)
    pred, phi, g = pl.forward_gradient(m)
    assert pl.status() == 0
    pl.close()
    om, od, oi, op = to_oracle(mesh, d, tinv, prior)
    opred, ophi, og = _oracle_grad(om, od, oi, op, m)
    sens_g, sens_p = _self_sensitivity(om, od, oi, op, m, og, opred)
    assert _rel(pred[0], opred) < max(TOL, 20 * sens_p)
    assert abs(phi[0] - ophi) / abs(ophi) < max(TOL, 20 * sens_p)
    assert _rel(g[0], og) < max(TOL, 20 * sens_g), (_rel(g[0], og), sens_g)


@pytest.mark.parametrize("solver", ["mf", "band"])
def test_impedance_rows_bit_identical(solver, monkeypatch):
    """Adding TZY rows changes no bit of the ZXY / ZYX predictions of the same model."""
    from hmcmt2d_b200 import api, synthetic
    monkeypatch.setenv("HMCMT_SOLVER", solver)
    mesh, data, inv, prior, d, tinv = _cfg2_tipper(nF=4, ny=40, nz=30, nRx=9)
    m = synthetic.stress_model(tinv)
    pz = api.Plan(mesh, data, inv, prior)
    pt = api.Plan(mesh, d, tinv, prior)
    assert np.array_equal(pz.forward_gradient(m)[0][0], pt.forward_gradient(m)[0][0][d.dtID != 3])
    pt.close()
    pz.close()


def test_jtvec_and_jacobian():
    """Plan.jtvec and Plan.jacobian against the CPU reference, and J^T v == jtvec(v) on the device; the predictions of the plan
    are intact after the adjoint passes."""
    from hmcmt2d_b200 import api
    mesh, data, inv, prior = tiny_problem(seed=19)
    d, tinv = tipper_problem(mesh, data, inv)
    for comps in (["ZXY", "ZYX", "TZY"], ["ZYX", "TZY"], ["TZY"]):
        sd, si = _subset(d, tinv, comps)
        pm, pd, pi, pp = to_product(mesh, sd, si, prior)
        m = si.strModel + 0.2 * np.random.default_rng(20).standard_normal(len(si.strModel))
        pl = api.Plan(pm, pd, pi, pp)
        pred, _, _ = pl.forward(m=m, fields=False)
        J = pl.jacobian()[0]
        mesh.sigma = si.activeCell @ np.exp(m) + si.bgModel
        opred, ofw = tpo.MT2DFwdSolver(mesh, sd)
        oJ = tpo.compJacMat(ofw.exTE, ofw.hxTM, mesh, sd, si.activeCell, ofw.AinvTE, ofw.AinvTM)
        assert J.shape == oJ.shape == (len(sd.dtID), len(m))
        assert _rel(pred[0], opred) < TOL and _rel(J, oJ) < TOL, comps
        rng = np.random.default_rng(2)
        v = rng.standard_normal(len(sd.dtID)) + 1j * rng.standard_normal(len(sd.dtID))
        g = pl.jtvec(v)[0]
        og = tpo.compJacTMatVec(ofw.exTE, ofw.hxTM, v, mesh, sd, si.activeCell, ofw.AinvTE, ofw.AinvTM)
        assert _rel(g, og) < TOL, comps
        assert _rel(np.real(J.T @ np.conj(v)), g) < 1e-11
        pred2, _, _ = pl.forward(m=m, fields=False)
        assert np.array_equal(pred2, pred)
        pl.close()


def test_leapfrog_and_hamiltonian():
    from hmcmt2d_b200 import api
    mesh, data, inv, prior = tiny_problem(seed=21)
    d, tinv = tipper_problem(mesh, data, inv)
    pm, pd, pi, pp = to_product(mesh, d, tinv, prior)
    rng = np.random.default_rng(22)
    m0 = tinv.strModel + 0.2 * rng.standard_normal(len(tinv.strModel))
    p0 = np.clip(rng.standard_normal(len(m0)), -2.5, 2.5)
    om, op = tpo.proposeLeapfrog(m0.copy(), p0.copy(), mesh, d, tinv, prior, 3)
    gm, gp = api.proposeLeapfrog(api.HMCParameter(len(m0), m0.copy(), p0.copy()), pm, pd, pi, pp, intstep=3)
    assert np.abs(gm - om).max() < 1e-9 * max(1.0, np.abs(om).max())
    assert np.abs(gp - op).max() < 1e-8 * max(1.0, np.abs(op).max())
    od, ok, oh, omn, opred = tpo.getHamiltonian(d, mesh, tinv, prior, op)
    gd, gk, gh, gmn, gpred = api.getHamiltonian(pd, pm, pi, pp, api.HMCParameter(len(m0), gm, gp))
    assert abs(gd - od) / od < 1e-8 and abs(gk - ok) / ok < 1e-8 and abs(gh - oh) / abs(oh) < 1e-8
    assert _rel(gpred, opred) < 1e-8


def test_short_chain_parity():
    """runHMCSampler with injected draws, 5 samples: accept flags, models, statistics and hmcdata."""
    from hmcmt2d_b200 import api
    from oracle import sampler as osamp
    mesh, data, inv, prior = tiny_problem(seed=31)
    prior.dt = 0.02
    d, tinv = tipper_problem(mesh, data, inv)
    ns, n = 5, len(tinv.strModel)
    st = osamp.make_streams(7, n, ns, prior.timestep)
    pm, pd, pi, pp = to_product(mesh, d, tinv, prior)
    omodel, ostats, odata = tpo.runHMCSampler(mesh, d, copy.copy(tinv), prior, st, nsamples=ns)
    gs = api.RandomStreams(st.u_start, st.z_init, st.intsteps, st.u_accept, st.z_momentum)
    gmodel, gstat, gdata = api.runHMCSampler(pm, pd, pi, pp, gs, nsamples=ns)
    assert gdata.shape == odata.shape == (len(d.dtID), ns + 1)
    assert np.array_equal(gstat.acceptstats, ostats["acceptstats"])
    assert np.abs(gmodel - omodel).max() < 1e-7
    assert _rel(gstat.hmstats, ostats["hmstats"]) < 1e-7
    assert _rel(gdata, odata) < 1e-7


def test_mirror_antisymmetry_on_the_device():
    """synthetic.make_mesh(150, 20) and true_model are mirror-symmetric about the core centre y0: with receivers at y0 -/+ a the
    device's T is odd and its ZXY even, to round-off (tests/test_oracle_tipper.py on the CPU)."""
    from hmcmt2d_b200 import api, fileio, synthetic
    mesh, data, inv, prior = synthetic.make_problem(150, 20, 3, nRx=4)
    y0 = 0.5 * (150 - 16) * 200.0
    a = np.array([30.0, 170.0, 290.0, 530.0])
    rx = np.stack([np.concatenate([y0 - a, y0 + a]), np.zeros(8)], axis=1)
    d = fileio.MTData(rx, data.freqs, "Impedance", ["ZXY", "ZYX", "TZY"], *[np.asarray(v, dtype=np.int64) for v in (
        np.tile(np.repeat(np.arange(1, 9), 3), 3), np.repeat(np.arange(1, 4), 24), np.tile([1, 2, 3], 24))],
        np.ones(72, dtype=bool), True, True)
    mesh.sigma = synthetic.true_model(mesh)
    pred, _ = api.MT2DFwdSolver(mesh, d)
    p = pred.reshape(3, 8, 3)
    Z, T = p[:, :, 0], p[:, :, 2]
    assert np.abs(T).max() > 1e-3
    assert np.abs(T[:, 4:] + T[:, :4]).max() <= 1e-10 * np.abs(T).max()
    assert np.abs(Z[:, 4:] - Z[:, :4]).max() <= 1e-10 * np.abs(Z).max()


def test_execution_modes_are_bit_identical(monkeypatch):
    """A tipper plan goes through the captured graph like an impedance plan: one stream vs groups of systems, eager launches vs
    graph replay, with and without pruned right-hand sides, device-resident leapfrog steps and host-buffer evaluations give the
    same bits; so do 3 batched chains and 3 single-chain plans."""
    from hmcmt2d_b200 import api, synthetic
    mesh, _, _, prior, d, tinv = _cfg2_tipper(nF=4, ny=70, nz=50, nRx=9)
    m0 = synthetic.stress_model(tinv)
    p0 = np.clip(np.random.default_rng(0).standard_normal(len(m0)), -2.5, 2.5)
    results = []
    for groups, graph, prune in [("3", "1", "1"), ("1", "1", "1"), ("3", "0", "1"), ("3", "1", "0")]:
        monkeypatch.setenv("HMCMT_SOLVER", "mf")
        monkeypatch.setenv("HMCMT_GROUPS", groups)
        monkeypatch.setenv("HMCMT_GRAPH", graph)
        monkeypatch.setenv("HMCMT_MF_PRUNE", prune)
        pl = api.Plan(mesh, d, tinv, prior)
        assert pl.info(11) == 1
        pl.set_state(m0, p0, m0)
        pl.leapfrog_steps_device(prior.dt, 4)
        assert pl.status() == 0
        m, p = pl.get_state()
        outs = [pl.forward_gradient(m0) for _ in range(3)]          # eager, captured, replayed
        for o in outs[1:]:
            assert all(np.array_equal(a, b) for a, b in zip(o, outs[0]))
        results.append((m.copy(), p.copy()) + tuple(np.array(a) for a in outs[0]))
        pl.close()
    for r in results[1:]:
        assert all(np.array_equal(a, b) for a, b in zip(r, results[0]))
    for k in ("HMCMT_GROUPS", "HMCMT_GRAPH", "HMCMT_MF_PRUNE"):
        monkeypatch.delenv(k)
    ms = m0[None, :] + 0.3 * np.random.default_rng(13).standard_normal((3, len(m0)))
    pl3 = api.Plan(mesh, d, tinv, prior, nChains=3)
    pred3, phi3, g3 = pl3.forward_gradient(ms)
    pl3.close()
    pl1 = api.Plan(mesh, d, tinv, prior, nChains=1)
    for c in range(3):
        pred, phi, g = pl1.forward_gradient(ms[c])
        assert np.array_equal(pred[0], pred3[c]) and phi[0] == phi3[c] and np.array_equal(g[0], g3[c])
    pl1.close()


def test_response_toggle_keeps_the_tipper_complex():
    """The response toggle of a plan with a tipper gives (rho_a, phase) on the impedance slots and (Re T, Im T) on the tipper
    slots."""
    from hmcmt2d_b200 import api, lib, synthetic
    mesh, data, inv, prior, d, tinv = _cfg2_tipper(nF=3, ny=40, nz=30, nRx=5)
    pl = api.Plan(mesh, d, tinv, prior)
    m = synthetic.stress_model(tinv)
    pred, _, _ = pl.forward(m=m, fields=False)
    lib.check(pl.L.hmcmt_set_response_kind(pl.h, 1), "hmcmt_set_response_kind")
    pl.forward(m=m, fields=False)
    out = np.zeros((1, 3, 5, 3, 2))
    lib.check(pl.L.hmcmt_get_responses(pl.h, lib.f64(out)), "hmcmt_get_responses")
    z = pred[0].reshape(3, 5, 3)
    assert np.array_equal(out[0, :, :, 2, 0] + 1j * out[0, :, :, 2, 1], z[:, :, 2])
    om = 2 * np.pi * d.freqs[:, None]
    assert np.allclose(out[0, :, :, 0, 0], np.abs(z[:, :, 0]) ** 2 / (om * 4e-7 * np.pi), rtol=1e-12, atol=0)
    pl.close()


def _problem_struct(comp_modes):
    """A valid hmcmt_problem of the tiny problem with compMode `comp_modes` (one row per component), arrays kept alive."""
    from hmcmt2d_b200 import lib
    mesh, data, inv, prior = tiny_problem(seed=3)
    pm, pd, pi, pp = to_product(mesh, data, inv, prior)
    n = len(comp_modes)
    keep = dict(yLen=np.array(pm.yLen), zLen=np.array(pm.zLen), freqs=np.array(pd.freqs), rx=np.ascontiguousarray(pd.rxLoc),
                comp=np.array(comp_modes, dtype=np.int32), fid=np.ones(n, dtype=np.int64), rid=np.ones(n, dtype=np.int64),
                did=np.arange(1, n + 1, dtype=np.int64), obs=np.ones(2 * n), err=np.ones(n),
                act=np.asarray(pi.activeCell.tocsc().indices, dtype=np.int32), bg=np.array(pi.bgModel))
    Wm = pi.Wm.tocsr()
    keep.update(wp=Wm.indptr.astype(np.int32), wi=Wm.indices.astype(np.int32), wv=Wm.data.astype(np.float64))
    pr = lib.Problem()
    pr.ny, pr.nz = pm.gridSize
    pr.yLen, pr.zLen = lib.f64(keep["yLen"]), lib.f64(keep["zLen"])
    pr.origin[0], pr.origin[1] = float(pm.origin[0]), float(pm.origin[1])
    pr.nFreq, pr.freqs = len(keep["freqs"]), lib.f64(keep["freqs"])
    pr.nRx, pr.rxLoc = keep["rx"].shape[0], lib.f64(keep["rx"])
    pr.nComp, pr.compMode = n, lib.i32(keep["comp"])
    pr.nData, pr.freqID, pr.rxID, pr.dtID = n, lib.i64(keep["fid"]), lib.i64(keep["rid"]), lib.i64(keep["did"])
    pr.obsData, pr.dataErr = lib.f64(keep["obs"]), lib.f64(keep["err"])
    pr.nAC, pr.activeIdx, pr.bgModel = len(keep["act"]), lib.i32(keep["act"]), lib.f64(keep["bg"])
    pr.wmRowPtr, pr.wmColIdx, pr.wmVal = lib.i32(keep["wp"]), lib.i32(keep["wi"]), lib.f64(keep["wv"])
    pr.regParam, pr.sigBounds[0], pr.sigBounds[1] = 1.0, 1e-4, 1.0
    pr.nChains, pr.device = 1, 0
    return pr, keep


def test_plan_creation_rules():
    """compMode 2 (TZY): at most once and last, after at most two impedance components, impedance plans only (-3 otherwise)."""
    from hmcmt2d_b200 import lib
    L = lib.load()
    for modes, want in (([0, 1, 2], 0), ([0, 2], 0), ([1, 2], 0), ([2], 0), ([0, 1], 0), ([1], 0),
                        ([2, 0], -3), ([0, 2, 1], -3), ([2, 2], -3), ([0, 1, 2, 2], -3), ([1, 1, 2], -3)):
        pr, keep = _problem_struct(modes)
        h = C.c_void_p()
        rc = L.hmcmt_plan_create(C.byref(pr), C.byref(h))
        assert rc == want, (modes, rc)
        if rc == 0:
            L.hmcmt_destroy(h)
    pr, keep = _problem_struct([0, 2])
    keep["did"][:] = [1, 2]
    keep["obs"] = np.ones(2)
    pr.obsData = lib.f64(keep["obs"])
    h = C.c_void_p()
    assert L.hmcmt_plan_create_rho_phase(C.byref(pr), C.byref(h)) == -3


def test_startup_file_through_the_sampler(tmp_path):
    """A TZY data file (the coprod2 example with tipper rows from the CPU reference added) through readstartupFile, runHMCSampler,
    outputHMCSamples and parallelHMCSampler."""
    import shutil
    from hmcmt2d_b200 import api, fileio
    src = os.path.join(GOLDEN, "coprod2")
    mesh, data, inv, prior = load_example("coprod2")
    d, tinv = tipper_problem(mesh, data, inv)
    fileio.writeMT2DData(str(tmp_path / "coprod2t.dat"), d, tinv.obsData, 1.0 / tinv.dataW)
    shutil.copy(os.path.join(src, "coprod2.mod"), tmp_path / "coprod2.mod")
    text = open(os.path.join(src, "startupfile")).read().replace("coprod2data.dat", "coprod2t.dat")
    (tmp_path / "startupfile").write_text(text)
    pmesh, mdata, minv, pprior = api.readstartupFile(str(tmp_path / "startupfile"))
    assert mdata.dataComp == ["ZXY", "ZYX", "TZY"] and mdata.compTE and mdata.compTM
    model, stats, hmcdata = api.runHMCSampler(pmesh, mdata, minv, pprior, nsamples=2, seed=3)
    assert model.shape == (len(minv.strModel), 2) and hmcdata.shape == (len(minv.obsData), 3)
    assert np.isfinite(stats.hmstats).all() and np.isfinite(hmcdata).all()
    api.outputHMCSamples(model, stats, hmcdata, outdir=str(tmp_path))
    assert (tmp_path / "hmcsamples_id1.data").read_text().count("\n") == 3
    pmesh, mdata, minv, pprior = api.readstartupFile(str(tmp_path / "startupfile"))
    out = tmp_path / "parallel"
    out.mkdir()
    models, _, _ = api.parallelHMCSampler(pmesh, mdata, minv, pprior, [2], nsamples=1, outdir=str(out))
    assert models[0].shape == (len(minv.strModel), 1) and (out / "hmcstatistics_id1.log").exists()


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _shard_worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from hmcmt2d_b200 import api, synthetic
    mesh, _, _, prior, d, tinv = _cfg2_tipper(nF=4, ny=48, nz=40, nRx=8)
    m = synthetic.stress_model(tinv)
    sp = api.FreqShardedPlan(mesh, d, tinv, prior, rank, world, device=rank)
    pred, phi, g = sp.forward_gradient(m)
    sp.close()
    if rank == 0:
        np.savez(out, pred=pred, phi=phi, g=g)
    dist.barrier()
    dist.destroy_process_group()


def test_freq_sharded_plan_two_devices(tmp_path):
    """FreqShardedPlan over 2 devices (a ZXY + TZY rank and a ZYX rank) equals the unsharded evaluation."""
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 visible GPUs")
    from hmcmt2d_b200 import api, synthetic
    out = str(tmp_path / "sharded.npz")
    mp.spawn(_shard_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    r = np.load(out)
    mesh, _, _, prior, d, tinv = _cfg2_tipper(nF=4, ny=48, nz=40, nRx=8)
    m = synthetic.stress_model(tinv)
    pl = api.Plan(mesh, d, tinv, prior)
    pred, phi, g = pl.forward_gradient(m)
    pl.close()
    assert np.array_equal(r["pred"], pred[0])
    assert abs(float(r["phi"]) - phi[0]) <= 1e-12 * phi[0]
    assert _rel(r["g"], g[0]) < 1e-12
