"""The device sampler at the shapes where its kernels change behaviour, against the float64 restatement of one step in
tests/hmc_reference.py.  Every dynamic comparison is teacher-forced (one step from a state set on the host), so chaos cannot
accumulate and the bounds are round-off bounds.

Kernel paths, with nAC = ny x (nz - 7 air layers) and drift blocks = clamp(ceil(nAC / 1024), 1, 128):
- nAC 255 (17 x 22) and 261 (29 x 16): one drift block; k_kick / k_clip_momentum / k_bandL_matvec at one and two x-blocks of 256.
- nAC 1023 (31 x 40) and 1025 (25 x 48): one drift block, then two, the second holding one element; k_energies / k_accept with
  1023 and 1025 elements over 1024 threads.
- nAC 4000 (50 x 87): four drift blocks, the last partial; the mass matrix's multifrontal tree has several levels.
- nAC 131 460 (420 x 320): 129 blocks needed, 128 launched, so the grid-stride loops of k_drift_max / k_drift run a second pass.
One step: nChains 1 and 3 at every shape.  Chains, trajectories and the staging ring: nAC 1025, nChains 3 (2 for rho / phase and
tipper plans), 7 samples, staging chunks of 1, 2, 3 and 7 samples (7, 4, 3 and 1 chunks)."""
import math

import numpy as np
import pytest
import scipy.sparse.linalg as spla

from tests import hmc_reference as ref

pytestmark = pytest.mark.gpu

SHAPES = [(17, 22), (29, 16), (31, 40), (25, 48), (50, 87), (420, 320)]
WIDE = (1e-4, 1.0)                      # sigma bounds: ln sigma in [ln 1e-4, 0]
EPS = np.finfo(np.float64).eps


def _problem(ny, nz, bounds=WIDE, nF=1, seed=7):
    """Synthetic mesh, one mode (TE: ZXY), nF low frequencies, 8 receivers, half-space observations."""
    from hmcmt2d_b200 import api, fileio, synthetic
    mesh = synthetic.make_mesh(ny, nz)
    full = synthetic.make_survey(mesh, nF, nRx=8, fmax_exp=-1.0, fmin_exp=-2.0)
    te = np.asarray(full.dtID) == 1
    data = fileio.MTData(np.array(full.rxLoc), np.array(full.freqs), "Impedance", ["ZXY"], np.asarray(full.rxID)[te],
                         np.asarray(full.freqID)[te], np.asarray(full.dtID)[te], np.ones(int(te.sum()), dtype=bool), True, False)
    obs, err = synthetic.halfspace_data(data, seed=seed)
    inv = api.setupInverseDataModel(mesh, [1e-8], bounds[0], bounds[1], obs, err)
    prior = fileio.HMCPrior(burninsamples=0, totalsamples=10, sigBounds=list(bounds), dt=0.05, timestep=[1, 3], regParam=0.8)
    assert len(inv.strModel) == ny * (nz - 7)
    return mesh, data, inv, prior


def _plan(prob, nChains, mass=0):
    from hmcmt2d_b200 import api, lib
    pl = api.Plan(*prob, nChains=nChains)
    lib.check(pl.L.hmcmt_set_mass_matrix(pl.h, mass), "hmcmt_set_mass_matrix")
    return pl


def _blocks(n):
    return max(1, min(128, -(-n // 1024)))


def _start(inv, prior, nChains, rng, margin=0.05):
    lo, hi = math.log(prior.sigBounds[0]), math.log(prior.sigBounds[1])
    m = inv.strModel[None, :] + 0.3 * rng.standard_normal((nChains, len(inv.strModel)))
    return np.clip(m, lo + margin, hi - margin), lo, hi


def _check_step(pl, prior, m0, p0, mref, dt, exact_m=False):
    """One device step from (m0, p0) against the reference drift and a kick with the plan's own gradient at the new model."""
    lo, hi = math.log(prior.sigBounds[0]), math.log(prior.sigBounds[1])
    pl.set_state(m0, p0, mref)
    pl.leapfrog_steps_device(dt, 1)
    assert pl.status() == 0
    gm, gp = pl.get_state()
    _, _, g = pl.forward_gradient(gm, total=True)
    nb_all = []
    for c in range(len(m0)):
        rm, rp, nb, guard = ref.drift(m0[c], p0[c], dt, lo, hi)
        assert not guard
        if exact_m:
            assert np.array_equal(gm[c], rm), c
        assert np.abs(gm[c] - rm).max() <= 1e-14, c
        pd = gp[c] + dt * g[c]                        # the device's momentum after its drift, before the kick
        assert np.array_equal(np.signbit(pd), np.signbit(rp)), c
        assert np.array_equal(np.signbit(pd) != np.signbit(p0[c]), nb % 2 == 1), c
        want = ref.kick(rp, g[c], dt)
        assert np.abs(gp[c] - want).max() <= 1e-12 * np.abs(want).max(), c
        nb_all.append(nb)
    return nb_all


@pytest.mark.parametrize("nChains", [1, 3])
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: f"{s[0]}x{s[1]}")
def test_one_step_teacher_forced(shape, nChains):
    """No clip; a clip whose maximum sits in the last, partial block of chain 1 and in a middle block of chain 2 while chain 0
    is not clipped (chain 0 carries it with one chain); the tie max |dt p| = 3.0, not clipped; bounds 0.4 wide in ln sigma."""
    prob = _problem(*shape)
    mesh, data, inv, prior = prob
    n = len(inv.strModel)
    rng = np.random.default_rng(n + nChains)
    m0, lo, hi = _start(inv, prior, nChains, rng)
    mref = inv.strModel[None, :] + 0.1 * rng.standard_normal((nChains, n))
    pl = _plan(prob, nChains)
    base = np.clip(rng.standard_normal((nChains, n)), -2.5, 2.5)
    _check_step(pl, prior, m0, base, mref, 0.05)                                   # no clip
    p = base.copy()
    mid = ((_blocks(n) - 1) // 2) * 1024 + 17                   # the middle block; the first of two
    big = [9.0, -11.0] if nChains == 3 else []
    if nChains == 3:
        p[1, n - 1], p[2, mid] = big
        assert 0.5 * np.abs(p[0]).max() < 3.0
    else:
        p[0, n - 1] = 9.0
    _check_step(pl, prior, m0, p, mref, 0.5)                                       # clip
    p = base.copy()
    for c in range(nChains):
        p[c, (337 * c + 5) % n], p[c, (911 * c + n // 3) % n] = 6.0, -6.0
    _check_step(pl, prior, m0, p, mref, 0.5, exact_m=True)                         # tie: dt p exact, no rescale
    pl.close()
    narrow = (0.01, 0.01 * math.exp(0.4))
    prob = _problem(*shape, bounds=narrow)
    pl = _plan(prob, nChains)
    m0, lo, hi = _start(prob[2], prob[3], nChains, rng, margin=0.0)
    p = 6.0 * (2.0 * rng.random((nChains, n)) - 1.0)
    p[:, 0] = 6.0
    nb = _check_step(pl, prob[3], m0, p, mref, 0.5)
    pl.close()
    nb = np.concatenate(nb)
    assert {0, 1, 2} <= set(nb.tolist()) and nb.max() >= 7


def test_bounce_guard_reports_once_and_clears():
    """Bounds narrower than 3/1000 in ln sigma: a step of 3 outlasts the 500 iterations of the reflection loop.  status() reports
    -21 once; the next evaluation succeeds and equals the same evaluation on a fresh plan."""
    narrow = (0.01, 0.01 * math.exp(0.002))
    prob = _problem(25, 48, bounds=narrow)
    inv, prior = prob[2], prob[3]
    lo = math.log(narrow[0])
    n = len(inv.strModel)
    m0 = np.full((1, n), lo + 0.001)
    p0 = np.zeros((1, n))
    p0[0, n // 2] = 6.0
    assert ref.drift(m0[0], p0[0], 0.5, lo, math.log(narrow[1]))[3]
    pl = _plan(prob, 1)
    pl.set_state(m0, p0, m0)
    pl.leapfrog_steps_device(0.5, 1)
    assert pl.status() == -21
    assert pl.status() == 0
    again = pl.forward_gradient(m0, total=True)
    pl.close()
    fresh = _plan(prob, 1)
    fresh.set_state(m0, p0, m0)
    want = fresh.forward_gradient(m0, total=True)
    fresh.close()
    assert all(np.array_equal(a, b) for a, b in zip(again, want))


def _cond(Wm):
    """An upper bound of cond(Wm): Gershgorin's bound of the largest eigenvalue over the smallest one."""
    lmax = np.abs(Wm).sum(axis=1).max()
    lmin = spla.eigsh(Wm, k=1, sigma=0.0, which="LM", return_eigenvectors=False)[0]
    return lmax / lmin


@pytest.mark.parametrize("mass", [0, 1], ids=["diagonal", "nondiagonal"])
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: f"{s[0]}x{s[1]}")
def test_energies_at_scale(shape, mass):
    """leapfrog_trajectory(dt = 0, one step) leaves (m, p) unchanged and returns [phi_d, phi_m, K, H] at the state that was set.
    phi_m to 1e-13; K to 1e-13 with the identity mass matrix, and to 1e-13 + 8 eps cond(Wm) with M = Wm (K = 1/2 p^T Wm^-1 p
    from the multifrontal solve against a sparse LU solve)."""
    prob = _problem(*shape)
    inv, prior = prob[2], prob[3]
    n = len(inv.strModel)
    rng = np.random.default_rng(3 * n)
    m0, _, _ = _start(inv, prior, 3, rng)
    mref = inv.strModel[None, :] + 0.1 * rng.standard_normal((3, n))
    p0 = rng.standard_normal((3, n))
    pl = _plan(prob, 3, mass)
    pl.set_state(m0, p0, mref)
    stats, _ = pl.leapfrog_trajectory(0.0, 1, want_pred=False)
    m1, p1 = pl.get_state()
    pl.close()
    assert np.array_equal(m1, m0) and np.array_equal(p1, p0)
    invM, tolK = None, 1e-13
    if mass:
        lu = spla.splu(inv.Wm.tocsc())
        invM = spla.LinearOperator((n, n), matvec=lu.solve)
        tolK = 1e-13 + 8 * EPS * _cond(inv.Wm)
    for c in range(3):
        K, phim = ref.energies(m0[c], mref[c], p0[c], inv.Wm, prior.regParam, invM)
        assert abs(stats[c, 1] - phim) <= 1e-13 * phim, (c, stats[c, 1], phim)
        assert abs(stats[c, 2] - K) <= tolK * K, (c, stats[c, 2], K, tolK)
        assert stats[c, 3] == stats[c, 0] + stats[c, 2] + stats[c, 1]


# ---- several chains in one plan ----------------------------------------------------------------------------------------------

NS = 7
INTSTEPS = np.array([1, 3, 2, 1, 2, 3, 1], dtype=np.int32)


def _chain_setup(prob, nChains, seed):
    """Per-chain streams: chain 0 accepts whenever exp(hdif) > 0 (u = 0), chain 1 only when hdif > 0 (u = 1 - 2^-53), chain 2
    draws.  Start models differ per chain except in their first cell, from which the oracle derives rhoref."""
    n = len(prob[2].strModel)
    rng = np.random.default_rng(seed)
    u = rng.random((nChains, NS))
    u[0] = 0.0
    if nChains > 1:
        u[1] = 1.0 - 2.0 ** -53
    st = dict(u_start=float(rng.random()), z_init=rng.standard_normal((nChains, n)), u_accept=u,
              z_mom=rng.standard_normal((NS, nChains, n)))
    rng = np.random.default_rng(seed + 1)
    ms = np.log(0.01) + 0.05 * rng.standard_normal((nChains, n))
    ms[:, 0] = ms[0, 0]
    st["m_start"] = ms
    rho0 = 1.0 / np.exp(ms[0, 0])
    st["rhoref"] = float(np.round(rho0 * 0.5 + (rho0 * 1.5 - rho0 * 0.5) * st["u_start"]))
    return st


def _run(pl, st, dt, reuse, chain=None):
    c = slice(None) if chain is None else slice(chain, chain + 1)
    return pl.run_chain(dt, NS, st["rhoref"], st["z_init"][c], INTSTEPS, st["u_accept"][c], st["z_mom"][:, c],
                        reuse_last_forward=reuse, m_start=st["m_start"][c])


def _assert_chains_equal_single(prob, nChains, dt, reuse, mass=0, seed=11):
    """run_chain with nChains chains equals, bit for bit, one single-chain plan run on each chain's slice of the streams."""
    st = _chain_setup(prob, nChains, seed)
    pl = _plan(prob, nChains, mass)
    many = _run(pl, st, dt, reuse)
    pl.close()
    one = _plan(prob, 1, mass)
    for c in range(nChains):
        single = _run(one, st, dt, reuse, chain=c)
        for a, b in zip(many, single):
            assert np.array_equal(a[c], b[0]), c
    one.close()
    return st, many


@pytest.mark.parametrize("reuse", [True, False])
def test_chains_are_independent(reuse):
    """3 chains at nAC 1025 equal three 1-chain plans (model, statistics, accept flags, packed data), with one chain accepting
    where another rejects in the same iteration; each chain also against oracle.sampler.runHMCSampler at 1e-7."""
    import copy
    from oracle import sampler as osamp
    from tests.helpers import to_oracle
    prob = _problem(25, 48)
    mesh, data, inv, prior = prob
    dt = 0.05
    st, (model, stats, acc, pdata) = _assert_chains_equal_single(prob, 3, dt, reuse)
    assert acc[0].all() and np.any(~acc[1].astype(bool)), acc
    om, od, oi, op = to_oracle(mesh, data, inv, prior)
    op.dt = dt
    for c in range(3):
        oi_c = copy.copy(oi)
        oi_c.strModel = st["m_start"][c].copy()
        ost = osamp.RandomStreams(st["u_start"], st["z_init"][c], INTSTEPS, st["u_accept"][c], st["z_mom"][:, c])
        omodel, ostats, odata = osamp.runHMCSampler(om, od, oi_c, op, ost, nsamples=NS)
        assert np.array_equal(acc[c].astype(bool), ostats["acceptstats"]), c
        assert np.abs(model[c].T - omodel).max() < 1e-7, c
        assert np.abs(stats[c].T - ostats["hmstats"]).max() / np.abs(ostats["hmstats"]).max() < 1e-7, c
        assert np.abs(pdata[c].T - odata).max() / np.abs(odata).max() < 1e-7, c


@pytest.mark.parametrize("kind", ["rho_phase", "tipper"])
def test_chains_are_independent_real_and_tipper_data(kind):
    """k_accept<double> packs the real rho / phase rows; a tipper plan adds TZY rows to the complex ones.  2 chains."""
    from hmcmt2d_b200 import synthetic
    mesh, data, inv, prior = _problem(25, 48)
    if kind == "rho_phase":
        data, inv = synthetic.rho_phase_problem(data, inv)
    else:
        rng = np.random.default_rng(5)
        t = 0.02 * (rng.standard_normal(8) + 1j * rng.standard_normal(8))
        data, inv = synthetic.tipper_problem(data, inv, t)
    _, (_, _, acc, pdata) = _assert_chains_equal_single((mesh, data, inv, prior), 2, 0.05, True)
    assert pdata.dtype == (np.float64 if kind == "rho_phase" else np.complex128)
    assert acc[0].all() and np.any(~acc[1].astype(bool))


def test_trajectory_three_chains_equal_single_chains():
    prob = _problem(25, 48)
    inv = prob[2]
    n = len(inv.strModel)
    rng = np.random.default_rng(17)
    m0, _, _ = _start(inv, prob[3], 3, rng)
    p0 = np.clip(rng.standard_normal((3, n)), -2.5, 2.5)
    mref = np.broadcast_to(inv.strModel, (3, n))
    pl = _plan(prob, 3)
    pl.set_state(m0, p0, mref)
    stats, pred = pl.leapfrog_trajectory(0.1, 3)
    m3, p3 = pl.get_state()
    pl.close()
    one = _plan(prob, 1)
    for c in range(3):
        one.set_state(m0[c], p0[c], mref[c])
        s1, d1 = one.leapfrog_trajectory(0.1, 3)
        m1, p1 = one.get_state()
        assert np.array_equal(s1[0], stats[c]) and np.array_equal(d1[0], pred[c]), c
        assert np.array_equal(m1[0], m3[c]) and np.array_equal(p1[0], p3[c]), c
    one.close()


def test_staging_ring_chunks(monkeypatch):
    """HMCMT_RUN_CHAIN_STAGE_BYTES sized to 1, 2 and 3 samples of draws: the two slots alternate, the last chunk is partial for 2
    and 3, and every run equals the single-chunk run bit for bit (3 chains, 7 samples)."""
    prob = _problem(25, 48)
    n = len(prob[2].strModel)
    st = _chain_setup(prob, 3, 23)
    pl = _plan(prob, 3)
    monkeypatch.delenv("HMCMT_RUN_CHAIN_STAGE_BYTES", raising=False)
    whole = _run(pl, st, 0.1, True)
    for chunk in (1, 2, 3):
        monkeypatch.setenv("HMCMT_RUN_CHAIN_STAGE_BYTES", str(chunk * 3 * n * 8))
        got = _run(pl, st, 0.1, True)
        assert all(np.array_equal(a, b) for a, b in zip(got, whole)), chunk
    pl.close()


@pytest.mark.parametrize("shape", [(25, 48), (50, 87)], ids=lambda s: f"{s[0]}x{s[1]}")
def test_nondiagonal_mass_at_a_real_tree(shape):
    """M = Wm with 3 chains: p = sqrtM clip(z_last) after run_chain against a dense Cholesky of Wm; Wm^-1 p from one drift
    without clipping against a sparse solve; then 3 chains against three 1-chain plans, bit for bit."""
    prob = _problem(*shape)
    inv, prior = prob[2], prob[3]
    n = len(inv.strModel)
    st = _chain_setup(prob, 3, 31)
    pl = _plan(prob, 3, 1)
    _run(pl, st, 0.05, True)
    _, p = pl.get_state()
    L = np.linalg.cholesky(inv.Wm.toarray())
    for c in range(3):
        want = L @ np.clip(st["z_mom"][NS - 1, c], -2.5, 2.5)
        assert np.abs(p[c] - want).max() <= 1e-12 * np.abs(want).max(), c
    rng = np.random.default_rng(41)
    m0, _, _ = _start(inv, prior, 3, rng, margin=3.5)
    p0 = rng.standard_normal((3, n))
    x = np.stack([spla.spsolve(inv.Wm.tocsc(), p0[c]) for c in range(3)])
    dt = 2.5 / np.abs(x).max()
    pl.set_state(m0, p0, m0)
    pl.leapfrog_steps_device(dt, 1)
    assert pl.status() == 0
    m1, _ = pl.get_state()
    pl.close()
    cond = _cond(inv.Wm)
    tol = 4 * EPS * np.abs(m0).max() / (dt * np.abs(x).max()) + 8 * EPS * cond
    for c in range(3):
        got = (m1[c] - m0[c]) / dt
        assert np.abs(got - x[c]).max() <= tol * np.abs(x[c]).max(), (c, np.abs(got - x[c]).max() / np.abs(x[c]).max(), tol)
    _assert_chains_equal_single(prob, 3, 0.05, True, mass=1)
