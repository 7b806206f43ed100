"""Forward-mode J dsig (Plan.jvec / hmcmt_jvec) and the Gauss-Newton product D Re(J^H Wd^2 J) D v (Plan.gn_hessvec /
hmcmt_gn_hessvec) on the device: against the explicit Jacobian the plan builds and the oracle's, on both solvers, for impedance,
rho / phase and tipper plans; the dot-product identity with J^T at the benchmark shape; a problem where the 1-D boundary
recursion's overflow guard fires; central differences; symmetry of the GN product; and that the entry points leave the plan's
state, its graph and its chains exactly as they were."""
import numpy as np
import pytest

from tests.helpers import load_example, tiny_problem, to_product
from tests import rho_phase_oracle as rpo
from tests import tipper_oracle as tpo
from tests.rho_phase_helpers import ragged_mask, rho_phase_problem
from tests.tipper_helpers import survey, tipper_problem

pytestmark = pytest.mark.gpu
TOL = 1e-9
KINDS = ["impedance", "rho_phase", "tipper", "tipper_only"]


def _problem(kind, seed=19, mesh_data=None):
    """(oracle mesh, oracle data, oracle inv, prior, oracle module) of one data type on the tiny mesh."""
    from oracle import jacobian as ojac
    mesh, data, inv, prior = mesh_data or tiny_problem(seed=seed)
    if kind == "impedance":
        return mesh, data, inv, prior, ojac
    if kind == "rho_phase":
        _, d, rinv, _ = rho_phase_problem(mesh, data, prior, keep=ragged_mask(data, seed=5))
        return mesh, d, rinv, prior, rpo
    d, tinv = tipper_problem(mesh, data, inv)
    comps = ["ZXY", "ZYX", "TZY"] if kind == "tipper" else ["TZY"]
    comp = np.array([d.dataComp[k - 1] for k in d.dtID])
    sel = np.isin(comp, comps)
    nF, nRx = len(d.freqs), d.rxLoc.shape[0]
    keep = np.asarray(d.dataID, dtype=bool).reshape(nF, nRx, len(d.dataComp))[:, :, [d.dataComp.index(c) for c in comps]]
    sd = survey(d, comps, keep.reshape(-1))
    si = type(tinv)(tinv.obsData[sel], tinv.dataW[sel], tinv.strModel.copy(), tinv.refModel.copy(), tinv.activeCell, tinv.bgModel,
                    tinv.Wm)
    return mesh, sd, si, prior, tpo


def _model(inv, seed=20):
    return inv.strModel + 0.2 * np.random.default_rng(seed).standard_normal(len(inv.strModel))


def _plan(mesh, data, inv, prior, nChains=1):
    from hmcmt2d_b200 import api
    pm, pd, pi, pp = to_product(mesh, data, inv, prior)
    return api.Plan(pm, pd, pi, pp, nChains=nChains), (pm, pd, pi, pp)


def _check_against_jacobian(mesh, data, inv, prior, m=None, seed=4):
    pl, _ = _plan(mesh, data, inv, prior)
    m = _model(inv) if m is None else m
    pl.forward(m=m, fields=False)
    J = pl.jacobian()[0]
    dsig = np.random.default_rng(seed).standard_normal(pl.nAC) * np.exp(m)
    jv = pl.jvec(dsig)[0]
    want = J @ dsig
    assert jv.dtype == J.dtype and jv.shape == want.shape
    err = np.abs(jv - want).max() / np.abs(want).max()
    pl.close()
    return err


@pytest.mark.parametrize("solver", ["band", "mf"])
@pytest.mark.parametrize("kind", KINDS)
def test_jvec_equals_explicit_jacobian(kind, solver, monkeypatch):
    """jvec(dsig) == jacobian() @ dsig: impedance, rho / phase with a ragged mask, [ZXY, ZYX, TZY] and [TZY] alone."""
    monkeypatch.setenv("HMCMT_SOLVER", solver)
    mesh, data, inv, prior, _ = _problem(kind)
    err = _check_against_jacobian(mesh, data, inv, prior)
    assert err <= 1e-10, (kind, solver, err)


@pytest.mark.parametrize("kind", KINDS)
def test_jvec_against_oracle(kind):
    """jvec against the oracle's explicit Jacobian (compJacMat and its rho / phase and tipper twins) times dsig."""
    from oracle import forward as ofwd
    mesh, data, inv, prior, omod = _problem(kind)
    pl, _ = _plan(mesh, data, inv, prior)
    m = _model(inv)
    pl.forward(m=m, fields=False)
    dsig = np.random.default_rng(6).standard_normal(pl.nAC) * np.exp(m)
    jv = pl.jvec(dsig)[0]
    pl.close()
    mesh.sigma = inv.activeCell @ np.exp(m) + inv.bgModel
    _, ofw = (tpo if kind.startswith("tipper") else ofwd).MT2DFwdSolver(mesh, data)
    oJ = omod.compJacMat(ofw.exTE, ofw.hxTM, mesh, data, inv.activeCell, ofw.AinvTE, ofw.AinvTM)
    want = oJ @ dsig
    assert np.abs(jv - want).max() / np.abs(want).max() < TOL, kind


def test_reference_named_entry_point():
    """compJacMatVec: the oracle's compJacMat @ dsig through the MT2DFwdSolver handles, an activeCell mapped by cell index, the
    stale-handle and Rho_Pha refusals."""
    from hmcmt2d_b200 import api
    from oracle import forward as ofwd
    from oracle import jacobian as ojac
    mesh, data, inv, prior = tiny_problem(seed=19)
    pm, pd, pi, pp = to_product(mesh, data, inv, prior)
    pred, fwd = api.MT2DFwdSolver(pm, pd)
    dsig = np.random.default_rng(8).standard_normal(inv.activeCell.shape[1]) * 0.01
    jv = api.compJacMatVec(fwd.exTE, fwd.hxTM, dsig, pm, pd, pi.activeCell, fwd.AinvTE, fwd.AinvTM)
    _, ofw = ofwd.MT2DFwdSolver(mesh, data)
    oJ = ojac.compJacMat(ofw.exTE, ofw.hxTM, mesh, data, inv.activeCell, ofw.AinvTE, ofw.AinvTM)
    assert jv.shape == pred.shape
    assert np.abs(jv - oJ @ dsig).max() / np.abs(oJ @ dsig).max() < TOL
    # a selector over a subset of the cells in another order: the perturbation lands on the cells it names
    import scipy.sparse as sp
    act = pi.activeCell.tocsc().indices
    sub = act[::-1][: len(act) // 2]
    sel = sp.csr_matrix((np.ones(len(sub)), (sub, np.arange(len(sub)))), shape=(pi.activeCell.shape[0], len(sub)))
    d2 = np.random.default_rng(9).standard_normal(len(sub)) * 0.01
    full = np.zeros(pi.activeCell.shape[0])
    full[sub] = d2
    jv2 = api.compJacMatVec(fwd.exTE, fwd.hxTM, d2, pm, pd, sel, fwd.AinvTE, fwd.AinvTM)
    want = oJ @ full[act]
    assert np.abs(jv2 - want).max() / np.abs(want).max() < TOL
    api.MT2DFwdSolver(pm, pd)
    with pytest.raises(RuntimeError):
        api.compJacMatVec(fwd.exTE, fwd.hxTM, dsig, pm, pd, pi.activeCell, fwd.AinvTE, fwd.AinvTM)
    _, d, rinv, _ = rho_phase_problem(mesh, data, prior)
    rm, rd, ri, rp = to_product(mesh, d, rinv, prior)
    _, rfwd = api.MT2DFwdSolver(rm, rd)
    with pytest.raises(NotImplementedError):
        api.compJacMatVec(rfwd.exTE, rfwd.hxTM, dsig, rm, rd, ri.activeCell, rfwd.AinvTE, rfwd.AinvTM)


def test_dot_product_identity_at_benchmark_shape(monkeypatch):
    """cfg2 mesh (200 x 100 cells) on the default multifrontal solver: Re<w, J dsig> == <jtvec(w), dsig>."""
    from hmcmt2d_b200 import api, synthetic
    monkeypatch.delenv("HMCMT_SOLVER", raising=False)
    mesh, data, inv, prior = synthetic.make_problem(200, 100, 4)
    pl = api.Plan(mesh, data, inv, prior)
    assert pl.info(11) == 1
    m = synthetic.stress_model(inv)
    pl.forward_gradient(m)
    rng = np.random.default_rng(11)
    dsig = rng.standard_normal(pl.nAC) * np.exp(m)
    w = rng.standard_normal(pl.nData) + 1j * rng.standard_normal(pl.nData)
    jv = pl.jvec(dsig)[0]
    g = pl.jtvec(w)[0]
    lhs = np.real(np.vdot(w, jv))
    rhs = float(g @ dsig)
    assert abs(lhs - rhs) <= 1e-10 * float(np.sum(np.abs(w) * np.abs(jv))), (lhs, rhs)
    pl.close()


def _guard_problem():
    """tiny mesh with a 10x more conductive earth at 10 kHz and 10 Hz: the 1-D recursions' overflow guard fires above the last
    layer at 10 kHz (the two deepest rows of the boundary derivative are zero) and not at all at 10 Hz."""
    mesh, data, inv, prior = tiny_problem(seed=19, nF=2)
    s = np.array(mesh.sigma)
    s[s > 1e-6] *= 10.0
    mesh.sigma = s
    data.freqs = np.array([1e4, 10.0])
    inv.strModel = np.log(s[inv.activeCell.tocsc().indices])
    return mesh, data, inv, prior


@pytest.mark.parametrize("solver", ["band", "mf"])
def test_overflow_guard(solver, monkeypatch):
    """A (frequency, mode, profile) whose guard fires (zero rows below some depth of the oracle's getBCDerivMatrix) and one whose
    does not, in one plan: jvec against the plan's and the oracle's explicit Jacobian."""
    from oracle import forward as ofwd
    from oracle import jacobian as ojac
    from oracle import sensitivity as osens
    monkeypatch.setenv("HMCMT_SOLVER", solver)
    mesh, data, inv, prior = _guard_problem()
    ny, nz = mesh.gridSize
    fired = {}
    for f in data.freqs:
        for src in "EH":
            dBC, bc = osens.getBCDerivMatrix(f, mesh.yLen, mesh.zLen, mesh.sigma, src)
            left = dBC[ny + 1:ny + nz + 1]
            zero = [not r.any() for r in left]
            fired[(f, src)] = (bc[ny + nz] == 0, sum(zero), zero[0])
    assert fired[(1e4, "E")] == fired[(1e4, "H")] == (True, 2, False)
    assert fired[(10.0, "E")] == fired[(10.0, "H")] == (False, 0, False)
    m = inv.strModel.copy()
    err = _check_against_jacobian(mesh, data, inv, prior, m)
    assert err <= 1e-10, err
    pl, _ = _plan(mesh, data, inv, prior)
    pl.forward(m=m, fields=False)
    dsig = np.random.default_rng(12).standard_normal(pl.nAC) * np.exp(m)
    jv = pl.jvec(dsig)[0]
    pl.close()
    _, ofw = ofwd.MT2DFwdSolver(mesh, data)
    want = ojac.compJacMat(ofw.exTE, ofw.hxTM, mesh, data, inv.activeCell, ofw.AinvTE, ofw.AinvTM) @ dsig
    assert np.abs(jv - want).max() / np.abs(want).max() < TOL


def test_finite_differences():
    """coprod2 geometry: central differences (h = 1e-5 in ln sigma) of the predicted data along a direction on 10 probe cells away
    from the bottom 5 cell rows (the selection of test_gpu_parity.py::test_cfg5_finite_difference_check) against jvec(sigma v)."""
    from hmcmt2d_b200 import api
    mesh, data, inv, prior = load_example("coprod2")
    pm, pd, pi, pp = to_product(mesh, data, inv, prior)
    rng = np.random.default_rng(5)
    m = np.log(0.01) + 0.7 * rng.standard_normal(len(inv.strModel))
    ny, nz = mesh.gridSize
    nrows = nz - len(mesh.airLayer)
    rows = rng.integers(0, nrows - 5, size=10)
    cols = rng.integers(2, ny - 2, size=10)
    v = np.zeros(len(m))
    v[rows * ny + cols] = rng.standard_normal(10)
    pl = api.Plan(pm, pd, pi, pp)
    pl.forward(m=m, fields=False)
    jv = pl.jvec(np.exp(m) * v)[0]
    h = 1e-5
    fd = (pl.forward(m=m + h * v, fields=False)[0][0] - pl.forward(m=m - h * v, fields=False)[0][0]) / (2 * h)
    assert np.abs(fd - jv).max() < 1e-4 * np.abs(jv).max(), np.abs(fd - jv).max() / np.abs(jv).max()
    pl.close()


@pytest.mark.parametrize("kind", ["impedance", "rho_phase", "tipper"])
def test_gauss_newton_product(kind):
    """gn_hessvec(v) == D Re(J^H Wd^2 J) D v (+ beta Wm v) formed from jacobian(); symmetric and positive semi-definite."""
    mesh, data, inv, prior, _ = _problem(kind)
    pl, (pm, pd, pi, pp) = _plan(mesh, data, inv, prior)
    m = _model(inv)
    pl.forward(m=m, fields=False)
    J = pl.jacobian()[0]
    D = np.exp(m)
    w2 = np.abs(np.asarray(pi.dataW)) ** 2
    H = D[:, None] * np.real(np.conj(J).T @ (w2[:, None] * J)) * D[None, :]
    rng = np.random.default_rng(13)
    u, v = rng.standard_normal(len(m)), rng.standard_normal(len(m))
    hv, hu = pl.gn_hessvec(v)[0], pl.gn_hessvec(u)[0]
    assert np.abs(hv - H @ v).max() <= 1e-10 * np.abs(H @ v).max()
    ht = pl.gn_hessvec(v, total=True)[0]
    want = H @ v + pp.regParam * (pi.Wm @ v)
    assert np.abs(ht - want).max() <= 1e-10 * np.abs(want).max()
    assert abs(u @ hv - hu @ v) <= 1e-12 * np.linalg.norm(u) * np.linalg.norm(hv)
    assert v @ hv >= 0.0 and u @ hu >= 0.0
    pl.close()


def _responses(pl):
    from hmcmt2d_b200 import lib as _lib
    out = np.zeros((pl.nChains, pl.nFreq * pl._keep["rx"].shape[0] * len(pl._keep["comp"]) * 2))
    _lib.check(pl.L.hmcmt_get_responses(pl.h, _lib.f64(out)), "hmcmt_get_responses")
    return out


@pytest.mark.parametrize("solver", ["band", "mf"])
def test_state_and_determinism(solver, monkeypatch):
    """After jvec / gn_hessvec the responses, predictions, jtvec, the next forward_gradient (graph replay) and get_state are
    bit-identical to a plan that never called them; repeated calls are bit-identical; chain c of a 3-chain plan equals a 1-chain
    plan; -3 before any forward evaluation and on NULL arguments."""
    from hmcmt2d_b200 import lib as _lib
    monkeypatch.setenv("HMCMT_SOLVER", solver)
    mesh, data, inv, prior = tiny_problem(seed=7)
    rng = np.random.default_rng(14)
    m = _model(inv)
    m2 = _model(inv, seed=21)
    p0 = rng.standard_normal(len(m))
    dsig = rng.standard_normal(len(m)) * np.exp(m)
    v = rng.standard_normal(len(m))
    w = rng.standard_normal(len(data.dtID)) + 1j * rng.standard_normal(len(data.dtID))
    a, _ = _plan(mesh, data, inv, prior)
    b, _ = _plan(mesh, data, inv, prior)
    with pytest.raises(_lib.HmcmtError) as e:
        a.jvec(dsig)
    assert e.value.code == -3
    with pytest.raises(_lib.HmcmtError) as e:
        a.gn_hessvec(v)
    assert e.value.code == -3
    for pl in (a, b):
        pl.set_state(m, p0, inv.strModel)
        pl.forward_gradient(m)
        r0 = pl.forward_gradient(m)                       # the second evaluation captures the graph
    jv = a.jvec(dsig)
    hv = a.gn_hessvec(v, total=True)
    assert np.array_equal(a.jvec(dsig), jv) and np.array_equal(a.gn_hessvec(v, total=True), hv)
    assert np.array_equal(a.gn_hessvec(v), a.gn_hessvec(v))
    assert a.L.hmcmt_jvec(a.h, None, None) == -3 and a.L.hmcmt_gn_hessvec(a.h, None, 0, None) == -3
    assert np.array_equal(_responses(a), _responses(b))
    assert np.array_equal(a.jtvec(w), b.jtvec(w))
    ra, rb = a.forward_gradient(m2), b.forward_gradient(m2)          # graph replay
    for x, y in zip(ra, rb):
        assert np.array_equal(x, y)
    for x, y in zip(a.get_state(), b.get_state()):
        assert np.array_equal(x, y)
    assert all(np.array_equal(x, y) for x, y in zip(r0, a.forward_gradient(m)))
    a.close()
    b.close()
    # chain c of a 3-chain plan against a 1-chain plan
    M = np.stack([m, m2, _model(inv, seed=22)])
    D = np.stack([dsig, -dsig, 2 * dsig])
    V = np.stack([v, 2 * v, -v])
    c3, _ = _plan(mesh, data, inv, prior, nChains=3)
    c3.forward(m=M, fields=False)
    jv3, hv3 = c3.jvec(D), c3.gn_hessvec(V, total=True)
    c3.close()
    for c in range(3):
        c1, _ = _plan(mesh, data, inv, prior)
        c1.forward(m=M[c], fields=False)
        assert np.array_equal(c1.jvec(D[c])[0], jv3[c]) and np.array_equal(c1.gn_hessvec(V[c], total=True)[0], hv3[c]), c
        c1.close()
