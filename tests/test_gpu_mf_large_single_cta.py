"""Fronts of more than 144 rows on the single-CTA path (mf_small_kernel<8/16> with M' in shared memory, mf_small_stream_kernel
with M' streamed through the factor arena), against an extended-precision reference and against the same systems with every such
front on the global-memory path (HMCMT_MF_FSMALL=144).  tests/test_mf_large_single_cta_cpu.py checks on the CPU that the
matrices below reach both layouts and a front that misses the shared-memory limit by size and stays global."""
import numpy as np
import pytest

from tests import mf_class_cases as mc
from tests.test_gpu_mf_kernel_classes import EPS, reference, relres, solve

pytestmark = pytest.mark.gpu

# MT-like 2-D system and 3-D div-grad whose Level-1 analyses reach, at the default knobs, resident and streamed single-CTA fronts
# above 144 rows and a front of at most 256 rows that stays global because its pivot columns do not fit
LARGE_CASES = {
    "mt2d_150x150": lambda real: mc.mt2d(150, 150, 6, real),
    "divgrad_16x16x16": lambda real: mc.divgrad3d(16, 16, 16, 3, real),
}


@pytest.fixture
def default_knobs(monkeypatch):
    """every knob at the library's default (HMCMT_MF_FSMALL unset), multifrontal path forced; returns a setter for FSMALL"""
    for k in mc.KNOBS:
        monkeypatch.delenv(k, raising=False)
    monkeypatch.setenv("HMCMT_SHIM_SOLVER", "mf")
    return lambda v: monkeypatch.setenv("HMCMT_MF_FSMALL", v)


@pytest.mark.parametrize("real", [False, True], ids=["complex", "real"])
@pytest.mark.parametrize("name", sorted(LARGE_CASES))
def test_large_single_cta_fronts_against_reference(default_knobs, name, real):
    A = LARGE_CASES[name](real)
    n = A.shape[0]
    rng = np.random.default_rng(21)
    b = rng.standard_normal(n) if real else rng.standard_normal(n) + 1j * rng.standard_normal(n)
    xref, kappa = reference(A, b)
    bound = 100 * EPS * kappa
    assert bound <= 1e-9, (name, kappa)
    xs = {}
    for fs in ("256", "144"):
        default_knobs(fs)
        x = solve(A, b)
        assert x.dtype == (np.float64 if real else np.complex128)
        err = np.abs(x - xref).max() / np.abs(xref).max()
        assert err <= bound, (name, fs, err, bound)
        assert relres(A, x, b) < 1e-14, (name, fs, relres(A, x, b))
        xs[fs] = x
    d = np.abs(xs["256"] - xs["144"]).max() / np.abs(xs["144"]).max()
    print(f"\n[large fronts] {name} {'real' if real else 'complex'}: n {n}  kappa_1 ~ {kappa:.2e}  bound {bound:.1e}  "
          f"fSmall 256 vs 144: {d:.2e}")
    assert d <= bound, (name, d, bound)


def test_cfg2_plan_default_matches_fsmall_144(monkeypatch):
    """The benchmarked plan (cfg2: 200 x 100 cells, 30 frequencies, TE + TM, stress model): predicted data, misfit and gradient
    with the large fronts on the single-CTA path equal those with every front above 144 rows in global memory to 1e-9
    (gradient: max-normalised).  Only the summation order of the large fronts' Schur products differs."""
    from hmcmt2d_b200 import api, synthetic
    monkeypatch.delenv("HMCMT_SOLVER", raising=False)
    mesh, data, inv, prior = synthetic.make_problem(200, 100, 30)
    m = synthetic.stress_model(inv)
    out = {}
    for fs in ("256", "144"):
        monkeypatch.setenv("HMCMT_MF_FSMALL", fs)
        pl = api.Plan(mesh, data, inv, prior)
        assert pl.info(11) == 1
        out[fs] = pl.forward_gradient(m)
        assert pl.status() == 0
        pl.close()
    (p1, f1, g1), (p0, f0, g0) = out["256"], out["144"]
    e_p = float((np.abs(p1[0] - p0[0]) / np.abs(p0[0])).max())
    e_f = abs(f1[0] - f0[0]) / abs(f0[0])
    e_g = float(np.abs(g1[0] - g0[0]).max() / np.abs(g0[0]).max())
    print(f"\n[large fronts] cfg2 fSmall 256 vs 144: pred {e_p:.2e}  misfit {e_f:.2e}  gradient {e_g:.2e}")
    assert e_p < 1e-9 and e_f < 1e-9 and e_g < 1e-9, (e_p, e_f, e_g)
