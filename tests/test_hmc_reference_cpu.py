"""tests/hmc_reference.py against the oracle's restatement of HMCSampler.jl (CPU): the drift with its clip and reflections, element
for element, and the energies."""
import copy
import math

import numpy as np
import pytest

from oracle import sampler as osamp
from tests import hmc_reference as ref
from tests.helpers import tiny_problem


def _prior(lo_sigma, hi_sigma):
    prior = copy.copy(tiny_problem(seed=1)[3])
    prior.sigBounds = [lo_sigma, hi_sigma]
    return prior, math.log(lo_sigma), math.log(hi_sigma)


def _oracle_drift(m, p, dt, prior):
    dm = dt * p
    mx = np.abs(dm).max()
    if mx > 3.0:
        dm = dm / mx * 3.0
    return osamp.checkParameterBound(m + dm, p.copy(), prior)


@pytest.mark.parametrize("bounds", [(2e-3, 5e-2), (1e-2, 1.5e-2), (0.1, 0.104)])
@pytest.mark.parametrize("dt", [0.05, 0.5])
def test_drift_equals_check_parameter_bound(bounds, dt):
    """Momenta of four scales land 0, 1, 2 and many reflections away; the first elements sit exactly on lo / hi with p = 0."""
    prior, lo, hi = _prior(*bounds)
    rng = np.random.default_rng(int(1000 * dt) + int(1e4 * bounds[0]))
    n = 4000
    m = lo + (hi - lo) * rng.random(n)
    p = rng.standard_normal(n) * rng.choice([0.1, 1.0, 4.0, 12.0], n)
    m[:2], p[:2] = [lo, hi], 0.0
    gm, gp, nb, guard = ref.drift(m, p, dt, lo, hi)
    om, op = _oracle_drift(m.copy(), p.copy(), dt, prior)
    assert not guard
    assert np.array_equal(gm, om) and np.array_equal(gp, op)
    assert np.array_equal(np.signbit(gp) != np.signbit(p), nb % 2 == 1)
    assert np.all((gm >= lo) & (gm <= hi)) and np.array_equal(gm[:2], [lo, hi])
    if dt == 0.5 and bounds[0] != 2e-3:
        assert {0, 1, 2} <= set(nb.tolist()) and nb.max() >= 5


def test_drift_clip_tie_and_exact_bounds():
    """max |dt p| == 3.0 exactly is not rescaled; one element above 3.0 rescales every element; a step that ends exactly on hi
    stays there without a reflection."""
    prior, lo, hi = _prior(1e-4, 1.0)
    assert hi == 0.0
    m = np.full(6, -4.0)
    p = np.array([6.0, -6.0, 1.0, 0.5, -2.0, 0.0])
    gm, gp, nb, _ = ref.drift(m, p, 0.5, lo, hi)
    assert np.array_equal(gm, m + 0.5 * p) and nb.sum() == 0          # the tie: dm = p / 2 unchanged
    om, op = _oracle_drift(m.copy(), p.copy(), 0.5, prior)
    assert np.array_equal(gm, om) and np.array_equal(gp, op)
    p2 = p.copy()
    p2[2] = 6.5
    gm, _, _, _ = ref.drift(m, p2, 0.5, lo, hi)
    assert np.array_equal(gm, m + (0.5 * p2) / 3.25 * 3.0)
    m3, p3 = np.array([-1.0, -1.0, lo + 0.5]), np.array([2.0, 2.5, -2.0])     # v = hi exactly; v = 0.25 -> -0.25; v = lo - 0.5
    gm, gp, nb, _ = ref.drift(m3, p3, 0.5, lo, hi)
    om, op = _oracle_drift(m3.copy(), p3.copy(), 0.5, prior)
    assert np.array_equal(gm, om) and np.array_equal(gp, op)
    assert np.array_equal(nb, [0, 1, 1]) and gm[0] == hi and gm[1] == -0.25


def test_drift_bounce_guard():
    """An iteration of the reflection loop reflects at most twice (lo, then hi), so with bounds narrower than 3/1000 a step of 3
    outlasts the 500 iterations.  The reference reports the guard; the oracle raises (HMCSampler.jl loops forever)."""
    prior, lo, _ = _prior(0.01, 0.01 * math.exp(0.002))
    hi = math.log(prior.sigBounds[1])
    m = np.array([lo + 0.001, lo + 0.0005])
    p = np.array([6.0, 0.001])
    _, _, nb, guard = ref.drift(m, p, 0.5, lo, hi)
    assert guard and nb[0] >= 500 and nb[1] == 0
    with pytest.raises(RuntimeError):
        osamp.checkParameterBound(m + 0.5 * p, p.copy(), prior)


@pytest.mark.parametrize("mass", ["diagonal", "nondiagonal"])
def test_energies_equal_oracle(mass):
    mesh, data, inv, prior = tiny_problem(seed=5)
    prior.massType = mass
    prior.regParam = 0.7
    invM, sqrtM = osamp.setMassMatrix(inv, prior)
    rng = np.random.default_rng(6)
    n = len(inv.strModel)
    m = inv.strModel + 0.3 * rng.standard_normal(n)
    mref = inv.strModel + 0.1 * rng.standard_normal(n)
    p = rng.standard_normal(n) if sqrtM is None else sqrtM @ rng.standard_normal(n)
    K, phim = ref.energies(m, mref, p, inv.Wm, prior.regParam, invM)
    oK = osamp.getKineticEnergy(p, invM)
    d = m - mref
    ophim = 0.5 * float(d @ (inv.Wm @ d)) * prior.regParam
    assert abs(K - oK) <= 1e-13 * abs(oK) and abs(phim - ophim) <= 1e-13 * abs(ophim)


def test_accept_rule():
    assert ref.accept(1.0, 0.5, 0.999)                     # hdif > 0 always accepts
    assert ref.accept(1.0, 2.0, 0.0)                       # u = 0 accepts unless exp(hdif) underflows to 0
    assert not ref.accept(0.0, 746.0, 0.0)
    assert not ref.accept(1.0, 1.5, 1.0 - 2.0 ** -53)
    assert ref.accept(1.0, 1.0, 1.0 - 2.0 ** -53)           # hdif = 0: u < exp(0) = 1
