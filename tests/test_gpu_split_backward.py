"""The gradient evaluation on the multifrontal path back-substitutes x on the receiver path first and the rest of x together with
the adjoint lam in one pass over the factor (Solver::backward_pair).  The timed evaluation (Plan.kernel_time(reset=1)) keeps
the complete forward and adjoint solves, one after the other, on the same plan and factors: both orders must give the same
bits, for every data type and execution mode."""
import copy

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

MODES = [("1", "0", "0"), ("1", "1", "1"), ("3", "0", "1"), ("3", "1", "0"), ("8", "1", "1")]


def _problem(kind):
    from hmcmt2d_b200 import api, synthetic
    mesh, data, inv, prior = synthetic.make_problem(70, 50, 4, nRx=9)
    if kind == "rho_phase":
        data, inv = synthetic.rho_phase_problem(data, inv)
    elif kind == "tipper":
        nF = 4
        d0, _ = synthetic.tipper_problem(data, inv, np.zeros(nF * data.rxLoc.shape[0]))
        tm = copy.copy(mesh)
        tm.sigma = synthetic.true_model(mesh)
        pred, _ = api.MT2DFwdSolver(tm, d0)
        data, inv = synthetic.tipper_problem(data, inv, pred[d0.dtID == 3])
    return mesh, data, inv, prior


@pytest.mark.parametrize("kind", ["impedance", "rho_phase", "tipper"])
def test_split_backward_matches_complete_solves(kind, monkeypatch):
    from hmcmt2d_b200 import api, synthetic
    mesh, data, inv, prior = _problem(kind)
    m0 = synthetic.stress_model(inv)
    m1 = m0 + 0.2 * np.random.default_rng(5).standard_normal(len(m0))
    first = None
    for groups, graph, prune in MODES:
        monkeypatch.setenv("HMCMT_SOLVER", "mf")
        monkeypatch.setenv("HMCMT_GROUPS", groups)
        monkeypatch.setenv("HMCMT_GRAPH", graph)
        monkeypatch.setenv("HMCMT_MF_PRUNE", prune)
        pl = api.Plan(mesh, data, inv, prior)
        assert pl.info(11) == 1
        split = [pl.forward_gradient(m) for m in (m0, m1, m0, m1)]      # eager, captured, replayed (graph on)
        fields = pl.forward(m1)                                          # forward-only after a split evaluation
        pl.kernel_time(reset=1)                                          # complete solves from here on
        ref = [pl.forward_gradient(m) for m in (m0, m1)]
        pl.kernel_time(reset=-1)
        ref_fields = pl.forward(m1)
        assert pl.status() == 0
        pl.close()
        for s, r in zip(split, ref + ref):
            for a, b in zip(s, r):
                assert np.array_equal(a, b), (kind, groups, graph, prune)
        for a, b in zip(fields, ref_fields):
            assert (a is None and b is None) or np.array_equal(a, b)
        if first is None:
            first = ref
        for s, r in zip(ref, first):
            assert all(np.array_equal(a, b) for a, b in zip(s, r))
