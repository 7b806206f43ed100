"""Kernel-class coverage of the multifrontal GPU tests, checked on the CPU: tests/cpp/mf_classes.cpp runs the Level-1 analysis and
the launch-schedule rules of the solver (mf_symbolic.h) on every matrix of tests/test_gpu_mf_kernel_classes.py under every knob
setting that test uses, and each matrix must reach the classes it is declared to cover.  A change of a threshold or of the
ordering that moves a matrix out of its class fails here, on any machine, instead of leaving a kernel untested."""
import pytest

from tests import mf_class_cases as mc


@pytest.fixture(scope="module")
def helper(tmp_path_factory):
    d = tmp_path_factory.mktemp("mf_classes")
    return mc.helper_exe(d), d


def reached(helper, A, name):
    exe, d = helper
    got = {}
    for r, env in mc.ROUTINGS.items():
        fronts, depths = mc.run_helper(exe, A, env, d, f"{name}_{r}")
        got[r] = mc.classes_of(fronts, depths)
    return got


@pytest.mark.parametrize("name", sorted(mc.CASES))
def test_case_reaches_declared_classes(helper, name):
    build, declared = mc.CASES[name]
    got = reached(helper, build(), name)
    union = set().union(*got.values())
    print(f"\n{name}: " + "  ".join(f"{r}: {','.join(sorted(c))}" for r, c in got.items()))
    assert declared <= union, f"{name} no longer reaches {sorted(declared - union)}"
    # the forced routings do what they claim: every single-CTA launch of routing w<W> runs W warps
    for r in mc.WARP_ROUTINGS:
        assert {c for c in got[r] if c in ("w1", "w2", "w4", "w8", "w16")} == {r}, (r, got[r])
    assert not any(c.startswith("w") and not c.startswith("ws") for c in got["fsmall0"]), got["fsmall0"]
    assert {c for c in got["t128"] if c.startswith("cta")} <= {"cta128"}
    assert {c for c in got["t256"] if c.startswith("cta")} <= {"cta256"}


def test_cases_cover_every_class():
    declared = set().union(*(c for _, c in mc.CASES.values()))
    assert declared == mc.ALL_CLASSES, sorted(mc.ALL_CLASSES ^ declared)


def test_real_twins_share_the_pattern():
    for name, (build, _) in mc.CASES.items():
        a, b = build(), build(True)
        assert (a.indptr == b.indptr).all() and (a.indices == b.indices).all(), name
        assert a.imag.count_nonzero() > 0 and b.dtype.kind == "f", name
