"""Assembly of the mid-size fronts on the CPU (no GPU): tests/cpp/mf_mid_gather_check.cpp checks, on the multifrontal tables, that
the children's rows landing in the pivot columns are a prefix, that the restricted extend-add and the inverse row maps together
reach every child entry exactly once, and that F22 gathered in child order equals the scattered F22 bit for bit."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def checker(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("mf") / "mf_mid_gather_check")
    subprocess.run(["g++", "-O2", "-std=c++17", "-o", exe, os.path.join(ROOT, "tests", "cpp", "mf_mid_gather_check.cpp")], check=True)
    return exe


@pytest.mark.parametrize("args", [
    ("grid", "199", "99", "16", "144", "0", "2"),    # cfg2 system with the plan's ordering
    ("grid", "799", "299", "16", "144", "0", "2"),   # cfg4 system
    ("grid", "199", "99", "16", "144", "0", "0"),    # cfg2 without pushed leaf excess
    ("grid", "60", "47", "16", "144", "13", "2"),    # cross-shaped separators (four children per front)
    ("graph3d", "20", "16", "12", "16", "144"),      # level-set bisection of a 3-D grid (Level-1 shim ordering, four children)
])
def test_gather_equals_scatter(checker, args):
    res = subprocess.run([checker, *args], capture_output=True, text=True)
    assert res.returncode == 0, res.stdout + res.stderr
    assert "bit-identical" in res.stdout
