"""Selected inversion on the CPU (no GPU): tests/cpp/mf_selinv_check.cpp factorises from the multifrontal tables, runs the
top-down recursion of Solver::inverse_diag in extended precision (roots first, Z(U, U) gathered from the parent through `rel`,
chunks last to first) and compares every entry of every front's Z, and the diagonal, with a dense inverse; padded rows and
columns must come out exactly zero (padded pivots exactly the identity)."""
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def checker(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("mf") / "mf_selinv_check")
    subprocess.run(["g++", "-O2", "-std=c++17", "-o", exe, os.path.join(ROOT, "tests", "cpp", "mf_selinv_check.cpp")], check=True)
    return exe


@pytest.mark.parametrize("args,min_chunks", [
    (("grid", "40", "37", "16", "144", "0", "2"), 1),       # grid ordering as the MT systems use it (leaf excess pushed)
    (("grid", "40", "37", "16", "144", "0", "0"), 1),       # push 0
    (("grid", "44", "45", "16", "144", "13", "2"), 1),      # cross-shaped separators (four children per front)
    (("active", "40", "50", "16", "144", "3"), 1),          # five-point active-cell graph through mf_order_graph (Wm's route)
    (("active", "31", "60", "16", "144", "8"), 1),
    (("graph3d", "11", "12", "13", "16", "144"), 1),        # 3-D div-grad pattern: fronts above fSmall, many children
    (("graph3d", "10", "10", "12", "16", "0"), 1),          # fSmall = 0: every front global
    (("grid", "40", "30", "300", "0"), 3),                  # fSmall = 0 with supernodes of up to 300 pivots: 2-4 chunks per front
    (("grid", "36", "30", "200", "0"), 2),
])
def test_selected_inversion_every_entry(checker, args, min_chunks):
    res = subprocess.run([checker, *args], capture_output=True, text=True)
    assert res.returncode == 0, res.stdout + res.stderr
    assert "matches the dense inverse" in res.stdout
    assert int(re.search(r"maxChunks (\d+)", res.stdout).group(1)) >= min_chunks, res.stdout
