"""Split backward substitution of the gradient evaluation on the CPU (no GPU): tests/cpp/mf_split_backward_check.cpp runs, on the
multifrontal tables, the receiver-path sweep of x followed by one sweep over x and the adjoint that skips x on the receiver path,
and checks that it gives the complete backward substitutions bit for bit, that the receiver path holds both receiver rows and is
closed under parents, and that back-substituting x a second time on the receiver path would be caught."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def checker(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("mf") / "mf_split_backward_check")
    subprocess.run(["g++", "-O2", "-std=c++17", "-o", exe, os.path.join(ROOT, "tests", "cpp", "mf_split_backward_check.cpp")], check=True)
    return exe


@pytest.mark.parametrize("args", [
    ("199", "99", "16", "144", "0", "2", "6"),     # cfg2 system with the default ordering, receiver node rows 7, 8
    ("199", "99", "16", "144", "0", "0", "6"),     # the same without pushed leaf excess
    ("60", "47", "16", "144", "13", "2", "3"),     # cross-shaped separators (four children per front)
    ("64", "45", "9", "144", "0", "7", "0"),       # every leaf excess pushed; receiver rows at the grid's edge
    ("64", "50", "16", "0", "0", "0", "10"),       # every front through the large-front path, chunked pivots
])
def test_split_order_equals_complete_backward(checker, args):
    res = subprocess.run([checker, *args], capture_output=True, text=True)
    assert res.returncode == 0, res.stdout + res.stderr
    assert "bit-identical" in res.stdout
