"""Fronts of more than 144 rows on the single-CTA path, checked on the CPU: tests/cpp/mf_large_fronts.cpp prints the classification
of mf_symbolic.h and the single-CTA launch of every depth as Solver::build() forms it (warps, resident or streamed M', shared
memory), and a hash of the tables and of that schedule."""
import os
import subprocess

import pytest
import scipy.sparse as sp

from tests.test_gpu_mf_large_single_cta import LARGE_CASES

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SMEM_MAX = 227 * 1024
CFG2 = ("199", "99", "16")     # the cfg2 system (200 x 100 cells) with the plan's ordering: leaf 16, no cross, push 2
CFG4 = ("799", "299", "16")
# hash of the tables and schedule at fSmall = 144, computed with the classification that had no single-CTA front above 144 rows
HASH_144 = {CFG2 + ("0", "2"): "f0e7033423c9282a", CFG4 + ("0", "2"): "2438c5194a7d5b96", CFG2 + ("0", "0"): "0ec7f3289a28f997",
            ("60", "47", "16", "13", "2"): "0492d41301a6eb01"}


@pytest.fixture(scope="module")
def helper(tmp_path_factory):
    d = tmp_path_factory.mktemp("mf_large")
    exe = str(d / "mf_large_fronts")
    subprocess.run(["g++", "-O2", "-std=c++17", "-o", exe, os.path.join(ROOT, "tests", "cpp", "mf_large_fronts.cpp")], check=True)
    return exe, d


def run(exe, *args):
    res = subprocess.run([exe, *args], capture_output=True, text=True)
    assert res.returncode == 0, res.stdout + res.stderr
    depths, fronts, h = [], [], None
    for line in res.stdout.splitlines():
        tok = line.split()
        if tok[0] == "hash":
            h = tok[1]
            continue
        rec = {tok[i]: tok[i + 1] for i in range(0, len(tok), 2)}
        rec = {k: (v if k == "layout" else int(v)) for k, v in rec.items()}
        (depths if tok[0] == "depth" else fronts).append(rec)
    return depths, fronts, h


def grid(exe, dims, fs, cross="0", push="2"):
    return run(exe, "grid", *dims, str(fs), cross, push)


@pytest.mark.parametrize("args", sorted(HASH_144))
def test_fsmall_144_keeps_the_tables(helper, args):
    exe, _ = helper
    depths, fronts, h = run(exe, "grid", *args[:3], "144", *args[3:])
    assert h == HASH_144[args]
    assert all(f["big"] for f in fronts) and not any(d["stream"] for d in depths)


def test_cfg2_depths_2_to_4_single_cta(helper):
    exe, _ = helper
    depths, fronts, _ = grid(exe, CFG2, 256)
    by = {d["depth"]: d for d in depths}
    assert by[1]["nBig"] == 2 and by[1]["nSmall"] == 0
    for d in (2, 3, 4):
        assert by[d]["nBig"] == 0 and by[d]["warps"] == 16, by[d]
    assert by[2]["stream"] == 1 and by[3]["stream"] == 1 and by[4]["stream"] == 0
    moved = [f for f in fronts if not f["big"]]
    assert len(fronts) == 26 and len(moved) == 24
    assert all(f["nChunk"] == 1 for f in moved)
    assert {f["depth"] for f in fronts if f["big"]} == {1}


def test_cfg4_moved_fronts(helper):
    exe, _ = helper
    depths, fronts, _ = grid(exe, CFG4, 256)
    moved = [f for f in fronts if not f["big"]]
    assert len(fronts) == 341 and len(moved) == 250
    assert {f["layout"] for f in moved} == {"resident", "streamed"}
    assert {f["depth"] for f in moved} == {6, 7, 8}
    assert all(f["nChunk"] == 1 for f in moved)


@pytest.mark.parametrize("fs", [144, 152, 208, 256])
@pytest.mark.parametrize("dims", [CFG2, CFG4])
def test_single_cta_shared_memory_fits(helper, dims, fs):
    exe, _ = helper
    depths, fronts, _ = grid(exe, dims, fs)
    for d in depths:
        assert d["smem"] <= SMEM_MAX, d
        if d["maxFpSmall"] > 144:
            assert d["warps"] >= 8, d
    assert all(f["big"] or f["sp"] + f["up"] <= fs for f in fronts)


@pytest.mark.parametrize("name", sorted(LARGE_CASES))
def test_level1_cases_reach_both_layouts(helper, name):
    exe, d = helper
    A = sp.csc_matrix(LARGE_CASES[name](False))
    A.sort_indices()
    path = os.path.join(str(d), f"{name}.pattern")
    with open(path, "w") as f:
        f.write(f"{A.shape[0]}\n")
        f.write(" ".join(map(str, A.indptr + 1)) + "\n")
        f.write(" ".join(map(str, A.indices + 1)) + "\n")
    depths, fronts, _ = run(exe, "csc", path, "16", "256")
    got = {f["layout"] for f in fronts if not f["big"]}
    assert got == {"resident", "streamed"}, got
    # a front within fSmall and the child limit that stays global because its pivot columns do not fit
    assert any(f["big"] and f["sp"] + f["up"] <= 256 and f["nChild"] <= 4 for f in fronts), fronts
    assert all(dd["smem"] <= SMEM_MAX for dd in depths)


@pytest.mark.parametrize("args", [
    ("grid", "199", "99", "16", "256", "0", "2"),    # cfg2
    ("grid", "799", "299", "16", "256", "0", "2"),   # cfg4
    ("grid", "60", "47", "16", "256", "13", "2"),    # cross-shaped separators
    ("graph3d", "20", "16", "12", "16", "256"),      # level-set bisection of a 3-D grid
])
def test_gather_equals_scatter_above_144(helper, args):
    """tests/cpp/mf_mid_gather_check.cpp (prefix of the pivot-column rows, coverage of the restricted scatter and of the inverse
    maps, gathered F22 bit-identical to the scattered one) on the fronts that fSmall = 256 moves to the single-CTA path"""
    _, d = helper
    exe = str(d / "mf_mid_gather_check")
    if not os.path.exists(exe):
        subprocess.run(["g++", "-O2", "-std=c++17", "-o", exe, os.path.join(ROOT, "tests", "cpp", "mf_mid_gather_check.cpp")], check=True)
    res = subprocess.run([exe, *args], capture_output=True, text=True)
    assert res.returncode == 0, res.stdout + res.stderr
    assert "bit-identical" in res.stdout
