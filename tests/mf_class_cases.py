"""Matrices of the multifrontal kernel-class tests (tests/test_gpu_mf_kernel_classes.py on the GPU, tests/test_mf_classes_cpu.py
on the CPU) and the kernel classes each of them is declared to reach.  The classes are read from the output of
tests/cpp/mf_classes.cpp, which runs the Level-1 analysis and the launch-schedule rules of the solver on the host."""
import os
import subprocess

import numpy as np
import scipy.sparse as sp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MU0 = 4e-7 * np.pi

# knob settings every matrix is factorised under (the Level-1 shim reads them when it analyses a pattern and builds a solver):
# each small front forced through 1, 2, 4, 8 and 16 warps, every front through the global-memory path, and the CTA solves with
# 128 and 256 threads
_WARPS_OFF = {"HMCMT_MF_FSMALL": "144", "HMCMT_MF_SOLVE_THREADS": "0"}
ROUTINGS = {
    "w1": dict(_WARPS_OFF, HMCMT_MF_FP1="1000", HMCMT_MF_FP2="1000", HMCMT_MF_FP4="1000", HMCMT_MF_FP8="1000"),
    "w2": dict(_WARPS_OFF, HMCMT_MF_FP1="0", HMCMT_MF_FP2="1000", HMCMT_MF_FP4="1000", HMCMT_MF_FP8="1000"),
    "w4": dict(_WARPS_OFF, HMCMT_MF_FP1="0", HMCMT_MF_FP2="0", HMCMT_MF_FP4="1000", HMCMT_MF_FP8="1000"),
    "w8": dict(_WARPS_OFF, HMCMT_MF_FP1="0", HMCMT_MF_FP2="0", HMCMT_MF_FP4="0", HMCMT_MF_FP8="1000"),
    "w16": dict(_WARPS_OFF, HMCMT_MF_FP1="0", HMCMT_MF_FP2="0", HMCMT_MF_FP4="0", HMCMT_MF_FP8="0"),
    "fsmall0": {"HMCMT_MF_FSMALL": "0"},
    "t128": {"HMCMT_MF_SOLVE_THREADS": "128"},
    "t256": {"HMCMT_MF_SOLVE_THREADS": "256"},
}
WARP_ROUTINGS = ("w1", "w2", "w4", "w8", "w16")
KNOBS = ("HMCMT_MF_LEAF", "HMCMT_MF_FSMALL", "HMCMT_MF_FP1", "HMCMT_MF_FP2", "HMCMT_MF_FP4", "HMCMT_MF_FP8", "HMCMT_MF_SOLVE_THREADS")
DEFAULTS = {"HMCMT_MF_LEAF": "16", "HMCMT_MF_FSMALL": "144", "HMCMT_MF_FP1": "40", "HMCMT_MF_FP2": "40", "HMCMT_MF_FP4": "64",
            "HMCMT_MF_FP8": "96", "HMCMT_MF_SOLVE_THREADS": "0"}

# every class of the multifrontal numeric phase:
#   w<W>           a launch of mf_small_kernel<W>
#   mid_cpiv_part  a front of the 8 / 16-warp (pivot-column) layout with a child whose update rows fall partly into the pivot
#                  columns (scattered) and partly into F22 (gathered in the Schur product); mid_cpiv_all: all of them into the pivot
#                  columns.  (No child has cPiv = 0: a child's parent is the front holding its first update row.)
#   npb1, nub0     a single-CTA front of one pivot tile / without update rows
#   big_fp, big_children   a global-memory front taken there for fp > fSmall / for more than kSmallChildren children
#   chunks1/2/3    a global-memory front of 1, 2, >= 3 pivot chunks (kChunkMax = 96); tail8: last chunk of 8 pivots;
#                  root_mr0: a global-memory root (its last chunk has no rows below it)
#   ws8/16/32      a warp solve of width 8, 16, 32 (mf_bwd_warp_front); ws_u_gt40: a warp solve with more than kDescRows = 40
#                  update rows (the rows beyond 40 read from global memory)
#   cta128/256     CTA solves launched with 128 / 256 threads
ALL_CLASSES = {
    "w1", "w2", "w4", "w8", "w16", "mid_cpiv_part", "mid_cpiv_all", "npb1", "nub0", "big_fp", "big_children",
    "chunks1", "chunks2", "chunks3", "tail8", "root_mr0", "ws8", "ws16", "ws32", "ws_u_gt40", "cta128", "cta256",
}


def _laplacian_1d(h):
    """cell-centred second difference on cells of widths h, Dirichlet outside: (n x n) matrix of face coefficients"""
    dist = np.concatenate(([h[0] / 2], (h[:-1] + h[1:]) / 2, [h[-1] / 2]))
    c = 1.0 / dist
    return sp.diags([c[:-1] + c[1:], -c[1:-1], -c[1:-1]], [0, 1, -1])


def mt2d(nl, nf, seed, real=False):
    """MT-like 5-point system on an nl x nf tensor mesh: a core of unit cells padded on every side by cells growing by 1.3,
    div-grad with the cell geometry as coefficients plus i omega mu0 sigma area on the diagonal, sigma log-uniform over four
    decades.  The real part is positive definite (weakly diagonally dominant off the boundary), so the pivot-free factorisation
    is well defined.  real=True: the real twin, omega mu0 sigma area added as a real shift."""
    rng = np.random.default_rng(seed)

    def widths(n):
        pad = min(6, n // 4)
        g = 1.3 ** np.arange(1, pad + 1)
        return np.concatenate((g[::-1], np.ones(n - 2 * pad), g))

    hl, hf = widths(nl), widths(nf)
    Ll, Lf = _laplacian_1d(hl), _laplacian_1d(hf)
    # q = l * nf + f: the geometric factors of a face (length / distance) from the Kronecker structure
    A = sp.kron(Ll, sp.diags(hf)) + sp.kron(sp.diags(hl), Lf)
    area = np.outer(hl, hf).ravel()
    sigma = 10.0 ** rng.uniform(-3.0, 1.0, nl * nf)
    shift = 2 * np.pi * 0.5 * MU0 * 1e6 * sigma * area          # omega mu0 sigma area, lengths in units of 1 km
    A = A + sp.diags(shift if real else 1j * shift)
    return sp.csc_matrix(A)


def divgrad3d(n1, n2, n3, seed, real=False):
    """3-D div-grad of MUMPS/test/getDivGrad.jl (7-point, Dirichlet) plus a random diagonal, imaginary (complex) or real"""
    def ddx(n):
        return sp.diags([-np.ones(n), np.ones(n)], [0, 1], shape=(n, n + 1))
    I = sp.identity
    D = sp.hstack([sp.kron(I(n3), sp.kron(I(n2), ddx(n1))), sp.kron(I(n3), sp.kron(ddx(n2), I(n1))),
                   sp.kron(ddx(n3), sp.kron(I(n2), I(n1)))])
    d = np.random.default_rng(seed).random(n1 * n2 * n3)
    return sp.csc_matrix(D @ D.T + sp.diags(d if real else 1j * d))


def hub(spokes, length, width, seed, real=False):
    """`spokes` strips of length x width grid nodes, each joined at one end to a hub node: the level-set bisection cuts the
    strips across, and the strips' far parts fall apart into components whose fronts are all children of one separator front"""
    rng = np.random.default_rng(seed)
    n = 1 + spokes * length * width
    rows, cols = [], []
    for s in range(spokes):
        base = 1 + s * length * width
        for a in range(length):
            for b in range(width):
                q = base + a * width + b
                if b + 1 < width:
                    rows.append(q); cols.append(q + 1)
                if a + 1 < length:
                    rows.append(q); cols.append(q + width)
                if a == 0:
                    rows.append(0); cols.append(q)
    W = sp.coo_matrix((np.ones(len(rows)), (rows, cols)), shape=(n, n))
    W = (W + W.T).tocsr()
    L = sp.diags(np.asarray(W.sum(axis=1)).ravel()) - W
    d = 0.5 + rng.random(n)
    return sp.csc_matrix(L + sp.diags(d if real else 1j * d))


# name -> (builder, classes the matrix is declared to reach over ROUTINGS); real=True builds the real twin of the same pattern
CASES = {
    "mt2d_37x53": (lambda real=False: mt2d(37, 53, 1, real),
                   {"w1", "w2", "w4", "w8", "w16", "mid_cpiv_part", "mid_cpiv_all", "npb1", "nub0", "big_fp", "big_children",
                    "chunks1", "root_mr0", "ws8", "ws16", "ws32", "ws_u_gt40", "cta128", "cta256"}),
    "mt2d_21x19": (lambda real=False: mt2d(21, 19, 2, real),
                   {"w1", "w2", "w4", "w8", "w16", "mid_cpiv_part", "mid_cpiv_all", "npb1", "nub0", "big_fp", "chunks1", "root_mr0",
                    "ws8", "ws16", "ws32", "cta128"}),
    "divgrad_20x20x20": (lambda real=False: divgrad3d(20, 20, 20, 3, real),
                         {"w1", "w2", "w4", "w8", "w16", "mid_cpiv_part", "npb1", "big_fp", "big_children", "chunks1", "chunks2",
                          "chunks3", "tail8", "root_mr0", "ws8", "ws16", "ws_u_gt40", "cta128", "cta256"}),
    "divgrad_9x10x11": (lambda real=False: divgrad3d(9, 10, 11, 4, real),
                        {"w1", "w2", "w4", "w8", "w16", "mid_cpiv_part", "mid_cpiv_all", "npb1", "nub0", "big_fp", "chunks1",
                         "root_mr0", "ws8", "ws16", "ws_u_gt40", "cta128", "cta256"}),
    "hub_7x9x3": (lambda real=False: hub(7, 9, 3, 5, real),
                  {"w1", "w2", "w4", "w8", "w16", "mid_cpiv_part", "mid_cpiv_all", "npb1", "big_fp", "big_children", "chunks1",
                   "root_mr0", "ws8", "ws16", "ws32", "cta128", "cta256"}),
}


def helper_exe(tmpdir):
    exe = os.path.join(str(tmpdir), "mf_classes")
    subprocess.run(["g++", "-O2", "-std=c++17", "-o", exe, os.path.join(ROOT, "tests", "cpp", "mf_classes.cpp")], check=True)
    return exe


def knob_values(env):
    """the helper's knob arguments for a routing (unset knobs at the library's defaults)"""
    v = dict(DEFAULTS)
    v.update(env)
    return [v[k] for k in KNOBS]


def run_helper(exe, A, env, tmpdir, tag):
    """fronts and depths of A's analysis under the knob settings env, as the Level-1 shim would build them"""
    A = sp.csc_matrix(A)
    A.sort_indices()
    path = os.path.join(str(tmpdir), f"{tag}.pattern")
    with open(path, "w") as f:
        f.write(f"{A.shape[0]}\n")
        f.write(" ".join(map(str, A.indptr + 1)) + "\n")
        f.write(" ".join(map(str, A.indices + 1)) + "\n")
    res = subprocess.run([exe, path, *knob_values(env)], capture_output=True, text=True)
    assert res.returncode == 0, res.stdout + res.stderr
    fronts, depths = [], []
    for line in res.stdout.splitlines():
        tok = line.split()
        rec = {tok[i]: tok[i + 1] for i in range(2, len(tok), 2)}
        for k, v in rec.items():
            if k not in ("why", "cpiv", "solve"):
                rec[k] = int(v)
        (fronts if tok[0] == "front" else depths).append(rec)
    return fronts, depths


def classes_of(fronts, depths):
    """kernel classes reached by one analysis + schedule"""
    c = set()
    for d in depths:
        if d["nSmall"]:
            c.add(f"w{d['warps']}")
        if d["nSolveCta"]:
            c.add(f"cta{d['threads']}")
    for f in fronts:
        if f["big"]:
            c.add("big_" + f["why"])
            c.add("chunks%d" % min(f["nChunk"], 3))
            if f["nChunk"] >= 2 and f["lastChunk"] == 8:
                c.add("tail8")
            if f["u"] == 0:
                c.add("root_mr0")
        else:
            if f["sp"] == 8:
                c.add("npb1")
            if f["u"] == 0:
                c.add("nub0")
            if f["warps"] >= 8 and f["cpiv"] != "-":
                for pc in f["cpiv"].split(","):
                    p, cu = map(int, pc.split("/"))
                    c.add("mid_cpiv_all" if p == cu else "mid_cpiv_part")
        if f["solve"] == "warp":
            c.add(f"ws{f['width']}")
            if f["u"] > 40:
                c.add("ws_u_gt40")
    return c
