"""Selected inversion (hmcmt_factor_inverse_diag / lib.inverse_diag) on one GPU at the size of the plan's Wm: a five-point
operator on an active-cell grid of cfg2 size (200 x 93 = 18 600 cells) and of cfg4 size (800 x 293 = 234 400 cells), real
symmetric positive definite (graph Laplacian + 1e-2 on the diagonal), factorised on the multifrontal path (HMCMT_SHIM_SOLVER=mf).

CUDA events on the default stream (the stream the Level-1 entries launch on) around factorMUMPS and around inverse_diag, after a
warm-up call of each, medians of `rounds` rounds.  Both calls include their host work (factorMUMPS: conversion of the values and
the host-to-device copy; inverse_diag: the output buffer and its device-to-host copy of n values), so the sweep's rate is a lower
bound.  Reports the flop counts of the factorisation and of the sweep (padded front sizes), TFLOP/s against them, the sweep's
bit-identity across rounds, and the card and its power limit.

Then the plan (synthetic.make_problem at cfg2 200 x 100 and cfg4 800 x 300 cells, two frequencies: the Wm parts do not depend on
them), host clock around calls that end in a stream synchronisation:
  - set_mass_matrix(1) on a fresh plan: the plan's Wm set-up (analysis on the host, upload, multifrontal factorisation, banded
    Cholesky);
  - the first hmcmt_posterior_variance (prior only) after it: inverse_diag of the plan's Wm factor, kept on the plan, and the copy;
  - a later call with all three outputs after gn_eig(16, 32): the combine kernels alone (medians of `rounds`).

    python tools/dev/t_selinv.py [rounds] [cfg2|cfg4|both]
"""
import json
import os
import sys

import numpy as np
import scipy.sparse as sp

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from hmcmt2d_b200 import lib  # noqa: E402
from tools.dev.t_rho_phase import card  # noqa: E402

CONFIGS = {"cfg2": (200, 93), "cfg4": (800, 293)}


def wm_like(nl, nf):
    def lap(n):
        return sp.diags([2.0 * np.ones(n), -np.ones(n - 1), -np.ones(n - 1)], [0, 1, -1])
    A = sp.kron(lap(nl), sp.identity(nf)) + sp.kron(sp.identity(nl), lap(nf)) + 1e-2 * sp.identity(nl * nf)
    return sp.csc_matrix(A)


def run(cfg, rounds):
    import torch
    nl, nf = CONFIGS[cfg]
    A = wm_like(nl, nf)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    tf, ts, ref = [], [], None
    fl = np.zeros(2)
    for r in range(rounds + 1):
        torch.cuda.synchronize()
        ev[0].record()
        F = lib.factorMUMPS(A, 1)
        ev[1].record()
        ev[2].record()
        d = lib.inverse_diag(F)
        ev[3].record()
        torch.cuda.synchronize()
        h = lib.C.c_int64(F.ptr)
        lib.check(lib.load().hmcmt_debug_factor_flops(lib.C.byref(h), fl.ctypes.data_as(lib._f64p)), "hmcmt_debug_factor_flops")
        lib.destroyMUMPS(F)
        if r == 0:
            ref = d
            continue
        tf.append(ev[0].elapsed_time(ev[1]))
        ts.append(ev[2].elapsed_time(ev[3]))
        assert np.array_equal(d, ref)
    f_ms, s_ms = float(np.median(tf)), float(np.median(ts))
    return dict(config=cfg, n=nl * nf, rounds=rounds, factor_ms=round(f_ms, 3), inverse_diag_ms=round(s_ms, 3),
                ratio=round(s_ms / f_ms, 2), factor_gflop=round(fl[0] / 1e9, 3), selinv_gflop=round(fl[1] / 1e9, 3),
                factor_tflops=round(fl[0] / f_ms / 1e9, 3), selinv_tflops=round(fl[1] / s_ms / 1e9, 3),
                diag_min=float(d.min()), diag_max=float(d.max()), bit_identical_rounds=True)


def run_plan(cfg, rounds):
    import time
    from hmcmt2d_b200 import api, synthetic
    ny, nz = {"cfg2": (200, 100), "cfg4": (800, 300)}[cfg]
    mesh, data, inv, prior = synthetic.make_problem(ny, nz, 2)
    pl = api.Plan(mesh, data, inv, prior)

    def timed(fn):
        t0 = time.perf_counter()
        fn()
        return 1000.0 * (time.perf_counter() - t0)
    t_wm = timed(lambda: pl.set_mass_matrix(1))
    t_first = timed(lambda: pl.posterior_variance(prior=True, posterior=False, resolution=False))
    pl.set_mass_matrix(0)
    pl.forward(m=np.array(inv.strModel), fields=False)
    pl.gn_eig(16, 32, seed=1)
    pl.posterior_variance()
    t_call = float(np.median([timed(lambda: pl.posterior_variance()) for _ in range(rounds)]))
    out = dict(config=cfg + " plan", nAC=pl.nAC, wm_setup_ms=round(t_wm, 2), first_posterior_variance_ms=round(t_first, 2),
               posterior_variance_k16_ms=round(t_call, 3))
    pl.close()
    return out


def main():
    rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 3
    which = sys.argv[2] if len(sys.argv) > 2 else "both"
    os.environ["HMCMT_SHIM_SOLVER"] = "mf"
    name, limit = card()
    print(f"[t_selinv] {name}, power limit {limit}")
    for cfg in (("cfg2", "cfg4") if which == "both" else (which,)):
        res = run(cfg, rounds)
        res.update(card=name, power_limit=limit)
        print(json.dumps(res))
        res = run_plan(cfg, rounds)
        res.update(card=name, power_limit=limit)
        print(json.dumps(res))


if __name__ == "__main__":
    main()
