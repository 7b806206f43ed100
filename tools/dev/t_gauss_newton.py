"""Projected Gauss-Newton-CG on one GPU (hmcmt_gauss_newton) at cfg2 (synthetic.make_problem(200, 100, 30), 60 systems) and
cfg4 (800 x 300 cells, 60 frequencies: all 120 systems on one GPU), data of synthetic.true_model with 5 % noise
(synthetic.true_model_data), started from the homogeneous model:

- one CG iteration inside hmcmt_gauss_newton: (t(max_cg = 12) - t(max_cg = 2)) / 10 of one-iteration runs with one line-search
  trial, against one Plan.gn_hessvec call (what a host CG loop pays per iteration for the product alone);
- one outer iteration with the default options: t(max_iter = 1) - t(max_iter = 0);
- a 10-iteration run: its time, and U = phi_d + phi_m and |P g| per iteration.

Host clock around the calls (each ends in a stream synchronisation), after a warm-up call of each, medians of `rounds` rounds
with the variants alternated.  Prints the card and its power limit beside the numbers.

    python tools/dev/t_gauss_newton.py [rounds] [cfg2|cfg4|both]
"""
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from hmcmt2d_b200 import api, synthetic  # noqa: E402
from tools.dev.t_rho_phase import card  # noqa: E402

CONFIGS = {"cfg2": (200, 100, 30, 40), "cfg4": (800, 300, 60, 40)}


def timed(fn):
    t0 = time.perf_counter()
    fn()
    return 1000.0 * (time.perf_counter() - t0)


def run(cfg, rounds):
    ny, nz, nf, nrx = CONFIGS[cfg]
    mesh, data, inv, prior = synthetic.make_problem(ny, nz, nf, nrx)
    fw = api.Plan(mesh, data, inv, prior)
    obs, err = synthetic.true_model_data(data, fw.forward(sigma=synthetic.true_model(mesh), fields=False)[0][0])
    fw.close()
    mesh, data, inv, prior = synthetic.make_problem(ny, nz, nf, nrx, obs=obs, err=err)
    pl = api.Plan(mesh, data, inv, prior)
    m0 = np.array(inv.strModel)
    v = np.random.default_rng(3).standard_normal(pl.nAC)
    pl.forward_gradient(m0)
    calls = {"gn_hessvec": lambda: pl.gn_hessvec(v, total=True),
             "cg2": lambda: pl.gauss_newton(m0, max_iter=1, max_cg=2, max_ls=1),
             "cg12": lambda: pl.gauss_newton(m0, max_iter=1, max_cg=12, max_ls=1),
             "iter0": lambda: pl.gauss_newton(m0, max_iter=0),
             "iter1": lambda: pl.gauss_newton(m0, max_iter=1)}
    for fn in calls.values():
        fn()
    t = {k: [] for k in calls}
    for _ in range(rounds):
        for k, fn in calls.items():
            t[k].append(timed(fn))
    med = {k: float(np.median(x)) for k, x in t.items()}
    _, h1, _ = pl.gauss_newton(m0, max_iter=1)
    t0 = time.perf_counter()
    m, h, info = pl.gauss_newton(m0, max_iter=10)
    t10 = 1000.0 * (time.perf_counter() - t0)
    n = int(info[0, 0])
    out = dict(config=cfg, mesh=f"{ny}x{nz} cells", frequencies=nf, receivers=nrx, systems=pl.info(7), nAC=pl.nAC, nData=pl.nData,
               solver="multifrontal" if pl.info(11) else "band", rounds=rounds,
               raw_ms={k: [round(x, 3) for x in v_] for k, v_ in t.items()},
               gn_hessvec_call_ms=round(med["gn_hessvec"], 3), cg_iteration_ms=round((med["cg12"] - med["cg2"]) / 10, 3),
               outer_iteration_ms=round(med["iter1"] - med["iter0"], 3), outer_iteration_trials=int(h1[0, 1, 5]),
               outer_iteration_cg=int(h1[0, 1, 3]), run10_ms=round(t10, 1), run10_info=[int(x) for x in info[0]],
               run10_U=[float(x) for x in h[0, : n + 1, 0] + h[0, : n + 1, 1]], run10_Pg=[float(x) for x in h[0, : n + 1, 2]],
               run10_trials=[int(x) for x in h[0, 1 : n + 1, 5]], run10_cg=[int(x) for x in h[0, 1 : n + 1, 3]])
    assert pl.status() == 0
    pl.close()
    return out


def main(rounds=5, which="both"):
    name, limit = card()
    res = [run(c, rounds) for c in (["cfg2", "cfg4"] if which == "both" else [which])]
    for r in res:
        print(f"{r['config']} ({r['mesh']}, {r['systems']} systems, {r['solver']}): CG iteration in gauss_newton {r['cg_iteration_ms']} ms, "
              f"gn_hessvec call {r['gn_hessvec_call_ms']} ms, outer iteration {r['outer_iteration_ms']} ms "
              f"({r['outer_iteration_cg']} CG, {r['outer_iteration_trials']} trials), 10-iteration run {r['run10_ms']} ms, info {r['run10_info']}")
        for k, (u, g) in enumerate(zip(r["run10_U"], r["run10_Pg"])):
            print(f"   it {k}: U {u:.6e}  |P g| {g:.6e}")
    print(f"card {name}, power limit {limit}")
    print(json.dumps(dict(card=name, power_limit=limit, results=res)))


if __name__ == "__main__":
    main(int(sys.argv[1]) if len(sys.argv) > 1 else 5, sys.argv[2] if len(sys.argv) > 2 else "both")
