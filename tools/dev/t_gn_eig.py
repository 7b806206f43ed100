"""The low-rank Gauss-Newton Hessian on one GPU (hmcmt_gn_eig) at cfg2 (synthetic.make_problem(200, 100, 30), 60 systems) and cfg4
(800 x 300 cells, 60 frequencies: all 120 systems on one GPU), at the homogeneous start model:

- one hmcmt_gn_eig call for r = 32 and 64 (k = r / 2), split into its Gauss-Newton products (r + r' Plan.gn_hessvec-equivalent
  products, timed as gn_hessvec calls), its r Wm solves (timed as one-step drifts with mass kind 1 minus kind 0) and the rest
  (the small kernels, by difference);
- leapfrog steps/s at cfg2 with mass kinds 0, 1 and 2 (leapfrog_steps_device, 20 steps per call).

Host clock around the calls (each ends in a stream synchronisation), after a warm-up call of each, medians of `rounds` rounds.
Prints the card and its power limit beside the numbers.

    python tools/dev/t_gn_eig.py [rounds] [cfg2|cfg4|both]
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
STEPS = 20


def timed(fn):
    t0 = time.perf_counter()
    fn()
    return 1000.0 * (time.perf_counter() - t0)


def med(fn, rounds):
    fn()
    return float(np.median([timed(fn) for _ in range(rounds)]))


def run(cfg, rounds):
    ny, nz, nf, nrx = CONFIGS[cfg]
    mesh, data, inv, prior = synthetic.make_problem(ny, nz, nf, nrx)
    pl = api.Plan(mesh, data, inv, prior)
    m0 = np.array(inv.strModel)
    p0 = np.random.default_rng(1).standard_normal(pl.nAC)
    pl.forward_gradient(m0)
    v = np.random.default_rng(3).standard_normal(pl.nAC)
    out = dict(config=cfg, mesh=f"{ny}x{nz} cells", systems=pl.info(7), nAC=pl.nAC, solver="multifrontal" if pl.info(11) else "band",
               rounds=rounds)
    out["gn_hessvec_ms"] = med(lambda: pl.gn_hessvec(v), rounds)
    # one Wm solve: a 1-step drift with M = Wm minus the same with M = I (one solve each for the drift and the energies' kinetic
    # term would be two; leapfrog_steps_device drifts once per step)
    def steps(kind, n):
        pl.set_mass_matrix(kind)
        pl.set_state(m0, 0.01 * p0, m0)
        pl.leapfrog_steps_device(1e-3, n)
    t0, t1 = med(lambda: steps(0, 1), rounds), med(lambda: steps(1, 1), rounds)
    out["wm_solve_ms"] = max(t1 - t0, 0.0)
    pl.set_mass_matrix(0)
    for r in (32, 64):
        k = r // 2
        om = np.random.default_rng(r).standard_normal((1, r, pl.nAC))
        pl.forward_gradient(m0)
        res = {}
        t = med(lambda: res.update(zip(("lam", "V", "info"), pl.gn_eig(k, r, omega=om))), rounds)
        rk = int(res["info"][0, 0])
        prod = (r + rk) * out["gn_hessvec_ms"]
        solves = r * out["wm_solve_ms"]
        out[f"r{r}"] = dict(k=k, total_ms=round(t, 2), info=[int(x) for x in res["info"][0]], gn_products_ms=round(prod, 2),
                            wm_solves_ms=round(solves, 2), rest_ms=round(t - prod - solves, 2),
                            lam_head=[float(x) for x in res["lam"][0, :4]])
    if cfg == "cfg2":
        pl.forward_gradient(m0)
        pl.gn_eig(16, 32, seed=0)
        for kind in (0, 1, 2):
            ms = med(lambda: steps(kind, STEPS), rounds)
            out[f"steps_per_s_kind{kind}"] = round(STEPS / (ms / 1000.0), 1)
    assert pl.status() == 0
    pl.close()
    return out


def main(rounds=5, which="both"):
    name, limit = card()
    res = [run(c, rounds) for c in (["cfg2", "cfg4"] if which == "both" else [which])]
    for r in res:
        print(f"{r['config']} ({r['mesh']}, {r['systems']} systems, nAC {r['nAC']}, {r['solver']}): gn_hessvec {r['gn_hessvec_ms']:.3f} ms, "
              f"Wm solve {r['wm_solve_ms']:.3f} ms")
        for key in ("r32", "r64"):
            x = r[key]
            print(f"   {key}: gn_eig {x['total_ms']} ms = GN products {x['gn_products_ms']} + Wm solves {x['wm_solves_ms']} + rest "
                  f"{x['rest_ms']} (info {x['info']})")
        if "steps_per_s_kind0" in r:
            print(f"   leapfrog steps/s: kind 0 {r['steps_per_s_kind0']}, kind 1 {r['steps_per_s_kind1']}, kind 2 {r['steps_per_s_kind2']}")
    print(f"card {name}, power limit {limit}")
    print(json.dumps(dict(card=name, power_limit=limit, results=res)))


if __name__ == "__main__":
    main(int(sys.argv[1]) if len(sys.argv) > 1 else 5, sys.argv[2] if len(sys.argv) > 2 else "both")
