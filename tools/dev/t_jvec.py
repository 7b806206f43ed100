"""Call times of the derivative entry points on one GPU: hmcmt_jvec (J dsig), hmcmt_gn_hessvec (D Re(J^H Wd^2 J) D v),
hmcmt_jtvec (Re J^T conj w) and one hmcmt_forward_gradient (graph replay), at cfg2 (synthetic.make_problem(200, 100, 30), 60
systems) and cfg4 (800 x 300 cells, 60 frequencies: all 120 systems on one GPU), stress model; hmcmt_jacobian at cfg2 as well.
Host clock around the calls, each of which ends in a stream synchronisation (they return host buffers), after two warm-up calls
of each, `rounds` rounds with the entry points alternated.  Prints the card and its power limit beside the numbers.

    python tools/dev/t_jvec.py [rounds] [cfg2|cfg4|both]
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
    pl = api.Plan(mesh, data, inv, prior)
    m = synthetic.stress_model(inv)
    rng = np.random.default_rng(3)
    dsig = rng.standard_normal(pl.nAC) * np.exp(m)
    v = rng.standard_normal(pl.nAC)
    w = rng.standard_normal(pl.nData) + 1j * rng.standard_normal(pl.nData)
    calls = {"forward_gradient": lambda: pl.forward_gradient(m), "jvec": lambda: pl.jvec(dsig),
             "gn_hessvec": lambda: pl.gn_hessvec(v), "jtvec": lambda: pl.jtvec(w)}
    for _ in range(2):
        for fn in calls.values():
            fn()
    t = {k: [] for k in calls}
    for _ in range(rounds):
        for k, fn in calls.items():
            t[k].append(timed(fn))
    out = dict(config=cfg, mesh=f"{ny}x{nz} cells", frequencies=nf, receivers=nrx, systems=pl.info(7), nAC=pl.nAC, nData=pl.nData,
               solver="multifrontal" if pl.info(11) else "band", rounds=rounds)
    for k, v_ in t.items():
        out[k] = dict(ms=[round(x, 3) for x in v_], median_ms=round(float(np.median(v_)), 3))
    if cfg == "cfg2":
        pl.forward_gradient(m)
        pl.jacobian()
        out["jacobian"] = dict(ms=[round(timed(pl.jacobian), 1) for _ in range(2)])
        out["jacobian"]["median_ms"] = float(np.median(out["jacobian"]["ms"]))
    assert pl.status() == 0
    pl.close()
    return out


def main(rounds=5, which="both"):
    name, limit = card()
    res = [run(c, rounds) for c in (["cfg2", "cfg4"] if which == "both" else [which])]
    for r in res:
        line = "  ".join(f"{k} {r[k]['median_ms']} ms" for k in ("forward_gradient", "jvec", "gn_hessvec", "jtvec", "jacobian") if k in r)
        print(f"{r['config']} ({r['mesh']}, {r['systems']} systems, {r['solver']}): {line}")
    print(f"card {name}, power limit {limit}")
    print(json.dumps(dict(card=name, power_limit=limit, results=res)))


if __name__ == "__main__":
    main(int(sys.argv[1]) if len(sys.argv) > 1 else 5, sys.argv[2] if len(sys.argv) > 2 else "both")
