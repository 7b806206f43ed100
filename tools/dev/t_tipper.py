"""Device-resident leapfrog rate of the cfg2 workload (synthetic.make_problem(200, 100, 30), stress model) with impedance data
and with the same survey plus TZY rows (synthetic.tipper_problem: the tipper of the device forward of true_model, absolute error
0.02), both plans in one process, alternated for `rounds` rounds after warm-up.  ms / step from CUDA events on the plan's stream
(timer_start / timer_stop around leapfrog_steps_device).  Prints the card and its power limit beside the numbers, and the largest
difference of the final states between the rounds of each plan (0: graph replay is deterministic).

    python tools/dev/t_tipper.py [steps] [warmup] [rounds]
"""
import copy
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from hmcmt2d_b200 import api, synthetic  # noqa: E402
from tools.dev.t_rho_phase import card  # noqa: E402


def main(steps=20, warmup=3, rounds=3):
    mesh, data, inv, prior = synthetic.make_problem(200, 100, 30)
    m0 = synthetic.stress_model(inv)
    p0 = np.clip(np.random.default_rng(0).standard_normal(len(m0)), -2.5, 2.5)
    d0, _ = synthetic.tipper_problem(data, inv, np.zeros(len(data.freqs) * data.rxLoc.shape[0]))
    tm = copy.copy(mesh)
    tm.sigma = synthetic.true_model(mesh)
    pred, _ = api.MT2DFwdSolver(tm, d0)
    tdata, tinv = synthetic.tipper_problem(data, inv, pred[d0.dtID == 3])
    plans = {"impedance": api.Plan(mesh, data, inv, prior), "tipper": api.Plan(mesh, tdata, tinv, prior)}

    def run(pl, n):
        pl.set_state(m0, p0, m0)
        pl.timer_start()
        pl.leapfrog_steps_device(prior.dt, n)
        ms = pl.timer_stop()
        status = pl.status()
        m, p = pl.get_state()
        return ms / n, status, np.concatenate([m[0], p[0]])

    for pl in plans.values():
        run(pl, warmup)
    times = {k: [] for k in plans}
    finals = {k: [] for k in plans}
    statuses = {k: set() for k in plans}
    for _ in range(rounds):
        for k, pl in plans.items():
            ms, st, state = run(pl, steps)
            times[k].append(ms)
            finals[k].append(state)
            statuses[k].add(st)
    name, limit = card()
    out = dict(card=name, power_limit=limit, workload="cfg2 200x100 cells, 30 frequencies, TE+TM, 40 receivers, stress model; "
               "tipper: the same survey + TZY at every (frequency, receiver)", steps=steps, warmup=warmup, rounds=rounds)
    for k in plans:
        t = np.array(times[k])
        out[k] = dict(ms_per_step=[round(float(v), 4) for v in t], median_ms=round(float(np.median(t)), 4),
                      steps_per_s=round(1000.0 / float(np.median(t)), 2), spread_pct=round(100.0 * float(t.max() - t.min()) / float(t.min()), 2),
                      max_final_state_diff=float(max(np.abs(f - finals[k][0]).max() for f in finals[k])), status=sorted(statuses[k]))
        print(f"{k:10s} ms/step {out[k]['ms_per_step']}  median {out[k]['median_ms']} ms = {out[k]['steps_per_s']} steps/s  "
              f"spread {out[k]['spread_pct']} %  final-state diff between rounds {out[k]['max_final_state_diff']}  status {out[k]['status']}")
    print(f"card {name}, power limit {limit}")
    print(json.dumps(out))
    for pl in plans.values():
        pl.close()


if __name__ == "__main__":
    main(*(int(a) for a in sys.argv[1:4]))
