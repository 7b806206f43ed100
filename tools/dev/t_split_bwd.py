"""Backward-substitution time of one cfg2 gradient evaluation (synthetic.make_problem(200, 100, 30), stress model), un-grouped
and eagerly launched (HMCMT_GROUPS=1 HMCMT_GRAPH=0): the split order of the gradient evaluation (receiver path of x, then the
paired sweep over x and lam) against the complete solves one after the other, which the same plan runs while its factorisation
is being timed (Plan.kernel_time(reset=1)).  Kernel times from torch.profiler (CUDA activities), summed per solve kernel over
`reps` evaluations and divided by reps; evaluation time from CUDA events on the plan's stream (timer_start / timer_stop).  The
two orders alternate for `rounds` rounds.  Prints the card and its power limit beside the numbers, and whether both orders gave
the same bits.

    python tools/dev/t_split_bwd.py [reps] [rounds]
"""
import json
import os
import subprocess
import sys
from collections import defaultdict

import numpy as np

os.environ["HMCMT_GROUPS"] = "1"
os.environ["HMCMT_GRAPH"] = "0"
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from hmcmt2d_b200 import api, synthetic  # noqa: E402


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = "unknown"
    return name, limit


def main(reps=20, rounds=3):
    import torch
    from torch.profiler import ProfilerActivity, profile
    mesh, data, inv, prior = synthetic.make_problem(200, 100, 30)
    m = synthetic.stress_model(inv)
    pl = api.Plan(mesh, data, inv, prior)

    def route(complete):
        pl.kernel_time(reset=1 if complete else -1)

    def evaluate(complete, n):
        route(complete)
        pl.timer_start()
        outs = [pl.forward_gradient(m) for _ in range(n)]
        return pl.timer_stop() / n, outs[-1]

    def kernels(complete):
        route(complete)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(reps):
                pl.forward_gradient(m)
            torch.cuda.synchronize()
        acc = defaultdict(float)
        for e in prof.key_averages():
            name = e.key
            for k in ("mf_bwd_pair_warp_kernel", "mf_bwd_pair_kernel", "mf_bwd_warp_kernel", "mf_bwd_kernel",
                      "mf_fwd_warp_kernel", "mf_fwd_kernel"):
                if k + "(" in name or name.endswith(k):
                    acc[k] += e.device_time_total / 1000.0 / reps
                    break
        return dict(acc)

    for c in (False, True):
        evaluate(c, 3)
    res = {"split": defaultdict(list), "complete": defaultdict(list)}
    outs = {}
    for _ in range(rounds):
        for key, c in (("split", False), ("complete", True)):
            ms, outs[key] = evaluate(c, reps)
            res[key]["eval_ms"].append(round(ms, 4))
            k = kernels(c)
            res[key]["bwd_ms"].append(round(sum(v for n, v in k.items() if "bwd" in n), 4))
            res[key]["fwd_ms"].append(round(sum(v for n, v in k.items() if "fwd" in n), 4))
            res[key]["kernels_ms"] = {n: round(v, 4) for n, v in sorted(k.items())}
    route(False)
    same = all(np.array_equal(a, b) for a, b in zip(outs["split"], outs["complete"]))
    pl.close()
    name, limit = card()
    out = dict(card=name, power_limit=limit, workload="cfg2 200x100 cells, 30 frequencies, TE+TM, 40 receivers, stress model, "
               "one gradient evaluation, HMCMT_GROUPS=1 HMCMT_GRAPH=0", reps=reps, rounds=rounds, bit_identical=same,
               **{k: dict(v) for k, v in res.items()})
    for k in ("split", "complete"):
        print(f"{k:9s} evaluation ms {res[k]['eval_ms']}  backward sweeps ms {res[k]['bwd_ms']}  forward eliminations ms {res[k]['fwd_ms']}")
        print(f"          per kernel (last round) {res[k]['kernels_ms']}")
    print(f"bit-identical outputs: {same}; card {name}, power limit {limit}")
    print(json.dumps(out))


if __name__ == "__main__":
    main(*[int(a) for a in sys.argv[1:3]])
