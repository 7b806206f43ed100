"""Mid-size fronts of one cfg2 gradient evaluation (synthetic.make_problem(200, 100, 30), stress model), un-grouped and eagerly
launched (HMCMT_GROUPS=1 HMCMT_GRAPH=0), for two source trees alternated: `mf_small_kernel<8>` / `<16>` times from
torch.profiler (CUDA activities, summed over `reps` evaluations and divided by reps), the evaluation time from CUDA events on the
plan's stream, and the HMCMT_MF_PROF=1 phase cycles per front of every mf_small_kernel instantiation (a separate run: the
counters slow the kernels).  Each tree runs in its own process, built in place.  Prints the card and its power limit beside the
numbers, and whether both trees gave the same bits.

    python tools/dev/t_mid_fronts.py <other tree> [reps] [rounds]
"""
import json
import os
import subprocess
import sys
import tempfile
from collections import defaultdict

import numpy as np

HERE = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def child(tree, reps, out):
    os.environ["HMCMT_GROUPS"] = "1"
    os.environ["HMCMT_GRAPH"] = "0"
    sys.path.insert(0, tree)
    import torch
    from torch.profiler import ProfilerActivity, profile
    from hmcmt2d_b200 import api, synthetic
    mesh, data, inv, prior = synthetic.make_problem(200, 100, 30)
    m = synthetic.stress_model(inv)
    pl = api.Plan(mesh, data, inv, prior)
    res = {}
    if os.environ.get("HMCMT_MF_PROF"):
        pl.forward_gradient(m)
    else:
        for _ in range(3):
            pl.forward_gradient(m)
        pl.timer_start()
        outs = [pl.forward_gradient(m) for _ in range(reps)]
        res["eval_ms"] = pl.timer_stop() / reps
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(reps):
                pl.forward_gradient(m)
            torch.cuda.synchronize()
        acc = defaultdict(float)
        for e in prof.key_averages():
            for nw in (1, 2, 4, 8, 16):
                if f"mf_small_kernel<{nw}>" in e.key:
                    acc[f"mf_small_kernel<{nw}>"] += e.device_time_total / 1000.0 / reps
        res["kernels_ms"] = dict(acc)
        np.save(out + ".npy", np.concatenate([np.ascontiguousarray(x).ravel().view(np.float64) for x in outs[-1]]))
    pl.close()
    with open(out + ".json", "w") as f:
        json.dump(res, f)


def run(tree, reps, tmp, tag, prof=False):
    env = dict(os.environ)
    if prof:
        env["HMCMT_MF_PROF"] = "1"
    subprocess.run([sys.executable, "-c", f"import sys; sys.path.insert(0, {tree!r}); import __graft_entry__ as g; g.build()"],
                   cwd=tree, env=env, check=True, capture_output=True)
    out = os.path.join(tmp, tag)
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", tree, str(reps), out], env=env, capture_output=True, text=True)
    if r.returncode:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError(f"{tree} failed")
    with open(out + ".json") as f:
        res = json.load(f)
    if prof:
        res["phases"] = [ln.split("] ", 1)[-1] for ln in r.stderr.splitlines() if "cycles per" in ln]
    return res


def main(other, reps=20, rounds=3):
    import torch
    trees = {"this": HERE, "other": os.path.abspath(other)}
    res = {k: defaultdict(list) for k in trees}
    with tempfile.TemporaryDirectory() as tmp:
        for r in range(rounds):
            for k, t in trees.items():
                x = run(t, reps, tmp, k)
                res[k]["eval_ms"].append(round(x["eval_ms"], 4))
                for n, v in x["kernels_ms"].items():
                    res[k][n].append(round(v, 4))
        same = np.array_equal(np.load(os.path.join(tmp, "this.npy")), np.load(os.path.join(tmp, "other.npy")))
        phases = {k: run(t, 1, tmp, k + "_prof", prof=True)["phases"] for k, t in trees.items()}
    name = torch.cuda.get_device_name(0)
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = "unknown"
    for k in trees:
        print(f"{k:6s} {dict(res[k])}")
        for ln in phases[k]:
            print(f"       {ln}")
    print(f"bit-identical outputs: {same}; card {name}, power limit {limit}")
    print(json.dumps(dict(card=name, power_limit=limit, reps=reps, rounds=rounds, bit_identical=same, trees=trees,
                          workload="cfg2 200x100 cells, 30 frequencies, TE+TM, stress model, one gradient evaluation, "
                                   "HMCMT_GROUPS=1 HMCMT_GRAPH=0", **{k: dict(v) for k, v in res.items()}, phases=phases)))


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "--child":
        child(sys.argv[2], int(sys.argv[3]), sys.argv[4])
    else:
        main(sys.argv[1], *[int(a) for a in sys.argv[2:4]])
