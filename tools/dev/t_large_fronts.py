"""Fronts above 144 rows on the single-CTA path: one gradient evaluation of cfg2 (synthetic.make_problem(200, 100, 30)) or cfg4
(800, 300, 60), stress model, un-grouped and eagerly launched (HMCMT_GROUPS=1 HMCMT_GRAPH=0), for several settings alternated,
each in its own process: two source trees (this one and `--other TREE`, e.g. the parent commit, built in place), or several
HMCMT_MF_FSMALL values in this tree (`--fsmall 144 152 208 256`).  Reports per setting
  * the factorisation time per evaluation from the plan's factor timing (CUDA events around the factorisation alone),
  * the evaluation time (CUDA events on the plan's stream),
  * the per-kernel device times of the factorisation from torch.profiler (CUDA activities, a separate pass),
and the card and its power limit, and the largest relative difference of predicted data, misfit and gradient against the first
setting.

    python tools/dev/t_large_fronts.py [--config cfg2|cfg4] [--other TREE | --fsmall V ...] [--reps N] [--rounds R]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
from collections import defaultdict

import numpy as np

HERE = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
SIZES = {"cfg2": (200, 100, 30), "cfg4": (800, 300, 60)}
KERNELS = ("mf_small_kernel", "mf_small_stream_kernel", "mf_asm_gather_kernel", "mf_asm_orig_kernel", "mf_inv_kernel", "mf_gemm_kernel")


def child(tree, config, reps, out):
    os.environ["HMCMT_GROUPS"] = "1"
    os.environ["HMCMT_GRAPH"] = "0"
    sys.path.insert(0, tree)
    import torch
    from torch.profiler import ProfilerActivity, profile
    from hmcmt2d_b200 import api, synthetic
    mesh, data, inv, prior = synthetic.make_problem(*SIZES[config])
    m = synthetic.stress_model(inv)
    pl = api.Plan(mesh, data, inv, prior)
    for _ in range(3):
        pl.forward_gradient(m)
    res = {}
    pl.kernel_time(reset=1)
    for _ in range(reps):
        pl.forward_gradient(m)
    res["factor_ms"] = pl.kernel_time_split()[0] / reps
    pl.kernel_time(reset=-1)
    pl.timer_start()
    outs = [pl.forward_gradient(m) for _ in range(reps)]
    res["eval_ms"] = pl.timer_stop() / reps
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            pl.forward_gradient(m)
        torch.cuda.synchronize()
    acc = defaultdict(float)
    for e in prof.key_averages():
        for k in KERNELS:
            if e.key.startswith(k + "<") or e.key.startswith(k + "(") or e.key == k or ("::" + k + "(") in e.key or ("::" + k + "<") in e.key:
                name = e.key.split("(")[0].replace("hmcmt::mf::", "").replace("void ", "")
                acc[name] += e.device_time_total / 1000.0 / reps
    res["kernels_ms"] = dict(acc)
    pred, phi, g = outs[-1]
    np.savez(out + ".npz", pred=np.asarray(pred), phi=np.asarray(phi), g=np.asarray(g))
    pl.close()
    with open(out + ".json", "w") as f:
        json.dump(res, f)


def run(tree, config, reps, env_extra, tmp, tag):
    env = dict(os.environ, **env_extra)
    subprocess.run([sys.executable, "-c", f"import sys; sys.path.insert(0, {tree!r}); import __graft_entry__ as g; g.build()"],
                   cwd=tree, env=env, check=True, capture_output=True)
    out = os.path.join(tmp, tag)
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", tree, config, str(reps), out], env=env,
                       capture_output=True, text=True)
    if r.returncode:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError(f"{tag} failed")
    with open(out + ".json") as f:
        return json.load(f)


def rel_diff(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-300))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="cfg2", choices=sorted(SIZES))
    ap.add_argument("--other")
    ap.add_argument("--fsmall", nargs="*", default=[])
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    if a.other:
        settings = {"this": (HERE, {}), "other": (os.path.abspath(a.other), {})}
    else:
        settings = {f"fsmall{v}": (HERE, {"HMCMT_MF_FSMALL": v}) for v in (a.fsmall or ["144", "256"])}
    import torch
    res = {k: defaultdict(list) for k in settings}
    with tempfile.TemporaryDirectory() as tmp:
        for _ in range(a.rounds):
            for k, (tree, env) in settings.items():
                x = run(tree, a.config, a.reps, env, tmp, k)
                res[k]["factor_ms"].append(round(x["factor_ms"], 4))
                res[k]["eval_ms"].append(round(x["eval_ms"], 4))
                for n, v in x["kernels_ms"].items():
                    res[k][n].append(round(v, 4))
        first = next(iter(settings))
        ref = np.load(os.path.join(tmp, first + ".npz"))
        diffs = {}
        for k in settings:
            o = np.load(os.path.join(tmp, k + ".npz"))
            diffs[k] = {n: rel_diff(o[n], ref[n]) for n in ("pred", "phi", "g")}
    name = torch.cuda.get_device_name(0)
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = "unknown"
    for k in settings:
        print(f"{k:10s} {dict(res[k])}  rel. diff vs {first}: {diffs[k]}")
    print(f"card {name}, power limit {limit}")
    print(json.dumps(dict(card=name, power_limit=limit, config=a.config, reps=a.reps, rounds=a.rounds,
                          settings={k: dict(tree=t, env=e) for k, (t, e) in settings.items()},
                          workload=f"{a.config} {SIZES[a.config]}, TE+TM, stress model, one gradient evaluation, HMCMT_GROUPS=1 HMCMT_GRAPH=0",
                          results={k: dict(v) for k, v in res.items()}, rel_diff=diffs)))


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "--child":
        child(sys.argv[2], sys.argv[3], int(sys.argv[4]), sys.argv[5])
    else:
        main()
