#!/usr/bin/env python
"""bench.py — HMC leapfrog steps/s of the HMCMT2D forward + adjoint hot path on B200.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched by torchrun, one rank per GPU)
    python bench.py --impl reference --gpus N --steps K --warmup W

One "step" = one leapfrog step of the reference sampler (HMCSampler.jl:235-265): position drift with step clipping and bound
reflection, one compDataGradient-equivalent evaluation (forward + adjoint over all frequencies x TE/TM), prior gradient,
momentum kick.

Headline workload = BASELINE.json configs[1]/[2] ("cfg2"): synthetic 200x100-cell mesh, 30 frequencies, TE+TM, one independent
chain per GPU (weak scaling, no data-path collective: "replicas only", as parallelHMC.jl).  Observations = forward(true model)
(1 + 5 % noise), evaluation model = the stress model of SURVEY.md 8(d).

`value` : steps/s with the chain state resident in HBM (hmcmt_leapfrog_steps_device), CUDA events on the library's stream,
          max over ranks.
`e2e`   : the same step through the reference-facing call (compDataGradient-equivalent through the C ABI) with HOST buffers:
          the model goes host->device and predicted data / misfit / gradient come back every step; drift, bound reflection and
          kick run on the host as in the reference's proposeLeapfrog.  The gradient that comes back is data + model-norm part
          (hmcmt_forward_gradient_total: the library forms beta Wm (m - m_ref) on the device in every evaluation anyway).
`validated` : the device loop's error flags are clear, its states are finite, one device step and one host step from the same
          (m0, p0) agree to 1e-9, three steps to 1e-7, and the final states of the two timed arms (W+K steps each) are still on the
          same trajectory (the dynamics amplify round-off differences step by step: reported, bounded at 1e-2); on every rank.
`strong_scaling` : the SAME json line also carries BASELINE.json configs[3] ("cfg4": 800x300 cells, 60 frequencies, one chain,
          the 120 (frequency, mode) systems sharded over the N GPUs, one ncclAllReduce of [gradient | misfit] per step issued by
          the library on its own stream) with its own value / e2e / roofline / clocks, so that the driver's 1/2/4/8-GPU runs hold
          a strong-scaling curve next to the weak-scaling one.   `--config cfg4` prints that record as the main line instead.
`--dump-outputs DIR` : after the run, the chain state the last timed step of the main line left on the device (what
          hmcmt_get_state hands a caller of hmcmt_leapfrog_steps_device), rank 0's, as DIR/model.npy and DIR/momentum.npy (float64,
          [chains, active cells]).  The inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "leapfrog_steps_per_sec"
UNIT = "steps/s"
WORKLOAD = dict(workload="cfg2: synthetic 200x100-cell mesh, 30 frequencies, TE+TM, 1 HMC chain per GPU",
                ny=200, nz=100, nfreq=30, nrx=40, modes="TE+TM", chains_per_gpu=1)
CFG4 = dict(workload="cfg4: synthetic 800x300-cell mesh, 60 frequencies, TE+TM, 1 HMC chain, the 120 (frequency, mode) systems "
                     "sharded over the GPUs (one NCCL sum-all-reduce of [gradient | misfit] per step)",
            ny=800, nz=300, nfreq=60, nrx=40, modes="TE+TM", chains_per_gpu=1)
# dram__bytes_read + dram__bytes_write of the factorisation group per step at cfg2 (band kernel): FM_OWN capture + its
# back-substitution sweep, ncu --set full (profiles/r01_final_factor_own_ncu.txt, profiles/r01_final_solve_own_ncu.txt)
NCU_FACTOR_DRAM_BYTES = (24.28e6 + 2.250943e9) + (2.278771e9 + 23.64e6)
# the same for the multifrontal path at cfg2 (60 systems): the 59 launches from mf_mt_vals_kernel to the end of the forward solve,
# ncu dram__bytes_read.sum + dram__bytes_write.sum per launch (profiles/r02_cfg2_launches.csv, summary beside it)
NCU_MF_FACTOR_DRAM_BYTES = 5.044e9
NCU_MF_FACTOR_ONLY_DRAM_BYTES = 3.700e9         # the 33 launches of the factorisation alone
NCU_MF_FWD_SOLVE_DRAM_BYTES = 1.344e9           # the 26 launches of the forward solve
FP64_DMMA_PEAK_TFLOPS = 37.1     # measured on this pool's B200 with DMMA.8x8x4 (profiles/r01_fp64_peak_ubench.txt)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as fh:
            return json.load(fh), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe).  nvidia-smi needs a moment
    to start, so it is launched ahead of the warm-up (`start`), `mark` records when the timed region begins, and `stop` keeps
    the samples whose own timestamps fall inside the region (or, if the region was shorter than one sampling period, the
    samples taken under the identical load right before it — `window` says which)."""
    Q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.t_mark = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            import select
            if select.select([self.proc.stdout], [], [], 5.0)[0]:      # wait (bounded) until nvidia-smi is up:
                self.proc.stdout.readline()                             # its first sample
        except Exception:
            self.proc = None

    def mark(self):
        self.t_mark = time.time()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        t_end = time.time()
        time.sleep(0.06)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        import datetime
        rows = []
        for ln in out.splitlines():
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 10:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                rows.append((ts, float(f[2]), float(f[3]), f[6:10]))
            except ValueError:
                continue
        t0 = self.t_mark if self.t_mark is not None else 0.0
        inside = [r for r in rows if t0 <= r[0] <= t_end + 0.06]
        window = "timed region"
        if not inside:
            inside = rows[-3:]                   # same load (warm-up steps of the same workload) right before the region
            window = "timed region shorter than the sampling period: last samples under the same load before it"
        sm, mx, reasons = [], [], set()
        for _, a, b, flags in inside:
            sm.append(a); mx.append(b)
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), flags):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "window": window}


# ------------------------------------------------------------------------------------------------------
# workload: mesh / survey of SURVEY.md 8(d); observations = forward(true model) (1 + 0.05 N), err = 0.05 |Z|

def build_problem_gpu(cfg, device):
    """Problem with true-model observations; the forward of the true model runs on this GPU through the library."""
    from hmcmt2d_b200 import api, synthetic
    mesh, data, inv, prior = synthetic.make_problem(cfg["ny"], cfg["nz"], cfg["nfreq"], cfg["nrx"])
    truth = synthetic.true_model(mesh)
    mesh_t = type(mesh)(mesh.yLen, mesh.zLen, mesh.airLayer, mesh.gridSize, mesh.origin, truth)
    pl0 = api._forward_only_plan(mesh_t, data, device)
    pred_true, _ = api.MT2DFwdSolver(mesh_t, data, plan=pl0)
    pl0.close()
    data.__dict__.pop("_fwd_plans", None)
    obs, err = synthetic.true_model_data(data, pred_true)
    return synthetic.make_problem(cfg["ny"], cfg["nz"], cfg["nfreq"], cfg["nrx"], obs=obs, err=err)


# ------------------------------------------------------------------------------------------------------
# CPU arm: the oracle (restated reference algorithm, SciPy SuperLU in place of UMFPACK/MUMPS) on host cores.

def _best_cpu_factor(A):
    """SuperLU with the settings that measured fastest on these complex-symmetric systems (symmetric-mode minimum degree on
    A^T + A, no diagonal pivoting: 0.11-0.15 s vs 0.16-0.18 s per factorisation with the default COLAMD at cfg2)."""
    import scipy.sparse.linalg as spla
    return spla.splu(A.tocsc(), permc_spec="MMD_AT_PLUS_A", diag_pivot_thresh=0.0, options=dict(SymmetricMode=True))


_JOB_CACHE = {}


def _cpu_freq_job(args):
    """forward + adjoint for ONE frequency (TE+TM) of the workload — the unit the host cores are farmed over.  The problem
    of a frequency (mesh, survey row subset, true-model observations) is set up once per worker and cached: untimed."""
    fidx, seed, cfg = args
    sys.path.insert(0, ROOT)
    from hmcmt2d_b200 import synthetic
    from oracle import fileio as ofio
    from oracle import forward as ofwd
    from oracle import sampler as osamp
    key = (fidx, cfg["ny"], cfg["nz"], cfg["nfreq"])
    if key not in _JOB_CACHE:
        mesh, data, inv, prior = synthetic.make_problem(cfg["ny"], cfg["nz"], cfg["nfreq"], cfg["nrx"])
        keep = data.freqID == fidx + 1
        od = ofio.MTData(data.rxLoc, data.freqs[fidx:fidx + 1], data.dataType, data.dataComp, data.rxID[keep],
                         np.ones(int(keep.sum()), np.int64), data.dtID[keep], np.ones(int(keep.sum()), bool), True, True)
        tmesh = ofio.TensorMesh2D(mesh.yLen, mesh.zLen, mesh.airLayer, mesh.gridSize, mesh.origin, synthetic.true_model(mesh))
        pred_true, _ = ofwd.MT2DFwdSolver(tmesh, od, _best_cpu_factor)
        noise = np.random.default_rng(7).standard_normal(len(data.freqID))[keep]         # the rows of synthetic.true_model_data
        obs, err = pred_true * (1.0 + 0.05 * noise), 0.05 * np.abs(pred_true)
        omesh = ofio.TensorMesh2D(mesh.yLen, mesh.zLen, mesh.airLayer, mesh.gridSize, mesh.origin, mesh.sigma)
        oinv = osamp.setupInverseDataModel(omesh, [1e-8], obs, err)
        oinv.strModel = synthetic.stress_model(inv, seed)
        _JOB_CACHE[key] = (omesh, od, oinv)
    omesh, od, oinv = _JOB_CACHE[key]
    t0 = time.perf_counter()
    osamp.compDataGradient(omesh, od, oinv, ofio.HMCPrior(), factor_fn=_best_cpu_factor)
    return time.perf_counter() - t0


def _pool(nworkers):
    import multiprocessing as mp
    # one process per core, ONE thread per process: the workers inherit these (spawn) before they import numpy / scipy —
    # without them every worker starts a full BLAS / OpenMP team and the oversubscribed host takes minutes per sample
    for var in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS", "NUMEXPR_NUM_THREADS"):
        os.environ[var] = "1"
    return mp.get_context("spawn").Pool(nworkers)


def cpu_one_core_sample(cfg):
    """One frequency (TE+TM forward + adjoint) on one host core -> steps/s of the whole step by multiplication."""
    with _pool(1) as pool:
        pool.map(_cpu_freq_job, [(0, 1, cfg)])                        # set-up + warm-up of the worker
        t0 = time.perf_counter()
        pool.map(_cpu_freq_job, [(0, 1, cfg)])
        wall = time.perf_counter() - t0
    return 1.0 / (wall * cfg["nfreq"]), wall


def run_reference(args, rank):
    """Reference arm: WHOLE steps of the workload (all frequencies, TE+TM, forward + adjoint) on all host cores, frequencies
    farmed over one single-threaded process per core — the fairest stand-in available for the reference's MUMPS + OpenMP path
    (neither Julia nor MUMPS exists on the box).  `steps` is what was actually run: as many of the requested K as fit a
    ~150 s budget."""
    if rank != 0:
        return
    cfg = WORKLOAD
    cores = os.cpu_count() or 1
    nw = min(cores, cfg["nfreq"])
    jobs = [(f, 1, cfg) for f in range(cfg["nfreq"])]
    times = []
    with _pool(nw) as pool:
        pool.map(_cpu_freq_job, jobs)                                 # untimed: per-frequency problem set-up (cached) + warm-up step
        t_start = time.perf_counter()
        for _ in range(max(1, args.steps)):
            t0 = time.perf_counter()
            pool.map(_cpu_freq_job, jobs)
            times.append(time.perf_counter() - t0)
            if time.perf_counter() - t_start + times[-1] > 150.0:
                break
    step = float(np.mean(times))
    value = 1.0 / step
    sample = (f"{len(times)} whole steps: all {cfg['nfreq']} frequencies (TE+TM forward + adjoint each) farmed over {nw} single-threaded "
              f"host processes ({cores} cores; {-(-cfg['nfreq'] // nw)} wave(s) per step), no extrapolation; restated CPU path (oracle, SciPy "
              f"SuperLU with symmetric-mode MMD ordering, the fastest of the SuperLU settings tried) — not MUMPS / UMFPACK, not Julia")
    line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=args.gpus, steps=len(times), warmup=1,
                ms_per_step=1000.0 * step, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f64 (complex128)",
                data="synthetic", config=dict(WORKLOAD), impl="reference",
                cpu_baseline=dict(value=value, unit=UNIT, cores=nw, kind="port", sample=sample),
                e2e=dict(value=value, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------

class Dist:
    """torch.distributed plumbing: barrier + max over ranks."""

    def __init__(self, rank, world, local_rank):
        import torch
        self.torch, self.rank, self.world = torch, rank, world
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device — hmcmt2d_b200 has no CPU path")
        torch.cuda.set_device(local_rank)
        if world > 1:
            import torch.distributed as dist
            self.dist = dist
            dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local_rank))

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max(self, x):
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def host_stepper(evaluate, inv, prior, m0, dt, total_gradient=False):
    """The reference's proposeLeapfrog inner step on the host (HMCSampler.jl:235-265) around a host-buffer gradient call.
    total_gradient: `evaluate` already returns data + model-norm gradient (hmcmt_forward_gradient_total: the library forms
    beta Wm (m - m_ref) on the device in every evaluation anyway), otherwise the host adds the model-norm part as the reference does."""
    lo, hi = np.log(prior.sigBounds[0]), np.log(prior.sigBounds[1])
    Wm, beta = inv.Wm, prior.regParam

    def step(m, p):
        dm = dt * p
        mx = max(dm.max(), -dm.min())
        if mx > 3.0:
            dm = dm / mx * 3.0
        m = m + dm
        for _ in range(500):                                   # checkParameterBound! (HMCSampler.jl:515-559)
            if m.min() >= lo and m.max() <= hi:
                break
            low = m < lo
            m = np.where(low, 2 * lo - m, m); p = np.where(low, -p, p)
            high = m > hi
            m = np.where(high, 2 * hi - m, m); p = np.where(high, -p, p)
        pred, phi, g = evaluate(m)                             # H2D m ; D2H pred, phi, grad  (pinned staging inside)
        if not total_gradient:
            g += beta * (Wm @ (m - m0))
        g *= dt
        p = p - g
        return m, p, phi
    return step


def factor_pass(pl, run_steps, K):
    """The roofline's kernel time.  In the timed region the systems of a step run as groups on their own streams and overlap each
    other (HMCMT_GROUPS), so no pair of events brackets one factorisation alone; right after it the same K steps run once more
    with the library's factor timing switched on, which keeps every launch on the plan's stream: CUDA events around the
    factorisation + forward solve of each step, and around the whole pass.  Returns (factor ms total, launches timed, pass ms)."""
    pl.kernel_time(reset=1)
    pl.timer_start()
    run_steps(K)
    serial_ms = pl.timer_stop()
    pl._factor_split = pl.kernel_time_split()      # (factorisation alone, forward solve alone), same events
    factor_ms, factor_n = pl.kernel_time(reset=-1)
    return factor_ms, factor_n, serial_ms


def factor_roofline(pl, factor_ms, factor_n, step_ms, peaks, peak_src):
    """Roofline record of the factorisation phase (the dominant kernel group), timed with CUDA events inside the library."""
    N, b, nsys, mf = pl.info(0), pl.info(4), pl.info(7), pl.info(11)
    fac_ms = factor_ms / max(1, factor_n)
    band_flops = (4.0 * N * b * b + 16.0 * N * b) * nsys            # SURVEY.md 8(d): banded LDL^T + fused forward solve
    if mf:
        flops = float(pl.info(12)) * nsys                             # counted from the symbolic structure of the ordering used
        fbytes = 2.0 * pl.info(9) * nsys                              # factor written once + read once by the forward solve
        kernel = ("factorisation of this rank's systems on the nested-dissection multifrontal path: mf_small_kernel (shared-memory fronts), "
                  "mf_asm_*/mf_inv_kernel/mf_gemm_kernel (DMMA.8x8x4 64x64x16 tiles) per depth and pivot chunk, + the forward solve "
                  "(mf_fwd_*/mf_bwd_*), timed as one unit")
        traffic, tsrc = None, None
        if N == 19701 and nsys == 60:
            traffic = NCU_MF_FACTOR_DRAM_BYTES
            tsrc = ("sum of dram__bytes_read.sum + dram__bytes_write.sum over the launches of one factorisation + forward solve at this "
                    "workload (profiles/r02_cfg2_launches.csv): factor written and read back once, update matrices of the fronts "
                    "written by the children and read by the parents, assembly of the large fronts in global memory")
    else:
        flops, fbytes = band_flops, 2.0 * 16.0 * N * (b + 1) * nsys
        kernel = ("factorisation of the systems = band_factor_kernel<14> FM_OWN + FM_SEP (FP64 DMMA.8x8x4 block LDL^T, fused assembly + "
                  "forward elimination) + band_solve_kernel<14> SM_BACKZ_OWN (its back-substitution), timed as one unit")
        traffic = NCU_FACTOR_DRAM_BYTES
        tsrc = ("dram__bytes_read.sum + dram__bytes_write.sum of ncu --set full captures at this workload: FM_OWN launch "
                "(profiles/r01_final_factor_own_ncu.txt) + one factor-streaming sweep (profiles/r01_final_solve_own_ncu.txt)")
    achieved = flops / (fac_ms * 1e-3) / 1e12
    parts = None
    split = getattr(pl, "_factor_split", None)
    if mf and split and split[0] > 0 and split[1] > 0:
        # the two halves of the unit, from the same events: the factorisation alone against the tensor roof, the forward solve
        # (sparse forward elimination + complete backward substitution) against the HBM roof
        f_ms, s_ms = split[0] / max(1, factor_n), split[1] / max(1, factor_n)
        cfg2 = N == 19701 and nsys == 60
        sbytes = float(pl.info(9)) * nsys                             # >= : the backward substitution streams the whole factor once
        parts = dict(
            factorisation=dict(bound="tensor", achieved=flops / (f_ms * 1e-3) / 1e12, peak=FP64_DMMA_PEAK_TFLOPS, unit="TFLOP/s",
                               frac=flops / (f_ms * 1e-3) / 1e12 / FP64_DMMA_PEAK_TFLOPS, avg_launch_ms=f_ms,
                               traffic=NCU_MF_FACTOR_ONLY_DRAM_BYTES if cfg2 else None),
            forward_solve=dict(bound="hbm", achieved=sbytes / (s_ms * 1e-3) / 1e9, peak=peaks.get("hbm_gbs"), unit="GB/s",
                               frac=sbytes / (s_ms * 1e-3) / 1e9 / peaks.get("hbm_gbs", 6650.0), avg_launch_ms=s_ms,
                               algorithmic_bytes_per_launch=sbytes, traffic=NCU_MF_FWD_SOLVE_DRAM_BYTES if cfg2 else None))
    return dict(bound="tensor", kernel=kernel, parts=parts, achieved=achieved, peak=FP64_DMMA_PEAK_TFLOPS, unit="TFLOP/s",
                frac=achieved / FP64_DMMA_PEAK_TFLOPS,
                peak_source="measured FP64 DMMA m8n8k4 rate on this pool's B200 (profiles/r01_fp64_peak_ubench.txt); "
                            "MEASURED_PEAKS.json holds only bf16/HBM peaks: " + peak_src,
                traffic=traffic, traffic_source=tsrc, algorithmic_flops_per_launch=flops,
                banded_count_flops_per_launch=band_flops, banded_count_frac=band_flops / (fac_ms * 1e-3) / 1e12 / FP64_DMMA_PEAK_TFLOPS,
                algorithmic_bytes_per_launch=fbytes, hbm_achieved_gbs=fbytes / (fac_ms * 1e-3) / 1e9, hbm_peak_gbs=peaks.get("hbm_gbs"),
                avg_launch_ms=fac_ms, launches_timed=factor_n, share_of_step=fac_ms / step_ms,
                timing="CUDA events on the library's stream around the factorisation + forward solve of every step of a separate "
                       "un-grouped pass of the same steps, run inside bench.py right after the timed region (in the timed region "
                       "groups of systems overlap on several streams); share_of_step is relative to that pass "
                       f"({step_ms:.3f} ms per step)",
                ordering="nested dissection (multifrontal)" if mf else "band, short axis fastest, two halves per system")


def rel_diff(a, b):
    return float(np.abs(np.asarray(a) - np.asarray(b)).max() / max(1e-300, np.abs(np.asarray(b)).max()))


def run_cfg2(args, D, local_rank):
    """Weak scaling: one chain of the cfg2 workload per GPU."""
    from hmcmt2d_b200 import api, synthetic
    rank, world = D.rank, D.world
    mesh, data, inv, prior = build_problem_gpu(WORKLOAD, local_rank)
    pl = api.Plan(mesh, data, inv, prior, nChains=1, device=local_rank)
    rng = np.random.default_rng(100 + rank)
    m0 = synthetic.stress_model(inv, seed=1 + rank)            # chains differ per GPU (seeds 1..N, cfg3)
    p0 = np.clip(rng.standard_normal(len(m0)), -2.5, 2.5)
    dt = prior.dt
    K, W = args.steps, max(3, args.warmup)
    step = host_stepper(lambda m: (lambda r: (r[0], float(r[1][0]), r[2][0]))(pl.forward_gradient(m, total=True)), inv, prior, m0, dt,
                        total_gradient=True)

    # ---------------- validation (untimed): device-resident steps vs host-loop steps from the same state ----------------
    # one step: same state in -> same state out at the north_star tolerance (1e-9); three steps: the chain stays together while the
    # dynamics amplify the round-off difference of the two loops (prior gradient summed on the host / on the device), bound 1e-7
    pl.set_state(m0, p0, m0)
    pl.leapfrog_steps_device(dt, 1)
    md1, pd1 = pl.get_state()
    pl.leapfrog_steps_device(dt, 2)
    status3 = pl.status()
    md3, pd3 = pl.get_state()
    m, p = m0.copy(), p0.copy()
    m, p, _ = step(m, p)
    one_diff = max(rel_diff(md1[0], m), rel_diff(pd1[0], p))
    for _ in range(2):
        m, p, _ = step(m, p)
    short_diff = max(rel_diff(md3[0], m), rel_diff(pd3[0], p))

    # ---------------- device-resident arm (`value`) ----------------
    sampler = ClockSampler(local_rank)
    sampler.start()
    pl.set_state(m0, p0, m0)
    pl.leapfrog_steps_device(dt, W)
    pl.sync()
    launches0 = pl.info(10)
    D.barrier()
    sampler.mark()
    pl.timer_start()
    pl.leapfrog_steps_device(dt, K)
    ms = pl.timer_stop()
    D.barrier()
    clocks = sampler.stop()
    launches = pl.info(10) - launches0
    status = pl.status()                                       # device error flags of the whole timed loop
    m_dev, p_dev = pl.get_state()
    ms = D.max(ms)
    value = world * K / (ms * 1e-3)
    factor_ms, factor_n, serial_ms = factor_pass(pl, lambda n: pl.leapfrog_steps_device(dt, n), K)

    # ---------------- end-to-end arm through the host-buffer C ABI ----------------
    m, p = m0.copy(), p0.copy()
    for _ in range(W):
        m, p, _ = step(m, p)
    D.barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        m, p, phi = step(m, p)
    D.torch.cuda.synchronize()
    e2e_s = D.max(time.perf_counter() - t0)
    D.barrier()
    e2e_value = world * K / e2e_s
    h2d = pl.nAC * 8
    d2h = pl.nData * 16 + 8 + pl.nAC * 8
    # both arms integrated W+K steps from (m0, p0): their end states agree up to the round-off the dynamics amplify
    final_diff = max(rel_diff(m_dev[0], m), rel_diff(p_dev[0], p))
    finite = bool(np.isfinite(m_dev).all() and np.isfinite(p_dev).all() and np.isfinite(m).all() and np.isfinite(phi))
    # The gate is the one-step comparison at 1e-9 (north_star tolerance) and the three-step one at 1e-7.  Over the W+K steps of the timed arms the leapfrog dynamics
    # amplify the round-off difference between the two loops (prior gradient summed on the host vs on the device) by ~1.4x per step,
    # chain dependent: the end states are reported and only required to stay on the same trajectory (1e-2), not gated at 1e-9.
    validated = bool(status == 0 and status3 == 0 and finite and one_diff < 1e-9 and short_diff < 1e-7 and final_diff < 1e-2)
    validated = bool(D.max(0.0 if validated else 1.0) == 0.0)
    # worst rank (every GPU integrates its own chain): what the gate saw
    worst = dict(one_step_device_vs_host_rel=D.max(one_diff), three_step_device_vs_host_rel=D.max(short_diff),
                 final_state_device_vs_host_rel=D.max(final_diff),
                 device_status=int(-D.max(-float(min(status, status3)))), states_finite=bool(D.max(0.0 if finite else 1.0) == 0.0))

    peaks, peak_src = load_peaks()
    roofline = factor_roofline(pl, factor_ms, factor_n, serial_ms / K, peaks, peak_src)
    line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=K, warmup=W, ms_per_step=ms / K,
                higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f64 (complex128)", data="synthetic",
                config=dict(WORKLOAD),
                l2_policy=f"inputs larger than L2: each step streams the {pl.info(9) * pl.info(7) / 1e9:.2f} GB factor of the "
                          f"{pl.info(7)} systems (written once, read by the four sweeps of the two solves) through the 126 MB L2",
                parallelism=f"chains x{world} (replicas only, no data-path collective)",
                solver="multifrontal" if pl.info(11) else "band",
                e2e=dict(value=e2e_value, unit=UNIT, h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h, ms_per_step=1000 * e2e_s / K),
                gpu_launches=int(launches), clocks=clocks, roofline=roofline, validated=validated,
                validation=dict(worst_rank=worst, device_status=int(status), states_finite=finite, one_step_device_vs_host_rel=one_diff,
                                three_step_device_vs_host_rel=short_diff,
                                final_state_device_vs_host_rel=final_diff, steps_compared=W + K,
                                observations="forward(true model) x (1 + 0.05 N), err = 0.05 |Z| (SURVEY.md 8d)"))
    pl.close()
    return line, dict(model=m_dev, momentum=p_dev)


def run_cfg4(args, D, local_rank, K, nfreq=0):
    """Strong scaling: one chain of the cfg4 workload, its (frequency, mode) systems sharded over the ranks, K timed steps."""
    from hmcmt2d_b200 import api, synthetic
    rank, world = D.rank, D.world
    cfg = dict(CFG4)
    if nfreq:
        cfg["nfreq"] = nfreq
        cfg["workload"] += f" [reduced to {nfreq} frequencies]"
    mesh, data, inv, prior = synthetic.make_problem(cfg["ny"], cfg["nz"], cfg["nfreq"], cfg["nrx"])
    sp = api.FreqShardedPlan(mesh, data, inv, prior, rank, world, device=local_rank)
    pl = sp.plan
    m0 = synthetic.stress_model(inv, seed=1)                                   # the same chain state on every rank
    p0 = np.clip(np.random.default_rng(100).standard_normal(len(m0)), -2.5, 2.5)
    dt = prior.dt
    W = 3

    sampler = ClockSampler(local_rank)
    sampler.start()
    sp.set_state(m0, p0, m0)
    sp.leapfrog_steps_device(dt, W)
    sp.sync()
    launches0 = pl.info(10)
    D.barrier()
    sampler.mark()
    pl.timer_start()
    sp.leapfrog_steps_device(dt, K)
    ms = pl.timer_stop()
    D.barrier()
    clocks = sampler.stop()
    launches = pl.info(10) - launches0
    status = pl.status()
    ms = D.max(ms)
    value = K / (ms * 1e-3)
    m_end, p_end = sp.get_state()
    csum = float(np.abs(m_end).sum())
    spread = D.max(csum) - (-D.max(-csum))
    factor_ms, factor_n, serial_ms = factor_pass(pl, lambda n: sp.leapfrog_steps_device(dt, n), K)

    # end to end: compDataGradient through host buffers (H2D model, D2H data / misfit / gradient, all-reduce) + host leapfrog
    step = host_stepper(lambda m: sp.forward_gradient(m), inv, prior, m0, dt)
    Ke = max(1, min(K, 5))
    m, p = m0.copy(), p0.copy()
    m, p, _ = step(m, p)
    D.barrier()
    t0 = time.perf_counter()
    for _ in range(Ke):
        m, p, phi = step(m, p)
    D.torch.cuda.synchronize()
    e2e_s = D.max(time.perf_counter() - t0)
    D.barrier()
    finite = bool(np.isfinite(m_end).all() and np.isfinite(p_end).all() and np.isfinite(phi))
    validated = bool(D.max(0.0 if (status == 0 and finite and spread == 0.0) else 1.0) == 0.0)

    peaks, peak_src = load_peaks()
    roofline = factor_roofline(pl, factor_ms, factor_n, serial_ms / K, peaks, peak_src)
    nsys = int(pl.info(7))
    line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=K, warmup=W, ms_per_step=ms / K, higher_is_better=True,
                scaling="strong", vs_baseline=None, dtype="f64 (complex128)", data="synthetic", config=cfg,
                systems_per_gpu=nsys, factor_gb_per_gpu=pl.info(9) * nsys / 1e9,
                l2_policy="inputs larger than L2: each rank streams the multifrontal factors of its systems",
                parallelism=(f"(frequency, mode) systems x{world}; one sum-all-reduce of [gdata | phi_d] = {8 * (pl.nAC + 1)} B per step, "
                             + ("ncclAllReduce issued by the library on its own stream" if sp.in_library_nccl else
                                "single GPU: no exchange" if world == 1 else "torch.distributed all_reduce")),
                state_spread_between_ranks=spread, solver="multifrontal" if pl.info(11) else "band",
                e2e=dict(value=Ke / e2e_s, unit=UNIT, h2d_bytes_per_step=pl.nAC * 8, d2h_bytes_per_step=pl.nData * 16 + 8 + pl.nAC * 8,
                         ms_per_step=1000 * e2e_s / Ke, steps=Ke),
                gpu_launches=int(launches), clocks=clocks, roofline=roofline, validated=validated,
                validation=dict(device_status=int(status), states_finite=finite, observations="analytic half-space + 5 % noise"))
    sp.close()
    return line, dict(model=m_end, momentum=p_end)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-strong-scaling", action="store_true", help="skip the cfg4 record appended to the cfg2 line")
    ap.add_argument("--config", default="cfg2", choices=["cfg2", "cfg4"])
    ap.add_argument("--nfreq", type=int, default=0, help="cfg4 only: reduced number of frequencies (testing)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the chain state left by the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world == 1 and args.gpus > 1:
        # convenience: re-launch under torchrun when called directly with --gpus N
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1",
               "--master-port", "29511", os.path.abspath(__file__), "--gpus", str(args.gpus), "--steps", str(args.steps),
               "--warmup", str(args.warmup), "--config", args.config, "--nfreq", str(args.nfreq)]
        cmd += ["--no-strong-scaling"] if args.no_strong_scaling else []
        cmd += ["--dump-outputs", args.dump_outputs] if args.dump_outputs else []
        raise SystemExit(subprocess.call(cmd))
    D = Dist(rank, world, local_rank)
    if args.config == "cfg4":
        line, outputs = run_cfg4(args, D, local_rank, args.steps, args.nfreq)
    else:
        line, outputs = run_cfg2(args, D, local_rank)
        if not args.no_strong_scaling:
            try:
                # a short record next to the headline: 3 to 10 timed steps whatever --steps says
                line["strong_scaling"] = run_cfg4(args, D, local_rank, max(3, min(args.steps, 10)), args.nfreq)[0]
            except Exception as e:                                   # never lose the headline line to the second workload
                line["strong_scaling"] = dict(error=repr(e))
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cfg = line["config"]
        v1, wall1 = cpu_one_core_sample(cfg)
        line["cpu_baseline"] = dict(value=v1, unit=UNIT, cores=1, kind="port",
                                    sample=f"1 of {cfg['nfreq']} frequencies (TE+TM forward+adjoint, {wall1:.2f} s) on one host core, "
                                           f"multiplied by {cfg['nfreq']}; restated CPU path (oracle, SciPy SuperLU symmetric-mode MMD), not MUMPS. "
                                           f"All-core figure: `bench.py --impl reference` ({os.cpu_count()} cores on this box)")
    if rank == 0 and args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in outputs.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))
    if rank == 0:
        print(json.dumps(line), flush=True)
    D.close()


if __name__ == "__main__":
    main()
