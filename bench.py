#!/usr/bin/env python
"""bench.py — headline benchmark of the DeMethify deconvolution hot path on B200.

Workload (BASELINE.json metric "... at 1M CpG x K x N", configs[4] shape): partial-reference deconvolution,
M = 1,000,000 CpGs x N = 256 samples, K = 6 known + n_u = 2 unknown cell types, fp64, synthetic data
(recipe of test/gen_data.ipynb cell 5).  One STEP = one fit of OUTER_PER_STEP = 100 outer iterations of mdwbssmf_deconv
(deconvolution.py:206-221) with n_iter2 = 20: 20 update_u + 20 update_alpha inner iterations + cost_f_w each,
tol = 0 so no step stops early (the reference's fixture fits need 54-166 outer iterations at its default tolerance).
metric = update iterations / second (inner iterations of U and alpha); fits/s = value / 4000.

  value     : inputs resident in HBM when the timed region starts; the library's default engine (fused: per outer iteration
              ONE streaming pass - row statistics -> 20 update_u iterations -> Gram panel on a single visit of every row tile,
              csrc/dmf_fused.cuh - followed by the per-sample alpha kernel)
  e2e       : the public call demethify_b200.deconvolution.mdwbssmf_deconv with HOST (pinned) numpy buffers;
              H2D of X, d_x, R_trunc, u0, alpha0 and D2H of u, alpha inside the timed region
  roofline  : dominant kernel of the timed region (the fused pass): algorithmic bytes (SURVEY 8 d4 "fused outer iteration")
              and algorithmic FP64 flops / CUDA-event duration against the measured HBM and FP64 peaks; `bound` names the larger
              fraction (SURVEY 8 d3); `stream_passes` = the reference-shaped one-launch-per-inner-iteration kernels timed in the
              same run
  parity_sample : the SAME arrays and initial iterate as the GPU arm, first CPU_SAMPLE_ROWS rows: one outer iteration by the
              oracle on the host and by the library on the GPU -> max |d alpha|, max |d u|, cost (SURVEY 8 d2 / d5)
  cpu_baseline / --impl reference : the numpy port of the reference loop (oracle/) on the host cores, on a
              bounded row sample of the same workload (cost is linear in M; the sample and the scaling are stated)

N > 1 GPUs: the headline `value` is ONE fit with its CpG rows sharded over the GPUs (BASELINE config 5's partitioning, SURVEY 8 e1
(ii)): per outer iteration one fused pass over a rank's rows, one all-reduce of the per-sample statistics (in-kernel over NVLink peer
memory), then the identical test / alpha iterations on every rank -> "scaling": "strong".  The leg first checks, on 5 outer
iterations, that alpha is bit-identical on all ranks and equals the one-GPU fit of the same data to 1e-9 (`row_sharded.parity`).
`fit_sharded` = the other partitioning (independent fits, one per GPU, no collective; weak scaling) as an extra key.

--dump-outputs DIR: after the timed steps, the u (M x n_u), alpha (K + n_u x N) and cost of the fit behind `value` (the resident
arm's fit on one GPU, the row-sharded fit with u gathered in row order on several; with --impl reference, the oracle's fit on its
row sample) go to DIR/{u,alpha,cost}.npy in float64.  The inputs are drawn from fixed seeds, so two builds run with the same
arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

if "reference" in sys.argv:          # torchrun exports OMP_NUM_THREADS=1: the CPU arm is meant to use every host core
    for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[_v] = str(os.cpu_count() or 1)

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

M_FULL, N_S, K_KNOWN, N_UNK = 1_000_000, 256, 6, 2
N_ITER2 = 20
OUTER_PER_STEP = 100
CPU_SAMPLE_ROWS = 100_000
METRIC = "update_iters_per_sec"
UNIT = "inner update iterations/s at 1M CpG x 256 samples (K=6, n_u=2)"
DUMP_BYTES = 60 << 20          # --dump-outputs: the .npy files stay under 64 MB in all, headers included


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--rows", type=int, default=M_FULL, help="override M (debug)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--precision", default="fp64", choices=["fp64", "fp32"])
    ap.add_argument("--profile", action="store_true", help="resident arm only (for runs under ncu): no e2e, no CPU leg")
    ap.add_argument("--outer", type=int, default=OUTER_PER_STEP, help="outer iterations per step (default: one 100-iteration fit)")
    ap.add_argument("--engine", default="auto", choices=["auto", "fused", "gram", "stream"], help="device engine of the timed region")
    ap.add_argument("--boot-resamples", type=int, default=1000, help="resamples of the BASELINE config-4 bootstrap leg (0 = skip the leg)")
    ap.add_argument("--boot-rows", type=int, default=500_000, help="CpG rows of the bootstrap leg (debug)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write u, alpha and cost of the timed fit as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    return args


def workload_config(M, extra=None):
    cfg = {"workload": "partial-reference deconvolution (mdwbssmf_deconv), BASELINE configs[4] shape",
           "M_cpg": M, "N_samples": N_S, "K_known": K_KNOWN, "n_unknown": N_UNK, "n_iter2": N_ITER2,
           "outer_iterations_per_step": OUTER_PER_STEP, "update_iters_per_step": 2 * N_ITER2 * OUTER_PER_STEP,
           "tol": 0.0, "init": "uniform_", "cache": "inputs (>= 2.6 GB per pass) exceed the 126 MB L2"}
    if extra:
        cfg.update(extra)
    return cfg


def dump_outputs(out_dir, arrays):
    """Write `arrays` as out_dir/<name>.npy in float64 so that two builds can be compared output for output.  An array larger than
    its share of DUMP_BYTES is replaced by a fixed, seeded sample of its rows, with the sampled row indices in <name>_rows.npy."""
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // len(arrays)
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float64)
        if a.nbytes > share:
            n_keep = share // (a.nbytes // a.shape[0] + 8)
            rows = np.sort(np.random.RandomState(0).choice(a.shape[0], n_keep, replace=False))
            np.save(os.path.join(out_dir, f"{name}_rows.npy"), rows.astype(np.float64))
            a = a[rows]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def synth_host(M, seed=0):
    """Small-M synthetic problem on the host (CPU baseline sample)."""
    rs = np.random.RandomState(seed)
    a = rs.uniform(0.2, 1.0, size=K_KNOWN + N_UNK)
    Rf = rs.beta(a, a, size=(M, K_KNOWN + N_UNK))
    unk = rs.uniform(0, 0.9, size=N_S)
    Ak = rs.dirichlet(np.ones(K_KNOWN), N_S).T * (1 - unk)
    Au = rs.dirichlet(np.ones(N_UNK), N_S).T * unk
    D = rs.poisson(50, size=(M, N_S)) + 1
    X = rs.binomial(D, np.clip(Rf @ np.vstack([Ak, Au]), 0, 1)) / D
    return X, D.astype(np.int64), np.ascontiguousarray(Rf[:, :K_KNOWN])


def blas_threads():
    """Use every host core for the CPU arm whatever the launcher exported (torchrun sets OMP_NUM_THREADS=1)."""
    n = os.cpu_count() or 1
    try:
        import threadpoolctl
        threadpoolctl.threadpool_limits(limits=n)
        used = max([p.get("num_threads", 1) for p in threadpoolctl.threadpool_info()] or [1])
    except Exception:
        used = n
    return used


def cpu_reference_leg(steps, warmup, rows=CPU_SAMPLE_ROWS, data=None):
    """The reference algorithm's numpy port (oracle/bssmf_numpy.py, pinned to the reference by
    tests/test_oracle_golden.py) timed on the host cores.  One step = ONE outer iteration on a row sample.
    `data` = (X, D, Rk, u0, a0) host arrays of the GPU arm (first `rows` rows); else a problem of the same recipe is drawn."""
    if data is not None:
        data = (data[0], np.asarray(data[1]).astype(np.int64), data[2], data[3], data[4])
    from oracle import bssmf_numpy as orc
    threads = blas_threads()
    if data is None:
        X, D, Rk = synth_host(rows)
        u0, R0, a0 = orc.draw_init("uniform_", X, D, Rk, N_UNK, seed=1)
    else:
        X, D, Rk, u0, a0 = data
        R0 = np.c_[Rk, u0]
    Df = D.astype(np.float64)
    times, out = [], None
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        tr = {}
        out = orc.solve_partial_reference(u0.copy(), R0, a0.copy(), X, Df, Rk, N_UNK, 1, N_ITER2, 0.0, trace=tr)
        times.append(time.perf_counter() - t0)
        out = out + (tr,)
    t = float(np.mean(times[warmup:]))
    its_sample = 2 * N_ITER2 / t
    cores = threads
    return {"result": out, "value": its_sample * rows / M_FULL, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{rows} of {M_FULL} CpG rows x {N_S} samples, 1 outer iteration (40 inner updates + cost) per step, "
                      f"{its_sample:.2f} it/s on the sample scaled by {rows}/{M_FULL} (cost linear in M); numpy/OpenBLAS threads",
            "s_per_step_sample": t}


class ClockSampler:
    QUERY = "clocks.sm,clocks.max.sm,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
            "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.proc, self.t_begin = index, [], None, None

    def start(self):
        """Launch nvidia-smi in loop mode.  Called BEFORE the warm-up steps: the tool needs a few hundred ms before its first line, and
        the timed region of the headline is well under a second."""
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def mark_begin(self):
        self.t_begin = time.perf_counter()          # start of the timed region: only later samples count

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        t_end = time.perf_counter()
        time.sleep(0.15)
        self.proc.terminate()
        t0 = self.t_begin if self.t_begin is not None else 0.0
        inside = [r for t, r in self.rows if t0 <= t <= t_end + 0.1]
        window = "timed region"
        if not inside:                               # region shorter than the sampling period: the warm-up steps ran the same kernels
            inside, window = [r for _t, r in self.rows], "warm-up + timed region (no sample fell inside the timed region)"
        sm = [float(r[0]) for r in inside if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in inside if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in inside if len(r) >= 7 for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm), "window": window}


def run_reference(args, rank, world):
    if rank != 0:
        return
    leg = cpu_reference_leg(args.steps, args.warmup)
    if args.dump_outputs:
        u_last, a_last, tr = leg["result"]
        dump_outputs(args.dump_outputs, {"u": u_last, "alpha": a_last, "cost": tr["costs"][-1]})
    line = {"impl": "reference", "metric": METRIC, "value": leg["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": leg["s_per_step_sample"] * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload_config(M_FULL),
            "cpu_baseline": {k: leg[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": leg["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line))


def hbm_peak_gbs():
    """(GB/s, where it comes from): the driver's measured copy bandwidth of this pool's B200s, else the profiling recipe's fallback."""
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        return json.load(open(peaks_path))["hbm_gbs"], "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
    return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


def bootstrap_leg(args, dev, rank, world):
    """BASELINE config 4: bootstrap confidence intervals, 500k CpG x 64 samples, K = 6, n_u = 1, CLI defaults (10000 x 20, tol 1e-2,
    init uniform_, seed 1 -> the reference's seed sequence 1, 2, 4, 7, ...), boot_resamples resamples, percentiles included
    (bootstrap.py:26-54, :77-78).  Fit-sharded over the ranks (resample b on rank b mod world, no data-path collective; the alpha
    and u stacks are all-gathered for the percentiles).  Wall clock of the public pieces bt_ci is made of, host work included."""
    import torch
    import torch.distributed as dist
    from demethify_b200.bootstrap import bootstrap_fits, bootstrap_seeds, merge_resample_stacks, percentile_bounds_device, shard_of
    from demethify_b200.engine import DeviceProblem
    Mb, Nb, Kb, nub, B = args.boot_rows, 64, K_KNOWN, 1, args.boot_resamples
    gen = torch.Generator(device=dev)
    gen.manual_seed(4321)
    conc = torch.rand(Kb + 1, device=dev, generator=gen, dtype=torch.float64) * 0.8 + 0.2
    g1 = torch._standard_gamma(conc.expand(Mb, Kb + 1).contiguous(), generator=gen)
    g2 = torch._standard_gamma(conc.expand(Mb, Kb + 1).contiguous(), generator=gen)
    Rf = g1 / (g1 + g2)
    unk = torch.rand(Nb, device=dev, generator=gen, dtype=torch.float64) * 0.9
    ek = -torch.log1p(-torch.rand(Kb, Nb, device=dev, generator=gen, dtype=torch.float64))
    A_true = torch.cat([ek / ek.sum(0) * (1 - unk), unk[None]], 0)
    D = torch.poisson(torch.full((Mb, Nb), 50.0, device=dev), generator=gen).to(torch.int64) + 1
    X = torch.binomial(D.to(torch.float64), (Rf @ A_true).clamp_(0, 1), generator=gen) / D.to(torch.float64)
    Rk = Rf[:, :Kb].contiguous()
    prob = DeviceProblem(X, D, Rk)
    Xh, Rh = X.cpu().numpy(), Rk.cpu().numpy()               # bootstrap_fits takes the reference's host arrays (shapes / data-dependent inits)
    del g1, g2, Rf, X, D
    seeds = shard_of(bootstrap_seeds(1, B), rank, world)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    alphas, us, n_outer = bootstrap_fits(len(seeds), nub, Xh, None, Rh, "uniform_", 10000, 20, 1e-2, None, 1, prob=prob, on_device=True,
                                         seeds=seeds)
    torch.cuda.synchronize()
    t_fit = time.perf_counter() - t0
    if world > 1:
        alphas = merge_resample_stacks(alphas, B)
        us = merge_resample_stacks(us, B)
    lo, hi = percentile_bounds_device(alphas, 2.5, 97.5)
    ulo, uhi = percentile_bounds_device(us, 2.5, 97.5)
    torch.cuda.synchronize()
    t_all = time.perf_counter() - t0
    tt = torch.tensor([t_fit, t_all, float(sum(n_outer))], dtype=torch.float64, device=dev)
    if world > 1:
        tmax = tt.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(tt, op=dist.ReduceOp.SUM)
        t_fit, t_all, total_outer = float(tmax[0]), float(tmax[1]), float(tt[2])
    else:
        total_outer = float(tt[2])
    ok = bool(np.isfinite(lo).all() and np.isfinite(uhi).all() and (hi >= lo).all() and (uhi >= ulo).all())
    # algorithmic FP64 work of one outer iteration of one resample (n_u = 1): the fused-pass count of SURVEY 8 d4 with n_u = 1
    flops_outer = 2.0 * Mb * Nb * (Kb + 2 + 1 + 1 + 1 + 1 + Kb + 1)
    fp64_peak = 37.1
    fpath = os.path.join(ROOT, "profiles", "fp64_peak.json")
    if os.path.exists(fpath):
        fp64_peak = json.load(open(fpath))["fp64_tflops"]
    tf = flops_outer * total_outer / t_fit / 1e12 / world
    # materialised form: every resample streams its own gathered copy of X, d_x, R_trunc once per outer iteration (SURVEY 8 d4, fused pass)
    bytes_outer = Mb * (8 * (Nb + Kb + 4 * nub) + 2 * Nb)
    gbs = bytes_outer * total_outer / t_fit / 1e9 / world
    hbm_peak, _src = hbm_peak_gbs()
    return {"workload": "BASELINE configs[3]: bootstrap CIs, 500k CpG x 64 samples, K=6, n_u=1, 10000 x 20 iterations, tol 1e-2, uniform_ init",
            "M_cpg": Mb, "N_samples": Nb, "resamples": B, "n_gpus": world, "parallelism": f"fit-sharded x{world} (resample b on rank b mod {world})",
            "seconds_total": t_all, "seconds_fits": t_fit, "seconds_percentiles_and_gather": t_all - t_fit,
            "resample_fits_per_sec": B / t_all, "seconds_per_1000_resamples": t_all * 1000.0 / max(B, 1),
            "mean_outer_iterations": total_outer / max(B, 1), "bounds_finite_and_ordered": ok,
            "form": "materialised form (every resample of a wave owns a gathered copy of X, d_x, R_trunc; device MT19937 draws), fused one-pass engine, "
                    "32-row tiles of the N <= 64 width class",
            "roofline": {"bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak,
                         "algorithmic_bytes_per_fit_outer_iteration": bytes_outer,
                         "frac_fp64": tf / fp64_peak, "achieved_fp64_tflops": tf, "peak_fp64_tflops": fp64_peak,
                         "algorithmic_fp64_flops_per_fit_outer_iteration": flops_outer,
                         "note": "per GPU, wall clock of the fits (set-up of the waves, polling and the tails of the waves included)"}}


def run_b200(args, rank, world, local_rank):
    if os.environ.get("DMF_BENCH_GRAPH", "0") == "1":
        # NCCL's user-buffer registration for captured collectives hung the 500k-row all-reduce on this pool (NCCL 2.28.9)
        os.environ.setdefault("NCCL_GRAPH_REGISTER", "0")
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    import __graft_entry__ as g
    if world > 1:               # one process compiles (a no-op when the shipped library is current), the others wait
        if rank == 0:
            g.build()
        dist.barrier()
    g.build()
    import demethify_b200
    from demethify_b200 import deconvolution as dec
    from demethify_b200.engine import DeviceProblem, FitBatch
    demethify_b200.set_precision(args.precision)
    M = args.rows
    tdt = torch.float64 if args.precision == "fp64" else torch.float32

    # ---- synthetic inputs, generated on the device (same recipe as synth_host), then mirrored into pinned host memory
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234)          # the SAME problem on every rank: at N > 1 the headline is ONE fit with its rows sharded
    Kt = K_KNOWN + N_UNK
    conc = torch.rand(Kt, device=dev, generator=gen, dtype=torch.float64) * 0.8 + 0.2
    g1 = torch._standard_gamma(conc.expand(M, Kt).contiguous(), generator=gen)
    g2 = torch._standard_gamma(conc.expand(M, Kt).contiguous(), generator=gen)
    Rf = g1 / (g1 + g2)
    del g1, g2
    unk = torch.rand(N_S, device=dev, generator=gen, dtype=torch.float64) * 0.9
    ek = -torch.log1p(-torch.rand(K_KNOWN, N_S, device=dev, generator=gen, dtype=torch.float64))
    eu = -torch.log1p(-torch.rand(N_UNK, N_S, device=dev, generator=gen, dtype=torch.float64))
    A_true = torch.cat([ek / ek.sum(0) * (1 - unk), eu / eu.sum(0) * unk], 0)
    D = torch.poisson(torch.full((M, N_S), 50.0, device=dev), generator=gen).to(torch.int64) + 1
    P = (Rf @ A_true).clamp_(0, 1)
    cnt = torch.binomial(D.to(torch.float64), P, generator=gen)
    X = cnt / D.to(torch.float64)
    del P, cnt
    Rk = Rf[:, :K_KNOWN].contiguous()
    del Rf
    hX = torch.empty(X.shape, dtype=torch.float64, pin_memory=True); hX.copy_(X)
    # coverage as the CLI reader stages it (demethify_b200/demethify.py read_inputs): uint16 in page-locked memory
    hD = torch.empty(D.shape, dtype=torch.uint16, pin_memory=True); hD.view(torch.int16).copy_(D.to(torch.int16))      # (values < 2^15: the int16 view is exact)
    hR = torch.empty(Rk.shape, dtype=torch.float64, pin_memory=True); hR.copy_(Rk)
    u0, R0_unused, a0 = None, None, None
    rs = np.random.RandomState(1)
    u0 = rs.uniform(size=(M, N_UNK)); a0 = rs.dirichlet(np.ones(Kt), N_S).T.copy()
    hU = torch.empty(u0.shape, dtype=torch.float64, pin_memory=True); hU.copy_(torch.from_numpy(u0))
    hA = torch.empty(a0.shape, dtype=torch.float64, pin_memory=True); hA.copy_(torch.from_numpy(a0))
    torch.cuda.synchronize()

    # ---- resident arm
    demethify_b200.set_engine(args.engine)
    prob = DeviceProblem(X, D, Rk, precision=args.precision)
    del X, D
    batch = FitBatch(prob, N_UNK, [hU], [hA])
    engine = batch.engine
    geom = batch.geometry()
    sT = 8 if args.precision == "fp64" else 4
    sW = 2 if prob.wtype == 1 else sT
    NG = N_UNK + N_UNK * (N_UNK + 1) // 2
    bytes_u = M * (sT * (N_S + K_KNOWN + 3 * N_UNK) + sW * N_S)          # SURVEY 8 d4, U inner iteration
    bytes_a = M * (sT * (N_S + Kt) + sW * N_S)                             # alpha inner iteration / cost
    bytes_rowgram = M * (sT * (N_S + Kt) + sW * N_S + 8 * NG)              # read X, d_x, R_trunc, u; write b_m, H_m
    bytes_panel = M * (sT * (N_S + Kt) + sW * N_S)                         # read X, d_x, R_trunc, u
    bytes_fused = M * (sT * (N_S + K_KNOWN + 4 * N_UNK) + sW * N_S)        # SURVEY 8 d4 fused outer iteration: + u, u_ read, u, u_ written
    tri = N_UNK * (N_UNK + 1) // 2
    # algorithmic FP64 work of the fused pass per (row, sample): c (K) + d c (1) + cost (1) + b (n_u) + H (tri) | d x (1) + bx_u (n_u)
    # + G_uk (n_u K) + G_uu (tri) multiply-adds
    flops_fused = 2.0 * M * N_S * (K_KNOWN + 2 + N_UNK + tri + 1 + N_UNK + N_UNK * K_KNOWN + tri)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def ev():
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        return e

    def one_step(evs=None):
        for _ in range(OUTER_PER_STEP):
            if engine == "fused":
                e0 = ev() if evs is not None else None
                batch.fused_pass(N_ITER2, 0.0)
                e1 = ev() if evs is not None else None
                batch.gram_alpha_inner(N_ITER2)
                e2 = ev() if evs is not None else None
                e3 = e4 = e2
            elif engine == "gram":
                e0 = ev() if evs is not None else None
                batch.gram_u_inner(N_ITER2)
                e1 = ev() if evs is not None else None
                batch.gram_panels(False)
                e2 = ev() if evs is not None else None
                batch.gram_alpha_inner(N_ITER2)
                e3 = ev() if evs is not None else None
                batch.gram_rowgram(False, 0.0)
                e4 = ev() if evs is not None else None
            else:
                e0 = ev() if evs is not None else None
                for _i in range(N_ITER2):
                    batch.pass_u()
                e1 = ev() if evs is not None else None
                for _i in range(N_ITER2):
                    batch.pass_alpha()
                e2 = ev() if evs is not None else None
                e3 = e2
                batch.pass_cost(0.0)
                e4 = ev() if evs is not None else None
            if evs is not None:
                evs.append((e0, e1, e2, e3, e4))

    if engine in ("gram", "fused"):
        batch.gram_init()
    else:
        batch.pass_init()
    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(args.warmup):
        one_step()
    barrier()
    sampler.mark_begin()
    launches0 = batch.launch_count()
    evs = []
    t_start, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_start.record()
    for _ in range(args.steps):
        one_step(evs)
    t_end.record()
    barrier()
    clocks = sampler.stop()
    elapsed_ms = t_start.elapsed_time(t_end)
    launches = batch.launch_count() - launches0
    seg = [float(np.mean([e[k].elapsed_time(e[k + 1]) for e in evs])) for k in range(4)]
    if engine == "fused":
        batch.fused_finish(0.0)           # cost of the last iterate (outside the timed region: one extra pass per FIT, not per step)
    st = batch.states()[0]
    assert st.n_outer == (args.warmup + args.steps) * OUTER_PER_STEP and np.isfinite(st.cost)
    if engine == "fused":
        kern = {"fused_outer_kernel": seg[0], "alpha_inner_kernel": seg[1]}
    elif engine == "gram":
        kern = {"u_inner_kernel": seg[0], "gram_panel_kernel": seg[1], "alpha_inner_kernel": seg[2], "rowgram4_kernel": seg[3]}
    else:
        kern = {"u_pass_kernel": seg[0] / N_ITER2, "alpha_pass_kernel": seg[1] / N_ITER2, "cost_kernel": seg[3]}

    # ---- the reference-shaped one-launch-per-inner-iteration passes, same data, timed on their own
    stream = None
    if engine in ("gram", "fused") and not args.profile:
        sb = FitBatch(prob, N_UNK, [hU], [hA], engine="stream")
        sb.pass_init()
        for fn in (sb.pass_u, sb.pass_alpha, lambda: sb.pass_cost(0.0)):
            for _ in range(3):
                fn()
        tms = []
        for fn in (sb.pass_u, sb.pass_alpha, lambda: sb.pass_cost(0.0)):
            torch.cuda.synchronize()
            a0_, n_rep = ev(), 10
            for _ in range(n_rep):
                fn()
            a1_ = ev()
            torch.cuda.synchronize()
            tms.append(a0_.elapsed_time(a1_) / n_rep)
        stream = {"u_pass_kernel": {"ms_per_launch": tms[0], "achieved": bytes_u / tms[0] / 1e6, "algorithmic_bytes_per_launch": int(bytes_u)},
                  "alpha_pass_kernel": {"ms_per_launch": tms[1], "achieved": bytes_a / tms[1] / 1e6, "algorithmic_bytes_per_launch": int(bytes_a)},
                  "cost_kernel": {"ms_per_launch": tms[2], "achieved": bytes_a / tms[2] / 1e6, "algorithmic_bytes_per_launch": int(bytes_a)},
                  "update_iters_per_sec": 2 * N_ITER2 / ((tms[0] + tms[1]) * N_ITER2 + tms[2]) * 1e3}
        sb.close()
        del sb

    # ---- N > 1: CpG-row sharding of ONE 1M-row fit over the ranks (BASELINE config 5's partitioning; strong scaling).  Rank r holds
    # rows row_range(M, r, world) of X, d_x, R_trunc, u and a replica of alpha; per outer iteration ONE fused pass over its rows, ONE
    # all-reduce of [G_j | bx_j | cost, ||u||^2] (in-kernel over NVLink peer memory; NCCL if symmetric memory is unavailable) and the
    # per-sample kernel that tests / commits / iterates identically on every rank.
    row_sharded = None
    if world > 1 and engine in ("gram", "fused") and not args.profile:
        from demethify_b200.sharded import GpuShardBackend, RowShardedFit, row_range
        lo, hi = row_range(M, rank, world)
        sprob = prob.row_slice(lo, hi)

        def sharded_fit(n_outer):
            be = GpuShardBackend(sprob, None, None, N_UNK, hU[lo:hi], hA)
            peer = os.environ.get("DMF_BENCH_PEER", "1") == "1" and be.enable_peer_exchange(None)
            fit = RowShardedFit(be)
            fit.init()
            be.reserve((n_outer + 2) * N_ITER2 + 4 * N_ITER2)
            return be, fit, peer

        # parity inside the leg: 5 outer iterations sharded vs the same 5 on one GPU (every rank holds the whole problem here)
        k_par = 5
        be, fit, use_peer = sharded_fit(k_par)
        for _ in range(k_par):
            fit.outer(N_ITER2, 0.0)
        fit.finish(0.0)
        (_, a_sh, n_sh, c_sh), = be.results()
        be.close()
        ref_b = FitBatch(prob, N_UNK, [hU], [hA])
        (_, a_1, n_1, c_1), = ref_b.results(ref_b.fit(k_par, N_ITER2, 0.0))
        ref_b.close()
        a_all = [torch.empty_like(torch.from_numpy(a_sh).to(dev)) for _ in range(world)]
        dist.all_gather(a_all, torch.from_numpy(a_sh).to(dev))
        replicated = all(bool(torch.equal(a_all[0], t)) for t in a_all)
        parity = {"outer_iterations": k_par, "alpha_bit_identical_on_all_ranks": bool(replicated),
                  "max_abs_d_alpha_vs_1gpu": float(np.abs(a_sh - a_1).max()), "n_outer_sharded": int(n_sh), "n_outer_1gpu": int(n_1),
                  "cost_rel_diff_vs_1gpu": float(abs(c_sh - c_1) / c_1)}
        assert replicated and parity["max_abs_d_alpha_vs_1gpu"] <= 1e-9 and n_sh == n_1 == k_par, parity
        # timed: warm-up step, then args.steps steps of OUTER_PER_STEP outer iterations
        n_total = (args.steps + 1) * OUTER_PER_STEP
        be, fit, use_peer = sharded_fit(n_total)
        for _ in range(OUTER_PER_STEP):
            fit.outer(N_ITER2, 0.0)
        barrier()
        l0 = be.batch.launch_count()
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        r0.record()
        for _ in range(args.steps * OUTER_PER_STEP):
            fit.outer(N_ITER2, 0.0)
        r1.record()
        barrier()
        rs_launches = be.batch.launch_count() - l0
        rs_ms = torch.tensor([r0.elapsed_time(r1)], dtype=torch.float64, device=dev)
        dist.all_reduce(rs_ms, op=dist.ReduceOp.MAX)
        fit.finish(0.0)
        st_rs = be.batch.states()[0]
        assert st_rs.n_outer == n_total and np.isfinite(st_rs.cost)
        if args.dump_outputs:
            (u_rows, a_rs, _n, c_rs), = be.results()
            u_parts = [None] * world
            dist.all_gather_object(u_parts, u_rows)             # rank order = row order (row_range)
            if rank == 0:
                dump_outputs(args.dump_outputs, {"u": np.concatenate(u_parts), "alpha": a_rs, "cost": c_rs})
        row_sharded = {"value": 2 * N_ITER2 * OUTER_PER_STEP * args.steps / (float(rs_ms[0]) * 1e-3), "unit": UNIT, "scaling": "strong",
                       "ms_per_step": float(rs_ms[0]) / args.steps, "rows_per_gpu": hi - lo,
                       "ms_per_outer_iteration": float(rs_ms[0]) / (args.steps * OUTER_PER_STEP),
                       "engine": "fused" if be.fused else "gram", "collectives_per_outer_iteration": 1 if be.fused else 2,
                       "launches_per_outer_iteration": rs_launches / (args.steps * OUTER_PER_STEP), "gpu_launches": int(rs_launches),
                       "allreduce": "one kernel over NVLink peer memory (dmf_gram_exchange: push, flag, rank-ordered sum)" if use_peer else "NCCL",
                       "allreduce_doubles_per_outer_iteration": int(Kt * (Kt + 1) * N_S + 8),
                       "parity": parity}
        torch.cuda.synchronize()
        be.close()
        del be, sprob

    if args.dump_outputs and row_sharded is None and rank == 0:
        (u_last, a_last, _n, c_last), = batch.results()
        dump_outputs(args.dump_outputs, {"u": u_last, "alpha": a_last, "cost": c_last})
    if args.profile:
        if rank == 0:
            print(json.dumps({"profile_run": True, "engine": engine, "ms": kern}))
        return
    # ---- end-to-end arm: public API, host buffers in, host arrays out
    nX, nD, nR, nU, nA = hX.numpy(), hD.numpy(), hR.numpy(), hU.numpy(), hA.numpy()
    batch.close()
    del batch
    # ---- parity sample: the first rows of the SAME arrays / initial iterate, one outer iteration on the GPU (CPU side below)
    parity_gpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        ms = min(CPU_SAMPLE_ROWS, M)
        pb = FitBatch(prob.row_slice(0, ms), N_UNK, [nU[:ms]], [nA])
        (pu, pa, pn, pc), = pb.results(pb.fit(1, N_ITER2, 0.0))
        parity_gpu = (ms, pu, pa, pn, pc, pb.engine)
        pb.close()
        del pb
    del prob
    torch.cuda.empty_cache()
    e2e_times = []
    for i in range(2 + min(args.steps, 3)):
        barrier()
        t0 = time.perf_counter()
        if world > 1:       # the row-sharded public call: every rank passes ITS rows (host buffers), gets its rows of u and alpha back
            from demethify_b200.sharded import mdwbssmf_deconv_sharded, row_range
            lo, hi = row_range(M, rank, world)
            os.environ.setdefault("DMF_PEER_XCHG", "1")
            u_out, a_out, _n, _c = mdwbssmf_deconv_sharded(nU[lo:hi], nA, nX[lo:hi], nD[lo:hi], nR[lo:hi], N_UNK, n_iter1=OUTER_PER_STEP,
                                                           n_iter2=N_ITER2, tol=0.0)
        else:
            lo, hi = 0, M
            u_out, a_out = dec.mdwbssmf_deconv(nU, None, nA, nX, nD, nR, N_UNK, n_iter1=OUTER_PER_STEP, n_iter2=N_ITER2, tol=0.0)
        torch.cuda.synchronize()
        e2e_times.append(time.perf_counter() - t0)
    e2e_s = float(np.mean(e2e_times[2:]))
    rows_here = hi - lo
    h2d = rows_here * (N_S * 8 + N_S * 2 + K_KNOWN * 8 + N_UNK * 8) + hA.numel() * 8
    d2h = u_out.nbytes + a_out.nbytes

    # ---- reduce over ranks: device time = max over ranks, work = sum over ranks
    its_per_step = 2 * N_ITER2 * OUTER_PER_STEP
    tmax = torch.tensor([elapsed_ms, e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    elapsed_ms, e2e_s = float(tmax[0]), float(tmax[1])
    fit_sharded_value = world * its_per_step * args.steps / (elapsed_ms * 1e-3)
    if world > 1 and row_sharded is not None:
        value, step_ms, scaling = row_sharded["value"], row_sharded["ms_per_step"], "strong"      # ONE fit, rows sharded
        e2e_value = its_per_step / e2e_s
        h2d_total = torch.tensor([float(h2d), float(d2h)], dtype=torch.float64, device=dev)
        dist.all_reduce(h2d_total)
        h2d, d2h = int(h2d_total[0]), int(h2d_total[1])
    else:
        value, step_ms, scaling = fit_sharded_value, elapsed_ms / args.steps, "weak"
        e2e_value = world * its_per_step / e2e_s

    boot = None
    if args.boot_resamples > 0 and not args.profile and engine in ("gram", "fused") and args.precision == "fp64":
        boot = bootstrap_leg(args, dev, rank, world)
    if rank == 0:
        peak, peak_src = hbm_peak_gbs()
        flops = {}
        if engine == "fused":
            passes = {"fused_outer_kernel": (kern["fused_outer_kernel"], bytes_fused)}
            flops = {"fused_outer_kernel": flops_fused}
        elif engine == "gram":
            passes = {"rowgram4_kernel": (kern["rowgram4_kernel"], bytes_rowgram), "gram_panel_kernel": (kern["gram_panel_kernel"], bytes_panel)}
        else:
            passes = {"u_pass_kernel": (kern["u_pass_kernel"], bytes_u), "alpha_pass_kernel": (kern["alpha_pass_kernel"], bytes_a)}
        dom = max(passes, key=lambda k: passes[k][0])
        dom_ms, dom_bytes = passes[dom]
        ach = dom_bytes / (dom_ms * 1e-3) / 1e9
        # FP64 peak of this pool's B200, measured by tools/fp64_peak.cu (DMMA; DFMA reaches 34.1): the second roofline (SURVEY 8 d3)
        fp64_peak, fp64_src = 37.1, "fallback: B200 FP64 37 TFLOP/s"
        fpath = os.path.join(ROOT, "profiles", "fp64_peak.json")
        if os.path.exists(fpath):
            fj = json.load(open(fpath))
            fp64_peak, fp64_src = fj["fp64_tflops"], fj["source"]
        traffic, traffic_src = None, None     # DRAM bytes per launch of the dominant kernel: ncu capture of this build and shape
        tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        if os.path.exists(tpath):
            tj = json.load(open(tpath))
            same = tj["shape"] == {"M_cpg": M, "N_samples": N_S, "K_known": K_KNOWN, "n_unknown": N_UNK,
                                   "dtype": "f64" if args.precision == "fp64" else "f32", "weights_storage": "u16" if sW == 2 else "float"}
            traffic = tj["kernels"].get(dom) if same else None
            traffic_src = tj.get("capture") if traffic is not None else None
        frac_hbm = ach / peak
        roof = {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": frac_hbm, "traffic": traffic,
                "traffic_source": traffic_src, "peak_source": peak_src, "algorithmic_bytes_per_launch": int(dom_bytes), "ms_per_launch": dom_ms,
                "frac_hbm": frac_hbm, "kernels_ms_per_launch": kern,
                "passes": {k: {"ms_per_launch": v[0], "achieved": v[1] / (v[0] * 1e-3) / 1e9, "frac": v[1] / (v[0] * 1e-3) / 1e9 / peak,
                               "algorithmic_bytes_per_launch": int(v[1])} for k, v in passes.items()}}
        if dom in flops:
            tf = flops[dom] / (dom_ms * 1e-3) / 1e12
            roof.update({"frac_fp64": tf / fp64_peak, "achieved_fp64_tflops": tf, "peak_fp64_tflops": fp64_peak, "peak_fp64_source": fp64_src,
                         "algorithmic_fp64_flops_per_launch": flops[dom]})
            if tf / fp64_peak > frac_hbm:       # the binding roofline is the larger fraction (SURVEY 8 d3)
                roof.update({"bound": "fp64", "achieved": tf, "peak": fp64_peak, "unit": "TFLOP/s", "frac": tf / fp64_peak,
                             "note": "bound/achieved/peak/frac describe the FP64 (DFMA + DMMA) pipe, the binding roofline of the fused "
                                     "pass; frac_hbm and algorithmic_bytes_per_launch give the HBM side"})
        if stream is not None:
            for k in ("u_pass_kernel", "alpha_pass_kernel", "cost_kernel"):
                stream[k]["frac"] = stream[k]["achieved"] / peak
            roof["stream_passes"] = stream
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": step_ms, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
            "dtype": "f64" if args.precision == "fp64" else "f32", "data": "synthetic",
            "config": workload_config(M, {"weights_storage": "u16" if prob_wtype_is_u16(sW, sT) else "float", "engine": engine,
                                          "parallelism": "one GPU" if world == 1 else f"ONE fit, CpG rows sharded over {world} GPUs (fit-sharded "
                                                         "weak-scaling number under fit_sharded)", "ctas_per_fit": geom["ctas_per_fit"],
                                          "tile_rows": geom["tile_rows"], "smem_bytes": geom["smem_bytes"]}),
            "fits_per_sec_at_100_outer": value / (2 * N_ITER2 * 100),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "s_per_call": e2e_s, "call": "demethify_b200.deconvolution.mdwbssmf_deconv(numpy in, numpy out)" if world == 1 else
                    "demethify_b200.sharded.mdwbssmf_deconv_sharded(this rank's rows: numpy in, numpy out), bytes summed over the ranks"},
            "gpu_launches": int(launches) if world == 1 else int(row_sharded["gpu_launches"]) if row_sharded else int(launches),
            "roofline": roof,
            "clocks": clocks,
        }
        if boot is not None:
            line["bootstrap_config4"] = boot
        if row_sharded is not None:
            line["row_sharded"] = row_sharded
            line["fit_sharded"] = {"value": fit_sharded_value, "unit": UNIT, "scaling": "weak", "ms_per_step": elapsed_ms / args.steps,
                                   "note": f"{world} independent fits, one per GPU, no data-path collective (restarts / sweep members)"}
        if not args.no_cpu and world == 1:
            ms = parity_gpu[0]
            leg = cpu_reference_leg(2, 1, rows=ms, data=(nX[:ms], nD[:ms], nR[:ms], nU[:ms], nA))
            line["cpu_baseline"] = {k: leg[k] for k in ("value", "unit", "cores", "kind", "sample")}
            cu, ca, ctr = leg["result"]
            _, pu, pa, pn, pc, peng = parity_gpu
            line["parity_sample"] = {"rows": ms, "outer_iterations": 1, "engine": peng, "same_arrays_and_init_as_gpu_arm": True,
                                     "max_abs_d_alpha": float(np.abs(pa - ca).max()), "max_abs_d_u": float(np.abs(pu - cu).max()),
                                     "n_outer_gpu": int(pn), "n_outer_cpu": int(ctr["n_outer"]),
                                     "cost_gpu": float(pc), "cost_cpu": float(ctr["costs"][-1]),
                                     "cost_rel_diff": float(abs(pc - ctr["costs"][-1]) / ctr["costs"][-1])}
        else:
            line["cpu_baseline"] = None
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def prob_wtype_is_u16(sW, sT):
    return sW == 2 and sT != 2


def main():
    global OUTER_PER_STEP
    args = parse()
    OUTER_PER_STEP = args.outer
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    run_b200(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
