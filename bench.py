#!/usr/bin/env python
"""bench.py - neg2loglik evaluations/sec (assembly + Cholesky + solves) at n = 50 000 (BASELINE.json).

    python bench.py --gpus 1 --steps K --warmup W                 our arm, one B200
    torchrun --nproc-per-node N ... bench.py --gpus N ...          our arm, N replicas (weak scaling)
    python bench.py --impl reference --steps K --warmup W          the reference's CPU path, host cores

A step is one full objective evaluation (GetNeg2loglikelihood, R/neg2loglikelihood.R:183-222) of
the synthetic nonstationary model of SURVEY.md §8(d) config 3 at a fresh theta (the optimiser's
finite-difference neighbours, R/optim.R:237-259).  With N GPUs every rank evaluates its own
theta on its own replica of the data - the reference's own fan-out, no data-path collective.
Prints ONE JSON line (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEED = 20261018
THETA = {"mean": np.zeros(5), "std.dev": np.array([0.2, 0.15, 0.10, -0.05, 0.05]),
         "scale": np.array([-1.6, 0.2, -0.15, 0.1, -0.1]), "aniso": np.array([0.1, 0.2, -0.1, 0.05, 0]),
         "tilt": np.array([0.3, -0.2, 0.1, 0.1, -0.1]), "smooth": np.array([0.2, 0.3, -0.2, 0.1, 0.1]),
         "nugget": np.array([-4, 0.1, 0.1, 0, 0])}
LIMITS = [0.5, 2.5]
DERIVED_FP64_PEAK_TFLOPS = 37.2  # 148 SM x 128 flop/clk x 1.965 GHz (SURVEY.md §8d)


def synthetic(n):
    """SURVEY.md §8(d) config 3: locs ~ U(-1,1)^2, four covariates, z ~ N(0,1), numpy PCG64 seed 20261018."""
    rng = np.random.default_rng(SEED)
    locs = rng.uniform(-1, 1, (n, 2))
    c1, c2 = (locs[:, 0] + 1) / 2, (locs[:, 1] + 1) / 2
    raw = np.column_stack([np.ones(n), c1, c2, c1 * c2,
                           0.5 + 0.5 * np.sin(np.pi * locs[:, 0]) * np.cos(np.pi * locs[:, 1])])
    mean, sd = raw.mean(axis=0), raw.std(axis=0, ddof=1)
    mean[0], sd[0] = 0.0, 1.0
    X = np.asfortranarray((raw - mean) / sd)  # getScale, R/getFunctions.R:376-436
    z = rng.standard_normal(n)
    return np.asfortranarray(locs), X, z


def theta_at(step, rank):
    """A distinct evaluation point per (step, rank): the base theta nudged the way a finite-difference
    gradient would nudge it (ndeps = eps^(1/4), R/profile.R:14)."""
    th = {k: v.copy() for k, v in THETA.items()}
    keys = ("std.dev", "scale", "aniso", "tilt", "smooth", "nugget")
    idx = (step * 131 + rank * 17) % 30
    th[keys[idx // 5]][idx % 5] += np.finfo(float).eps ** 0.25
    return th


def flops_chol(n):
    return n ** 3 / 3 + n ** 2 / 2 + n / 6


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        time.sleep(0.05)
        sm, smax, power, reasons = [], [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])), smax.append(float(r[2])), power.append(float(r[3]))
            except (ValueError, IndexError):
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7),
                              ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(smax)), "power_w_max": float(max(power)),
                "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------------------
# the reference's CPU path on the host cores (oracle/_ref = its own source compiled, + LAPACK)
# ---------------------------------------------------------------------------------------------
def _asm_sample(args):
    n_s, kind, n_full = args
    from oracle import cov
    locs, X, _ = synthetic(n_full)
    # a random subset of the sites of the full problem: the same per-pair branch mix as the full pair loop
    idx = np.sort(np.random.default_rng(os.getpid()).choice(n_full, n_s, replace=False))
    locs, X = np.asfortranarray(locs[idx]), np.asfortranarray(X[idx])
    t0 = time.perf_counter()
    cov.cov_rns(THETA, locs, X, LIMITS, kind=kind)
    return time.perf_counter() - t0


def host_ram_gb():
    try:
        with open("/proc/meminfo") as f:
            for line in f:
                if line.startswith("MemTotal"):
                    return int(line.split()[1]) / 1048576.0
    except OSError:
        pass
    return None


def cpu_reference_sample(n, n_asm=2200, n_chol=7000):
    """One BOUNDED sample of the reference's evaluation at size n on the host cores, scaled to n.

    assembly : the reference's single-threaded pair loop (src/cocons_full.cpp:257-313) on n_asm sites drawn
               from the n-site problem -> ns/pair, scaled to n(n-1)/2 pairs; run on every core at once (one
               sample per core) the way optimParallel's workers would run it (R/optim.R:117-121)
    cholesky : LAPACK dpotrf on an n_chol matrix -> flop/s, scaled to n^3/3; (a) one thread per worker,
               (b) one worker with every thread
    The evals/s returned is an EXTRAPOLATION from this sample (flagged as such); layout (a) is capped by
    the host RAM (every worker holds its own 8 n^2-byte matrix).
    """
    import multiprocessing as mpc

    import scipy.linalg as sla
    from threadpoolctl import threadpool_limits

    from oracle import cov
    cores = os.cpu_count() or 1
    kind = "reference" if cov.have_reference() else "restatement"
    with mpc.get_context("fork").Pool(cores) as pool:
        t_asm = float(np.mean(pool.map(_asm_sample, [(n_asm, kind, n)] * cores)))
    ns_pair = t_asm / (n_asm * (n_asm - 1) / 2) * 1e9
    t_asm_full = ns_pair * 1e-9 * n * (n - 1) / 2
    rng = np.random.default_rng(1)
    A = rng.standard_normal((n_chol, 64))
    S = A @ A.T + n_chol * np.eye(n_chol)
    with threadpool_limits(limits=cores):
        t0 = time.perf_counter()
        sla.cholesky(S, lower=True, check_finite=False)
        t_all = time.perf_counter() - t0
    gflops_all = flops_chol(n_chol) / t_all / 1e9
    with threadpool_limits(limits=1):
        m1 = 2500
        t0 = time.perf_counter()
        sla.cholesky(S[:m1, :m1], lower=True, check_finite=False)
        t_one = time.perf_counter() - t0
    gflops_one = flops_chol(m1) / t_one / 1e9
    ram = host_ram_gb()
    per_worker_gb = 8e-9 * n * n * 1.1
    workers = cores if ram is None else max(1, min(cores, int(ram * 0.9 / per_worker_gb)))
    # (a) `workers` single-threaded evaluations side by side (the reference's layout, RAM permitting)
    thr_workers = workers / (t_asm_full + flops_chol(n) / (gflops_one * 1e9))
    # (b) one worker, assembly single-threaded (it has no threads), LAPACK on every core
    thr_single = 1.0 / (t_asm_full + flops_chol(n) / (gflops_all * 1e9))
    best = max(thr_workers, thr_single)
    return {"value": best, "unit": "evals/s", "cores": cores, "kind": "reference" if kind == "reference" else "port",
            "extrapolated": True,
            "sample": ("EXTRAPOLATED to n=%d from a bounded sample: reference pair loop (general Bessel branch) on %d "
                       "of the n sites per core = %.0f ns/pair; LAPACK dpotrf n=%d all threads = %.0f GFLOP/s, n=%d one "
                       "thread = %.1f GFLOP/s; layouts: %d single-threaded workers (host RAM %s GB, %.0f GB per worker) "
                       "%.3e evals/s, one worker + threaded LAPACK %.3e evals/s"
                       % (n, n_asm, ns_pair, n_chol, gflops_all, m1, gflops_one, workers,
                          "%.0f" % ram if ram else "?", per_worker_gb, thr_workers, thr_single)),
            "ns_per_pair": ns_pair, "dpotrf_gflops_all_threads": gflops_all, "dpotrf_gflops_one_thread": gflops_one,
            "workers": workers, "host_ram_gb": ram}


def reference_full_eval(n_small):
    """ONE real end-to-end evaluation of the reference's CPU path at n_small sites (not extrapolated): its
    cov_rns (single-threaded, as the reference is) + LAPACK dpotrf / dtrtrs on every core
    (R/neg2loglikelihood.R:183-222); returns seconds and the value."""
    import scipy.linalg as sla

    from oracle import cov
    locs, X, z = synthetic(n_small)
    kind = "reference" if cov.have_reference() else "restatement"
    t0 = time.perf_counter()
    S = cov.cov_rns(THETA, locs, X, LIMITS, kind=kind)
    t1 = time.perf_counter()
    c = sla.cholesky(S, lower=True, check_finite=False, overwrite_a=True)
    y = sla.solve_triangular(c, z, lower=True, check_finite=False)
    v = n_small * np.log(2 * np.pi) + 2 * float(np.sum(np.log(np.diag(c)))) + float(y @ y)
    t2 = time.perf_counter()
    return {"n": n_small, "seconds": t2 - t0, "assembly_s": t1 - t0, "lapack_s": t2 - t1, "neg2loglik": v,
            "kind": kind, "note": "measured, not extrapolated: one full evaluation at this n"}


def run_reference(args, rank, world):
    if rank != 0:
        return
    from oracle import cov
    # load the checker library in THIS process (the samples run in forked workers)
    locs0, X0, _ = synthetic(64)
    cov.cov_rns(THETA, locs0, X0, LIMITS, kind="reference" if cov.have_reference() else "restatement")
    vals, t_steps = [], []
    res = None
    t_region0 = time.perf_counter()
    for s in range(args.warmup + args.steps):
        if s == args.warmup:
            t_region0 = time.perf_counter()
        t0 = time.perf_counter()
        res = cpu_reference_sample(args.n)
        if s >= args.warmup:
            vals.append(res["value"])
            t_steps.append(time.perf_counter() - t0)
    region = time.perf_counter() - t_region0
    v = float(np.mean(vals))
    res["value"] = v
    full = guarded(reference_full_eval, 4000)
    # the same model predicts the measured small evaluation: a check of the extrapolation's two rates
    pred = res["ns_per_pair"] * 1e-9 * 4000 * 3999 / 2 + flops_chol(4000) / (res["dpotrf_gflops_all_threads"] * 1e9)
    full["model_predicts_s"] = pred
    line = {"impl": "reference", "metric": "neg2loglik evals/sec (assembly+Cholesky) at n=50k", "value": v,
            "unit": "evals/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            # a step of this arm is one bounded SAMPLE of the workload: ms_per_step is its measured duration;
            # `value` is the evaluations/s at n the sample extrapolates to (1e3 / value = ms per full evaluation)
            "ms_per_step": region / args.steps * 1e3, "ms_per_eval_extrapolated": 1e3 / v, "extrapolated": True,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": "synthetic n=%d nonstationary Matern, 4 covariates (p=5), r=1, ML objective"
                                   % args.n, "n": args.n},
            "cpu_baseline": res, "measured_full_eval": full,
            "e2e": {"value": v, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "sample_seconds_per_step": float(np.mean(t_steps))}
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------
def dgemm_ceiling(torch, dev, n=8192, reps=4):
    a = torch.randn(n, n, dtype=torch.float64, device=dev)
    b = torch.randn(n, n, dtype=torch.float64, device=dev)
    torch.matmul(a, b)
    torch.cuda.synchronize()
    best = 0.0
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.matmul(a, b)
        e1.record()
        torch.cuda.synchronize()
        best = max(best, 2 * n ** 3 / e0.elapsed_time(e1) / 1e9)
    del a, b
    torch.cuda.empty_cache()
    return best


def load_goldens(n):
    """tests/golden/n2ll_large.json (oracle/make_golden_large.py: the reference's compiled cov_rns + LAPACK)."""
    try:
        with open(os.path.join(ROOT, "tests", "golden", "n2ll_large.json")) as f:
            cases = json.load(f)["cases"]
    except (OSError, ValueError, KeyError):
        return {}
    return {c["point"]: c for c in cases.values() if c["n"] == n}


def golden_theta(case):
    return {k: np.array(v, dtype=np.float64) for k, v in case["theta"].items()}


def north_star_problem(n_big):
    """Data of the n_big-site north-star evaluation: the first n_big sites of one synthetic stream of n_big + n_big / 5
    sites (the rest are the prediction sites of BASELINE configs[4]); theta = theta_at(0, 0)."""
    m_pred = n_big // 5
    locs_all, X_all, z_all = synthetic(n_big + m_pred)
    return (np.asfortranarray(locs_all[:n_big]), np.asfortranarray(X_all[:n_big]), z_all[:n_big],
            np.asfortranarray(locs_all[n_big:]), np.asfortranarray(X_all[n_big:]), theta_at(0, 0))


def sampled_sites(n, m=48, seed=7):
    return np.sort(np.random.default_rng(seed).choice(n, m, replace=False))


def sampled_factor_residual(ctx, n_big):
    """max |(L L^T - Sigma)_ab| / sqrt(Sigma_aa Sigma_bb) over all pairs of the sampled sites: L rows from the device
    factor, Sigma from the committed fixture tests/golden/sigma_samples.npz (the reference's compiled cov_rns on
    those sites, written by `python -m oracle.make_golden_large --sigma-samples`; an entry of cov_rns depends on its
    two sites and theta only).  Size-independent check of assembly + factorisation; None without a fixture."""
    try:
        fx = np.load(os.path.join(ROOT, "tests", "golden", "sigma_samples.npz"))
        sites, S = fx["sites_n%d" % n_big], fx["sigma_n%d" % n_big]
    except (OSError, KeyError):
        return None
    rows, _ = ctx.factor_rows(sites)
    G = rows @ rows.T
    d = np.sqrt(np.diag(S))
    return {"max_rel": float(np.max(np.abs(G - S) / np.outer(d, d))), "sampled_sites": int(len(sites)),
            "entries": int(len(sites) * (len(sites) + 1) // 2),
            "sigma_from": "tests/golden/sigma_samples.npz (reference's compiled cov_rns)",
            "what": "max |(L L^T - Sigma)_ab| / sqrt(Sigma_aa Sigma_bb)"}


def reference_datasets_record(local_rank):
    """BASELINE.json configs[0] / [1]: the reference's own data sets (holes n = 5570, stripes n = 11 977, shipped as
    tests/golden/datasets.npz) - the all-aspects ML objective against the committed golden (reference-compiled
    covariance + LAPACK), evaluations/s one at a time and with 8 in flight on this GPU (the optimiser's
    finite-difference points, R/optim.R:237-259)."""
    import cocons_b200 as cb
    from cocons_b200 import _lib
    D = np.load(os.path.join(ROOT, "tests", "golden", "datasets.npz"))
    with open(os.path.join(ROOT, "tests", "golden", "n2ll_cases.json")) as f:
        gold = {c["name"]: c for c in json.load(f)["cases"]}
    out = {}
    for name, key, cols in (("holes", "holes_training", [2, 3]), ("stripes", "stripes_training", [2, 3, 4])):
        c = gold[name + "_full_general"]
        M, n = D[key], c["n"]
        X = cb.getScale(np.column_stack([np.ones(n)] + [M[:n, k] for k in cols]))["std.covs"]
        pp = {k: (np.array(v, dtype=bool) if isinstance(v, list) else v) for k, v in c["par_pos"].items()}
        v = cb.GetNeg2loglikelihood(np.array(c["theta"]), pp, M[:n, :2], X, c["limits"], M[:n, -1], n, c["lambda"])
        tl = cb.getModelLists(np.array(c["theta"]), pp, "diff")
        pts = []
        for k in range(32):
            t = {a: x.copy() for a, x in tl.items()}
            t["scale"][0] += 1e-4 * k
            pts.append(t)

        def f(ctx, t):
            return ctx.terms(_lib.ML, t, c["limits"], t["mean"])["logdet"]
        rates, ref = {}, None
        for size in (1, 8):
            with cb.DenseLikelihoodPool(M[:n, :2], X, M[:n, -1], size=size, device=local_rank) as pool:
                pool.map(f, pts[:size])
                t0 = time.perf_counter()
                vals = pool.map(f, pts)
                rates[size] = len(pts) / (time.perf_counter() - t0)
            if ref is None:
                ref = vals
            same = bool(vals == ref)
        out[name] = {"n": n, "p": X.shape[1], "neg2loglik_rel_err_vs_golden": abs(v - c["values"]["ml"]) / abs(c["values"]["ml"]),
                     "evals_per_s_one_at_a_time": rates[1], "evals_per_s_8_in_flight": rates[8],
                     "pooled_values_bit_identical": same}
    cb._lib.lib().cocons_release_workspace()
    return out


def north_star_single(local_rank, n_big, with_predict=False):
    """north_star: one full evaluation at n = 100 000 on ONE B200 (80 GB matrix), device-timed phases, Cholesky
    phase against the FP64 peak, and the sampled-entry residual of its factor against the reference covariance."""
    import cocons_b200 as cb
    from cocons_b200 import _lib
    locs, X, z, lp, Xp, th = north_star_problem(n_big)
    m_pred = lp.shape[0]
    cfg4 = None
    with cb.DenseLikelihood(locs, X, z, device=local_rank) as ctx:
        t = ctx.terms(_lib.ML, th, LIMITS, th["mean"])
        tm = ctx.timings()
        resid = sampled_factor_residual(ctx, n_big)
        if with_predict:
            # BASELINE.json configs[4]: cocoPredict (type "pred") for n/5 new sites and one cocoSim draw on the KEPT
            # factor (R/predict.R:136-183, R/sim.R:87-121), with size-independent checks
            import torch
            r = z - X @ th["mean"]
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            sto, expl = ctx.predict(lp, Xp, r)
            t_pred = time.perf_counter() - t0
            prior = np.exp(Xp @ th["std.dev"]) + np.exp(Xp @ th["nugget"])
            rng = np.random.default_rng(SEED + 1)
            sub = np.sort(rng.choice(m_pred, 300, replace=False))
            s2, e2 = ctx.predict(lp[sub], Xp[sub], r)
            # kriging at TRAINING coordinates interpolates: a coincident pair takes variance + nugget
            # (src/cocons_full.cpp:284-286), so the predictor returns the residual itself and explains everything
            tr = np.sort(rng.choice(n_big, 64, replace=False))
            s3, e3 = ctx.predict(locs[tr], X[tr], r)
            prior_tr = np.exp(X[tr] @ th["std.dev"]) + np.exp(X[tr] @ th["nugget"])
            eps = rng.standard_normal((n_big, 1))
            t0 = time.perf_counter()
            draw = ctx.sim(eps)
            t_sim = time.perf_counter() - t0
            cfg4 = {"prediction_sites": m_pred, "predict_s": t_pred, "sim_s": t_sim,
                    "predict_tflops": 2.0 * m_pred * n_big * n_big / 2 / t_pred / 1e12,
                    "checks": {"finite": bool(np.all(np.isfinite(sto)) and np.all(np.isfinite(expl))),
                               "explained_within_prior": bool(np.all(expl >= 0) and np.all(expl <= prior * (1 + 1e-9))),
                               "subset_of_300_bit_identical": bool(np.array_equal(s2, sto[sub]) and np.array_equal(e2, expl[sub])),
                               "interpolation_at_64_training_sites_rel": float(np.max(np.abs(s3 - r[tr]) / np.abs(r[tr]))),
                               "explained_equals_prior_at_training_sites_rel": float(np.max(np.abs(e3 - prior_tr) / prior_tr)),
                               "draw_variance_over_model_variance": float(np.mean(
                                   draw[:, 0] ** 2 / (np.exp(X @ th["std.dev"]) + np.exp(X @ th["nugget"]))))}}
    tf = flops_chol(n_big) / (tm["factor_ms"] * 1e-3) / 1e12
    return {"n": n_big, "config4_predict_sim": cfg4,
            "eval_ms": tm["total_ms"], "assembly_ms": tm["assembly_ms"], "factor_ms": tm["factor_ms"],
            "solve_ms": tm["solve_ms"], "chol_tflops": tf, "frac_of_derived_fp64_peak": tf / DERIVED_FP64_PEAK_TFLOPS,
            "value": n_big * np.log(2 * np.pi) + 2 * t["logdet"] + float(t["quad"][0]),
            "factor_residual": resid}


def distributed_record(torch, dist, dev, rank, world, n_large):
    """BASELINE.json configs[3] / north_star (c): ONE matrix over all ranks (column-panel block-cyclic
    Cholesky, NCCL panel broadcast).  A golden-pinned evaluation at n = 20 000 through the same code, then
    one evaluation at n_large.  Times are the max over ranks of device-synchronised phases."""
    import cocons_b200 as cb  # noqa: F401
    from cocons_b200 import _lib
    from cocons_b200.distributed import DistributedDenseLikelihood

    def vmax(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    rec = {"layout": "512-wide column panels dealt in a snake over the ranks (1 x N block-cyclic), one NCCL "
                     "broadcast of the factored panel per step, one-panel look-ahead", "nccl_ranks": world}
    gold = load_goldens(20000)
    if gold:
        locs, X, z = synthetic(20000)
        worst = 0.0
        with DistributedDenseLikelihood(locs, X, z) as d:
            for name, c in sorted(gold.items()):
                th = golden_theta(c)
                t = d.terms(_lib.ML, th, LIMITS, th["mean"])
                v = 20000 * np.log(2 * np.pi) + 2 * t["logdet"] + float(t["quad"][0])
                worst = max(worst, abs(v - c["neg2loglik"]) / abs(c["neg2loglik"]))
        rec["parity_n20k_rel"] = worst
        rec["parity_n20k_points"] = sorted(gold)
    # the optimiser's fan-out (SURVEY §8f N1, R/optim.R:237-259): 2p + 1 = 61 finite-difference points of the n = 20 000
    # problem dealt over the ranks by distributed.fan_out (NCCL all_gather of the values), against rank 0's own values
    from cocons_b200.distributed import fan_out
    locs, X, z = synthetic(20000)
    pts = [theta_at(k, 0) for k in range(61)]
    with cb.DenseLikelihood(locs, X, z, device=dev.index) as ctx:
        def f(th):
            t = ctx.terms(_lib.ML, th, LIMITS, th["mean"])
            return 20000 * np.log(2 * np.pi) + 2 * t["logdet"] + float(t["quad"][0])
        f(pts[0])
        dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        vals = fan_out(pts, f)
        t_fan = vmax(time.perf_counter() - t0)
        local = [f(th) for th in pts[:8]] if rank == 0 else None
    if rank == 0:
        rec["fan_out"] = {"points": len(pts), "n": 20000, "seconds": t_fan, "evals_per_s": len(pts) / t_fan,
                          "bit_identical_to_rank0_on_first_8": bool(vals[:8] == local)}
    # the two drivers on the same n = 100 000 problem: rank 0 alone (look-ahead driver, one GPU), then all ranks
    n_mid = 100000
    single = None
    if rank == 0:
        single = north_star_single(dev.index, n_mid)
    dist.barrier()
    locs, X, z = north_star_problem(n_mid)[:3]
    with DistributedDenseLikelihood(locs, X, z) as d:
        t = d.terms(_lib.ML, theta_at(0, 0), LIMITS, THETA["mean"])
        v_dist = n_mid * np.log(2 * np.pi) + 2 * t["logdet"] + float(t["quad"][0])
        ph = {k: vmax(v) for k, v in d.last_phase_s.items()}
    if rank == 0:
        rec["agreement_n100k"] = {"single_gpu_value": single["value"], "distributed_value": v_dist,
                                  "rel_diff": abs(single["value"] - v_dist) / abs(single["value"]),
                                  "single_gpu": single, "distributed_eval_s": ph["assemble_factor_s"] + ph["solve_s"]}
    locs, X, z = synthetic(n_large)
    os.environ["COCONS_DIST_PROFILE"] = "1"
    with DistributedDenseLikelihood(locs, X, z) as d:
        dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        t = d.terms(_lib.ML, theta_at(0, 0), LIMITS, THETA["mean"])
        torch.cuda.synchronize()
        wall = vmax(time.perf_counter() - t0)
        ph = {k: vmax(v) for k, v in d.last_phase_s.items()}
        waits = d.last_wait_ms
    tf = flops_chol(n_large) / ph["assemble_factor_s"] / 1e12
    rec.update({"n": n_large, "eval_s": wall, "assemble_factor_s": ph["assemble_factor_s"], "solve_s": ph["solve_s"],
                "chol_tflops_all_gpus": tf, "chol_tflops_per_gpu": tf / world,
                "frac_of_derived_fp64_peak_per_gpu": tf / world / DERIVED_FP64_PEAK_TFLOPS,
                "note": "assembly included in the Cholesky-phase time; FP64 peak = derived %.1f TFLOP/s per GPU"
                        % DERIVED_FP64_PEAK_TFLOPS,
                "value": n_large * np.log(2 * np.pi) + 2 * t["logdet"] + float(t["quad"][0]),
                "bcast_wait_ms_rank0": waits})
    return rec


def guarded(fn, *a, **k):
    """Secondary records (CPU baseline, north-star sizes, the reference's data sets, the distributed evaluation) never
    cost the headline line: a failure is reported in place of the record and the device workspace is handed back."""
    try:
        return fn(*a, **k)
    except Exception as e:  # noqa: BLE001 - whatever it was, the measured headline is still printed
        try:
            from cocons_b200 import _lib
            _lib.lib().cocons_release_workspace()
        except Exception:  # noqa: BLE001
            pass
        return {"error": "%s: %s" % (type(e).__name__, str(e)[:300])}


def dump_outputs(out_dir, terms, value):
    """What the last timed step computed, one float64 DIR/<name>.npy per array: the terms DenseLikelihood.terms
    returned to its caller and the -2 loglik formed from them.  The data and the theta of every step are fixed by
    --sites, --warmup and --steps, so two builds run with the same arguments can be compared array by array."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"neg2loglik": value, "logdet": terms["logdet"], "quad": terms["quad"], "logdet_w": terms["logdet_w"],
              "rank": terms["rank"]}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.atleast_1d(np.asarray(a, dtype=np.float64)))


def cusolver_potrf_comparator(torch, dev, n):
    """SURVEY.md §8(d): the library bar - torch.linalg.cholesky (cuSOLVER potrf, FP64) on an SPD matrix of the same
    n.  Comparison only; nothing of it is on the product path."""
    try:
        g = torch.Generator(device=dev).manual_seed(1)
        M = torch.randn(n, 64, dtype=torch.float64, device=dev, generator=g)
        A = M @ M.T
        A.diagonal().add_(float(n))
        del M
        best = None
        for _ in range(2):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            Lc = torch.linalg.cholesky(A)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            best = ms if best is None else min(best, ms)
            del Lc
        del A
        torch.cuda.empty_cache()
        return {"routine": "torch.linalg.cholesky (cuSOLVER potrf), float64", "n": n, "ms": best,
                "tflops": flops_chol(n) / (best * 1e-3) / 1e12}
    except Exception as e:  # comparison only: never fail the bench for it
        torch.cuda.empty_cache()
        return {"routine": "torch.linalg.cholesky", "unavailable": str(e)[:200]}


def run_ours(args, rank, world, local_rank):
    import torch

    import cocons_b200 as cb
    from cocons_b200 import _lib
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - cocons_b200 has no CPU path to fall back to")
    torch.cuda.set_device(local_rank)
    os.environ["COCONS_DEVICE"] = str(local_rank)  # device of the one-shot (host-buffer) entry point
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        # NCCL writes its banner / debug lines to stdout by default; stdout carries the ONE JSON line
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    n = args.n
    locs, X, z = synthetic(n)
    p = X.shape[1]
    par_pos = {k: np.ones(p, dtype=bool) for k in ("mean", "std.dev", "scale", "aniso", "tilt", "smooth", "nugget")}
    lam = (0.0, 0.0, 0.0)
    L = _lib.lib()

    def point(step):
        """(optimiser-level theta vector, its getModelLists image): BOTH arms evaluate exactly this image, so
        their values must agree bit for bit (getModelLists' (a+b)/2 does not return theta_at()'s std.dev
        exactly, so the image - not theta_at() itself - is the evaluation point)."""
        x = theta_vec(theta_at(step, rank), par_pos)
        return x, cb.getModelLists(x, par_pos, "diff")

    def n2ll(t):
        return n * np.log(2 * np.pi) + 2 * t["logdet"] + float(t["quad"][0])

    peak = dgemm_ceiling(torch, dev) if (rank == 0 and not args.profile) else 0.0

    # ---- device-resident arm: inputs in HBM before the timed region --------------------------
    stream = torch.cuda.current_stream().cuda_stream
    ctx = cb.DenseLikelihood(locs, X, z, device=local_rank, stream=stream)
    # parity against the oracle's goldens at this very size (untimed; doubles as warm-up)
    parity = {}
    if rank == 0 and not args.profile:
        for name, c in sorted(load_goldens(n).items()):
            th = golden_theta(c)
            v = n2ll(ctx.terms(_lib.ML, th, LIMITS, th["mean"]))
            parity[name] = abs(v - c["neg2loglik"]) / abs(c["neg2loglik"])
    values = []
    for s in range(args.warmup):
        tl = point(s)[1]
        t = ctx.terms(_lib.ML, tl, LIMITS, tl["mean"])
    phases = {"assembly_ms": [], "factor_ms": [], "solve_ms": [], "kernel_ms": []}
    sampler = ClockSampler(local_rank)
    barrier()
    if rank == 0:
        sampler.start()
    launches0 = L.cocons_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s in range(args.steps):
        tl = point(args.warmup + s)[1]
        t = ctx.terms(_lib.ML, tl, LIMITS, tl["mean"])
        values.append(n2ll(t))
        tm = ctx.timings()
        for k in phases:
            phases[k].append(tm[k])
    e1.record()
    barrier()
    launches = L.cocons_launch_count() - launches0
    elapsed = max_over_ranks(e0.elapsed_time(e1) * 1e-3)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, t, values[-1])
    # run-to-run reproducibility of the device-resident arm: the first timed point once more, bit for bit
    tl = point(args.warmup)[1]
    again = n2ll(ctx.terms(_lib.ML, tl, LIMITS, tl["mean"]))
    mismatches = int(again != values[0])
    ctx.close()

    if args.profile:
        if rank == 0:
            print(json.dumps({"profile_run": True, "ms_per_step": elapsed / args.steps * 1e3,
                              "phases_ms": {k: float(np.mean(v)) for k, v in phases.items()},
                              "gpu_launches": int(launches)}))
        return
    # ---- end to end: the call an R user makes, host buffers in, scalar out, every step -------
    for s in range(min(args.warmup, 2)):
        cb.GetNeg2loglikelihood(point(s)[0], par_pos, locs, X, LIMITS, z, n, lam)
    barrier()
    worst = 0.0
    t0 = time.perf_counter()
    for s in range(args.steps):
        v = cb.GetNeg2loglikelihood(point(args.warmup + s)[0], par_pos, locs, X, LIMITS, z, n, lam)
        if v != values[s]:  # same theta, same kernels, another context: must be the same bits
            mismatches += 1
            worst = max(worst, abs(v - values[s]) / abs(v))
    torch.cuda.synchronize()
    e2e_elapsed = max_over_ranks(time.perf_counter() - t0)
    L.cocons_release_workspace()
    mismatches = int(max_over_ranks(float(mismatches)))
    worst = max_over_ranks(worst)
    barrier()

    distributed = None
    if dist is not None and not args.no_distributed:
        n_large = args.dist_sites or {2: 140000, 3: 170000}.get(world, 200000 if world >= 4 else 100000)
        distributed = guarded(distributed_record, torch, dist, dev, rank, world, n_large)

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        if mismatches:
            sys.exit(3)
        return
    value = world * args.steps / elapsed
    f_ms = float(np.mean(phases["factor_ms"]))
    phase_tflops = flops_chol(n) / (f_ms * 1e-3) / 1e12
    # dominant kernel: the largest trailing-update launch of each factorisation (C -= P P^T on the
    # (n_pad - 2K)^2 lower triangle, K = 768 at n = 50 000), bracketed by CUDA events inside the timed region
    n_pad = (n + 127) // 128 * 128
    # outer panel width, the rule of chol_outer() in csrc/chol.cu: 768 from 16 384 sites up, 512 from 8192, else 256
    kk = 128 * max(1, min(int(os.environ.get("COCONS_CHOL_OUTER",
                                             "6" if n_pad >= 16384 else ("4" if n_pad >= 8192 else "2"))), 16))
    rest = n_pad - 2 * kk
    kernel_flops = rest * (rest + 1) / 2 * 2 * kk  # algorithmic: lower triangle incl. diagonal
    k_ms = float(np.mean(phases["kernel_ms"]))
    achieved = kernel_flops / (k_ms * 1e-3) / 1e12 if k_ms > 0 else None
    traffic, traffic_src = None, None
    try:
        with open(os.path.join(ROOT, "profiles", "gemm_tma_ncu_traffic.json")) as f:
            tr = json.load(f)
        if tr.get("n") == n:
            traffic, traffic_src = tr["dram_bytes_per_launch"], tr["source"]
    except (OSError, ValueError, KeyError):
        pass
    cpu = guarded(cpu_reference_sample, n) if world == 1 and not args.no_cpu_baseline else None
    big = guarded(north_star_single, local_rank, 100000, with_predict=True) if (world == 1 and not args.no_large) else None
    small = guarded(reference_datasets_record, local_rank) if world == 1 else None
    lib_cmp = cusolver_potrf_comparator(torch, dev, n) if (world == 1 and not args.no_large) else None
    line = {
        "metric": "neg2loglik evals/sec (assembly+Cholesky) at n=50k", "value": value, "unit": "evals/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": elapsed / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "synthetic n=%d nonstationary Matern, 4 covariates (p=5), r=1, ML objective" % n,
                   "n": n, "p": p, "r": 1, "parallelism": "replicas x%d (one theta per GPU, no collective)" % world,
                   "l2": "working set %.1f GB per evaluation >> 126 MB L2; no flush needed" % (8e-9 * n * n),
                   "objective_value_step0": values[0]},
        "parity": {"golden": "tests/golden/n2ll_large.json (reference's compiled cov_rns + LAPACK, n=%d)" % n,
                   "rel_err": parity, "max_rel_err": max(parity.values()) if parity else None, "bar": 1e-8},
        "repro": {"checked": args.steps + 1, "mismatches": mismatches, "worst_rel": worst,
                  "what": "device-resident arm vs host-buffer arm at the same theta, every timed step, and the first "
                          "timed point evaluated twice: values must be bit-identical"},
        "phases_ms": {k: float(np.mean(v)) for k, v in phases.items() if k != "kernel_ms"},
        "assembly_pairs_per_s": n * (n - 1) / 2 / (float(np.mean(phases["assembly_ms"])) * 1e-3),
        "roofline": {"bound": "tensor",
                     "kernel": "gemm_nt_tma_kernel<64,2,0> (DMMA.8x8x4 trailing update, bulk-copy fed): the largest "
                               "launch of each factorisation, %d^2 lower triangle x K=%d" % (rest, kk),
                     "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                     "frac": achieved / peak if (peak and achieved) else None,
                     "traffic": traffic, "traffic_source": traffic_src,
                     "algorithmic_flops_per_launch": kernel_flops, "launch_ms": k_ms,
                     "peak_source": "same-run cuBLAS dgemm 8192^3 (torch.matmul float64), burst; "
                                    "MEASURED_PEAKS.json has no FP64 entry",
                     "derived_peak": DERIVED_FP64_PEAK_TFLOPS,
                     "frac_of_derived": achieved / DERIVED_FP64_PEAK_TFLOPS if achieved else None,
                     "dmma_pipe_peak": 36.9,  # tools/micro/dmma_peak.cu on this pool (register-only DMMA loop)
                     "cholesky_phase": {"achieved": phase_tflops, "frac": phase_tflops / peak if peak else None,
                                        "frac_of_derived": phase_tflops / DERIVED_FP64_PEAK_TFLOPS,
                                        "algorithmic_flops_per_eval": flops_chol(n), "ms": f_ms}},
        "e2e": {"value": world * args.steps / e2e_elapsed, "unit": "evals/s",
                "h2d_bytes_per_step": int(8 * (n * 2 + n * p + n + 7 * p)), "d2h_bytes_per_step": int(8 * 2 + 4)},
        "gpu_launches": int(launches), "clocks": clocks,
    }
    if cpu is not None:
        line["cpu_baseline"] = cpu
    if big is not None:
        line["north_star_n100k_1gpu"] = big
    if small is not None:
        line["reference_datasets"] = small
    if lib_cmp is not None:
        line["roofline"]["cholesky_phase"]["library_comparator"] = lib_cmp
    if distributed is not None:
        line["distributed"] = distributed
    print(json.dumps(line))
    sys.stdout.flush()
    if dist is not None:
        dist.destroy_process_group()
    if mismatches:
        sys.stderr.write("bench.py: %d evaluation(s) were not bit-reproducible (worst %.3e relative)\n"
                         % (mismatches, worst))
        sys.exit(3)


def theta_vec(tl, par_pos):
    """Optimiser-level theta vector whose getModelLists(type='diff') image is tl (all aspects free)."""
    a, b = tl["std.dev"] + tl["scale"], tl["std.dev"] - tl["scale"]
    parts = {"mean": tl["mean"], "std.dev": a, "scale": b, "aniso": tl["aniso"], "tilt": tl["tilt"],
             "smooth": tl["smooth"], "nugget": tl["nugget"]}
    return np.concatenate([parts[k] for k in ("mean", "std.dev", "scale", "aniso", "tilt", "smooth", "nugget")])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--sites", dest="n", type=int, default=50000, help="sites (the metric is quoted at 50 000)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-distributed", action="store_true",
                    help="N > 1: skip the one-matrix-over-all-GPUs record (BASELINE.json configs[3])")
    ap.add_argument("--dist-sites", type=int, default=0, help="N > 1: sites of the distributed evaluation")
    ap.add_argument("--no-large", action="store_true", help="N = 1: skip the n = 100 000 north-star evaluation")
    ap.add_argument("--profile", action="store_true",
                    help="profiling run: device-resident arm only (no DGEMM probe, no e2e leg, no CPU sample)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm times a CPU sample and computes no objective to dump")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
