"""Evaluations/s of the dense ML objective on the reference's own data sets (holes n = 5570, stripes n = 11 977) at the
2p + 1 finite-difference points of the golden theta, in one session, arms alternated pass by pass:
  single   one context, one point at a time (DenseLikelihood.terms)
  pool8    DenseLikelihoodPool of 8 contexts driven by host threads
  batchB   DenseLikelihoodBatch with B matrices, one terms_batch call per pass
Reports the median evaluations/s over the passes, the phase times of the last call (cocons_ctx_timings), launches per
point (cocons_launch_count), and checks that every arm returns the single context's values bit for bit.
Usage: python tools/batch_bench.py [--passes 7] [--out profiles/r05_batch.json]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import cocons_b200 as cb  # noqa: E402
from cocons_b200 import _lib  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def problem(name):
    D = np.load(os.path.join(ROOT, "tests", "golden", "datasets.npz"))
    gold = {c["name"]: c for c in json.load(open(os.path.join(ROOT, "tests", "golden", "n2ll_cases.json")))["cases"]}
    key, cols, case = {"holes": ("holes_training", [2, 3], "holes_full_general"),
                       "stripes": ("stripes_training", [2, 3, 4], "stripes_full_general")}[name]
    c = gold[case]
    M, n = D[key], c["n"]
    X = cb.getScale(np.column_stack([np.ones(n)] + [M[:n, k] for k in cols]))["std.covs"]
    pp = {k: (np.array(v, dtype=bool) if isinstance(v, list) else v) for k, v in c["par_pos"].items()}
    theta = np.array(c["theta"])
    pts = [theta]
    for i in range(len(theta)):
        for s in (1, -1):
            t = theta.copy()
            t[i] += s * np.finfo(float).eps ** 0.25
            pts.append(t)
    return M[:n, :2], X, M[:n, -1], [cb.getModelLists(t, pp, "diff") for t in pts], c["limits"]


def same(a, b):
    return a["logdet"] == b["logdet"] and np.array_equal(a["quad"], b["quad"])


def run(name, passes, batches):
    locs, X, z, lists, lim = problem(name)
    means = [t["mean"] for t in lists]
    L = _lib.lib()
    arms = {}
    single = cb.DenseLikelihood(locs, X, z)
    pool = cb.DenseLikelihoodPool(locs, X, z, size=8)
    arms["single"] = (lambda: [single.terms(_lib.ML, t, lim, t["mean"]) for t in lists], single)
    arms["pool8"] = (lambda: pool.map(lambda c, t: c.terms(_lib.ML, t, lim, t["mean"]), lists), None)
    bctx = {}
    for B in batches:
        bctx[B] = cb.DenseLikelihoodBatch(locs, X, z, B)
        arms["batch%d" % B] = (lambda B=B: bctx[B].terms_batch(_lib.ML, lists, lim, means), bctx[B])
    ref = arms["single"][0]()
    rates = {a: [] for a in arms}
    launches, phases, identical = {}, {}, {}
    for a, (fn, _) in arms.items():  # warm-up, launches per point and bits
        l0 = L.cocons_launch_count()
        got = fn()
        launches[a] = (L.cocons_launch_count() - l0) / len(lists)
        identical[a] = all(same(g, w) for g, w in zip(got, ref))
    for _ in range(passes):
        for a, (fn, _) in arms.items():
            t0 = time.perf_counter()
            fn()
            rates[a].append(len(lists) / (time.perf_counter() - t0))
    for a, (fn, ctx) in arms.items():
        if ctx is not None:
            phases[a] = ctx.timings() if isinstance(ctx, cb.DenseLikelihoodBatch) else {
                k: v for k, v in ctx.timings().items() if k.endswith("_ms") and k != "kernel_ms"}
    pool.close()
    single.close()
    for b in bctx.values():
        b.close()
    out = {"n": len(locs), "points": len(lists), "passes": passes,
           "evals_per_s_median": {a: float(np.median(v)) for a, v in rates.items()},
           "evals_per_s_all": {a: [round(x, 1) for x in v] for a, v in rates.items()},
           "launches_per_point": launches, "bit_identical_to_single": identical,
           "phase_ms_last_call": {a: {k: round(float(v), 3) for k, v in p.items()} for a, p in phases.items()}}
    print(name, json.dumps(out["evals_per_s_median"]), json.dumps(identical), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--passes", type=int, default=7)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_batch.json"))
    a = ap.parse_args()
    res = {"card": card(), "cmd": "python tools/batch_bench.py --passes %d" % a.passes,
           "holes": run("holes", a.passes, (8, 16)), "stripes": run("stripes", a.passes, (8, 16))}
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["card"]), "->", a.out)


if __name__ == "__main__":
    main()
