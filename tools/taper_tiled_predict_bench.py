"""Prediction and simulation on the tiled tapered context (cocons_predict_taper, cocons_sim_taper) on one GPU.
Bench sites (bench.synthetic), Wendland-1 taper of radius delta, m = 20 000 prediction sites uniform over the domain.

  python tools/taper_tiled_predict_bench.py --out profiles/r04_taper_tiled_predict_sim.json [--reps 3]

For n = 50 000 (delta = 0.25) and n = 200 000 (delta = 0.05), after factor_taper on a tiled context: predict_taper
without (cocoPredict type "mean") and with the explained variance (type "pred"), and sim_taper with k = 10; one
warm-up call each, then the median of `reps` calls, host clock around each call (it ends in a stream synchronise).
At n = 50 000 the same three calls on a dense context with the tapered factor run beside them, alternated.
The explained path's FP64 work is counted from the tile structure, as the forward substitution runs it: every block
of 128 prediction sites starts at the tile row of its first neighbour I0, and tile row I >= I0 costs one 128 x 128 x
128 product per stored tile (I, J) with I0 <= J < I plus one with the inverted diagonal tile (2 x 128^3 flops each).
Its rate is that count over the time of the type "pred" call minus the type "mean" call, so it includes the
assembly of the blocks' right-hand sides.  The card's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
import cocons_b200 as cb  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def morton(locs):
    """the context's site order (csrc/assembly.cu morton_order)"""
    lo, hi = locs.min(axis=0), locs.max(axis=0)
    span = hi - lo
    u = np.clip(np.where(span > 0, (locs - lo) / np.where(span > 0, span, 1), 0.0), 0, 1)
    q = (u * 4294967295.0).astype(np.uint64)

    def spread(v):
        v = v & np.uint64(0xFFFFFFFF)
        for s, m in ((16, 0x0000FFFF0000FFFF), (8, 0x00FF00FF00FF00FF), (4, 0x0F0F0F0F0F0F0F0F),
                     (2, 0x3333333333333333), (1, 0x5555555555555555)):
            v = (v | (v << np.uint64(s))) & np.uint64(m)
        return v
    return np.argsort(spread(q[:, 0]) | (spread(q[:, 1]) << np.uint64(1)), kind="stable")


def explained_flops(sp, pt, perm):
    """2 x 128^3 x the tile products of the explained solves (see the module docstring)"""
    n = sp.dimension[0]
    T = (n + 127) // 128
    inv = np.empty(n, dtype=np.int64)
    inv[perm] = np.arange(n)
    rp = sp.rowpointers.astype(np.int64) - 1
    cols = [set() for _ in range(T)]
    for r0 in range(0, n, 20000):  # the pattern's lower tiles, a slab of rows at a time
        r1 = min(n, r0 + 20000)
        i = np.repeat(np.arange(r0, r1), np.diff(rp[r0:r1 + 1]))
        j = sp.colindices[rp[r0]:rp[r1]].astype(np.int64) - 1
        keep = i >= j
        ti, tj = inv[i[keep]] // 128, inv[j[keep]] // 128
        key = np.unique(np.maximum(ti, tj) * T + np.minimum(ti, tj))
        for k in key[key // T != key % T]:
            cols[int(k % T)].add(int(k // T))
    for J in range(T):  # fill through the elimination tree
        if cols[J]:
            par = min(cols[J])
            cols[par] |= cols[J] - {par}
    rows = [[] for _ in range(T)]
    for J in range(T):
        for I in cols[J]:
            rows[I].append(J)
    rows = [np.sort(np.array(r, dtype=np.int64)) for r in rows]
    prp = pt.rowpointers.astype(np.int64) - 1
    first = np.full(pt.dimension[0], np.iinfo(np.int64).max)
    has = np.diff(prp) > 0
    pos = inv[pt.colindices.astype(np.int64) - 1]
    first[has] = np.minimum.reduceat(pos, prp[:-1][has])
    firsts = np.sort(first[has])
    total = 0
    for b in range(0, len(firsts), 128):
        I0 = int(firsts[b] // 128)
        total += sum(1 + int(np.count_nonzero(rows[I] >= I0)) for I in range(I0, T))
    return 2.0 * 128 ** 3 * total, int(T), len(firsts)


def timed(fn):
    t0 = time.perf_counter()
    out = fn()
    return time.perf_counter() - t0, out


def calls(ctx, lp, Xp, pt, resid, eps):
    return {"predict_mean_s": lambda: ctx.predict_taper(lp, Xp, pt, resid, want_explained=False),
            "predict_pred_s": lambda: ctx.predict_taper(lp, Xp, pt, resid),
            "sim_k10_s": lambda: ctx.sim_taper(eps)}


def run(n, delta, m, reps, dense):
    locs, X, z = bench.synthetic(n)
    tl = dict(bench.THETA)
    rng = np.random.default_rng(20261022)
    lp = rng.uniform(-1, 1, (m, 2))
    Xp = np.column_stack([np.ones(m), 0.5 * rng.standard_normal((m, 4))])
    sp = cb.cov_wend1(cb.nearest_dist(locs, delta=delta), (delta, 1))
    pt = cb.cov_wend1(cb.nearest_dist(lp, locs, delta=delta), (delta, 1))
    resid = z - X @ tl["mean"]
    eps = np.random.default_rng(1).standard_normal((n, 10))
    row = {"n": n, "delta": delta, "m": m, "pred_pattern_nnz": int(pt.entries.shape[0])}
    ctxs = {"tiled": cb.TaperedLikelihood(locs, X, z, sp)}
    if dense:
        ctxs["dense"] = cb.DenseLikelihood(locs, X, z)
        ctxs["dense"].set_taper(sp)
    try:
        for name, ctx in ctxs.items():
            s, _ = timed(lambda: ctx.factor_taper(tl, bench.LIMITS))
            row[name + "_factor_taper_s"] = s
            for fn in calls(ctx, lp, Xp, pt, resid, eps).values():
                fn()
        times = {name: {k: [] for k in calls(ctx, lp, Xp, pt, resid, eps)} for name, ctx in ctxs.items()}
        outs = {}
        for _ in range(reps):
            for name, ctx in ctxs.items():
                for k, fn in calls(ctx, lp, Xp, pt, resid, eps).items():
                    s, outs[(name, k)] = timed(fn)
                    times[name][k].append(s)
        for name in ctxs:
            row[name] = {k: float(np.median(v)) for k, v in times[name].items()}
            row[name]["all"] = times[name]
        row["tile_stats"] = ctxs["tiled"].tile_stats()
        if dense:
            ts, te = outs[("tiled", "predict_pred_s")]
            ds, de = outs[("dense", "predict_pred_s")]
            row["stochastic_abs_diff_over_max"] = float(np.max(np.abs(ts - ds)) / np.max(np.abs(ds)))
            row["explained_rel_diff"] = float(np.max(np.abs(te - de) / np.maximum(np.abs(de), 1e-300)))
            row["sim_abs_diff_over_max"] = float(np.max(np.abs(outs[("tiled", "sim_k10_s")] - outs[("dense", "sim_k10_s")]))
                                                 / np.max(np.abs(outs[("dense", "sim_k10_s")])))
    finally:
        for ctx in ctxs.values():
            ctx.close()
    flops, T, ms = explained_flops(sp, pt, morton(locs))
    dt = row["tiled"]["predict_pred_s"] - row["tiled"]["predict_mean_s"]
    row.update({"tile_columns": T, "sites_with_neighbours": ms, "explained_solve_flops": flops,
                "explained_fp64_tflops": flops / dt / 1e12 if dt > 0 else None})
    print(json.dumps({k: v for k, v in row.items() if k not in ("tiled", "dense")} | {
        "tiled": {k: v for k, v in row["tiled"].items() if k != "all"}}), flush=True)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--m", type=int, default=20000)
    ap.add_argument("--sizes", default="50000:0.25:dense,200000:0.05")
    a = ap.parse_args()
    rec = {"card": card(), "reps": a.reps, "runs": []}
    for spec in a.sizes.split(","):
        f = spec.split(":")
        rec["runs"].append(run(int(f[0]), float(f[1]), a.m, a.reps, len(f) > 2 and f[2] == "dense"))
    rec["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
