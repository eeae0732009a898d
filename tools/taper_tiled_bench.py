"""Tiled against dense tapered likelihood evaluations on one GPU, and the tiled context at a size whose dense matrix
does not fit (n = 200 000: 320 GB).  Bench sites (bench.synthetic), Wendland-1 taper of radius delta.

  python tools/taper_tiled_bench.py --out profiles/r03_taper_tiled.json [--reps 5]

n = 50 000, delta in {0.05, 0.11, 0.25}: one dense context (set_taper) and one tiled context on the same data, two
warm-up evaluations each, then `reps` evaluations of each, alternated; host clock around each call (the call ends
in a stream synchronise).  Reported: median, per-phase device times of the last evaluation, the tile statistics and
the update's FLOP rate (tile products x 2 x 128^3 over the event-timed factorisation, which also holds the POTRFs and
panel solves, so it is a lower bound of the update kernel's own rate).  n = 200 000, delta = 0.05: tiled only,
median time per evaluation and the device memory the context holds.  The card's name and power limit are read in
the same run."""
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


def device_used():
    import torch
    free, total = torch.cuda.mem_get_info()
    return total - free


def timed(ctx, tl):
    t0 = time.perf_counter()
    r = ctx.terms_taper(tl, bench.LIMITS, tl["mean"])
    return time.perf_counter() - t0, r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--skip-big", action="store_true")
    a = ap.parse_args()
    tl = dict(bench.THETA)
    rec = {"card": card(), "reps": a.reps, "n50k": [], "n200k": None}
    locs, X, z = bench.synthetic(50000)
    for delta in (0.05, 0.11, 0.25):
        sp = cb.cov_wend1(cb.nearest_dist(locs, delta=delta), (delta, 1))
        with cb.DenseLikelihood(locs, X, z) as d, cb.TaperedLikelihood(locs, X, z, sp) as t:
            d.set_taper(sp)
            for _ in range(2):
                timed(d, tl), timed(t, tl)
            td, tt = [], []
            for _ in range(a.reps):
                s, rd = timed(d, tl)
                td.append(s)
                s, rt = timed(t, tl)
                tt.append(s)
            st, ph = t.tile_stats(), t.timings()
            flops = st["tile_products"] * 2.0 * 128 ** 3
            row = {"delta": delta, "density": sp.entries.shape[0] / 50000 ** 2, "dense_s": float(np.median(td)),
                   "tiled_s": float(np.median(tt)), "tiled_over_dense": float(np.median(tt) / np.median(td)),
                   "tiled_phases_ms": ph, "dense_phases_ms": d.timings(), "tile_stats": st,
                   "stored_share_of_lower": st["stored_tiles"] / (st["tile_columns"] * (st["tile_columns"] + 1) / 2),
                   "update_tflops_lower_bound": flops / (ph["factor_ms"] * 1e-3) / 1e12,
                   "logdet_rel_diff": abs(rt["logdet"] - rd["logdet"]) / abs(rd["logdet"]),
                   "quad_rel_diff": float(abs(rt["quad"][0] - rd["quad"][0]) / abs(rd["quad"][0]))}
            print(json.dumps(row), flush=True)
            rec["n50k"].append(row)
    if not a.skip_big:
        locs, X, z = bench.synthetic(200000)
        sp = cb.cov_wend1(cb.nearest_dist(locs, delta=0.05), (0.05, 1))
        before = device_used()
        with cb.TaperedLikelihood(locs, X, z, sp) as t:
            held = device_used() - before
            timed(t, tl)
            ts = [timed(t, tl)[0] for _ in range(a.reps)]
            rec["n200k"] = {"delta": 0.05, "tiled_s": float(np.median(ts)), "all_s": ts, "context_bytes": held,
                            "tile_stats": t.tile_stats(), "phases_ms": t.timings()}
        print(json.dumps(rec["n200k"]), flush=True)
    rec["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
