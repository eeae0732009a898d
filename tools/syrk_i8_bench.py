"""Stand-alone timing of the K = 768 trailing update C (m x m) -= P P^T, DMMA against split-int8
(cocons_trailing_update, device-generated data), over a range of m; prints the card, its power limit and clocks.

  python tools/syrk_i8_bench.py [--sizes 4096 8192 ...] [--reps 5] [--out FILE]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from cocons_b200 import _lib  # noqa: E402

K, PAIRS = 768, 36  # panel width; slice products of 8 slices (weights 2..9)
INT8_DATASHEET_TOPS = 4500.0


def card():
    q = "name,power.limit,clocks.max.sm,clocks.sm"
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], text=True).strip()
    except (OSError, subprocess.CalledProcessError) as e:
        return "unknown (%s)" % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[4096, 8192, 16384, 32768, 49152])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    rows = []
    print("card:", card(), flush=True)
    for m in a.sizes:
        tiles = (m / 128) * (m / 128 + 1)  # 128 x 64 tiles of the lower triangle
        flops = tiles * 2 * 128 * 64 * K
        ms = {}
        for path in (0, 1, 0, 1):
            v = ctypes.c_double()
            _lib.check(_lib.lib().cocons_trailing_update(0, m, None, None, path, a.reps, ctypes.byref(v)))
            ms[path] = min(ms.get(path, 1e30), v.value)
        r = {"m": m, "dmma_ms": ms[0], "int8_ms": ms[1], "dmma_tflops": flops / ms[0] / 1e9,
             "int8_fp64_equiv_tflops": flops / ms[1] / 1e9, "int8_tops": PAIRS * flops / ms[1] / 1e9,
             "speedup": ms[0] / ms[1]}
        r["int8_share_of_datasheet"] = r["int8_tops"] / INT8_DATASHEET_TOPS
        rows.append(r)
        print(json.dumps(r), flush=True)
    print("card:", card(), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            json.dump({"card": card(), "rows": rows}, f, indent=1)


if __name__ == "__main__":
    main()
