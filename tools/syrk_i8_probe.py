"""Phase probe of the split-int8 trailing update (csrc/syrk_i8.cu): builds the library with -DCOCONS_I8_PROBE into a
temporary directory (the shipped build is not touched), runs the lower-triangle update of --rows rows (K = 768,
device-generated data) and prints where the cycles of a CTA go, summed over the launch and per tile, with the card,
its power limit and clocks.

  python tools/syrk_i8_probe.py [--rows 49152] [--reps 3] [-D COCONS_I8_CLUSTER_M=1 ...] [--csrc DIR] [--out FILE]

Counters (clock64, SM cycles), all from the update kernel:
  start_to_first_mma  per CTA: launch of the CTA to its first MMA (barrier set-up, TMEM allocation, first stage)
  mma_full_wait       the MMA-issuing thread waiting for a stage to arrive (the feed is the limit)
  producer_empty_wait the producer waiting for a stage to be freed (the tensor pipe is the limit)
  epilogue            per tile: the epilogue, from its accumulators being complete to its last store of C
  mma_tmem_wait       the MMA-issuing thread waiting for the epilogue to hand tensor memory back (epilogue exposed)
  stage_refill        per stage: the producer issuing a stage's copies to the stage's full barrier completing (the
                      refill latency; seen by an observer warp that only the probe build has)
"""
import argparse
import concurrent.futures
import ctypes
import glob
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
NAMES = ("start_to_first_mma", "mma_full_wait", "producer_empty_wait", "epilogue", "mma_tmem_wait", "cta_cycles",
         "tiles", "ctas", "stage_refill")
CHUNKS = 24  # stages per tile (K = 768 in chunks of 32)


def card():
    q = "name,power.limit,clocks.max.sm,clocks.sm"
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], text=True).strip()
    except (OSError, subprocess.CalledProcessError) as e:
        return "unknown (%s)" % e


def build(csrc, defines, out_dir):
    flags = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xcompiler", "-fPIC",
             "-DCOCONS_I8_PROBE"] + ["-D" + d for d in defines]
    srcs = sorted(glob.glob(os.path.join(csrc, "*.cu")))
    objs = [os.path.join(out_dir, os.path.basename(src)[:-3] + ".o") for src in srcs]
    with concurrent.futures.ThreadPoolExecutor(os.cpu_count() or 4) as ex:
        list(ex.map(lambda so: subprocess.check_call([NVCC] + flags + ["-c", so[0], "-o", so[1]]), zip(srcs, objs)))
    so = os.path.join(out_dir, "libcocons_probe.so")
    subprocess.check_call([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", so] + objs)
    return so


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=49152)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("-D", dest="defines", action="append", default=[], help="extra preprocessor definition")
    ap.add_argument("--csrc", default=os.path.join(ROOT, "cocons_b200", "csrc"))
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    with tempfile.TemporaryDirectory(prefix="syrk_i8_probe_") as tmp:
        L = ctypes.CDLL(build(a.csrc, a.defines, tmp))
    L.cocons_trailing_update.argtypes = [ctypes.c_int, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int,
                                         ctypes.c_int, ctypes.POINTER(ctypes.c_double)]
    L.cocons_last_error.restype = ctypes.c_char_p
    sums = (ctypes.c_ulonglong * len(NAMES))()
    before = card()
    ms = ctypes.c_double()
    if L.cocons_trailing_update(0, a.rows, None, None, 1, 1, ctypes.byref(ms)) != 0:  # warm-up
        sys.exit("trailing_update: %s" % L.cocons_last_error().decode())
    L.cocons_i8_probe_read(sums)  # zeroes the sums
    if L.cocons_trailing_update(0, a.rows, None, None, 1, a.reps, ctypes.byref(ms)) != 0:
        sys.exit("trailing_update: %s" % L.cocons_last_error().decode())
    if L.cocons_i8_probe_read(sums) != 0:
        sys.exit("could not read the probe counters")
    s = dict(zip(NAMES, (float(v) for v in sums)))
    tiles, ctas = s["tiles"], s["ctas"]
    per_tile = {k: s[k] / tiles for k in NAMES[:6]}
    r = {"rows": a.rows, "defines": a.defines, "ms_per_split_and_update": ms.value, "launches": a.reps + 1,
         "ctas_per_launch": ctas / (a.reps + 1), "tiles_per_launch": tiles / (a.reps + 1),
         "cycles_per_cta": {"start_to_first_mma": s["start_to_first_mma"] / ctas, "cta_cycles": s["cta_cycles"] / ctas},
         "cycles_per_tile": per_tile, "share_of_cta_cycles": {k: s[k] / s["cta_cycles"] for k in NAMES[:5]},
         "stage_refill_cycles": s["stage_refill"] / (tiles * CHUNKS),
         "card": before, "card_after": card()}
    print(json.dumps(r, indent=1), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(r, f, indent=1)


if __name__ == "__main__":
    main()
