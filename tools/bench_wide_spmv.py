#!/usr/bin/env python
"""Wide-Q SpMV + dot micro-benchmark (k_spmv_wide, the kernel of a Q with more than 32 diagonals) through
sipb_bench_spmv2 form 2: CDS arrays with the 125 diagonals of the A'A of a 3-D 27-point stencil, beyond L2
(256^3 Float32: about 8.4 GB of matrix per launch).  Prints one JSON line: CUDA-event ms per launch, algorithmic GB/s,
the fraction of the 6534 GB/s copy peak, and the GPU name and power limit read in the same run.
  python tools/bench_wide_spmv.py [--n 256] [--dtype f32] [--reps 20] [--warmup 3] [--flush 1]"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import sip_b200 as sip  # noqa: E402

COPY_PEAK_GBS = 6534.1      # measured device-to-device copy rate of one B200 (tools/bench_spmv.py uses the same figure)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        name, power = [v.strip() for v in out[0].split(",")]
        return name, power
    except Exception as e:          # the numbers are still reported; the record says what could not be read
        return "unknown (%s)" % type(e).__name__, "unknown"


ap = argparse.ArgumentParser()
ap.add_argument("--n", type=int, default=256)
ap.add_argument("--dtype", default="f32", choices=["f32", "f64"])
ap.add_argument("--reps", type=int, default=20)
ap.add_argument("--warmup", type=int, default=3)
ap.add_argument("--flush", type=int, default=1, help="overwrite a 256 MB buffer before every timed launch")
args = ap.parse_args()
L = sip._lib
ms, nb = C.c_double(0.0), C.c_int64(0)
n3 = (C.c_int64 * 3)(args.n, args.n, args.n)
L.check(L.load().sipb_bench_spmv2(L.ctx(), 0 if args.dtype == "f32" else 1, 3, n3, args.warmup, args.reps, args.flush,
                                  2, 0, C.byref(ms), C.byref(nb)))
gbs = nb.value / (ms.value * 1e-3) / 1e9
name, power = gpu_info()
print(json.dumps({"kernel": "k_spmv_wide<DOT>", "grid": args.n, "dtype": args.dtype, "diagonals": 125,
                  "l2_flush": bool(args.flush), "ms": round(ms.value, 4), "algorithmic_bytes": nb.value,
                  "GBps": round(gbs, 1), "frac_copy_peak": round(gbs / COPY_PEAK_GBS, 3), "gpu": name,
                  "power_limit": power}))
