#!/usr/bin/env python
"""Multilevel PARSDMM (BASELINE config 4: 3-D bounds ∩ D_z / D_x / D_y bounds, 3 levels, coarsening 2, options of
tools/run_configs.py config 4) on N GPUs, one z-slab per rank.  Setup and one warm-up call are untimed; the best of
--reps calls through PARSDMM_multi_level is reported.  Rank 0 prints one JSON line: world, grid, per-level iterations
and device seconds (rank 0's), the host time of each level transition, wall seconds, final feasibility, and the GPU
name and power limit read in the same run.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N tools/bench_multilevel.py [--size 400] [--reps 3]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import problems as pr  # noqa: E402
import sip_b200 as sip  # noqa: E402
from sip_b200 import distributed as dd  # noqa: E402


def gpu_info(device):
    import torch
    name = torch.cuda.get_device_name(device)
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(device), "--query-gpu=power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "unknown"
    return name, out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--size", type=int, default=400, help="grid edge of the finest level (n x n x n)")
    ap.add_argument("--levels", type=int, default=3)
    ap.add_argument("--reps", type=int, default=3, help="timed calls; the best is reported")
    args = ap.parse_args()
    import torch
    import torch.distributed as dist
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("gloo")
        dd.init(rank, world, local)

    def barrier():
        if world > 1:
            dist.barrier()

    TF = np.float32
    n = (args.size,) * 3
    spec = pr.spec_config4(n, TF)
    cg = sip.compgrid(tuple(spec["d"]), tuple(spec["n"]))
    cons = [sip.set_definitions(st, op, lo, hi, ("tensor", "")) for (st, op, lo, hi) in spec["sets"]]
    opt = sip.PARSDMM_options()
    opt.FL = TF
    opt.evol_rel_tol = 10 * float(np.finfo(TF).eps)
    opt.rho_ini = [1.0, 1000.0, 1000.0, 1000.0, 1.0]
    t = time.perf_counter()
    lv = sip.setup_multi_level_PARSDMM(spec["m"], args.levels, 2, cg, cons, opt)
    t_setup = time.perf_counter() - t
    sip.PARSDMM_multi_level(spec["m"].copy(), *lv[:5], opt)          # warm-up: device problems built and uploaded
    best = None
    for _ in range(args.reps):
        m = spec["m"].copy()
        barrier()
        t = time.perf_counter()
        x, log, _, _ = sip.PARSDMM_multi_level(m, *lv[:5], opt)
        wall = time.perf_counter() - t
        if best is None or wall < best[0]:
            best = (wall, log)
    wall, log = best
    name, power = gpu_info(local)
    if rank == 0:
        sf = log.set_feasibility
        line = {"tool": "bench_multilevel", "config": "4: multilevel PARSDMM, 3-D bounds + D_z/D_x/D_y bounds",
                "world": world, "grid": list(n), "level_grids": [list(map(int, g.n)) for g in lv[4]][::-1],
                "dtype": np.dtype(TF).name, "reps": args.reps, "setup_s": t_setup, "wall_s": wall,
                "level_iterations": log.timing["level_iterations"],
                "level_device_s": [lt["device_seconds"] for lt in log.timing["levels"]],
                "level_solve_s": [lt["solve_seconds"] for lt in log.timing["levels"]],
                "transition_s": log.timing["transition_seconds"],
                "final_feasibility": [float(v) for v in sf[max(sf.shape[0] - 2, 0)]],
                "gpu": name, "power_limit": power}
        print(json.dumps(line), flush=True)
    barrier()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
