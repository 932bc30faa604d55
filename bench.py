#!/usr/bin/env python
"""bench.py — PARSDMM iterations/s and time-to-tolerance on the 3-D intersection-projection workloads of BASELINE.json.

Default workload: BASELINE configs[2] — 3-D 512^3 Float32, bounds ∩ TV l1-ball ∩ cardinality of the discrete gradient
(k = 5 % of the rows) — the problem the north star scales over 1/2/4/8 B200, STRONG scaling at every N (the whole
problem fits one GPU).  A "step" is one complete PARSDMM projection (initial feasibility check, Q assembly, iterations
until the reference's stopping rules fire or maxit = 200 is reached — at 512^3 it is maxit, see config.stop).
value = PARSDMM iterations / second, plain, at every N.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload config3|config2] [--size n] [--impl reference]
                  [--dump-outputs DIR]

Device arm (default):
  value      problem and m resident in HBM, CUDA-event time of the K solves on the solver stream, max over ranks
  e2e        the same through the public API sip_b200.PARSDMM(m, ...) with pinned HOST buffers: H2D of m and D2H of
             x, l, y (the reference returns (x, log, l, y), PARSDMM.jl:257) and the log inside the timed region;
             e2e_x_only: the same call with return_ly=False
  roofline   the kernel class with the largest share of the solve (algorithmic bytes counted by the library at every
             launch / CUDA-event time from a profiled solve) against MEASURED_PEAKS.json, every streaming class and the
             whole solve beside it, and the CDS SpMV alone (BASELINE's second metric) in both matrix forms
  config2    BASELINE configs[1] (200^3 Float32, bounds ∩ anisotropic TV ∩ lateral slope bounds) on the same N GPUs:
             value, e2e and FULL-SIZE parity against the CPU oracle (x, iteration count, CG iteration counts)
  parity     configs[2] against the CPU oracle on a reduced grid (the oracle's sparse set-up of 512^3 alone takes
             minutes; tests/checks/parity_fullsize.py runs larger grids, logs under profiles/)
  cpu_baseline  N=1: the threaded C/OpenMP restatement of the reference algorithm on the box's host cores, bounded
             sample: the first iterations of a sub-volume of the same workload (see `sample`)
Reference arm (--impl reference): the CPU restatement alone (Julia is not installable here), same metric / config,
each step a bounded sample, extrapolated to the full grid by the plane ratio (stated in the line).

Multi-GPU (N>1, torchrun): one process per GPU, z-slabs; peer-memory CG collectives + NCCL (see DESIGN.md §6).

--dump-outputs DIR: after the timed legs, the return value (x, log, l, y) of the last step of the end-to-end leg
(device arm, one process; the resident leg computes the same projection but leaves x, l, y on the device) or of the
last CPU sample (reference arm) as DIR/<name>.npy, see output_arrays.  The inputs are seeded, so two builds run with
the same arguments can be compared output for output.

A run writes nothing into the tree (it may be read-only): the CPU baseline library is built in a temporary
directory when the tree holds none for this host, and no bytecode is cached.
"""
from __future__ import annotations

import argparse
import copy
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

F32_EPS = float(np.finfo(np.float32).eps)
WORKLOADS = {
    "config3": "3D %dx%dx%d Float32 bounds ∩ TV l1-ball ∩ cardinality of the discrete gradient, k = 5 %% of the rows (BASELINE configs[2])",
    "config2": "3D %dx%dx%d Float32 bounds ∩ anisotropic TV l1-ball ∩ D_x, D_y slope bounds (BASELINE configs[1], test_scaling_3D-style)",
}


def env_int(name, default):
    return int(os.environ.get(name, default))


def make_spec(workload, grid, TF=np.float32):
    import problems as pr
    return pr.spec_config3(tuple(grid), TF) if workload == "config3" else pr.spec_config2(tuple(grid), TF)


def tweak_options(o, maxit=200):
    o.evol_rel_tol = 10 * F32_EPS      # examples/test_scaling_3D.jl:25
    o.maxit = maxit
    return o


def relerr(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


DUMP_BYTES = 64 * 10 ** 6


def output_arrays(result):
    """{name: array} of one PARSDMM return value (x, log, l, y) for --dump-outputs: x, l_<i>, y_<i> and log_<field>
    for every array of the log (cg_it as float64; evol_x from iteration 2 on: iteration 1 starts from x = 0 with
    rhs = 0, so its entry is 0/0 = NaN by definition, as in the reference's log).  A vector larger than its share of
    DUMP_BYTES becomes a sample of its entries at seeded random positions, the same positions for the same arguments.
    Returns copies: the caller's buffers may be reused."""
    x, log, l, y = result
    out = {"log_" + k: np.asarray(v, dtype=np.float64 if v.dtype.kind in "biu" else v.dtype).copy()
           for k, v in vars(log).items() if isinstance(v, np.ndarray)}
    out["log_evol_x"] = out["log_evol_x"][1:]
    vecs = [("x", x)] + [("l_%d" % i, v) for i, v in enumerate(l or [])] + [("y_%d" % i, v) for i, v in enumerate(y or [])]
    room = DUMP_BYTES - sum(v.nbytes for v in out.values()) - 4096 * (len(out) + len(vecs))       # 4096: .npy header
    for seed, (name, v) in enumerate(vecs):
        v = np.asarray(v).ravel()
        keep = room // len(vecs) // v.itemsize
        out[name] = v[np.unique(np.random.default_rng(seed).integers(0, v.size, keep))] if v.size > keep else v.copy()
    return out


def write_outputs(path, arrays):
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.path = "/tmp/sipb_clocks_%d_%d.csv" % (os.getpid(), gpu_index)

    def start(self):
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=self.f,
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                t = [v.strip() for v in line.split(",")]
                if len(t) < 9:
                    continue
                try:
                    sm.append(float(t[1]))
                    mx.append(float(t[2]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), t[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.remove(self.path)
        except Exception:
            pass
        if sm:
            busy = [v for v in sm if v > 0.5 * max(sm)] or sm
            out["sm_mhz"] = float(np.median(busy))
            out["sm_max_mhz"] = float(max(mx))
        out["reasons"] = sorted(reasons)
        return out


# --------------------------------------------------------------------------------------------------
# CPU side (threaded C/OpenMP restatement of the reference algorithm, oracle/cpu_baseline.py)
# --------------------------------------------------------------------------------------------------
_CPU_CACHE = {}
_CPU_MODE = {"threaded": None}
CPU_IMPL = ("threaded C/OpenMP restatement of the reference's vector phases (oracle/c/ref_kernels.c: per-diagonal CDS "
            "passes, BLAS-1 style CG passes, sort-based l1 projection; gcc -O3%s) driven by the NumPy oracle's control flow")


def cpu_threaded_available():
    """The C/OpenMP baseline needs gcc (or a prebuilt oracle/_cbuild/libsipref*.so); without it the CPU legs fall back
    to the plain NumPy oracle and say so."""
    if _CPU_MODE["threaded"] is None:
        try:
            from oracle import cpu_baseline as cb
            cb.use_all_cores()           # torchrun exports OMP_NUM_THREADS=1; the baseline gets every host core
            _CPU_MODE["threaded"] = True
        except Exception as e:       # noqa: BLE001
            print("bench.py: threaded CPU baseline unavailable (%s); timing the NumPy oracle instead" % e, file=sys.stderr)
            _CPU_MODE["threaded"] = False
    return _CPU_MODE["threaded"]


def cpu_threads():
    if not cpu_threaded_available():
        return 1
    from oracle import cpu_baseline as cb
    return cb.threads()


def cpu_impl():
    if not cpu_threaded_available():
        return "NumPy/SciPy oracle (single-threaded apart from BLAS dot/norm)"
    from oracle import build_c
    native = build_c.is_native(build_c.runtime_library())
    return CPU_IMPL % (" -march=native, built on this box" if native else ", portable build (no gcc on this box)")


def cpu_solve(workload, grid, maxit, max_iterations=None, threads=None):
    """One CPU PARSDMM run of `workload` on `grid`.  Returns ((x, log, l, y), seconds of the iteration phases, seconds
    of set-up + PARSDMM_initialize).  The operator set-up is cached between calls (it is outside the PARSDMM call in the
    reference too)."""
    import problems as pr
    orc = pr.OracleAPI()
    t0 = time.perf_counter()
    key = (workload, tuple(grid))
    if key not in _CPU_CACHE:
        spec = make_spec(workload, grid)
        _CPU_CACHE[key] = (spec, pr.build(orc, spec, orc.PARSDMM_options()))
    spec, ob = _CPU_CACHE[key]
    opt = copy.deepcopy(ob["opt"])
    tweak_options(opt, maxit)
    t_setup = time.perf_counter() - t0
    if cpu_threaded_available():
        from oracle import cpu_baseline as cb
        if threads is None:
            cb.use_all_cores()
        else:
            cb.lib().sipref_set_threads(int(threads))
        res = cb.PARSDMM(spec["m"].copy(), ob["AtA"], ob["TD_OP"], ob["set_Prop"], ob["P_sub"], ob["cg"], opt,
                         constraint=ob["cons"], max_iterations=max_iterations)
        if threads is not None:
            cb.use_all_cores()
    else:
        if max_iterations:
            opt.maxit = min(opt.maxit, int(max_iterations))
        res = orc.PARSDMM(spec["m"].copy(), ob["AtA"], ob["TD_OP"], ob["set_Prop"], ob["P_sub"], ob["cg"], opt)
    log = res[1]
    t_iter = sum(v for k, v in log.timing.items() if k != "initialization")
    return res, t_iter, t_setup + log.timing.get("initialization", 0.0)


def cpu_sample_main(args):
    """Bounded CPU sample of the main workload: the first `--cpu-iters` PARSDMM iterations of a sub-volume of the grid
    (the first n/f planes), all host cores.  The rate of the FULL grid is extrapolated by the plane ratio f: every
    vector phase of the algorithm is linear in the number of grid points."""
    n = args.n
    f = max(1, args.cpu_sub)
    sub = (n, n, max(n // f, 8))
    f_eff = n / sub[2]
    iters = args.cpu_iters
    res, t_iter, t_setup = cpu_solve(args.workload, sub, 200, max_iterations=iters)
    done = len(res[1].obj)
    rate_sub = done / t_iter
    return {"value": rate_sub / f_eff, "measured_on_sample": rate_sub, "iterations": done, "t_iter": t_iter, "t_setup": t_setup,
            "sample_grid": list(sub), "factor": f_eff, "result": res}


def run_reference(args, rank, world):
    """Reference arm: the reference's CPU algorithm (C/OpenMP + NumPy port of the oracle — Julia cannot be installed here)
    on the host cores.  Every step is a bounded sample (see cpu_sample_main)."""
    if rank != 0:
        return
    n = args.n
    cores = cpu_threads()
    vals, secs = [], []
    t_start = time.perf_counter()
    budget_s = float(os.environ.get("SIPB_REFERENCE_BUDGET_S", "200"))      # keep the whole arm within a few minutes
    warm = min(args.warmup, 1)       # one warm-up builds and caches the operators (outside PARSDMM in the reference too)
    last = None
    for s in range(warm + args.steps):
        last = cpu_sample_main(args)
        if s >= warm:
            vals.append(last["value"])
            secs.append(last["t_iter"])
        if time.perf_counter() - t_start > budget_s and len(vals) >= 1:
            break
    value = float(len(vals) / sum(1.0 / v for v in vals))       # total iterations / total (extrapolated) time
    sample = ("first %d PARSDMM iterations of the %dx%dx%d sub-volume (1/%.0f of the planes) of the workload per step, %.2f s "
              "each; full-grid rate = measured / %.0f (all vector phases are linear in the grid points) — EXTRAPOLATED; %s; "
              "the rate counts the iteration phases only: operator set-up and PARSDMM_initialize are excluded, which "
              "favours the CPU" % (last["iterations"], *last["sample_grid"], last["factor"], float(np.mean(secs)), last["factor"],
                                   cpu_impl()))
    line = {
        "impl": "reference", "metric": "parsdmm_iterations_per_second", "value": value, "unit": "iterations/s",
        "n_gpus": args.gpus, "steps": len(vals), "warmup": warm, "steps_requested": args.steps,
        "ms_per_step": 1e3 * float(np.mean(secs)),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOADS[args.workload] % (n, n, n), "grid": [n, n, n],
                   "ran_on_grid": last["sample_grid"], "extrapolated": True, "extrapolation_factor": last["factor"],
                   "warmup_note": "one warm-up instead of %d: it only builds and caches the operators, which the reference does "
                                  "outside PARSDMM as well; the CPU has no clocks / caches to warm beyond that" % args.warmup,
                   "note": "CPU restatement of the reference algorithm on %d OpenMP threads; the Julia reference cannot "
                           "be installed in this image (no Julia, no network)" % cores},
        "cpu_baseline": {"value": value, "unit": "iterations/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if args.dump_outputs:
        write_outputs(args.dump_outputs, output_arrays(last["result"]))
    print(json.dumps(line))


# --------------------------------------------------------------------------------------------------
# device arm
# --------------------------------------------------------------------------------------------------
class DeviceProblem:
    """One workload built through the public host API (setup_constraints -> PARSDMM_precompute_distribute) with pinned
    host buffers for the end-to-end calls."""

    def __init__(self, sip, workload, grid, maxit=200):
        import problems as pr
        import torch
        self.sip, self.grid = sip, tuple(grid)
        t0 = time.perf_counter()
        self.spec = make_spec(workload, grid)              # synthetic model + the size of its l1 ball: bench input, not product
        self.input_s = time.perf_counter() - t0
        t0 = time.perf_counter()
        self.sb = pr.build(sip, self.spec, tweak_options(sip.PARSDMM_options(), maxit))     # setup_constraints + precompute
        self.m = self.spec["m"]
        self.setup_s = time.perf_counter() - t0
        t0 = time.perf_counter()
        self.x0, self.log0 = self.solve()[:2]             # first call uploads the operator tables ("distribute")
        self.first_call_s = time.perf_counter() - t0
        dev = self.sb["AtA"]._device
        self.dev = dev
        slab = getattr(dev, "slab", None)
        plane = grid[0] * grid[1]
        m_loc = self.m if slab is None else self.m[plane * slab[0]: plane * slab[1]]
        pin = lambda k: torch.empty(int(k), dtype=torch.float32).pin_memory().numpy()       # noqa: E731
        self.m_pin = pin(m_loc.size)
        self.m_pin[:] = m_loc
        self.x_pin = pin(dev.N)
        self.l_pin = [pin(r) for r in dev.rows]
        self.y_pin = [pin(r) for r in dev.rows]

    def solve(self, **kw):
        sb = self.sb
        kw.setdefault("return_ly", False)
        kw.setdefault("gather_result", False)
        return self.sip.PARSDMM(self.m, sb["AtA"], sb["TD_OP"], sb["set_Prop"], sb["P_sub"], sb["cg"], sb["opt"], **kw)

    def solve_e2e(self, return_ly):
        sb = self.sb
        if return_ly:      # zero_ini_guess: l, y are outputs only (PARSDMM.jl:257 returns them)
            return self.sip.PARSDMM(self.m_pin, sb["AtA"], sb["TD_OP"], sb["set_Prop"], sb["P_sub"], sb["cg"], sb["opt"],
                                    x=self.x_pin, l=self.l_pin, y=self.y_pin, return_ly=True, gather_result=False)
        return self.sip.PARSDMM(self.m_pin, sb["AtA"], sb["TD_OP"], sb["set_Prop"], sb["P_sub"], sb["cg"], sb["opt"],
                                x=self.x_pin, return_ly=False, gather_result=False)


def timed(fn, steps, barrier):
    """K calls of fn bracketed by barrier + synchronize; returns (wall s, summed device s, iterations, launches, h2d, d2h,
    return value of the last call)."""
    barrier()
    t0 = time.perf_counter()
    dev_s, its, launches, h2d, d2h = 0.0, 0, 0, 0, 0
    res = None
    for _ in range(steps):
        res = fn()
        lg = res[1]
        dev_s += lg.timing["device_seconds"]
        its += len(lg.obj)
        launches += lg.timing["total_launches"]
        h2d += lg.timing["h2d_bytes"]
        d2h += lg.timing["d2h_bytes"]
    barrier()
    return time.perf_counter() - t0, dev_s, its, launches, h2d, d2h, res


def run_device(args, rank, world, local_rank):
    import torch
    import sip_b200 as sip

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("cpu:gloo,cuda:nccl", device_id=torch.device("cuda", local_rank))
        from sip_b200 import distributed as dd
        dd.init(rank, world, local_rank)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(vals):
        t = torch.tensor(vals, dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t.tolist()]

    def gather_x(prob, x_local):
        if dist is None:
            return x_local
        from sip_b200 import distributed as dd
        return dd.gather_model(np.asarray(x_local))

    n = args.n
    grid = (n, n, n)
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, which = float(json.load(open(peaks_path))["hbm_gbs"]), "measured"
    else:
        peak, which = 6650.0, "fallback"

    # ---- main workload ---------------------------------------------------------------------------------------
    t_wall0 = time.perf_counter()
    prob = DeviceProblem(sip, args.workload, grid)
    iters_per_step = len(prob.log0.obj)
    for _ in range(max(args.warmup - 1, 0)):
        prob.solve(resident_io=True)
    sampler = ClockSampler(local_rank)
    sampler.start()
    try:
        wall_res, dev_s, its, launches, _, _, _ = timed(lambda: prob.solve(resident_io=True), args.steps, barrier)
        # end to end through the public API, pinned host buffers; the reference's return tuple includes l and y
        e_steps = args.steps if args.e2e_steps <= 0 else min(args.steps, args.e2e_steps)
        prob.solve_e2e(True)
        wall_e2e, _, e2e_its, _, h2d, d2h, e2e_last = timed(lambda: prob.solve_e2e(True), e_steps, barrier)
        dump = output_arrays(e2e_last) if args.dump_outputs else None       # before the next leg reuses x's buffer
        prob.solve_e2e(False)
        wall_x, _, x_its, _, h2d_x, d2h_x, _ = timed(lambda: prob.solve_e2e(False), e_steps, barrier)
    finally:
        clocks = sampler.stop()
    dev_s_max, wall_e2e_max, wall_x_max, wall_res_max = reduce_max([dev_s, wall_e2e, wall_x, wall_res])

    # ---- roofline of the dominant kernel class from one profiled solve (CUDA events around every launch) -------
    _, lgp, _, _ = prob.solve(resident_io=True, profile_kernels=True)      # every rank: the solve contains collectives
    roof, kernels = None, {}
    if rank == 0:
        kernels = lgp.timing["kernels"]
        kbytes = lgp.timing["kernel_bytes"]         # algorithmic bytes per class, counted by the library at launch
        tot_ms = sum(v[1] for v in kernels.values())
        streaming = {k: v for k, v in kernels.items() if kbytes.get(k) and v[1] > 0}
        if streaming:
            top = max(streaming, key=lambda k: streaming[k][1])       # the class with the largest share of the solve
            cnt_k, ms_k = streaming[top]
            alg = kbytes[top] / cnt_k
            avg_ms = ms_k / cnt_k
            ach = alg / (avg_ms * 1e-3) / 1e9
            traffic = None       # dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu capture
            tpath = os.path.join(ROOT, "profiles", "r02_kernel_traffic.json")
            if os.path.exists(tpath) and world == 1:
                tj = json.load(open(tpath))
                if tj.get("workload") == args.workload and tj.get("grid") == list(grid) and top in tj.get("kernels", {}):
                    traffic = tj["kernels"][top]["dram_bytes_per_launch"]
            roof = {"bound": "hbm", "kernel": top, "achieved": ach, "peak": peak, "peak_source": which,
                    "unit": "GB/s", "frac": ach / peak, "traffic": traffic, "algorithmic_bytes_per_launch": alg,
                    "avg_launch_ms": avg_ms, "launches": cnt_k, "share_of_kernel_time": ms_k / tot_ms if tot_ms else None,
                    "q_form": prob.dev.q_form,
                    "per_kernel": {k: {"launches": v[0], "ms": round(v[1], 3), "gbs": round(kbytes[k] / (v[1] * 1e-3) / 1e9, 1),
                                       "frac": round(kbytes[k] / (v[1] * 1e-3) / 1e9 / peak, 3)} for k, v in streaming.items()},
                    "whole_solve": {"algorithmic_gb": round(sum(kbytes.values()) / 1e9, 3), "kernel_ms": round(tot_ms, 3),
                                    "gbs": round(sum(kbytes.values()) / (tot_ms * 1e-3) / 1e9, 1),
                                    "frac": round(sum(kbytes.values()) / (tot_ms * 1e-3) / 1e9 / peak, 3)}}
    # BASELINE's second metric, "CDS-SpMV HBM GB/s": the SpMV + dot kernel of cg.jl on this grid, timed alone back to
    # back (sipb_bench_spmv2, CUDA events): stencil-class form (what the solve runs: tiled TMA-staged kernel, 2*N*s
    # algorithmic bytes) and CDS arrays (the reference's storage: generic streaming kernel, (nd+2)*N*s)
    if rank == 0 and world == 1 and roof is not None:
        import ctypes as C
        L = sip._lib
        spm = {}
        for name, form, tiled in (("classes_tiled", 1, 1), ("arrays", 0, 0)):
            try:
                ms_, nb_ = C.c_double(0.0), C.c_int64(0)
                L.check(L.load().sipb_bench_spmv2(L.ctx(), 0, 3, (C.c_int64 * 3)(*grid), 3, 20, 0, form, tiled, C.byref(ms_),
                                                  C.byref(nb_)))
                gbs = nb_.value / (ms_.value * 1e-3) / 1e9
                spm[name] = {"avg_launch_ms": ms_.value, "algorithmic_bytes_per_launch": nb_.value, "gbs": gbs,
                             "frac": gbs / peak, "launches": 20}
            except Exception as e:       # noqa: BLE001 - an auxiliary figure must never take the bench line down
                print("bench.py: CDS SpMV unit timing (%s) skipped (%s)" % (name, e), file=sys.stderr)
        roof["cds_spmv"] = spm

    # ---- parity of the main workload on a reduced grid (every N) ----------------------------------------------
    parity = {}
    pg = (args.parity_size,) * 3
    if args.parity_size > 0 and pg[2] >= 2 * world:
        try:
            pmaxit = args.parity_iters
            pp_ = DeviceProblem(sip, args.workload, pg, maxit=pmaxit)
            xs, ls, _, _ = pp_.solve()
            xg = gather_x(pp_, xs)
            if rank == 0:
                (xo, lo, _, _), _, _ = cpu_solve(args.workload, pg, pmaxit)
                parity[args.workload + "_reduced"] = {
                    "grid": list(pg), "maxit": pmaxit, "rel_l2": relerr(xg, xo), "iters_equal": len(ls.obj) == len(lo.obj),
                    "cg_it_equal": bool(np.array_equal(ls.cg_it, lo.cg_it)), "iterations": len(ls.obj),
                    "note": "same workload and options on a reduced grid against the CPU oracle (the oracle's sparse set-up "
                            "of the full grid takes minutes; profiles/ holds full-size runs of tests/checks/parity_fullsize.py)"}
            del pp_
        except Exception as e:       # noqa: BLE001
            parity[args.workload + "_reduced"] = {"error": str(e)[:300]}

    # ---- BASELINE configs[1] (200^3) on the same GPUs: value, e2e, full-size parity ---------------------------
    c2 = None
    if args.workload != "config2" and not args.no_config2:
        try:
            g2 = (200, 200, 200)
            p2 = DeviceProblem(sip, "config2", g2)
            for _ in range(2):
                p2.solve(resident_io=True)
            w2, d2, it2, la2, _, _, _ = timed(lambda: p2.solve(resident_io=True), args.steps, barrier)
            p2.solve_e2e(True)
            we2, _, ite2, _, h2, dd2, _ = timed(lambda: p2.solve_e2e(True), args.steps, barrier)
            d2m, we2m = reduce_max([d2, we2])
            xs, ls, _, _ = p2.solve()
            xg = gather_x(p2, xs)
            if rank == 0:
                k2 = args.steps
                c2 = {"workload": WORKLOADS["config2"] % g2, "grid": list(g2), "steps": k2, "value": it2 / d2m,
                      "unit": "iterations/s", "ms_per_step": 1e3 * d2m / k2, "parsdmm_iterations_per_step": len(ls.obj),
                      "e2e": {"value": ite2 / we2m, "unit": "iterations/s", "ms_per_step": 1e3 * we2m / k2,
                              "h2d_bytes_per_step": h2 // k2, "d2h_bytes_per_step": dd2 // k2, "returns": "x, l, y, log"},
                      "gpu_launches_per_step": la2 // k2}
                if not args.no_cpu:
                    (xo, lo, _, _), t_iter, t_setup = cpu_solve("config2", g2, 200)
                    c2["parity"] = {"grid": list(g2), "rel_l2": relerr(xg, xo), "iters_equal": len(ls.obj) == len(lo.obj),
                                    "cg_it_equal": bool(np.array_equal(ls.cg_it, lo.cg_it)), "iterations": len(ls.obj),
                                    "oracle_iterations": len(lo.obj)}
                    c2["cpu_baseline"] = {"value": len(lo.obj) / t_iter, "unit": "iterations/s", "cores": cpu_threads(), "kind": "port",
                                          "sample": "one full projection of the same 200^3 workload (%d iterations, %.1f s of iteration "
                                                    "phases; %.1f s of set-up and initialization excluded); %s"
                                                    % (len(lo.obj), t_iter, t_setup, cpu_impl())}
                    if world == 1 and cpu_threaded_available():
                        (_, l4, _, _), t4, _ = cpu_solve("config2", g2, 200, max_iterations=8, threads=4)
                        c2["cpu_baseline"]["threads4"] = {"value": len(l4.obj) / t4, "unit": "iterations/s", "cores": 4,
                                                          "sample": "first %d iterations (JULIA_NUM_THREADS=4 of "
                                                                    "examples/test_scaling_3D.jl:3-4)" % len(l4.obj)}
            del p2
        except Exception as e:       # noqa: BLE001
            c2 = {"error": str(e)[:300]}

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    cpu = None
    if world == 1 and not args.no_cpu:
        try:
            s = cpu_sample_main(args)
            cpu = {"value": s["value"], "unit": "iterations/s", "cores": cpu_threads(), "kind": "port",
                   "measured_on_sample": s["measured_on_sample"], "extrapolation_factor": s["factor"],
                   "sample": "first %d PARSDMM iterations of the %dx%dx%d sub-volume (1/%.0f of the planes) of the same workload "
                             "(%.1f s of iteration phases; %.1f s of set-up and initialization excluded); full-grid rate = "
                             "measured / %.0f, EXTRAPOLATED (every vector phase is linear in the grid points); %s"
                             % (s["iterations"], *s["sample_grid"], s["factor"], s["t_iter"], s["t_setup"], s["factor"], cpu_impl())}
        except Exception as e:       # noqa: BLE001
            cpu = {"error": str(e)[:300]}

    value = its / dev_s_max
    maxit_bound = iters_per_step >= 200
    if world > 1:
        from sip_b200 import distributed as dd
        par = ("z-slabs over %d GPUs (%s), strong scaling" % (
            world, "peer-memory CG reductions + neighbour-plane bulk loads over NVLink (CUDA IPC), NCCL for the "
            "per-iteration halos / batched all-reduce" if dd.peer_path() else "NCCL send/recv halo planes + Float64 all-reduce"))
    else:
        par = "single GPU"
    line = {
        "metric": "parsdmm_iterations_per_second", "value": value, "unit": "iterations/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dev_s_max / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOADS[args.workload] % grid, "grid": list(grid),
                   "value_units": "PARSDMM iterations/s of the whole %dx%dx%d problem" % grid,
                   "step": "one full PARSDMM projection to the reference's stopping rules",
                   "parsdmm_iterations_per_step": iters_per_step, "time_to_tolerance_ms": 1e3 * dev_s_max / args.steps,
                   "stop": ("maxit = 200 reached before any stopping rule fired: time_to_tolerance_ms is time-to-maxit"
                            if maxit_bound else "the reference's stopping rules fired at iteration %d" % iters_per_step),
                   "cache": "working set %.1f GB per GPU >> 126 MB L2, no flush needed" % (prob.dev.N * 4 * 45 / 1e9),
                   "setup_seconds": {"synthetic_input": round(prob.input_s, 3), "host_setup_precompute": round(prob.setup_s, 3),
                                     "first_call_incl_upload": round(prob.first_call_s, 3)},
                   "parallelism": par},
        "e2e": {"value": e2e_its / wall_e2e_max, "unit": "iterations/s", "h2d_bytes_per_step": h2d // e_steps,
                "d2h_bytes_per_step": d2h // e_steps, "ms_per_step": 1e3 * wall_e2e_max / e_steps, "steps": e_steps,
                "returns": "x, l, y, log (the reference's return tuple, PARSDMM.jl:257) into pinned host buffers"},
        "e2e_x_only": {"value": x_its / wall_x_max, "unit": "iterations/s", "h2d_bytes_per_step": h2d_x // e_steps,
                       "d2h_bytes_per_step": d2h_x // e_steps, "ms_per_step": 1e3 * wall_x_max / e_steps, "steps": e_steps},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": roof,
        "parity": parity,
        "cpu_baseline": cpu,
        "config2": c2,
        "phase_ms_per_step": {k: round(1e3 * v, 3) for k, v in lgp.timing.items()
                              if k in sip._lib.PHASE_NAMES} if hasattr(sip, "_lib") else None,
        "kernel_table_ms": {k: [v[0], round(v[1], 3)] for k, v in kernels.items()},
        "resident_wall_ms_per_step": 1e3 * wall_res_max / args.steps,
        "bench_wall_s": round(time.perf_counter() - t_wall0, 1),
    }
    if dump is not None:
        write_outputs(args.dump_outputs, dump)
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="device", choices=["device", "reference"])
    ap.add_argument("--workload", default="config3", choices=["config3", "config2"],
                    help="config3 = BASELINE configs[2] (512^3, the north star's scaling problem; default); config2 = configs[1]")
    ap.add_argument("--size", "--n", dest="n", type=int, default=0,
                    help="grid width (default: 512 for config3, 200 for config2); use --size under torchrun (its parser claims --n)")
    ap.add_argument("--e2e-steps", type=int, default=3,
                    help="steps of the two end-to-end legs (each step is a full projection; 0 = as many as --steps)")
    ap.add_argument("--cpu-iters", type=int, default=3, help="PARSDMM iterations in the bounded CPU sample of the main workload")
    ap.add_argument("--cpu-sub", type=int, default=16, help="the CPU sample runs the first n/cpu_sub planes of the grid")
    ap.add_argument("--parity-size", type=int, default=96, help="grid width of the reduced-grid parity check (0 = skip)")
    ap.add_argument("--parity-iters", type=int, default=25, help="maxit of the reduced-grid parity check")
    ap.add_argument("--no-cpu", action="store_true", help="skip every CPU leg (cpu_baseline, oracle parity)")
    ap.add_argument("--no-config2", action="store_true", help="skip the configs[1] block")
    ap.add_argument("--scaling", default="strong", choices=["strong"], help="N>1 keeps the grid fixed")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the outputs of the last timed step as DIR/<name>.npy (at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.n <= 0:
        args.n = 512 if args.workload == "config3" else 200
    if args.no_cpu:
        args.parity_size = 0
    rank, world, local_rank = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if args.dump_outputs and args.impl == "device" and world > 1:
        ap.error("--dump-outputs needs a single process on the device arm (x, l and y stay in per-rank slabs)")
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_device(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
