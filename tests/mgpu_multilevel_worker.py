"""Worker of the multi-GPU multilevel tests; launched with
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 tests/mgpu_multilevel_worker.py
Every rank runs PARSDMM_multi_level on z-slabs (3 levels, coarsening 2) twice: with the device warm start
(sipb_problem_warm_from gathers the coarse vectors across ranks) and with the host warm start (distributed.gather_td +
interpolate_y_l).  The two must agree bit for bit; rank 0 also runs the CPU oracle on the full problem and compares
per-level iteration counts, cg_it, x and the gathered y."""
import copy
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import problems as pr  # noqa: E402
import sip_b200 as sip  # noqa: E402
from sip_b200 import distributed as dd  # noqa: E402
from sip_b200 import multilevel as ml  # noqa: E402

TOL = {np.float32: 1e-3, np.float64: 1e-5}
CONFIG4_RHO = [1.0, 1000.0, 1000.0, 1000.0, 1.0]


def relerr(a, b):
    return float(np.linalg.norm(a.astype(np.float64) - b.astype(np.float64)) / max(np.linalg.norm(b.astype(np.float64)), 1e-300))


def reads_across_ranks(grids, world):
    """True when at some level transition a rank's fine z planes read a coarse plane that another rank owns."""
    for k in range(len(grids) - 1):
        nf, nc = int(grids[k].n[2]), int(grids[k + 1].n[2])
        src = ml._nearest_table(nc, nf)
        for r in range(world):
            f0, f1 = dd.slab_range(nf, r, world)
            c0, c1 = dd.slab_range(nc, r, world)
            if np.any((src[f0:f1] < c0) | (src[f0:f1] >= c1)):
                return True
    return False


def options(api, TF, kw):
    opt = api.PARSDMM_options()
    opt.FL = TF
    for k, v in kw.items():
        setattr(opt, k, copy.deepcopy(v))
    return opt


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("cpu:gloo,cuda:nccl")
    dd.init(rank, world, local)
    orc = pr.OracleAPI() if rank == 0 else None
    from oracle import multilevel as om
    f32 = dict(maxit=40, evol_rel_tol=10 * np.finfo(np.float32).eps)
    cases = [
        ("config4_f32", pr.spec_config4((20, 18, 27), np.float32), dict(f32, rho_ini=CONFIG4_RHO)),
        ("config2_f32", pr.spec_config2((24, 20, 27), np.float32), f32),
        ("config2_f64", pr.spec_config2((16, 12, 27), np.float64), dict(maxit=60)),
        ("config4_100", pr.spec_config4((100, 100, 100), np.float32), dict(f32, rho_ini=CONFIG4_RHO)),
    ]
    ok = True
    for name, spec, kw in cases:
        TF = spec["TF"]
        cg = sip.compgrid(tuple(spec["d"]), tuple(spec["n"]))
        cons = [sip.set_definitions(st, op, lo, hi, ("tensor", "")) for (st, op, lo, hi) in spec["sets"]]
        s_opt = options(sip, TF, kw)
        lv = sip.setup_multi_level_PARSDMM(spec["m"], 3, 2, cg, cons, s_opt)
        TD_fine, grids = lv[0][0], lv[4]
        rho0 = copy.deepcopy(s_opt.rho_ini)
        xs, ls, l2, y2 = sip.PARSDMM_multi_level(spec["m"].copy(), *lv[:5], s_opt)
        xh, lh, l3, y3 = sip.PARSDMM_multi_level(spec["m"].copy(), *lv[:5], s_opt, device_resample=False)
        assert [float(v) for v in s_opt.rho_ini] == [float(v) for v in rho0]
        yg, lg = [dd.gather_td(v, A) for v, A in zip(y2, TD_fine)], [dd.gather_td(v, A) for v, A in zip(l2, TD_fine)]
        yh, lhg = [dd.gather_td(v, A) for v, A in zip(y3, TD_fine)], [dd.gather_td(v, A) for v, A in zip(l3, TD_fine)]
        checks = {
            "reads_across_ranks": world == 1 or reads_across_ranks(grids, world),
            "dev_vs_host_x": bool(np.array_equal(xs, xh)),
            "dev_vs_host_iters": ls.timing["level_iterations"] == lh.timing["level_iterations"],
            "dev_vs_host_ly": all(np.array_equal(a, b) for a, b in zip(yg + lg, yh + lhg)),
        }
        if rank == 0:
            o_opt = options(orc, TF, kw)
            o_cg = orc.compgrid(tuple(spec["d"]), tuple(spec["n"]))
            o_cons = [orc.set_definitions(st, op, lo, hi, ("tensor", "")) for (st, op, lo, hi) in spec["sets"]]
            olv = om.setup_multi_level_PARSDMM(spec["m"], 3, 2, o_cg, o_cons, o_opt, orc.types)
            xo, lo, ll, yy = om.PARSDMM_multi_level(spec["m"].copy(), *olv[:5], o_opt)
            tol = TOL[TF]
            checks.update({
                "level_iters": [len(g.obj) for g in lo.levels] == ls.timing["level_iterations"],
                "cg_it": bool(np.array_equal(ls.cg_it, lo.cg_it)),
                "x": relerr(xs, xo) < tol,
                "y": all(relerr(a, b) < 100 * tol for a, b in zip(yg, yy)),
            })
            print("[mgpu-ml %d ranks] %-12s levels=%s oracle=%s relerr_x=%.2e transitions_s=%s" % (
                world, name, ls.timing["level_iterations"], [len(g.obj) for g in lo.levels], relerr(xs, xo),
                ["%.4f" % t for t in ls.timing["transition_seconds"]]), flush=True)
        good = all(checks.values())
        ok = ok and good
        print("[mgpu-ml %d ranks] rank %d %-12s %s %s" % (world, rank, name, "OK " if good else "FAIL",
                                                          "" if good else str({k: v for k, v in checks.items() if not v})),
              flush=True)
    flag = torch.tensor([1 if ok else 0], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    dist.destroy_process_group()
    sys.exit(0 if int(flag.item()) == 1 else 1)


if __name__ == "__main__":
    main()
