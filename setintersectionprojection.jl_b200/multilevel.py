"""Coarse-to-fine multilevel PARSDMM — host driver over device solves.

Mirrors PARSDMM_multi_level.jl:8-89, setup_multi_level_PARSDMM.jl:7-137, constraint2coarse.jl:8-104 and
interpolate_y_l.jl:7-97.  Every level is one `PARSDMM` device solve (warm-started with x, l, y from the
coarser level); the nearest-neighbour resampling between levels is index work on the host arrays that the
reference API hands back between solves (separable `take` per axis).

Resampling rule: the reference evaluates `interpolate(A, BSpline(Constant()))` (Interpolations.jl 0.13) at
`range(1, stop=n_src, length=n_dst)`; that is nearest-neighbour with half-way positions rounded up.  The
index tables are built in exact integer arithmetic.
"""
from __future__ import annotations

import copy
import time

import numpy as np

from . import _lib
from . import distributed as dd
from .constraints import setup_constraints
from .precompute import PARSDMM_precompute_distribute
from .solver import PARSDMM, device_problem
from .types import compgrid


def _nearest_table(n_src: int, n_dst: int) -> np.ndarray:
    """Source index (0-based) of sample k of range(1, stop=n_src, length=n_dst): floor(pos + 1/2) - 1 with
    pos = 1 + k (n_src-1)/(n_dst-1), evaluated over the common denominator 2 (n_dst-1)."""
    if n_dst <= 1:
        return np.zeros(max(n_dst, 0), dtype=np.intp)
    k = np.arange(n_dst, dtype=np.int64)
    return ((3 * (n_dst - 1) + 2 * k * (n_src - 1)) // (2 * (n_dst - 1)) - 1).astype(np.intp)


def resample_nn(v: np.ndarray, shape_src, shape_dst) -> np.ndarray:
    """Nearest-neighbour resampling of vec(A) (column-major) from shape_src to shape_dst."""
    src = tuple(int(s) for s in shape_src)
    dst = tuple(int(s) for s in shape_dst)
    # the column-major box seen as a C-ordered array with the axes reversed: every `take` then copies contiguous runs
    # (slowest axis first, the gather along the fastest axis last, on the already reduced array) — 5-10x faster at 400^3
    # than taking along the axes of the Fortran-ordered view, same elements
    A = np.reshape(np.ascontiguousarray(v), src[::-1])
    for axis, (ns, nd) in enumerate(zip(src[::-1], dst[::-1])):
        A = np.take(A, _nearest_table(ns, nd), axis=axis)
    return np.ascontiguousarray(A.ravel())


def constraint2coarse(constraint, comp_grid, coarsening_factor):
    """constraint2coarse.jl:8-104: adapt constraint sizes to a coarser grid (in place)."""
    n = tuple(comp_grid.n)
    dim3 = len(n) == 3 and n[2] > 1
    for c in constraint:
        if c.set_type == "rank":
            c.max = min(c.max, min(n))                                   # :15-19
        elif c.set_type == "cardinality":
            c.max = min(c.max, int(np.prod(n)))                          # :22-26
        elif c.set_type == "l1":
            c.max = c.max / (coarsening_factor ** (3 if dim3 else 2))    # :47-51 / :73-77
        elif c.set_type == "l2":
            c.max = c.max / (np.sqrt(coarsening_factor ** 3) if dim3 else coarsening_factor)   # :54-58 / :80-84
        elif c.set_type == "nuclear" and not dim3:
            c.max = c.max / 2.7                                          # :87-91
    return constraint


def setup_multi_level_PARSDMM(m, n_levels, coarsening_factor, comp_grid, constraint, options):
    """-> (TD_OP_levels, AtA_levels, P_sub_levels, set_Prop_levels, comp_grid_levels, constraint_level)
    (setup_multi_level_PARSDMM.jl:7-14,135)."""
    TF = m.dtype.type
    grids = [comp_grid]
    for lev in range(1, n_levels):
        n = tuple(int(np.round(v / coarsening_factor ** lev)) for v in comp_grid.n)           # :66
        d = tuple((vn / nn) * vd for vn, nn, vd in zip(comp_grid.n, n, comp_grid.d))          # :82
        grids.append(compgrid(d, n))
    if dd.active() and len(comp_grid.n) == 3:
        for lev, grid in enumerate(grids):
            if int(grid.n[2]) < dd.world():
                raise ValueError("level %d (grid %s) has %d z planes, fewer than the %d ranks of the slab decomposition; "
                                 "use fewer levels or fewer ranks" % (lev, tuple(int(v) for v in grid.n), int(grid.n[2]),
                                                                      dd.world()))
    out = ([], [], [], [], [])
    level_constraint = None
    for lev, grid in enumerate(grids):
        if lev == 0:
            cons = constraint
        else:
            if level_constraint is None:
                level_constraint = copy.deepcopy(constraint)             # :61 (after the fine-level TF cast)
            cons = level_constraint = constraint2coarse(level_constraint, grid, coarsening_factor)   # :87
        P_sub, TD_OP, set_Prop = setup_constraints(cons, grid, TF)
        TD_OP, AtA, _, _ = PARSDMM_precompute_distribute(TD_OP, set_Prop, grid, options)
        for lst, item in zip(out, (TD_OP, AtA, P_sub, set_Prop, grid)):
            lst.append(item)
    if level_constraint is None:
        level_constraint = copy.deepcopy(constraint)
    return (*out, level_constraint)


def interpolate_y_l(l, y, set_Prop_levels, comp_grid_levels, dim3, i):
    """interpolate_y_l.jl:7-97: bring l and y from level i+1 (coarser) to level i (finer); `i` is 0-based.
    TV vectors are cut into blocks shaped (n1-1,n2,n3),(n1,n2-1,n3),(n1,n2,n3-1) in that order — the
    reference's heuristic (the operator rows are ordered D_z, D_y, D_x), reproduced as is."""
    coarse, fine = tuple(comp_grid_levels[i + 1].n), tuple(comp_grid_levels[i].n)
    nax = 3 if dim3 else 2

    def minus_one(n, axis):
        return tuple(v - 1 if a == axis else v for a, v in enumerate(n[:nax]))

    for j in range(len(l)):
        if set_Prop_levels[i].tag[j][1] in ("TV", "D2D", "D3D"):
            parts_l, parts_y, start = [], [], 0
            for axis in range(nax):
                sc, sf = minus_one(coarse, axis), minus_one(fine, axis)
                stop = l[j].size if axis == nax - 1 else start + int(np.prod(sc))
                parts_l.append(resample_nn(l[j][start:stop], sc, sf))
                parts_y.append(resample_nn(y[j][start:stop], sc, sf))
                start = stop
            l[j], y[j] = np.concatenate(parts_l), np.concatenate(parts_y)
        else:
            src = tuple(set_Prop_levels[i + 1].TD_n[j])
            shrink = tuple(a - b for a, b in zip(fine, set_Prop_levels[i].TD_n[j]))           # :78
            dst = tuple(a - b for a, b in zip(fine, shrink))
            l[j], y[j] = resample_nn(l[j], src, dst), resample_nn(y[j], src, dst)
    return l, y


def _pad3(shape):
    return tuple(int(v) for v in shape) + (1,) * (3 - len(shape))


def warm_start_segments(set_Prop_levels, comp_grid_levels, dim3, i):
    """The boxes `interpolate_y_l` (and the x up-sampling) resample between level i+1 and level i, as
    (vector id, src offset, dst offset, src shape, dst shape); vector id -1 is x, otherwise the set index."""
    coarse, fine = tuple(comp_grid_levels[i + 1].n), tuple(comp_grid_levels[i].n)
    nax = 3 if dim3 else 2
    segs = [(-1, 0, 0, coarse[:nax], fine[:nax])]
    for j in range(len(set_Prop_levels[i].tag)):
        if set_Prop_levels[i].tag[j][1] in ("TV", "D2D", "D3D"):
            so = do = 0
            for axis in range(nax):
                sc = tuple(v - 1 if a == axis else v for a, v in enumerate(coarse[:nax]))
                sf = tuple(v - 1 if a == axis else v for a, v in enumerate(fine[:nax]))
                segs.append((j, so, do, sc, sf))
                so += int(np.prod(sc))
                do += int(np.prod(sf))
        else:
            src = tuple(set_Prop_levels[i + 1].TD_n[j])
            shrink = tuple(a - b for a, b in zip(fine, set_Prop_levels[i].TD_n[j]))
            segs.append((j, 0, 0, src, tuple(a - b for a, b in zip(fine, shrink))))
    return segs


def _host_warm_start(x, l, y, TD_OP_coarse, set_Prop_levels, comp_grid_levels, dim3, i):
    """x, l, y of level i+1 resampled on the host to level i (global vectors).  On slabs `l`, `y` are this rank's
    slabs: they are gathered into the reference's global order first (`x` is already global); PARSDMM scatters the
    global result again."""
    if dd.active():
        l = [dd.gather_td(v, A) for v, A in zip(l, TD_OP_coarse)]
        y = [dd.gather_td(v, A) for v, A in zip(y, TD_OP_coarse)]
    x = resample_nn(x, comp_grid_levels[i + 1].n, comp_grid_levels[i].n)       # :61-67
    l, y = interpolate_y_l(l, y, set_Prop_levels, comp_grid_levels, dim3, i)   # :74
    return x, l, y


def _device_warm_start(dev_fine, dev_coarse, segs):
    arr = (_lib.ResampleSeg * len(segs))()
    for q, (vec, so, do, ss, ds) in enumerate(segs):
        arr[q].vec, arr[q].src_off, arr[q].dst_off = vec, so, do
        arr[q].src_shape[:] = _pad3(ss)
        arr[q].dst_shape[:] = _pad3(ds)
    _lib.check(_lib.load().sipb_problem_warm_from(dev_fine.handle, dev_coarse.handle, arr, len(segs)))


def PARSDMM_multi_level(m, TD_OP_levels, AtA_levels, P_sub_levels, set_Prop_levels, comp_grid_levels, options,
                        x_ini=None, l_ini=None, y_ini=None, *, device_resample=True):
    """-> (x, log_PARSDMM, l, y) on the finest grid (PARSDMM_multi_level.jl:8-19,88).

    With `device_resample` (default) x, l, y never leave the GPU between levels: a resampling kernel writes the
    warm start straight into the finer problem's device buffers; only the finest level's x, l, y are copied back.
    Otherwise the host-side `resample_nn` / `interpolate_y_l` are used.

    Multi-GPU slabs (after `distributed.init`, 3-D problems): every level is slab-decomposed along z.  On the device
    path each transition gathers the coarse x, l, y on every rank (ncclSend / ncclRecv) and each rank resamples its
    own planes; the host path gathers l, y with `distributed.gather_td`.  As for `PARSDMM`, the returned x is global
    and l, y are this rank's slabs.

    `log.timing["transition_seconds"]` holds the host time of each level-to-level warm start, coarsest first."""
    TF = m.dtype.type
    n_levels = len(TD_OP_levels)
    rho_orig = copy.deepcopy(options.rho_ini)
    fine = tuple(comp_grid_levels[0].n)
    dim3 = len(fine) == 3 and fine[2] > 1
    m_levels = [m] + [resample_nn(m, fine, comp_grid_levels[k].n) for k in range(1, n_levels)]
    logs, transitions = [], []
    x, l, y = x_ini, l_ini, y_ini
    on_device = bool(device_resample) and not options.Minkowski
    try:
        for k in range(n_levels - 1, -1, -1):
            kw = {}
            t0 = time.perf_counter()
            if k == n_levels - 1:
                options.zero_ini_guess = True                                    # coarsest level: zero guess (:53)
            elif on_device:
                devs = [device_problem(m.dtype, AtA_levels[q], TD_OP_levels[q], set_Prop_levels[q], P_sub_levels[q],
                                       comp_grid_levels[q], options) for q in (k, k + 1)]
                t0 = time.perf_counter()
                _device_warm_start(devs[0], devs[1], warm_start_segments(set_Prop_levels, comp_grid_levels, dim3, k))
                options.zero_ini_guess = False                                   # :81
                x, l, y = None, None, None
                kw = dict(warm_resident=True)
            else:
                x, l, y = _host_warm_start(x, l, y, TD_OP_levels[k + 1], set_Prop_levels, comp_grid_levels, dim3, k)
                options.zero_ini_guess = False                                   # :81
            if k < n_levels - 1:
                transitions.append(time.perf_counter() - t0)
            if on_device and k > 0:
                kw["return_ly"] = False                                          # l, y stay on the device
                kw["gather_result"] = False                                      # slabs: x too
            x, log, l, y = PARSDMM(m_levels[k], AtA_levels[k], TD_OP_levels[k], set_Prop_levels[k], P_sub_levels[k],
                                   comp_grid_levels[k], options, x, l, y, **kw)
            options.rho_ini = [TF(v) for v in log.rho[-1, :]]                    # :57 / :83
            logs.append(log)
    finally:
        options.rho_ini = rho_orig                                               # :87
    log.timing["levels"] = [lg.timing for lg in logs]
    log.timing["level_iterations"] = [len(lg.obj) for lg in logs]
    log.timing["transition_seconds"] = transitions
    return x, log, l, y
