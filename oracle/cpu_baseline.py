"""Threaded CPU baseline: the oracle's PARSDMM with its vector phases in C/OpenMP (oracle/c/ref_kernels.c).

TEST / MEASUREMENT INFRASTRUCTURE ONLY — this is what bench.py's `cpu_baseline` and `--impl reference` legs time:
the reference algorithm with the reference's structure (one pass per CDS diagonal, CDS_MVp_MT.jl:9-25; separate
BLAS-1 passes in the CG, cg.jl:85-114; sort-based l1 projection, project_l1_Duchi!.jl:33-49; separate passes of
update_y_l.jl / adapt_rho_gamma.jl) on all host cores.  The control flow, the scalar rules (tolerances, stop
rules, rho/gamma adaptation, quirks) and the log bookkeeping are the NumPy oracle's own functions
(oracle/parsdmm.py); `tests/test_cpu_baseline.py` checks that both give the same iterates.

Differences to oracle/parsdmm.py that do not change the algorithm: reductions accumulate in Float64 with OpenMP
(order not fixed), the l1 cumulative sum runs in Float64.  Set types without a C projector fall back to the
oracle's NumPy projector on the same arrays.
"""
from __future__ import annotations

import ctypes as C
import time

import numpy as np
import scipy.sparse as sp

from . import build_c
from . import operators as ops
from . import parsdmm as P
from .sip_types import convert_options, eps, log_type_PARSDMM

_LIB = None
_i64p, _i32p, _dp, _vp = C.POINTER(C.c_int64), C.POINTER(C.c_int32), C.POINTER(C.c_double), C.c_void_p


def lib():
    global _LIB
    if _LIB is None:
        _LIB = C.CDLL(build_c.runtime_library())
        _LIB.sipref_threads.restype = C.c_int
        _LIB.sipref_set_threads.restype, _LIB.sipref_set_threads.argtypes = None, [C.c_int]
        for sfx, real in (("f32", C.c_float), ("f64", C.c_double)):
            def f(name, res, args):
                fn = getattr(_LIB, "sipref_%s_%s" % (name, sfx))
                fn.restype, fn.argtypes = res, args
            f("csr_matvec", None, [C.c_int64, _vp, _vp, _vp, _vp, _vp])
            f("csc_rmatvec", None, [C.c_int64, _vp, _vp, _vp, real, _vp, _vp, _vp, C.c_int])
            f("cds_mvp", None, [C.c_int64, C.c_int, _vp, _vp, _vp, _vp])
            f("dot", C.c_double, [C.c_int64, _vp, _vp])
            f("norm2", C.c_double, [C.c_int64, _vp])
            f("norm2_diff", C.c_double, [C.c_int64, _vp, _vp])
            f("norm1", C.c_double, [C.c_int64, _vp])
            f("copy", None, [C.c_int64, _vp, _vp])
            f("cg", C.c_int, [C.c_int64, C.c_int, _vp, _vp, _vp, _vp, real, C.c_int, _vp, C.POINTER(C.c_int), _dp])
            f("axpy_col", None, [C.c_int64, _vp, _vp, real])
            f("yl_pre", None, [C.c_int64, _vp, _vp, _vp, _vp, _vp, _vp, real, real])
            f("yl_post", C.c_double, [C.c_int64, _vp, _vp, _vp, _vp, _vp, real, real])
            f("project_bounds", None, [C.c_int64, _vp, real, real])
            f("prox_l2s", None, [C.c_int64, _vp, real, _vp])
            f("project_l1", C.c_int, [C.c_int64, _vp, real, _vp])
            f("adapt_sums", None, [C.c_int64, _vp, real, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _dp])
            f("l_hat", None, [C.c_int64, _vp, real, _vp, _vp, _vp])
    return _LIB


def threads() -> int:
    return int(lib().sipref_threads())


def use_all_cores() -> int:
    """Use every core this process may run on, whatever OMP_NUM_THREADS says (torchrun exports OMP_NUM_THREADS=1)."""
    import os
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    lib().sipref_set_threads(int(n))
    return threads()


class _K:
    """dtype-bound view of the C kernels."""

    def __init__(self, TF):
        self.TF = np.dtype(TF).type
        self.sfx = "f32" if self.TF == np.float32 else "f64"
        self.L = lib()

    def __getattr__(self, name):
        fn = getattr(self.L, "sipref_%s_%s" % (name, self.sfx))

        def call(*args):          # NumPy scalars -> Python scalars for ctypes
            return fn(*[a.item() if isinstance(a, np.generic) else a for a in args])
        self.__dict__[name] = call
        return call


def _p(a):
    return a.ctypes.data


class _Op:
    """CSR + CSC copies of one SparseMatrixCSC of the reference (TD_OP[i])."""

    def __init__(self, A, TF):
        A = sp.csc_matrix(A).astype(TF)
        A.sort_indices()
        R = sp.csr_matrix(A)
        R.sort_indices()
        self.shape = A.shape
        self.rp, self.ci, self.va = R.indptr.astype(np.int64), R.indices.astype(np.int32), np.ascontiguousarray(R.data, dtype=TF)
        self.cp, self.ri, self.vt = A.indptr.astype(np.int64), A.indices.astype(np.int32), np.ascontiguousarray(A.data, dtype=TF)


def _projector(k, constraint, P_sub_i, work):
    """In-place projector on a TF vector: the C routine for the set types of the bench workloads, else the
    oracle's NumPy projector."""
    TF = k.TF
    if constraint is not None and constraint.app_mode[0] in ("matrix", "tensor"):
        if constraint.set_type == "bounds" and np.ndim(constraint.min) == 0:
            lo, hi = TF(constraint.min), TF(constraint.max)
            return lambda v: k.project_bounds(v.size, _p(v), lo, hi)
        if constraint.set_type == "l1":
            b = TF(constraint.max)
            if b <= 0:
                raise ValueError("Radius of L1 ball is negative")
            return lambda v: k.project_l1(v.size, _p(v), b, _p(work))
    return lambda v: P_sub_i(v)


def PARSDMM(m, AtA, TD_OP, set_Prop, P_sub, comp_grid, options, constraint=None, max_iterations=None):
    """Same call and return as oracle.parsdmm.PARSDMM (serial, non-Minkowski, zero initial guess) plus
    `constraint` (the list given to setup_constraints: selects the C projectors) and `max_iterations`
    (bounded samples for bench.py).  Returns (x, log, l, y)."""
    TF = m.dtype.type
    k = _K(TF)
    t0 = time.perf_counter()
    if options.Minkowski or getattr(options, "parallel", False):
        raise NotImplementedError("threaded baseline: serial, non-Minkowski problems only")
    convert_options(options, TF)
    maxit = int(options.maxit)
    evol_rel_tol, feas_tol, obj_tol = options.evol_rel_tol, options.feas_tol, options.obj_tol
    rho_update_frequency = int(options.rho_update_frequency)
    gamma_ini = options.gamma_ini
    adjust_rho, adjust_gamma = bool(options.adjust_rho), bool(options.adjust_gamma)
    adjust_feasibility_rho = bool(options.adjust_feasibility_rho)
    feasibility_only = bool(options.feasibility_only)
    N = m.size
    p = len(TD_OP)
    pp = p if feasibility_only else p - 1
    rho = np.empty(p, dtype=TF)
    rho[:] = options.rho_ini[0] if len(options.rho_ini) == 1 else np.asarray(options.rho_ini, dtype=TF)
    ind_ref = maxit
    A = [_Op(TD_OP[i], TF) for i in range(p)]
    ly = [A[i].shape[0] for i in range(p)]
    key = np.uint32 if TF == np.float32 else np.uint64
    work = np.empty(2 * max(ly), dtype=key)
    cons = list(constraint) if constraint is not None else [None] * pp
    project = [_projector(k, cons[i] if i < len(cons) else None, P_sub[i], work) for i in range(pp)]

    def fwd(i, x, out):
        k.csr_matvec(ly[i], _p(A[i].rp), _p(A[i].ci), _p(A[i].va), _p(x), _p(out))

    zl = lambda: [np.zeros(n, dtype=TF) for n in ly]               # noqa: E731
    y, l, y_0, y_old, l_0, l_old, l_hat_0, l_hat = zl(), zl(), zl(), zl(), zl(), zl(), zl(), zl()
    x_hat, s_0, s, r_pri = zl(), zl(), zl(), zl()
    x = np.zeros(N, dtype=TF)
    x_old = np.zeros(N, dtype=TF)
    rhs = np.zeros(N, dtype=TF)
    cg_work = np.empty(3 * N, dtype=TF)
    tmpN = np.empty(N, dtype=TF)

    # initial feasibility (PARSDMM_initialize.jl:97-104)
    feasibility_initial = np.zeros(pp, dtype=TF)
    with np.errstate(all="ignore"):
        for ii in range(pp):
            fwd(ii, m, s[ii])
            k.copy(ly[ii], _p(s[ii]), _p(x_hat[ii]))
            project[ii](x_hat[ii])
            feasibility_initial[ii] = TF(k.norm2_diff(ly[ii], _p(x_hat[ii]), _p(s[ii]))) / (TF(k.norm2(ly[ii], _p(s[ii]))) + TF(100) * eps(TF))
    stop = bool(P._jl_maximum(feasibility_initial) < feas_tol)
    for ii in range(pp):
        if set_Prop.ncvx[ii]:
            rho_update_frequency, adjust_gamma, gamma_ini = 3, False, TF(0.75)
    gamma = np.full(p, gamma_ini, dtype=TF)

    Q, Q_offsets = ops.assemble_Q(AtA, set_Prop.AtA_offsets, rho)
    Q = np.asfortranarray(Q)
    Q_offsets = np.ascontiguousarray(Q_offsets, dtype=np.int64)
    AtA_F = [np.asfortranarray(a) for a in AtA]
    nd = Q_offsets.size

    log = log_type_PARSDMM(np.zeros((maxit, pp)), np.zeros((maxit, p)), np.zeros((maxit, p)), np.zeros(maxit),
                           np.zeros(maxit), np.zeros(maxit), np.zeros(maxit), np.zeros((maxit, p)),
                           np.zeros((maxit, p)), np.zeros(maxit, dtype=np.int64), np.zeros(maxit), {})
    log.set_feasibility[0, :] = feasibility_initial
    if stop:                                                        # PARSDMM.jl:63-82
        P._trim(log, 1, 1)
        log.timing = {"total": time.perf_counter() - t0}
        return m.copy(), log, l, y

    counter = 2
    x_solve_tol_ref = TF(1.0)
    timing = {kk: 0.0 for kk in ("initialization", "form rhs for linear system", "argmin x", "argmin y and l update",
                                 "stopping conditions check", "adjust rho and gamma", "Q-update")}
    timing["initialization"] = time.perf_counter() - t0
    it_limit = maxit if max_iterations is None else min(maxit, int(max_iterations))
    sums = np.zeros(6)
    cg_it, cg_res = C.c_int(0), C.c_double(0.0)

    for i in range(1, it_limit + 1):
        t = time.perf_counter()
        for ii in range(p):                                          # rhs_compose.jl:24-36
            k.csc_rmatvec(N, _p(A[ii].cp), _p(A[ii].ri), _p(A[ii].vt), rho[ii], _p(y[ii]), _p(l[ii]), _p(rhs), 0 if ii == 0 else 1)
        timing["form rhs for linear system"] += time.perf_counter() - t

        t = time.perf_counter()
        k.copy(N, _p(x), _p(x_old))                                  # PARSDMM.jl:106
        with np.errstate(all="ignore"):                              # argmin_x.jl:33-39
            k.cds_mvp(N, nd, _p(Q), _p(Q_offsets), _p(x), _p(tmpN))
            ratio = np.float64(0.1) * np.float64(TF(k.norm2_diff(N, _p(tmpN), _p(rhs)))) / np.float64(TF(k.norm2(N, _p(rhs))))
            cur = P._jl_max(ratio, np.float64(TF(10) * eps(TF)))
            x_solve_tol_ref = TF(cur) if i < 3 else TF(P._jl_min(cur, np.float64(x_solve_tol_ref)))
        k.cg(N, nd, _p(Q), _p(Q_offsets), _p(rhs), _p(x), x_solve_tol_ref, 1000, _p(cg_work), C.byref(cg_it), C.byref(cg_res))
        log.cg_it[i - 1] = cg_it.value
        log.cg_relres[i - 1] = cg_res.value
        timing["argmin x"] += time.perf_counter() - t

        t = time.perf_counter()
        for ii in range(p):                                          # update_y_l.jl:39-94
            fwd(ii, x, s[ii])
            k.yl_pre(ly[ii], _p(s[ii]), _p(y[ii]), _p(y_old[ii]), _p(l[ii]), _p(l_old[ii]), _p(x_hat[ii]), rho[ii], gamma[ii])
            if ii < pp:
                project[ii](y[ii])
            else:
                k.prox_l2s(ly[ii], _p(y[ii]), rho[ii], _p(m))         # always the current rho[p]
            log.r_pri[i - 1, ii] = TF(k.yl_post(ly[ii], _p(s[ii]), _p(y[ii]), _p(l[ii]), _p(x_hat[ii]), _p(r_pri[ii]), rho[ii], gamma[ii]))
            np.subtract(y[ii], y_old[ii], out=x_hat[ii])              # :82
            k.csc_rmatvec(N, _p(A[ii].cp), _p(A[ii].ri), _p(A[ii].vt), TF(1), _p(x_hat[ii]), None, _p(tmpN), 0)
            log.r_dual[i - 1, ii] = rho[ii] * TF(k.norm2(N, _p(tmpN)))   # :84
            if i % 10 == 0 and ii < pp:                               # :90-94
                k.copy(ly[ii], _p(s[ii]), _p(x_hat[ii]))
                project[ii](x_hat[ii])
                with np.errstate(all="ignore"):
                    log.set_feasibility[counter - 1, ii] = TF(k.norm2_diff(ly[ii], _p(x_hat[ii]), _p(s[ii]))) / (
                        TF(k.norm2(ly[ii], _p(s[ii]))) + TF(100) * eps(TF))
        if i % 10 == 0:
            counter += 1
        log.r_dual_total[i - 1] = P._tf_sum(log.r_dual[i - 1, :], TF)
        log.r_pri_total[i - 1] = P._tf_sum(log.r_pri[i - 1, :], TF)
        with np.errstate(all="ignore"):
            log.obj[i - 1] = TF(0.5) * TF(k.norm2_diff(N, _p(x), _p(m))) ** 2
            log.evol_x[i - 1] = TF(k.norm2_diff(N, _p(x_old), _p(x))) / TF(k.norm2(N, _p(x)))
        log.rho[i - 1, :] = rho
        log.gamma[i - 1, :] = gamma
        timing["argmin y and l update"] += time.perf_counter() - t

        t = time.perf_counter()
        stop, adjust_rho, adjust_gamma, adjust_feasibility_rho, ind_ref = P.stop_PARSDMM(
            log, i, evol_rel_tol, feas_tol, obj_tol, adjust_rho, adjust_gamma, adjust_feasibility_rho, ind_ref, counter, TF)
        timing["stopping conditions check"] += time.perf_counter() - t
        if stop or i == it_limit:
            P._trim(log, i, counter)
            log.timing = timing
            return x, log, l, y

        t = time.perf_counter()

        def snapshot(ii):
            k.copy(ly[ii], _p(l_hat[ii]), _p(l_hat_0[ii]))
            k.copy(ly[ii], _p(y[ii]), _p(y_0[ii]))
            k.copy(ly[ii], _p(s[ii]), _p(s_0[ii]))
            k.copy(ly[ii], _p(l[ii]), _p(l_0[ii]))

        if i == 1:                                                   # PARSDMM.jl:164-180
            for ii in range(p):
                k.l_hat(ly[ii], _p(l_old[ii]), rho[ii], _p(s[ii]), _p(y_old[ii]), _p(l_hat[ii]))
                snapshot(ii)
        if (adjust_rho or adjust_gamma) and i % rho_update_frequency == 0:   # :182-207
            for ii in range(p):
                k.adapt_sums(ly[ii], _p(l_old[ii]), rho[ii], _p(s[ii]), _p(y_old[ii]), _p(l_hat[ii]), _p(l_hat_0[ii]),
                             _p(s_0[ii]), _p(l[ii]), _p(l_0[ii]), _p(y[ii]), _p(y_0[ii]), sums.ctypes.data_as(_dp))
                rho[ii], gamma[ii] = P.adapt_decide(TF, TF(sums[0]), TF(sums[1]), TF(sums[2]), TF(sums[3]), TF(sums[4]),
                                                    TF(sums[5]), rho[ii], gamma[ii], adjust_rho, adjust_gamma)
            if i > 1:
                for ii in range(p):
                    snapshot(ii)
        if adjust_feasibility_rho and i % 10 == 0:                   # :213-223
            row = log.set_feasibility[counter - 2, :]
            if i > 10 and row.size:
                idx = P._jl_findmax_index(row)
                rho[idx] = TF(2.0) * rho[idx]
        rho = np.maximum(np.minimum(rho, TF(1e4)), TF(1e-2)).astype(TF)
        timing["adjust rho and gamma"] += time.perf_counter() - t

        t = time.perf_counter()
        logged = log.rho[i - 1, :].astype(TF)                        # Q_update!.jl:45-49
        for ii in np.nonzero(rho != logged)[0]:
            alpha = TF(rho[ii] - logged[ii])
            offs = set_Prop.AtA_offsets[ii]
            for kk in range(len(offs)):
                col = int(np.nonzero(Q_offsets == offs[kk])[0][0])
                k.axpy_col(N, Q.ctypes.data + col * N * Q.itemsize, AtA_F[ii].ctypes.data + kk * N * Q.itemsize, alpha)
        timing["Q-update"] += time.perf_counter() - t
    P._trim(log, it_limit, counter)
    log.timing = timing
    return x, log, l, y
