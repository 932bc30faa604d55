"""One PARSDMM iteration's vector phases, kernel by kernel, against exact references (sipb_iter_probe).

The probe runs, on a finalized single-GPU problem, the rhs gather (k_rhs / k_sparse_adjoint, rhs_compose.jl) and the y/l
update of every set (k_yl_multi, k_yl pass 1 / pass 2, the l1 gated pass 1, k_rdual, k_stop; update_y_l.jl:39-94 fused
with adapt_rho_gamma.jl:41-53 and the snapshots of PARSDMM.jl:164-207) exactly as sipb_solve runs them at iteration `it`,
from a state the test draws.  The references:
  * rhs: oracle.parsdmm.rhs_compose (the SciPy fold order k_op_adjoint matches): bit patterns equal;
  * s, v, y, l, l_hat and the snapshots: the update_y_l formulas in TF NumPy arithmetic (the library builds with
    -fmad=false) with the oracle projectors (element-wise and index sets) or, for l1 / l2 / annulus, the projection
    formula with the parameters the device found: bit-identical;
  * the l1 threshold and the l2 / annulus scale: exact roots from math.fsum, within the error of a Float64 sum plus one
    TF rounding;
  * every reduction (r_pri, r_dual fused and unfused, feasibility, the six adaptation sums, pass-1 statistics, stop
    sums): math.fsum of the Float64 products of the TF element values, within N 2^-52 sum|terms| (any partition).
Every case asserts from the launch counts of the call the regime it exists for."""
import copy
import ctypes as C
import math
import zlib

import numpy as np
import pytest

import problems as pr

pytestmark = pytest.mark.gpu

GROUP = {np.float32: 8, np.float64: 4}        # columns per thread of k_rhs (two 16-byte vectors)


@pytest.fixture(scope="module")
def orc():
    return pr.OracleAPI()


# ---------------------------------------------------------------------------------------------
# problems
# ---------------------------------------------------------------------------------------------
def build_pair(sip, orc, n, TF, sets, d=None, feasibility_only=False, sparse_idx=()):
    """sets: (set_type, TD_OP, min, max[, app_mode[, custom matrix]]).  Returns (oracle build, device build)."""
    d = d or (25.0,) * len(n)
    out = []
    for api in (orc, sip):
        cg = api.compgrid(d, n)
        cons = []
        for s in sets:
            mode = s[4] if len(s) > 4 else ("matrix", "")
            args = (s[0], s[1], copy.deepcopy(s[2]), copy.deepcopy(s[3]), mode)
            cons.append(api.set_definitions(*args, (s[5].copy(), False)) if len(s) > 5 else api.set_definitions(*args))
        opt = api.PARSDMM_options()
        opt.FL = TF
        opt.feasibility_only = feasibility_only
        P_sub, TD_OP, set_Prop = api.setup_constraints(cons, cg, TF)
        for ic in sparse_idx:
            set_Prop.AtA_diag[ic], set_Prop.dense[ic], set_Prop.banded[ic] = False, False, True
        TD_OP, AtA, _, _ = api.PARSDMM_precompute_distribute(TD_OP, set_Prop, cg, opt)
        out.append(dict(cg=cg, opt=opt, P_sub=P_sub, TD_OP=TD_OP, set_Prop=set_Prop, AtA=AtA, minkowski=False))
    return out


def build_mink(sip, orc, n, TF):
    ob = pr.build_minkowski(orc, n, TF)
    sb = pr.build_minkowski(sip, n, TF)
    for b in (ob, sb):
        b["minkowski"] = True
    return ob, sb


def device_handle(sip, sb, TF):
    return sip.solver.device_problem(np.dtype(TF), sb["AtA"], sb["TD_OP"], sb["set_Prop"], sb["P_sub"], sb["cg"],
                                     sb["opt"])


def set_kinds(sb):
    """Device set kind of every operator (the last one is the distance term unless feasibility_only)."""
    kinds = [P.set_kind for P in sb["P_sub"]]
    return kinds + [7] * (len(sb["TD_OP"]) - len(kinds))


# ---------------------------------------------------------------------------------------------
# the probe
# ---------------------------------------------------------------------------------------------
def run_probe(sip, dev, TF, st, it, do_adapt):
    """st: m, x, x_old, rho, gamma, and per set l, y, y_prev, snaps (4), inactive, warm (2), key."""
    L = sip._lib
    lib = L.load()
    p = len(st["l"])
    l = [a.copy() for a in st["l"]]
    y = [a.copy() for a in st["y"]]
    yp = [a.copy() for a in st["y_prev"]]
    snaps = [a.copy() for s in st["snaps"] for a in s]
    s_out = [np.zeros(a.size, dtype=TF) for a in st["l"]]
    rhs = np.empty(st["x"].size, dtype=TF)
    slots = np.zeros(512)
    params = np.zeros(3 * p)
    iparams = np.zeros(6 * p, dtype=np.int64)
    launches = np.zeros(L.N_KERNEL_CLASSES, dtype=np.int64)
    info = np.zeros(5, dtype=np.int32)
    VPA = lambda arrs: (C.c_void_p * len(arrs))(*[a.ctypes.data for a in arrs])      # noqa: E731
    dp = lambda a: np.ascontiguousarray(a, dtype=np.float64).ctypes.data_as(C.POINTER(C.c_double))   # noqa: E731
    rho = np.asarray(st["rho"], dtype=np.float64)
    gamma = np.asarray(st["gamma"], dtype=np.float64)
    warm = np.ascontiguousarray(np.asarray(st["warm"], dtype=np.float64).reshape(-1))
    inactive = np.asarray(st["inactive"], dtype=np.int32)
    keys = np.asarray(st["key"], dtype=np.uint64)
    rc = lib.sipb_iter_probe(
        dev.handle, it, int(do_adapt), st["m"].ctypes.data, st["x"].ctypes.data, st["x_old"].ctypes.data, dp(rho),
        dp(gamma), VPA(l), VPA(y), VPA(yp), VPA(snaps), inactive.ctypes.data_as(C.POINTER(C.c_int)), dp(warm),
        keys.ctypes.data_as(C.POINTER(C.c_uint64)), rhs.ctypes.data, VPA(s_out),
        slots.ctypes.data_as(C.POINTER(C.c_double)), params.ctypes.data_as(C.POINTER(C.c_double)),
        iparams.ctypes.data_as(C.POINTER(C.c_int64)), launches.ctypes.data_as(C.POINTER(C.c_int64)),
        info.ctypes.data_as(C.POINTER(C.c_int)))
    L.check(rc)
    names = {lib.sipb_kernel_class_name(i).decode(): int(launches[i]) for i in range(L.N_KERNEL_CLASSES)}
    return dict(rhs=rhs, l=l, y=y, snaps=[snaps[4 * s:4 * s + 4] for s in range(p)], s=s_out, slots=slots,
                theta=params[0::3], scale=params[1::3], fill=params[2::3], key_thr=iparams[0::6], launches=names,
                fuse_rdual=bool(info[0]), rdual_it=int(info[1]), fuse_stop=bool(info[2]), per_set=int(info[3]),
                glob=int(info[4]))


def draw_state(ob, TF, m, seed, scale=1.0, rho=None, gamma=None):
    """x near m (so bounds clip some rows), random multipliers, y^k, y^{k-1} and snapshots."""
    rng = np.random.default_rng(seed)
    ops = ob["TD_OP"]
    p = len(ops)
    N = ops[0].shape[1]
    npts = m.size
    x = np.zeros(N, dtype=TF)
    x[:npts] = m + TF(300) * rng.standard_normal(npts).astype(TF)
    if N > npts:
        x[npts:] = TF(200) * rng.standard_normal(N - npts).astype(TF)
    x_old = (x + TF(5) * rng.standard_normal(N).astype(TF)).astype(TF)
    st = dict(m=m.copy(), x=x, x_old=x_old, l=[], y=[], y_prev=[], snaps=[], inactive=[0] * p, warm=[(0.0, 0.0)] * p,
              key=[0] * p)
    st["rho"] = np.asarray(rho if rho is not None else rng.uniform(0.5, 4.0, p), dtype=TF)
    st["gamma"] = np.asarray(gamma if gamma is not None else [1.0 if i % 2 else 1.5 for i in range(p)], dtype=TF)
    for A in ops:
        M = A.shape[0]
        sx = np.asarray(A @ x.astype(np.float64)).ravel()
        sc = float(np.abs(sx).mean()) * scale + 1.0
        g = lambda s: (s * sc * rng.standard_normal(M)).astype(TF)      # noqa: E731
        st["l"].append(g(0.1))
        st["y"].append((sx + g(0.05)).astype(TF))
        st["y_prev"].append((sx + g(0.05)).astype(TF))
        st["snaps"].append([g(0.1), (sx + g(0.05)).astype(TF), g(0.1), (sx + g(0.05)).astype(TF)])
    return st


# ---------------------------------------------------------------------------------------------
# references
# ---------------------------------------------------------------------------------------------
def jl_sign(v):
    TF = v.dtype.type
    return np.where(v > 0, TF(1), np.where(v < 0, TF(-1), v)).astype(TF)


def jl_max0(a):
    """Julia max(a, 0) as t_max: NaN propagates, -0.0 -> +0.0."""
    TF = a.dtype.type
    return np.where(np.isnan(a), a, np.where(a > 0, a, TF(0))).astype(TF)


def bits_equal(a, b):
    a, b = np.asarray(a), np.asarray(b)
    assert a.dtype == b.dtype and a.shape == b.shape
    u = np.uint32 if a.dtype == np.float32 else np.uint64
    av, bv = a.view(u), b.view(u)
    nan = np.isnan(a) & np.isnan(b)
    bad = (av != bv) & ~nan
    return not bad.any(), (np.flatnonzero(bad)[:5], a[bad][:5], b[bad][:5])


def assert_bits(a, b, what):
    ok, why = bits_equal(a, b)
    assert ok, (what,) + why


def assert_sum(got, terms, what):
    """|s - exact| <= n 2^-52 sum|t_i| holds for any partition of a Float64 sum of the terms."""
    terms = np.asarray(terms, dtype=np.float64).ravel()
    if not np.all(np.isfinite(terms)):
        assert not np.isfinite(got), (what, got)
        return
    exact = math.fsum(terms)
    assert abs(got - exact) <= max(terms.size, 1) * 2.0 ** -52 * float(np.abs(terms).sum()), (what, got, exact)


def sq(a):
    a = a.astype(np.float64)
    return a * a


def l1_root(v, tau):
    """Exact soft threshold of project_l1_Duchi!.jl:21-52: theta* = (sum u_1..u_r - tau) / r with u sorted descending and
    r the largest index with u_r > (sum u_1..u_r - tau) / r; all entries active: the lv-1 cap.  Returns (theta*, r, u)."""
    u = np.sort(np.abs(v.astype(np.float64)))[::-1]
    cs = np.cumsum(u)
    j = np.arange(1, u.size + 1)
    cond = u > (cs - tau) / j
    r = int(np.flatnonzero(cond)[-1]) + 1
    if r == u.size and u.size >= 2:
        return max(0.0, (math.fsum(u[:-1]) - tau) / (u.size - 1)), u.size - 1, u
    return max(0.0, (math.fsum(u[:r]) - tau) / r), r, u


def reference_set(TF, kind, A, P_orc, P_sip, x, l, yk, rho, gamma, m_ext, dev_params):
    """update_y_l.jl:43-78 for one set in TF arithmetic.  Returns s, xh, v, y, l_new."""
    s = orc_spmv(A, x)
    relaxed = not (gamma == TF(1))
    rho1 = TF(TF(1.0) / rho)
    xh = (gamma * s + (TF(1.0) - gamma) * yk).astype(TF) if relaxed else s
    v = (xh - l * rho1).astype(TF)
    if kind == 7:
        y = _prox_l2s(v, rho, m_ext[:v.size])
    elif kind == 6:
        y = (jl_sign(v) * jl_max0((np.abs(v) - TF(TF(1) / TF(P_sip.max))).astype(TF))).astype(TF)
    elif kind == 2:
        th = TF(dev_params["theta"])
        y = v.copy() if th < 0 else (jl_sign(v) * jl_max0((np.abs(v) - th).astype(TF))).astype(TF)
    elif kind in (3, 4):
        fill, sc = TF(dev_params["fill"]), TF(dev_params["scale"])
        y = np.full_like(v, fill) if fill == fill else (v.copy() if sc == TF(1) else (v * sc).astype(TF))
    else:
        y = P_orc(v.copy())
    rp = (-s + y).astype(TF)
    ln = (l + rho * (-xh + y)).astype(TF) if relaxed else (l + rho * rp).astype(TF)
    return s, xh, v, y, rp, ln


def orc_spmv(A, x):
    import oracle.operators as oops
    return oops.spmv(A, x)


def orc_spmv_t(A, v):
    import oracle.operators as oops
    return oops.spmv_t(A, v)


def _prox_l2s(v, rho, m):
    import oracle.projectors as op
    return op.prox_l2s(v.copy(), rho, m)


def check_iteration(orc, ob, sb, TF, st, out, it, do_adapt, expect_sums=True):
    """Compares every output of one probe call with the references; returns per-set details for regime checks."""
    ops = ob["TD_OP"]
    p = len(ops)
    kinds = set_kinds(sb)
    feas_only = bool(sb["opt"].feasibility_only)
    fuse_adapt = it == 1 or do_adapt
    do_sums = do_adapt and it > 1
    feas_it = it % 10 == 0
    m_ext = np.concatenate([st["m"], np.zeros(st["x"].size - st["m"].size, dtype=TF)])
    rho, gamma = st["rho"], st["gamma"]
    # rhs (rhs_compose.jl:24-36), bit patterns
    rhs = orc.parsdmm.rhs_compose(np.zeros(st["x"].size, dtype=TF), st["l"], st["y"], rho, ops, p)
    assert_bits(out["rhs"], rhs, "rhs")
    slots, B, G0 = out["slots"], out["per_set"], out["glob"]
    det = []
    for i, A in enumerate(ops):
        kind = kinds[i]
        P_orc = ob["P_sub"][i] if i < len(ob["P_sub"]) else None
        P_sip = sb["P_sub"][i] if i < len(sb["P_sub"]) else None
        dpar = dict(theta=out["theta"][i], scale=out["scale"][i], fill=out["fill"][i])
        s, xh, v, y, rp, ln = reference_set(TF, kind, A, P_orc, P_sip, st["x"], st["l"][i], st["y"][i], rho[i],
                                            gamma[i], m_ext, dpar)
        assert_bits(out["y"][i], y, "y[%d]" % i)
        assert_bits(out["l"][i], ln, "l[%d]" % i)
        base = B * i
        elementwise = kind in (0, 1, 6, 7, 8)
        sparse = bool(getattr(sb["TD_OP"][i], "op_kind", 0) == 6)
        if not elementwise or sparse:
            if feas_it or sparse:
                assert_bits(out["s"][i], s, "s[%d]" % i)
        # snapshots (adapt_rho_gamma.jl:41, PARSDMM.jl:164-207)
        lh = (st["l"][i] + rho[i] * (-s + st["y"][i])).astype(TF)
        want = [lh, s, ln, y] if fuse_adapt else st["snaps"][i]
        for q, nm in enumerate(("l_hat_0", "s_0", "l_0", "y_0")):
            assert_bits(out["snaps"][i][q], want[q], "%s[%d]" % (nm, i))
        if not expect_sums:
            det.append(dict(v=v, s=s))
            continue
        assert_sum(slots[base + 0], sq(rp), "r_pri[%d]" % i)
        if do_sums:
            lh0, s0, l0, y0 = st["snaps"][i]
            dlh, dH = (lh - lh0).astype(TF), (s - s0).astype(TF)
            dl, dG = (ln - l0).astype(TF), (-(y - y0)).astype(TF)
            for q, (a, b) in enumerate(((dH, dlh), (dH, dH), (dlh, dlh), (dl, dl), (dG, dG), (dG, dl))):
                assert_sum(slots[base + 4 + q], a.astype(np.float64) * b.astype(np.float64), "adapt[%d][%d]" % (i, q))
        if not elementwise:                                   # pass-1 statistics of v
            assert_sum(slots[base + 10], np.abs(v.astype(np.float64)), "sum|v|[%d]" % i)
            if not feas_it:                   # (the in-loop feasibility reuses slots 11.. for the statistics of s)
                assert_sum(slots[base + 11], sq(v), "sum v^2[%d]" % i)
                assert_sum(slots[base + 12], (v != 0).astype(np.float64), "nnz(v)[%d]" % i)
        if feas_it and i < (p if feas_only else p - 1):
            assert_sum(slots[base + 2], sq(s), "feas den[%d]" % i)
            if kind not in (2, 3, 4):        # the feasibility projector's own l1 / l2 parameters are not returned
                ps = P_orc(s.copy())
                assert_sum(slots[base + 1], sq((ps - s).astype(TF)), "feas num[%d]" % i)
        if not out["fuse_rdual"]:             # k_rdual / k_sparse_rdual of this iteration
            assert out["rdual_it"] == it
            assert_sum(slots[base + 3], sq(orc_spmv_t(A, (y - st["y"][i]).astype(TF))), "r_dual[%d]" % i)
        elif it >= 2:                         # fused into the rhs gather: iteration it-1
            assert out["rdual_it"] == it - 1
            assert_sum(slots[G0 + 8 + i], sq(orc_spmv_t(A, (st["y"][i] - st["y_prev"][i]).astype(TF))),
                       "fused r_dual[%d]" % i)
        det.append(dict(v=v, s=s))
    if expect_sums:                           # stop sums (PARSDMM.jl:140-145)
        x, xo = st["x"], st["x_old"]
        npts = st["m"].size
        if ob["minkowski"]:
            o = ((TF(0) + x[:npts]) + x[npts:]).astype(TF) - st["m"]
        else:
            o = (x - st["m"]).astype(TF)
        assert_sum(slots[G0 + 0], sq(o), "||x-m||^2")
        assert_sum(slots[G0 + 1], sq((xo - x).astype(TF)), "||x_old-x||^2")
        assert_sum(slots[G0 + 2], sq(x), "||x||^2")
    return det


def check_launches(sb, out, it, inactive=None):
    """The path the call took: one k_yl_multi per 8 element-wise sets, two pass-1 launches for an l1 set whose guess
    says inactive, k_rdual per set when the dual residual is not fused, k_stop when no distance term reduces the stop
    sums, one gather per run of stencil sets and one k_sparse_adjoint per explicit sparse operator."""
    kinds = set_kinds(sb)
    p = len(kinds)
    sparse = [getattr(A, "op_kind", 0) == 6 for A in sb["TD_OP"]]
    ew = sum(k in (0, 1, 6, 7, 8) for k in kinds)
    red = p - ew
    inactive = inactive or [0] * p
    n_l1_skip = sum(1 for k, a in zip(kinds, inactive) if k == 2 and a)
    L = out["launches"]
    assert L["yl_update_fused"] == -(-ew // 8), L
    assert L["yl_update_pass2"] == red and L["yl_update_pass1"] == red + n_l1_skip, L
    fuse_rdual = p <= 8 and not any(sparse)
    assert out["fuse_rdual"] == fuse_rdual
    assert L["r_dual"] == (0 if fuse_rdual else p), L
    runs = sum(1 for i in range(p) if not sparse[i] and (i == 0 or sparse[i - 1]))
    assert L["rhs_compose"] == runs + sum(sparse), L
    assert L["stop_reduce"] == (0 if out["fuse_stop"] else 1), L
    return L


# ---------------------------------------------------------------------------------------------
# grids: the line groups of the rhs gather, both precisions
# ---------------------------------------------------------------------------------------------
def grid_cases():
    cases = []
    for TF in (np.float32, np.float64):
        g = GROUP[TF]
        for n0, tag in ((g // 2 + 1, "n0_lt_G"), (g, "n0_eq_G"), (g - 1, "n0_G_minus_1"), (g + 1, "n0_G_plus_1"),
                        (2, "n0_2"), (3 * g + 5, "tail")):
            cases.append((TF, (n0, 13), tag))
            cases.append((TF, (n0, 7, 5), tag))
        cases.append((TF, (37, 2), "two_lines"))
    return cases


def grid_sets(n):
    if len(n) == 2:
        return [("bounds", "identity", 1500.0, 4500.0), ("bounds", "D_x", -40.0, 40.0), ("bounds", "D_z", 0.0, 1e6),
                ("l1", "TV", 0.0, 1e3), ("bounds", "D_xz", -50.0, 50.0)] if n[0] > 2 and n[1] > 2 else \
               [("bounds", "identity", 1500.0, 4500.0), ("bounds", "D_x", -40.0, 40.0), ("l1", "TV", 0.0, 1e3)]
    return [("bounds", "identity", 1500.0, 4500.0), ("bounds", "D_x", -40.0, 40.0), ("bounds", "D_y", -30.0, 30.0),
            ("bounds", "D_z", 0.0, 1e6), ("l1", "TV", 0.0, 1e3)]


@pytest.mark.parametrize("TF,n,tag", grid_cases(), ids=lambda v: getattr(v, "__name__", str(v)))
@pytest.mark.parametrize("it,do_adapt", [(1, False), (4, True), (5, False), (10, True)])
def test_iteration_grids(sip, orc, TF, n, tag, it, do_adapt):
    m = pr.synthetic_model(n, TF)
    ob, sb = build_pair(sip, orc, n, TF, grid_sets(n))
    dev = device_handle(sip, sb, TF)
    st = draw_state(ob, TF, m, seed=zlib.crc32(repr((n, it)).encode()))
    out = run_probe(sip, dev, TF, st, it, do_adapt)
    check_launches(sb, out, it)
    check_iteration(orc, ob, sb, TF, st, out, it, do_adapt)
    g = GROUP[TF]
    assert (n[0] % g != 0) or tag in ("n0_eq_G",), "the grid must exercise groups that end or wrap a line"
    assert out["rdual_it"] == (it - 1 if out["fuse_rdual"] else it)


@pytest.mark.parametrize("TF", [np.float32, np.float64])
@pytest.mark.parametrize("it,do_adapt", [(1, False), (3, True), (10, False)])
def test_iteration_minkowski(sip, orc, TF, it, do_adapt):
    """Minkowski blocks [A 0], [0 A], [A A]; npts % G != 0, so a column group straddles the two halves; the stop sums go
    through k_stop."""
    n = (29, 11)
    assert (n[0] * n[1]) % GROUP[TF] != 0
    ob, sb = build_mink(sip, orc, n, TF)
    dev = device_handle(sip, sb, TF)
    st = draw_state(ob, TF, ob["m"].astype(TF), seed=7 + it)
    out = run_probe(sip, dev, TF, st, it, do_adapt)
    L = check_launches(sb, out, it)
    assert not out["fuse_stop"] and L["stop_reduce"] == 1
    check_iteration(orc, ob, sb, TF, st, out, it, do_adapt)


@pytest.mark.parametrize("TF,n", [(np.float32, (96, 96, 96)), (np.float64, (64, 64, 64))])
def test_iteration_large_grid(sip, orc, TF, n):
    """Config 2 sets on a grid whose reductions span many blocks, at an adapting iteration and at it = 10."""
    spec = pr.spec_config2(n, TF)
    m = spec["m"]
    ob, sb = build_pair(sip, orc, n, TF, spec["sets"])
    dev = device_handle(sip, sb, TF)
    for it, do_adapt in ((10, True),):
        st = draw_state(ob, TF, m, seed=3)
        out = run_probe(sip, dev, TF, st, it, do_adapt)
        check_launches(sb, out, it)
        check_iteration(orc, ob, sb, TF, st, out, it, do_adapt)


# ---------------------------------------------------------------------------------------------
# set counts: fused / unfused dual residual, one or two k_yl_multi launches, the most sets
# ---------------------------------------------------------------------------------------------
def many_sets(k):
    base = [("bounds", "identity", 1500.0, 4500.0), ("bounds", "D_x", -40.0, 40.0), ("bounds", "D_z", 0.0, 1e6),
            ("prox_l1", "D_x", 0.0, 3.0), ("bounds", "D_xz", -50.0, 50.0), ("prox_l1", "identity", 0.0, 0.5),
            ("bounds", "D_z", -20.0, 20.0), ("prox_l1", "D_z", 0.0, 1.5)]
    return [base[i % len(base)] for i in range(k)]


@pytest.mark.parametrize("TF", [np.float32, np.float64])
@pytest.mark.parametrize("p", [8, 9, 15])
@pytest.mark.parametrize("it,do_adapt", [(2, True), (7, False), (10, False)])
def test_iteration_set_counts(sip, orc, TF, p, it, do_adapt):
    n = (37, 23)
    m = pr.synthetic_model(n, TF)
    ob, sb = build_pair(sip, orc, n, TF, many_sets(p - 1))
    assert len(sb["TD_OP"]) == p
    dev = device_handle(sip, sb, TF)
    st = draw_state(ob, TF, m, seed=p * 31 + it)
    out = run_probe(sip, dev, TF, st, it, do_adapt)
    L = check_launches(sb, out, it)
    assert L["yl_update_fused"] == (1 if p <= 8 else 2)
    assert out["fuse_rdual"] == (p <= 8)
    check_iteration(orc, ob, sb, TF, st, out, it, do_adapt)


def every_kind_sets(n, TF):
    rng = np.random.default_rng(5)
    M = int(np.prod(n))
    lo = np.full(M, 1400.0)
    hi = np.full(M, 4000.0)
    hlo = np.sort(rng.uniform(1000.0, 2500.0, M))
    hhi = np.sort(hlo + rng.uniform(100.0, 2500.0, M))
    flo = np.linspace(1400.0, 1600.0, n[1])
    fhi = np.linspace(3000.0, 4700.0, n[1])
    return [("bounds", "identity", 1500.0, 4500.0), ("bounds", "identity", lo, hi), ("l1", "TV", 0.0, 2e3),
            ("l2", "D_x", 0.0, 200.0), ("annulus", "D_z", 3e4, 4e4), ("cardinality", "TV", 0, 100),
            ("prox_l1", "identity", 0.0, 2.0), ("histogram", "identity", hlo, hhi),
            ("bounds", "identity", flo, fhi, ("fiber", "z")), ("cardinality", "D_x", 0, 3, ("fiber", "x"))]


@pytest.mark.parametrize("TF", [np.float32, np.float64])
@pytest.mark.parametrize("it,do_adapt,fuse_stop_off", [(1, False, False), (6, True, True), (10, False, False),
                                                       (20, True, False)])
def test_iteration_every_set_kind(sip, orc, TF, it, do_adapt, fuse_stop_off, monkeypatch):
    if fuse_stop_off:
        monkeypatch.setenv("SIPB_FUSE_STOP_OFF", "1")
    n = (30, 26)
    m = pr.synthetic_model(n, TF)
    ob, sb = build_pair(sip, orc, n, TF, every_kind_sets(n, TF))
    dev = device_handle(sip, sb, TF)
    st = draw_state(ob, TF, m, seed=11 + it)
    out = run_probe(sip, dev, TF, st, it, do_adapt)
    L = check_launches(sb, out, it)
    assert out["fuse_stop"] == (not fuse_stop_off) and out["fuse_rdual"] is False      # p = 11
    assert L["yl_update_pass2"] == 6
    det = check_iteration(orc, ob, sb, TF, st, out, it, do_adapt)
    check_l1_theta(sb, out, det, 2)
    check_l2_scale(sb, out, det, 3, TF)
    check_l2_scale(sb, out, det, 4, TF)


@pytest.mark.parametrize("TF", [np.float32, np.float64])
def test_iteration_feasibility_only(sip, orc, TF):
    """No distance term: the stop sums go through k_stop and every set is logged for feasibility."""
    n = (21, 19)
    m = pr.synthetic_model(n, TF)
    ob, sb = build_pair(sip, orc, n, TF, grid_sets(n), feasibility_only=True)
    dev = device_handle(sip, sb, TF)
    st = draw_state(ob, TF, m, seed=2)
    out = run_probe(sip, dev, TF, st, 10, True)
    L = check_launches(sb, out, 10)
    assert L["stop_reduce"] == 1 and not out["fuse_stop"]
    check_iteration(orc, ob, sb, TF, st, out, 10, True)


@pytest.mark.parametrize("TF", [np.float32, np.float64])
@pytest.mark.parametrize("where", ["first", "middle"])
def test_iteration_sparse_operator(sip, orc, TF, where):
    """An explicit SparseOperator splits the stencil run: several gather launches, accumulate = 1, k_sparse_adjoint in
    between, r_dual unfused (k_sparse_rdual), s = A x by k_sparse_forward."""
    import scipy.sparse as sps
    n, d = (23, 17), (25.0, 6.0)
    m = pr.synthetic_model(n, TF)
    A, *_ = orc.get_TD_operator(orc.compgrid(d, n), "TV", TF)
    w = (1.0 + 0.5 * np.sin(np.arange(A.shape[0]) * 0.37)).astype(TF)
    W = sps.csc_matrix(sps.diags(w).astype(TF) @ A).astype(TF)
    W.sort_indices()
    sets = [("bounds", "identity", 1500.0, 4500.0), ("bounds", "D_x", -40.0, 40.0),
            ("bounds", "D_z", 0.0, 1e6)]
    cs = ("bounds", "identity", -30.0, 30.0, ("matrix", ""), W)
    ic = 0 if where == "first" else 1
    sets.insert(ic, cs)
    ob, sb = build_pair(sip, orc, n, TF, sets, d=d, sparse_idx=(ic,))
    dev = device_handle(sip, sb, TF)
    st = draw_state(ob, TF, m, seed=9)
    out = run_probe(sip, dev, TF, st, 4, True)
    L = check_launches(sb, out, 4)
    assert L["rhs_compose"] == (2 if where == "first" else 3) and L["r_dual"] == len(sets) + 1
    check_iteration(orc, ob, sb, TF, st, out, 4, True)


# ---------------------------------------------------------------------------------------------
# l1 ball: skip-v guess, gated pass 1, threshold search
# ---------------------------------------------------------------------------------------------
def check_l1_theta(sb, out, det, i):
    """The device threshold against the exact root: the error of a Float64 sum over M terms divided by the active count,
    plus one TF rounding."""
    TF = sb["opt"].FL
    tau = float(TF(sb["P_sub"][i].max))
    v = det[i]["v"]
    th = float(out["theta"][i])
    s1 = math.fsum(np.abs(v.astype(np.float64)))
    if TF(s1) <= TF(tau):
        assert th < 0, th                               # inside the ball: untouched
        return None
    root, r, u = l1_root(v, tau)
    bound = v.size * 2.0 ** -52 * float(u.sum()) / r + float(np.finfo(TF).eps) * abs(root) + 1e-300
    assert abs(th - root) <= bound, (th, root, r, bound)
    return r


def check_l2_scale(sb, out, det, i, TF):
    P = sb["P_sub"][i]
    v = det[i]["v"]
    nl2 = math.sqrt(math.fsum(sq(v)))
    sc, fill = float(out["scale"][i]), float(out["fill"][i])
    lo, hi = float(TF(P.min)), float(TF(P.max))
    if P.set_kind == 3:
        want = 1.0 if nl2 <= hi else hi / nl2
    elif lo <= nl2 <= hi:
        want = 1.0
    elif nl2 > hi:
        want = hi / nl2
    elif nl2 > 0:
        want = lo / nl2
    else:
        assert fill == float(TF(lo / math.sqrt(v.size)))
        return
    assert math.isnan(fill)
    assert abs(sc - want) <= 4 * float(np.finfo(TF).eps) * want, (sc, want)


def l1_vector(case, M, TF, rng):
    if case == "ties":
        return (rng.integers(1, 4, M) * rng.choice([-1.0, 1.0], M)).astype(TF)
    if case == "all_active":
        return ((1.0 + 0.01 * rng.random(M)) * rng.choice([-1.0, 1.0], M)).astype(TF)
    if case == "one_survivor":
        v = rng.standard_normal(M).astype(TF)
        v[M // 3] = TF(50.0)
        return v
    return (rng.standard_normal(M) * 3.0).astype(TF)


def l1_tau(case, v):
    s = math.fsum(np.abs(v.astype(np.float64)))
    TF = v.dtype.type
    if case == "inactive":
        return 1.5 * s
    if case == "just_above":
        return float(np.nextafter(TF(s), TF(0)) * (TF(1) - TF(4) * np.finfo(TF).eps))
    if case == "one_survivor":
        return 1e-3
    if case == "all_active":
        u = np.abs(v.astype(np.float64))
        return s - 0.5 * u.size * u.min()
    return 0.4 * s


@pytest.mark.parametrize("TF", [np.float32, np.float64])
@pytest.mark.parametrize("case,guess_inactive,warm", [
    ("inactive", 1, "zero"), ("inactive", 0, "zero"), ("active", 1, "zero"), ("active", 0, "zero"),
    ("active", 0, "left"), ("active", 0, "right"), ("just_above", 1, "zero"), ("one_survivor", 0, "right"),
    ("all_active", 0, "left"), ("ties", 1, "zero")])
def test_iteration_l1_regimes(sip, orc, TF, case, guess_inactive, warm):
    """l1 ball on the identity with l = 0, gamma = 1, so that v = x.  A guess that says inactive sets skip_v: pass 1 runs
    twice and the gated launch must write v when the ball is active (y_prev, left in the buffer, differs from v)."""
    n = (61, 33)
    M = n[0] * n[1]
    rng = np.random.default_rng(zlib.crc32(repr((case, guess_inactive, warm)).encode()))
    v = l1_vector(case, M, TF, rng)
    tau = l1_tau(case, v)
    m = pr.synthetic_model(n, TF)
    ob, sb = build_pair(sip, orc, n, TF, [("l1", "identity", 0.0, tau)])
    dev = device_handle(sip, sb, TF)
    st = draw_state(ob, TF, m, seed=1, gamma=[1.0, 1.0], rho=[1.0, 2.0])
    st["x"] = v.copy()
    st["l"][0] = np.zeros(M, dtype=TF)
    st["y_prev"][0] = (TF(7) + rng.random(M)).astype(TF)
    st["inactive"] = [guess_inactive, 0]
    root, _, _ = l1_root(v, float(TF(tau))) if case != "inactive" else (0.0, 0, None)
    st["warm"] = [({"zero": 0.0, "left": 0.5 * root, "right": 1.5 * root + 1e-3}[warm], 0.0), (0.0, 0.0)]
    out = run_probe(sip, dev, TF, st, 5, False)
    L = check_launches(sb, out, 5, inactive=st["inactive"])
    assert L["yl_update_pass1"] == 1 + guess_inactive
    det = check_iteration(orc, ob, sb, TF, st, out, 5, False)
    r = check_l1_theta(sb, out, det, 0)
    active = case != "inactive"
    assert (out["theta"][0] >= 0) == active
    if case == "one_survivor":
        assert r == 1 and np.count_nonzero(out["y"][0]) == 1
    if case == "all_active":
        assert r == M - 1


# ---------------------------------------------------------------------------------------------
# special values in the element-wise sets
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("TF", [np.float32, np.float64])
@pytest.mark.parametrize("it,do_adapt", [(3, True), (10, False)])
def test_iteration_special_values(sip, orc, TF, it, do_adapt):
    """+-0 in x and l, entries exactly on a bound, subnormals and a NaN (Julia max / min propagate it)."""
    n = (27, 19)
    N = n[0] * n[1]
    m = pr.synthetic_model(n, TF)
    sets = [("bounds", "identity", 1500.0, 4500.0), ("bounds", "identity", -1.0, 1.0), ("prox_l1", "identity", 0.0, 2.0),
            ("bounds", "D_x", -40.0, 40.0)]
    ob, sb = build_pair(sip, orc, n, TF, sets)
    dev = device_handle(sip, sb, TF)
    st = draw_state(ob, TF, m, seed=4, gamma=[1.0, 1.3, 1.0, 1.0, 1.7])
    rng = np.random.default_rng(4)
    tiny = np.finfo(TF).smallest_subnormal
    x = st["x"]
    idx = rng.permutation(N)
    x[idx[:20]] = TF(0.0)
    x[idx[20:40]] = -TF(0.0)
    x[idx[40:50]] = TF(1500.0)
    x[idx[50:60]] = TF(4500.0)
    x[idx[60:70]] = TF(1.0)
    x[idx[70:80]] = tiny * rng.integers(1, 100, 10).astype(TF)
    x[idx[80:90]] = -tiny * rng.integers(1, 100, 10).astype(TF)
    for l in st["l"]:
        l[:10] = -TF(0.0)
        l[10:20] = TF(0.0)
        l[20:25] = tiny
    out = run_probe(sip, dev, TF, st, it, do_adapt)
    check_launches(sb, out, it)
    check_iteration(orc, ob, sb, TF, st, out, it, do_adapt)
    # a NaN: every element-wise set and the distance term carry it to y and l; only the sums see it otherwise
    x[idx[100]] = TF(np.nan)
    out = run_probe(sip, dev, TF, st, it, do_adapt)
    check_iteration(orc, ob, sb, TF, st, out, it, do_adapt, expect_sums=False)
    assert np.isnan(out["y"][0][idx[100]]) and np.isnan(out["l"][-1][idx[100]])


# ---------------------------------------------------------------------------------------------
# the unfused dual residual in whole solves
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("TF", [np.float64, np.float32])
def test_parsdmm_nine_sets_parity(sip, orc, TF):
    """p = 9: k_rdual for every set and two k_yl_multi launches per iteration, a whole solve against the oracle."""
    from test_gpu_parity import check_parity
    n = (40, 34)
    spec = dict(n=n, d=(25.0, 6.0), TF=TF, m=pr.synthetic_model(n, TF), sets=many_sets(8), mode="matrix")
    o_opt, s_opt = orc.PARSDMM_options(), sip.PARSDMM_options()
    for o in (o_opt, s_opt):
        o.maxit = 60
    ob = pr.build(orc, copy.deepcopy(spec), o_opt)
    sb = pr.build(sip, copy.deepcopy(spec), s_opt)
    m = spec["m"]
    xo, lo, ll, yy = orc.PARSDMM(m.copy(), ob["AtA"], ob["TD_OP"], ob["set_Prop"], ob["P_sub"], ob["cg"], ob["opt"])
    xs, ls, l2, y2 = sip.PARSDMM(m.copy(), sb["AtA"], sb["TD_OP"], sb["set_Prop"], sb["P_sub"], sb["cg"], sb["opt"])
    assert len(sb["TD_OP"]) == 9
    its = len(ls.obj)
    k = ls.timing["kernels"]
    assert k["r_dual"][0] == 9 * its and k["yl_update_fused"][0] == 2 * its, k
    check_parity((xo, lo, ll, yy, ob), (xs, ls, l2, y2, sb), TF)
