"""GPU tests: custom (explicit sparse) operators inside generalized Minkowski sets, and Q / A'A wider than 32 diagonals.

Kernel by kernel against exact references (bit patterns, signs of zeros included) and whole solves against the oracle
to the standard of test_gpu_parity.py."""
import ctypes as C
import zlib

import numpy as np
import pytest
import scipy.sparse as sp

import problems as pr
import test_gpu_iteration as gi
from test_custom_wide_host import STENCIL5, STENCIL27, weighted_gradient, weighted_stencil
from test_gpu_parity import TOL, check_parity, relerr

pytestmark = pytest.mark.gpu

MODES = {"left": 1, "right": 2, "both": 3}


@pytest.fixture(scope="module")
def orc():
    return pr.OracleAPI()


def bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint32 if a.dtype == np.float32 else np.uint64)


def assert_bits(got, want, what=""):
    assert got.dtype == want.dtype and got.shape == want.shape, what
    bad = np.nonzero(bits(got) != bits(want))[0]
    assert bad.size == 0, "%s: %d entries differ, first at %d: %r vs %r" % (what, bad.size, bad[0], got[bad[0]], want[bad[0]])


def hcat(W, mode):
    Z = sp.csc_matrix(W.shape, dtype=W.dtype)
    B = sp.hstack({"left": [W, Z], "right": [Z, W], "both": [W, W]}[mode], format="csc", dtype=W.dtype)
    B.sort_indices()
    return B


def signed_input(n, TF, seed):
    """values of both signs with exact zeros of both signs"""
    v = (pr.splitmix_uniform(seed, n) - 0.5).astype(TF)
    v[::7] = TF(0.0)
    v[3::11] = -TF(0.0)
    return v


# ---------------------------------------------------------------------------------------------
# sipb_sparse_apply_block
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("TF", [np.float32, np.float64])
@pytest.mark.parametrize("mode", ["left", "right", "both"])
def test_sparse_apply_block_bit_exact(sip, orc, TF, mode):
    n, d = (13, 9, 5), (2.0, 3.0, 1.5)
    W = weighted_gradient(orc, n, d, TF).tolil()
    W[5, :] = 0                  # empty rows
    W[17, :] = 0
    W[:, 0] = 0                  # empty columns
    W[:, 40] = 0
    W = sp.csc_matrix(W)
    W.eliminate_zeros()
    W.sort_indices()
    op = sip.SparseOperator(W, n, d, TF).with_block(MODES[mode])
    B = hcat(W, mode)
    assert op.shape == B.shape
    for seed in (3, 4):
        x = signed_input(B.shape[1], TF, seed)
        v = signed_input(B.shape[0], TF, seed + 10)
        assert_bits(op @ x, orc.ops.spmv(B, x), "B x")
        assert_bits(op.T @ v, orc.ops.spmv_t(B, v), "B' v")
    # all-negative-zero input: every fold stays +0, like SparseArrays'
    z = np.full(B.shape[1], -TF(0.0))
    assert_bits(op @ z, orc.ops.spmv(B, z), "B (-0)")
    zt = np.full(B.shape[0], -TF(0.0))
    assert_bits(op.T @ zt, orc.ops.spmv_t(B, zt), "B' (-0)")
    with pytest.raises(ValueError):
        op @ np.zeros(W.shape[1], dtype=TF)


# ---------------------------------------------------------------------------------------------
# wide CDS kernels (nd > 32)
# ---------------------------------------------------------------------------------------------
def wide_cds(N, nd, TF, seed, symmetric=False):
    """nd distinct offsets in Q_offsets-like order (0 first, then a random order: NOT ascending), random values on the
    in-range part of every diagonal, zeros outside (mat2CDS padding)."""
    rng = np.random.default_rng(seed)
    pairs = None
    if symmetric:
        k = (nd - 1) // 2
        pos = rng.choice(np.arange(1, N // 3), size=k + (nd - 1 - 2 * k), replace=False)
        pairs = pos[:k]
        offs = np.concatenate([[0], pos[:k], -pos[:k], pos[k:]])       # an extra (even nd) diagonal is all zeros
    else:
        offs = np.concatenate([[0], rng.choice(np.concatenate([np.arange(-N // 2, 0), np.arange(1, N // 2)]),
                                               size=nd - 1, replace=False)])
    offs = offs.astype(np.int64)
    offs[1:] = rng.permutation(offs[1:])
    assert not np.all(np.diff(offs) > 0)
    R = np.zeros((N, nd), dtype=TF, order="F")
    r = np.arange(N)
    for j, o in enumerate(offs):
        ok = (r + o >= 0) & (r + o < N)
        R[ok, j] = rng.standard_normal(int(ok.sum())).astype(TF)
    if symmetric:
        R[:] = 0
        A = sp.lil_matrix((N, N), dtype=np.float64)
        for o in pairs:
            vals = 0.1 * rng.standard_normal(N - o)
            A.setdiag(vals, int(o))
            A.setdiag(vals, -int(o))
        A = sp.csr_matrix(A)
        A.setdiag(np.asarray(abs(A).sum(axis=1)).ravel() + 1.0)
        A = sp.coo_matrix(A)
        col = {int(o): j for j, o in enumerate(offs)}
        for i, c, v in zip(A.row, A.col, A.data):
            R[i, col[int(c - i)]] = TF(v)
    return R, offs


@pytest.mark.parametrize("TF", [np.float32, np.float64])
@pytest.mark.parametrize("nd", [33, 125, 400])
def test_cds_spmv_wide_bit_exact(sip, orc, TF, nd):
    N = 3001 if nd < 400 else 1203            # not a multiple of the vector width: the scalar tail runs too
    R, off = wide_cds(N, nd, TF, seed=nd)
    x = np.random.default_rng(nd + 1).standard_normal(N).astype(TF)
    x[::13] = -TF(0.0)
    want = orc.ops.CDS_MVp(N, nd, R, off, x, np.zeros(N, dtype=TF))
    got = sip.CDS_MVp(N, nd, R, off, x, np.zeros(N, dtype=TF))
    assert_bits(got, want, "CDS_MVp")
    native = R.astype(np.float64)
    ref = np.zeros(N)
    for j, o in enumerate(off):
        r0, r1 = max(0, -o), min(N, N - o)
        ref[r0:r1] += native[r0:r1, j] * x[r0 + o:r1 + o].astype(np.float64)
    assert np.allclose(got, ref, rtol=0, atol=nd * 4 * np.finfo(TF).eps * np.abs(native).max() * np.abs(x).max())


def test_cds_width_limits(sip):
    N, TF = 2000, np.float64
    R, off = wide_cds(N, 1000, TF, seed=1)
    with pytest.raises(Exception):
        sip.CDS_MVp(N, 1000, R, off, np.ones(N), np.zeros(N))
    R9, off9 = np.asfortranarray(R[:, :999]), off[:999]
    got = sip.CDS_MVp(N, 999, R9, off9, np.ones(N), np.zeros(N))
    import oracle.operators as oops
    assert_bits(got, oops.CDS_MVp(N, 999, R9, off9, np.ones(N), np.zeros(N)))


@pytest.mark.parametrize("TF", [np.float32, np.float64])
@pytest.mark.parametrize("nd", [33, 125, 400])
def test_cds_scaled_add_wide(sip, orc, TF, nd):
    N = 2003
    RB, oB = wide_cds(N, nd, TF, seed=2 * nd)
    # A holds B's diagonals in another order plus five more
    rng = np.random.default_rng(nd)
    extra = np.setdiff1d(np.arange(-N + 1, N), oB)[rng.choice(2 * N - 1 - nd, 5, replace=False)]
    oA = rng.permutation(np.concatenate([oB, extra])).astype(np.int64)
    RA = np.asfortranarray(rng.standard_normal((N, oA.size)).astype(TF))
    want = RA.copy(order="F")
    orc.ops.CDS_scaled_add(want, RB, oA, oB, 0.375)
    got = sip.CDS_scaled_add(RA.copy(order="F"), RB, oA, oB, 0.375)
    assert_bits(got.ravel(order="F"), want.ravel(order="F"), "CDS_scaled_add")
    with pytest.raises(Exception):
        sip.CDS_scaled_add(RB.copy(order="F"), RA, oB, oA, 1.0)


@pytest.mark.parametrize("TF", [np.float32, np.float64])
@pytest.mark.parametrize("nd", [33, 125, 400])
def test_cg_wide_matches_oracle(sip, orc, TF, nd):
    N = 2501
    R, off = wide_cds(N, nd, TF, seed=3 * nd, symmetric=True)
    rng = np.random.default_rng(nd)
    xt = rng.standard_normal(N).astype(TF)
    b = orc.ops.Ax_CDS(xt, R, off)
    tol = 1e-5 if TF == np.float32 else 1e-10
    x, flag, relres, it = sip.cg(R, off, b, tol=tol, maxIter=1000)
    assert flag == 0 and np.linalg.norm(orc.ops.Ax_CDS(x, R, off) - b) / np.linalg.norm(b) <= 2 * tol
    xo, fo, ro, ito = orc.parsdmm.cg(lambda v: orc.ops.Ax_CDS(v, R, off), b.copy(), TF(tol), 1000, np.zeros(N, dtype=TF))
    assert it == ito and relerr(x, xo) < TOL[TF]
    assert abs(float(relres) - float(ro)) <= 1e-2 * float(ro) + 1e-30
    x2, flag2, relres2, it2 = sip.cg(R, off, b, tol=tol, maxIter=1000, x=xt.copy())
    assert it2 == 1 and flag2 == 0 and np.array_equal(x2, xt) and relres2 == 0
    x3, flag3, relres3, it3 = sip.cg(R, off, np.zeros(N, dtype=TF), tol=tol, maxIter=10, x=xt.copy())
    assert flag3 == -9 and it3 == 0 and not x3.any()


# ---------------------------------------------------------------------------------------------
# problems with custom operators in Minkowski sets
# ---------------------------------------------------------------------------------------------
def build_minkowski_custom(api, n, TF, d, W1=None, W2=None, Ws=None, options=None):
    """config 5 (pr.build_minkowski) with custom-operator sets: W1 (bounds) in c1, W2 (bounds) in c2, Ws (an l1 ball)
    in the sum component."""
    m = pr.synthetic_model(n, TF)
    cg = api.compgrid(d, n)
    lo = np.full(n, 1500.0, dtype=TF)
    hi = np.full(n, 4500.0, dtype=TF)
    hi[:, : max(n[1] // 8, 1)] = 1500.0
    mode = ("matrix", "")
    c1 = [api.set_definitions("bounds", "identity", lo.ravel(order="F"), hi.ravel(order="F"), mode),
          api.set_definitions("bounds", "D_z", 0.0, 1e6, mode)]
    c2 = [api.set_definitions("bounds", "identity", -1500.0, 1500.0, mode),
          api.set_definitions("l1", "TV", 0.0, 0.15 * pr.tv_l1(n, d, TF, m), mode)]
    cs = [api.set_definitions("bounds", "identity", 1500.0, 4500.0, mode)]
    mf = m.ravel(order="F").astype(np.float64)
    custom = []
    if W1 is not None:
        c1.insert(1, api.set_definitions("bounds", "identity", -20.0, 20.0, mode, (W1.copy(), False)))
        custom.append((0, 1))
    if W2 is not None:
        c2.insert(1, api.set_definitions("bounds", "identity", -15.0, 15.0, mode, (W2.copy(), False)))
        custom.append((1, 1))
    if Ws is not None:
        tau = 0.5 * float(np.abs(Ws.astype(np.float64) @ mf).sum())
        cs.append(api.set_definitions("l1", "identity", 0.0, tau, mode, (Ws.copy(), False)))
        custom.append((2, len(cs) - 1))
    P1, T1, S1 = api.setup_constraints(c1, cg, TF)
    P2, T2, S2 = api.setup_constraints(c2, cg, TF)
    P3, T3, S3 = api.setup_constraints(cs, cg, TF)
    for comp, i in custom:
        S = (S1, S2, S3)[comp]
        S.AtA_diag[i], S.dense[i], S.banded[i] = False, False, True
    opt = options if options is not None else api.PARSDMM_options()
    opt.FL = TF
    opt.Minkowski = True
    opt.feas_tol, opt.obj_tol, opt.evol_rel_tol = 1e-3, 1e-3, 1e-5
    TD_OP, set_Prop, AtA, l, y = api.PARSDMM_precompute_distribute_Minkowski(T1, T2, T3, S1, S2, S3, cg, opt)
    return dict(cg=cg, opt=opt, P_sub=list(P1) + list(P2) + list(P3), TD_OP=TD_OP, set_Prop=set_Prop, AtA=AtA, l=l,
                y=y, m=m, minkowski=True)


def solve_both(sip, orc, ob, sb, TF, maxit_f64=300):
    for o in (ob["opt"], sb["opt"]):
        if TF == np.float32:
            o.maxit, o.feas_tol, o.obj_tol, o.evol_rel_tol = 40, 1e-12, 1e-12, 1e-14
        else:
            o.maxit = maxit_f64
    m = ob["m"].ravel(order="F") if ob["m"].ndim > 1 else ob["m"]
    xo, lo, ll, yy = orc.PARSDMM(m.copy(), ob["AtA"], ob["TD_OP"], ob["set_Prop"], ob["P_sub"], ob["cg"], ob["opt"])
    xs, ls, l2, y2 = sip.PARSDMM(m.copy(), sb["AtA"], sb["TD_OP"], sb["set_Prop"], sb["P_sub"], sb["cg"], sb["opt"])
    return (xo, lo, ll, yy, ob), (xs, ls, l2, y2, sb)


@pytest.mark.parametrize("TF", [np.float32, np.float64])
@pytest.mark.parametrize("it,do_adapt", [(1, False), (3, True), (10, False)])
def test_iteration_minkowski_custom(sip, orc, TF, it, do_adapt):
    """One iteration through sipb_iter_probe with custom operators in c1 ([A 0]) and in the sum set ([A A]): rhs, s, y,
    l and the snapshots bit for bit against the oracle's formulas on the hcat matrices."""
    n, d = (29, 11), (25.0, 6.0)
    W1 = weighted_gradient(orc, n, d, TF, seed=2)
    Ws = weighted_stencil(n, TF, STENCIL5, seed=3)
    ob = build_minkowski_custom(orc, n, TF, d, W1=W1, Ws=Ws)
    sb = build_minkowski_custom(sip, n, TF, d, W1=W1, Ws=Ws)
    dev = gi.device_handle(sip, sb, TF)
    assert dev.q_offsets.size > 32                            # Q of the [A A] 5-point stencil: the wide kernels
    st = gi.draw_state(ob, TF, ob["m"].ravel(order="F").astype(TF), seed=zlib.crc32(repr(("mc", it)).encode()))
    out = gi.run_probe(sip, dev, TF, st, it, do_adapt)
    L = gi.check_launches(sb, out, it)
    assert not out["fuse_stop"] and L["stop_reduce"] == 1
    gi.check_iteration(orc, ob, sb, TF, st, out, it, do_adapt)


@pytest.mark.parametrize("TF", [np.float64, np.float32])
def test_parsdmm_minkowski_custom_each_component(sip, orc, TF):
    """A 32 x 28 Minkowski problem with a custom operator in c1, in c2 and in the sum set."""
    n, d = (32, 28), (25.0, 6.0)
    W1 = weighted_gradient(orc, n, d, TF, seed=2)
    W2 = weighted_gradient(orc, n, d, TF, seed=4)
    Ws = weighted_gradient(orc, n, d, TF, seed=6)
    ob = build_minkowski_custom(orc, n, TF, d, W1=W1, W2=W2, Ws=Ws)
    sb = build_minkowski_custom(sip, n, TF, d, W1=W1, W2=W2, Ws=Ws)
    o, s = solve_both(sip, orc, ob, sb, TF)
    assert sb["AtA"]._device.q_form == "arrays"
    check_parity(o, s, TF)
    xs, ls = s[0], s[1]
    assert xs.size == 2 * ob["m"].size
    if TF == np.float64:
        assert len(ls.obj) < 300


@pytest.mark.parametrize("TF", [np.float64, np.float32])
def test_parsdmm_minkowski_wide_q(sip, orc, TF):
    """A 5-point custom stencil in the sum set: Q has more than 32 diagonals (wide SpMV, CG prologue and Q update)."""
    n, d = (32, 28), (25.0, 6.0)
    Ws = weighted_stencil(n, TF, STENCIL5, seed=8)
    ob = build_minkowski_custom(orc, n, TF, d, Ws=Ws)
    sb = build_minkowski_custom(sip, n, TF, d, Ws=Ws)
    o, s = solve_both(sip, orc, ob, sb, TF)
    assert sb["AtA"]._device.q_offsets.size > 32
    check_parity(o, s, TF)


@pytest.mark.parametrize("TF", [np.float64, np.float32])
def test_parsdmm_3d_27_point_custom(sip, orc, TF):
    """A plain 3-D problem: a 27-point weighted custom operator (125 A'A diagonals) next to TV-l1 and bounds."""
    n, d = (14, 12, 10), (10.0, 10.0, 10.0)
    m = pr.synthetic_model(n, TF).ravel(order="F")
    W = weighted_stencil(n, TF, STENCIL27, seed=9)
    tau_w = 0.4 * float(np.abs(W.astype(np.float64) @ m.astype(np.float64)).sum())

    def build(api):
        cg = api.compgrid(d, n)
        sets = [api.set_definitions("bounds", "identity", 1500.0, 4500.0, ("matrix", "")),
                api.set_definitions("l1", "identity", 0.0, tau_w, ("matrix", ""), (W.copy(), False)),
                api.set_definitions("l1", "TV", 0.0, 0.5 * pr.tv_l1(n, d, TF, m.reshape(n, order="F")), ("matrix", ""))]
        opt = api.PARSDMM_options()
        opt.FL = TF
        P_sub, TD_OP, set_Prop = api.setup_constraints(sets, cg, TF)
        set_Prop.AtA_diag[1], set_Prop.dense[1], set_Prop.banded[1] = False, False, True
        TD_OP, AtA, l, y = api.PARSDMM_precompute_distribute(TD_OP, set_Prop, cg, opt)
        return dict(cg=cg, opt=opt, P_sub=P_sub, TD_OP=TD_OP, set_Prop=set_Prop, AtA=AtA, m=m)

    ob, sb = build(orc), build(sip)
    assert sb["set_Prop"].AtA_offsets[1].size == 125
    o, s = solve_both(sip, orc, ob, sb, TF)
    assert sb["AtA"]._device.q_offsets.size == 125
    check_parity(o, s, TF)
