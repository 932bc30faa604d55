"""Custom (explicit sparse) operators inside generalized Minkowski sets and A'A wider than 32 diagonals — host side.

PARSDMM_precompute_distribute_Minkowski.jl:32-131 hcat's any operator into [A 0], [0 A] or [A A] and forms mat2CDS of
the 2N x 2N block matrices of A'A; PARSDMM_precompute_distribute.jl:44-55 forms mat2CDS(A'A) of any width up to the
999 rows of the offset table of PARSDMM_initialize.jl:217-221.  The device package must produce the same operators,
arrays, offsets and y / l sizes as the oracle restatement, bit for bit."""
import numpy as np
import pytest
import scipy.sparse as sp

import problems as pr


@pytest.fixture(scope="module")
def orc():
    return pr.OracleAPI()


def same_csc(A, B):
    A, B = sp.csc_matrix(A), sp.csc_matrix(B)
    A.sort_indices()
    B.sort_indices()
    return (A.shape == B.shape and A.dtype == B.dtype and np.array_equal(A.indptr, B.indptr) and
            np.array_equal(A.indices, B.indices) and np.array_equal(A.data, B.data))


def weighted_gradient(orc, n, d, TF, seed=5):
    """The discrete gradient with smoothly varying row weights: banded A'A whose values differ from row to row."""
    A, *_ = orc.get_TD_operator(orc.compgrid(d, n), "TV", TF)
    w = (1.0 + 0.5 * np.sin(np.arange(A.shape[0]) * 0.37 + seed)).astype(TF)
    W = sp.csc_matrix(sp.diags(w).astype(TF) @ A).astype(TF)
    W.sort_indices()
    return W


def weighted_stencil(n, TF, points, seed=7):
    """A stencil operator (one row per grid point, entries at the offsets `points` = (di, dj[, dk]) that stay inside the
    grid) with weights that vary from row to row, so A'A is banded but not constant per stencil class."""
    n3 = tuple(n) + (1,) * (3 - len(n))
    n0, n1, n2 = n3
    N = n0 * n1 * n2
    rng = np.random.default_rng(seed)
    idx = np.arange(N)
    i, j, k = idx % n0, (idx // n0) % n1, idx // (n0 * n1)
    rows, cols, vals = [], [], []
    for pt in points:
        di, dj, dk = tuple(pt) + (0,) * (3 - len(pt))
        ok = (i + di >= 0) & (i + di < n0) & (j + dj >= 0) & (j + dj < n1) & (k + dk >= 0) & (k + dk < n2)
        r = idx[ok]
        rows.append(r)
        cols.append(r + di + n0 * (dj + n1 * dk))
        vals.append(rng.uniform(0.5, 1.5, r.size) * (-1.0 if any(pt) else float(len(points) - 1)))
    W = sp.csc_matrix((np.concatenate(vals).astype(TF), (np.concatenate(rows), np.concatenate(cols))), shape=(N, N), dtype=TF)
    W.sort_indices()
    return W


STENCIL5 = [(0, 0), (-1, 0), (1, 0), (0, -1), (0, 1)]
STENCIL27 = [(di, dj, dk) for dk in (-1, 0, 1) for dj in (-1, 0, 1) for di in (-1, 0, 1)]


def minkowski_sets(api, n, d, TF, W, where):
    """config-5-like sets with the custom operator W (an l1 ball in its range) in c1, c2 or the sum component."""
    mode = ("matrix", "")
    custom = api.set_definitions("l1", "identity", 0.0, 1e3, mode, (W.copy(), False))
    c1 = [api.set_definitions("bounds", "identity", 1500.0, 4500.0, mode), api.set_definitions("bounds", "D_z", 0.0, 1e6, mode)]
    c2 = [api.set_definitions("bounds", "identity", -1500.0, 1500.0, mode), api.set_definitions("l1", "TV", 0.0, 1e4, mode)]
    cs = [api.set_definitions("bounds", "identity", 1500.0, 4500.0, mode)]
    {"c1": c1, "c2": c2, "sum": cs}[where].insert(1, custom)
    return c1, c2, cs


def minkowski_precompute(api, n, d, TF, W, where):
    cg = api.compgrid(d, n)
    c1, c2, cs = minkowski_sets(api, n, d, TF, W, where)
    P1, T1, S1 = api.setup_constraints(c1, cg, TF)
    P2, T2, S2 = api.setup_constraints(c2, cg, TF)
    P3, T3, S3 = api.setup_constraints(cs, cg, TF)
    S = {"c1": S1, "c2": S2, "sum": S3}[where]
    S.AtA_diag[1], S.dense[1], S.banded[1] = False, False, True
    opt = api.PARSDMM_options()
    opt.FL = TF
    opt.Minkowski = True
    return api.PARSDMM_precompute_distribute_Minkowski(T1, T2, T3, S1, S2, S3, cg, opt)


def as_csc(op):
    return op.tosparse() if hasattr(op, "tosparse") else op


@pytest.mark.parametrize("TF", [np.float32, np.float64])
@pytest.mark.parametrize("n,d", [((11, 9), (2.0, 3.0)), ((6, 5, 4), (2.0, 3.0, 1.5))])
@pytest.mark.parametrize("where", ["c1", "c2", "sum"])
def test_minkowski_precompute_with_custom_operator(sip, orc, TF, n, d, where):
    W = weighted_gradient(orc, n, d, TF)
    To, So, Ao, lo, yo = minkowski_precompute(orc, n, d, TF, W, where)
    Ts, Ss, As, ls, ys = minkowski_precompute(sip, n, d, TF, W, where)
    N = W.shape[1]
    assert len(To) == len(Ts) == len(As) == len(Ao)
    ic = {"c1": 1, "c2": 3, "sum": 5}[where]
    assert isinstance(Ts[ic], sip.SparseOperator)
    assert Ts[ic].shape == (W.shape[0], 2 * N) == To[ic].shape
    for a, b in zip(To, Ts):           # the hcat operators, including [A 0], [0 A], [A A] of the custom matrix
        assert same_csc(as_csc(b), a)
    for i, (a, b) in enumerate(zip(Ao, As)):
        a, b = np.asarray(a), np.asarray(b)
        assert a.shape[0] == 2 * N and a.dtype == b.dtype and np.array_equal(a, b), i
    for a, b in zip(So.AtA_offsets, Ss.AtA_offsets):
        assert np.array_equal(a, b)
    assert [v.size for v in ys] == [v.size for v in yo] and [v.size for v in ls] == [v.size for v in lo]
    assert ys[ic].size == W.shape[0]


def test_minkowski_custom_sum_widens_q(sip, orc):
    """A 2-D custom 5-point stencil in the sum component: its 13 A'A diagonals become 39 in the [A A] block matrix,
    so Q exceeds 32 diagonals; the host forms the arrays without a width limit below 999."""
    n, d, TF = (12, 10), (1.0, 1.0), np.float64
    W = weighted_stencil(n, TF, STENCIL5)
    Ts, Ss, As, ls, ys = minkowski_precompute(sip, n, d, TF, W, "sum")
    To, So, Ao, lo, yo = minkowski_precompute(orc, n, d, TF, W, "sum")
    assert sip.SparseOperator(W, n, d, TF).ata_cds()[1].size == 13
    assert Ss.AtA_offsets[5].size == 39 and np.array_equal(Ss.AtA_offsets[5], So.AtA_offsets[5])
    for a, b in zip(Ao, As):
        assert np.array_equal(np.asarray(a), np.asarray(b))
    import oracle.operators as oops
    q = oops.assemble_Q(Ao, So.AtA_offsets, np.ones(len(Ao)))[1]
    assert q.size > 32


@pytest.mark.parametrize("TF", [np.float32, np.float64])
def test_plain_precompute_27_point_stencil(sip, orc, TF):
    n, d = (7, 6, 5), (1.0, 1.0, 1.0)
    W = weighted_stencil(n, TF, STENCIL27)

    def run(api):
        cons = [api.set_definitions("l1", "identity", 0.0, 10.0, ("matrix", ""), (W.copy(), False)),
                api.set_definitions("l1", "TV", 0.0, 10.0, ("matrix", "")),
                api.set_definitions("bounds", "identity", 0.0, 1.0, ("matrix", ""))]
        opt = api.PARSDMM_options()
        P_sub, TD_OP, sP = api.setup_constraints(cons, api.compgrid(d, n), TF)
        sP.AtA_diag[0], sP.dense[0], sP.banded[0] = False, False, True
        TD_OP, AtA, l, y = api.PARSDMM_precompute_distribute(TD_OP, sP, api.compgrid(d, n), opt)
        return TD_OP, AtA, sP

    To, Ao, So = run(orc)
    Ts, As, Ss = run(sip)
    assert So.AtA_offsets[0].size == 125
    for a, b in zip(Ao, As):
        assert np.array_equal(np.asarray(a), np.asarray(b))
    for a, b in zip(So.AtA_offsets, Ss.AtA_offsets):
        assert np.array_equal(a, b)


def test_more_than_999_diagonals_rejected(sip):
    """A synthetic operator whose A'A has 1001 diagonals: outside the reference's offset table."""
    n, d, TF = (40, 40), (1.0, 1.0), np.float64
    N = n[0] * n[1]
    # one row per diagonal offset in {0, 1, ..., 500}: A'A has the offsets -500..500
    rows = np.concatenate([np.zeros(501, dtype=np.int64), np.ones(1, dtype=np.int64)])
    cols = np.concatenate([np.arange(501), [0]])
    W = sp.csc_matrix((np.ones(rows.size, dtype=TF), (rows, cols)), shape=(2, N), dtype=TF)
    cons = [sip.set_definitions("l1", "identity", 0.0, 10.0, ("matrix", ""), (W.copy(), False))]
    P_sub, TD_OP, sP = sip.setup_constraints(cons, sip.compgrid(d, n), TF)
    sP.AtA_diag[0], sP.dense[0], sP.banded[0] = False, False, True
    assert TD_OP[0].ata_cds()[1].size == 1001
    with pytest.raises(NotImplementedError):
        sip.PARSDMM_precompute_distribute(TD_OP, sP, sip.compgrid(d, n), sip.PARSDMM_options())
