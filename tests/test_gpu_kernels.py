"""Kernel-by-kernel tests of the two single-GPU hot paths against exact references.

1. The tiled SpMV of the CG (spmv_tile.cuh) in the stencil-class form the solver runs (sipb_tile_probe): y = Q x and
   dot(x, y) (MODE 1), the CG prologue r = b - Q x, p = r, x_old = x, dot(b,b), dot(r,r) (MODE 2), against CDS_MVp
   (CDS_MVp.jl:9-28) on the class table expanded to CDS arrays.  Every grid asserts, from the plan the library reports,
   the regime it is there for.
2. The cardinality projection as the PARSDMM loop runs it (sipb_select_probe): speculative select levels in pass 1 of
   the y/l update, the radix search, the per-chunk tie counts, the chunk on the quota boundary settled in place and the
   surplus ties zeroed by pass 2, against a stable argsort (project_cardinality!.jl:3-21), signs of zeros included.
3. Whole solves under the switches that select alternate single-GPU paths (SIPB_SEL_SPEC, SIPB_L1_SKIPV): bit-identical."""
import copy
import ctypes as C
import math
import os
import sys
import zlib

import numpy as np
import pytest

import problems as pr

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
import select_model  # noqa: E402

pytestmark = pytest.mark.gpu

F32_STAGE_BUDGET = 226 * 1024 // 2 - 3 * 1024       # plan_tile: shared memory per CTA beside the static part


@pytest.fixture(scope="module")
def lib(sip):
    return sip._lib


@pytest.fixture(scope="module")
def orc():
    return pr.OracleAPI()


# ---------------------------------------------------------------------------------------------
# tiled SpMV
# ---------------------------------------------------------------------------------------------
ORDERS = {"q": lambda n0, P: [0, -P, -n0, -1, 1, n0, P], "z": lambda n0, P: [0, -P, P, -1, 1, -n0, n0],
          "sorted": lambda n0, P: [-P, -n0, -1, 0, 1, n0, P]}


def row_classes(n):
    """Stencil class of every row: (c(k)*3 + c(j))*3 + c(i), c = 0 / 1 / 2 on the first / an interior / the last index."""
    def c(m):
        v = np.ones(m, dtype=np.int64)
        v[0], v[-1] = 0, 2
        return v
    n0, n1, n2 = n
    return ((c(n2)[:, None, None] * 3 + c(n1)[None, :, None]) * 3 + c(n0)[None, None, :]).ravel()


def tile_probe(lib, TF, n, off, x, tab=None, R=None, b=None, mode=1, tiled=1):
    N = int(np.prod(n))
    out = {k: np.empty(N, dtype=TF) for k in ("y", "r", "p", "x_old")}
    sums = np.zeros(2)
    geom = np.zeros(8, dtype=np.int32)
    ptr = lambda a: None if a is None else a.ctypes.data      # noqa: E731
    rc = lib.load().sipb_tile_probe(
        lib.ctx(), lib.dtype_code(TF), (C.c_int64 * 3)(*n), off.size, off.ctypes.data_as(C.POINTER(C.c_int64)), ptr(tab),
        ptr(R), x.ctypes.data, ptr(b), mode, tiled, out["y"].ctypes.data, out["r"].ctypes.data, out["p"].ctypes.data,
        out["x_old"].ctypes.data, sums.ctypes.data_as(C.POINTER(C.c_double)), geom.ctypes.data_as(C.POINTER(C.c_int)))
    lib.check(rc)
    out["sums"] = sums
    out["geom"] = dict(zip(("ok", "TJ", "JT", "KC", "NS", "grid", "gpl", "LPP"), (int(v) for v in geom)))
    return out


def assert_sum(got, a, b):
    """|s - exact| <= N 2^-52 sum|a_i b_i|: holds for any partition of a Float64 sum of the products."""
    prod = a.astype(np.float64) * b.astype(np.float64)
    exact = math.fsum(prod)
    assert abs(got - exact) <= a.size * 2.0 ** -52 * float(np.abs(prod).sum()), (got, exact)


# (name, Float32 grid, Float64 grid): the regime each grid exists for is asserted in check_regime
GRIDS = [("one_group_per_line", (4, 9, 5), (2, 9, 5)),
         ("no_interior_line_or_plane", (8, 2, 2), (4, 2, 2)),
         ("uneven_z_chunks", (16, 37, 11), (8, 37, 11)),
         ("short_last_tile", (32, 40, 37), (16, 40, 37)),
         ("multi_unit_ctas", (1024, 1200, 3), (512, 600, 3)),
         ("widest_lines", (1024, 1100, 3), (512, 64, 6)),
         ("line_too_wide", (1028, 8, 3), (514, 8, 3)),
         ("bench_size", (200, 200, 200), (128, 128, 128))]


def check_regime(name, TF, n, g):
    n0, n1, n2 = n
    s = np.dtype(TF).itemsize
    if name == "line_too_wide":
        assert g["ok"] == 0 and n0 // (16 // s) == 257
        return
    assert g["ok"] == 1
    # the ring depth follows the planner's formula for the chosen tile height
    assert g["NS"] == min(5, (F32_STAGE_BUDGET - 27 * 8 * s) // ((g["TJ"] + 2) * n0 * s)), g
    assert g["JT"] == -(-n1 // g["TJ"])
    if name == "one_group_per_line":
        assert g["gpl"] == 1
    elif name == "no_interior_line_or_plane":
        assert n1 == 2 and n2 == 2
    elif name == "uneven_z_chunks":
        assert g["KC"] > 1 and n2 % g["KC"] != 0
    elif name == "short_last_tile":
        assert n1 % g["TJ"] != 0 and g["KC"] > 1 and n2 % g["KC"] != 0
    elif name == "multi_unit_ctas":
        assert g["gpl"] == 256 and g["JT"] * g["KC"] > g["grid"], g
    elif name == "widest_lines":
        assert g["gpl"] == 256 and g["LPP"] == 1
        if TF == np.float32:
            assert g["NS"] == 4, g        # (TJ + 2) lines of 4 KB: the fewest stages any tiled grid gets
    elif name == "bench_size":
        assert g["grid"] > 128


def make_table(rng, TF, nd, single_diag=None):
    """[27][nd]: a distinct random value for every class and diagonal, or (single_diag = j) classes that agree on every
    diagonal except j."""
    if single_diag is None:
        return rng.uniform(0.5, 2.0, (27, nd)).astype(TF)
    tab = np.repeat(rng.uniform(0.5, 2.0, (1, nd)), 27, axis=0)
    tab[:, single_diag] = rng.uniform(0.5, 2.0, 27)
    return tab.astype(TF)


def tile_cases():
    out = []
    for TF in (np.float32, np.float64):
        for name, g32, g64 in GRIDS:
            n = g32 if TF == np.float32 else g64
            small = int(np.prod(n)) < 2_000_000
            for order in (("q", "z", "sorted") if small else ("q",)):
                for table in (("random", "single_diag") if small else ("random",)):
                    out.append(pytest.param(TF, name, n, order, table, id="%s-%s-%s-%s" % (np.dtype(TF).name, name, order, table)))
    return out


@pytest.mark.parametrize("TF,name,n,order,table", tile_cases())
def test_tiled_spmv_class_form(lib, orc, TF, name, n, order, table):
    n0, n1, n2 = n
    N, P = n0 * n1 * n2, n0 * n1
    off = np.array(ORDERS[order](n0, P), dtype=np.int64)
    nd = off.size
    rng = np.random.default_rng(zlib.crc32(("%s/%s/%s/%s" % (name, order, table, np.dtype(TF).name)).encode()))
    # single_diag: the +1 diagonal, where the first / middle / last element of a 16-byte group take different registers
    tab = make_table(rng, TF, nd, single_diag=None if table == "random" else int(np.nonzero(off == 1)[0][0]))
    R = np.asfortranarray(tab[row_classes(n)])                  # the same matrix as CDS arrays (wrapping entries included)
    x = rng.standard_normal(N).astype(TF)
    b = rng.standard_normal(N).astype(TF)
    want = orc.ops.CDS_MVp(N, nd, R, off, x, np.zeros(N, dtype=TF))

    generic = tile_probe(lib, TF, n, off, x, tab=tab, tiled=0)
    generic_arr = tile_probe(lib, TF, n, off, x, R=R, tiled=0)
    check_regime(name, TF, n, generic["geom"])
    assert np.array_equal(generic["y"], want) and np.array_equal(generic_arr["y"], want)
    runs = [generic, generic_arr]
    if generic["geom"]["ok"]:
        cls = tile_probe(lib, TF, n, off, x, tab=tab)
        arr = tile_probe(lib, TF, n, off, x, R=R)
        assert cls["geom"] == arr["geom"] == generic["geom"]
        assert np.array_equal(cls["y"], want) and np.array_equal(arr["y"], want)
        runs += [cls, arr]
    else:
        with pytest.raises(lib.SipbError):
            tile_probe(lib, TF, n, off, x, tab=tab)
    for run in runs:
        assert_sum(run["sums"][0], x, want)

    # MODE 2, the CG prologue: r = b - Ax_CDS(x) as argmin_x / cg compute it, p = r, x_old = x
    r_want = b - orc.ops.Ax_CDS(x, R, off)
    for tiled in ((0, 1) if generic["geom"]["ok"] else (0,)):
        for form in (("tab", "R") if not tiled else ("tab",)):
            kw = {form: tab if form == "tab" else R}
            o = tile_probe(lib, TF, n, off, x, b=b, mode=2, tiled=tiled, **kw)
            assert np.array_equal(o["r"], r_want) and np.array_equal(o["p"], r_want) and np.array_equal(o["x_old"], x)
            assert_sum(o["sums"][0], b, b)
            assert_sum(o["sums"][1], r_want, r_want)


def test_tiled_cg_prologue_has_no_array_body(lib):
    n = (8, 6, 5)
    off = np.array(ORDERS["q"](8, 48), dtype=np.int64)
    R = np.ones((240, 7), dtype=np.float32, order="F")
    x = np.ones(240, dtype=np.float32)
    with pytest.raises(lib.SipbError) as e:
        tile_probe(lib, np.float32, n, off, x, R=R, b=x, mode=2, tiled=1)
    assert e.value.code == lib.SIPB_E_UNSUPPORTED


# ---------------------------------------------------------------------------------------------
# cardinality select
# ---------------------------------------------------------------------------------------------
UINT = {np.float32: np.uint32, np.float64: np.uint64}


def mag_keys(v):
    return (v.view(UINT[v.dtype.type]) & np.array(np.iinfo(UINT[v.dtype.type]).max >> 1, dtype=UINT[v.dtype.type])).astype(np.uint64)


def select_probe(lib, v, k, guess, path):
    y = np.empty_like(v)
    st = np.zeros(8, dtype=np.int64)
    lib.check(lib.load().sipb_select_probe(lib.ctx(), lib.dtype_code(v.dtype), v.size, v.ctypes.data, int(k), int(guess),
                                           path, y.ctypes.data, st.ctypes.data_as(C.POINTER(C.c_int64))))
    return y, dict(zip(("key", "quota", "count_eq", "need_ties", "levels", "table_valid", "chunk", "cross"),
                       (int(s) for s in st)))


def chunk_of(lib, TF, M):
    return select_probe(lib, np.zeros(M, dtype=TF), 0, 0, 2)[1]["chunk"]


def guesses(keys, thr, KB):
    top = KB - 11
    hi, lo = int(keys.max()), int(keys.min())
    return {"exact": thr, "zero": 0, "all_ones": (1 << KB) - 1,
            "second_digit": thr ^ (1 << (top - 1)),           # same top digit, another second digit
            "low_bits": thr ^ 1,                              # the top 22 bits agree
            "above_all": min(((hi >> top) + 1) << top, (1 << KB) - 1),
            "below_all": (((lo >> top) - 1) << top) if lo >> top else 0}


def check_select(lib, orc, v, k):
    TF = v.dtype.type
    KB = 8 * v.dtype.itemsize
    M = v.size
    keys = mag_keys(v)
    # pass 1 of the y/l update forms s = 0 + A x (update_y_l.jl:43 as SparseArrays computes it): a -0.0 entry enters the
    # loop's select as +0.0; sipb_project takes the vector as it is
    want_proj = orc.proj.project_cardinality(v.copy(), k)
    want_loop = orc.proj.project_cardinality(v + TF(0), k)
    if 0 < k < M:
        srt = np.sort(keys)[::-1]
        thr = int(srt[k - 1])
        quota = k - int(np.count_nonzero(keys > thr))
        count_eq = int(np.count_nonzero(keys == thr))
        exp = dict(key=thr, quota=quota, count_eq=count_eq, need_ties=int(count_eq > quota))
    else:
        thr = 0
        exp = dict(key=0, quota=0, count_eq=0, need_ties=0)
    ys = []
    for gname, guess in guesses(keys, thr, KB).items():
        for path in (1, 0, 2):
            y, st = select_probe(lib, v, k, guess, path)
            ctx = (M, k, gname, path, st)
            want = want_proj if path == 2 else want_loop
            assert np.array_equal(y, want), ctx
            assert np.array_equal(np.signbit(y), np.signbit(want)), ctx
            assert {q: st[q] for q in exp} == exp, ctx
            if 0 < k < M:
                levels = select_model.select(keys, k, KB, guess, spec=path == 1)[1]
            else:
                levels = 0
            assert st["levels"] == levels, ctx
            assert st["table_valid"] == int(levels > 0), ctx
            c = st["chunk"]
            cross = -1
            if path != 2 and exp["need_ties"] and exp["quota"] > 0:
                idx = np.nonzero(keys == thr)[0]
                a, b = idx[exp["quota"] - 1] // c, idx[exp["quota"]] // c
                cross = int(a) if a == b else -1
            assert st["cross"] == cross, ctx
            if path != 2:
                ys.append(y)
            if gname != "exact":
                break                  # the guess matters to the speculative path only
    for y in ys[1:]:
        assert np.array_equal(y.view(UINT[TF]), ys[0].view(UINT[TF]))
    return exp, st


def tie_vector(TF, M, ties, n_above, rng):
    """Small background values, `n_above` entries larger than the tie magnitude 3.0 (at positions outside `ties`), and
    +-3.0 at the sorted positions `ties`."""
    v = (rng.uniform(0.1, 1.0, M) * rng.choice([-1, 1], M)).astype(TF)
    free = np.setdiff1d(np.arange(M), ties)
    v[rng.choice(free, n_above, replace=False)] = TF(7.0)
    v[ties] = (TF(3.0) * rng.choice([-1, 1], len(ties))).astype(TF)
    return v


@pytest.mark.parametrize("TF", [np.float32, np.float64])
def test_select_sizes_and_edges(lib, orc, TF):
    rng = np.random.default_rng(21)
    c = chunk_of(lib, TF, 1024)
    assert c % 256 == 0
    sizes = [1, 7, 255, 256, 257, 1001, 5 * c - 1, 5 * c + 1]
    for M in sizes:
        if M > 7:
            assert chunk_of(lib, TF, M) == c
        v = rng.standard_normal(M).astype(TF)
        v[rng.integers(0, M, M // 4)] = v[0]                       # ties with the first entry
        for k in sorted({0, 1, M // 3, M - 1, M, M + 1}):
            check_select(lib, orc, v.copy(), k)
    assert (5 * c - 1) % c == c - 1 and (5 * c + 1) % c == 1


@pytest.mark.parametrize("TF", [np.float32, np.float64])
def test_select_all_equal(lib, orc, TF):
    v = np.full(1000, TF(1.5))
    v[::3] = -v[::3]
    for k in (1, 255, 256, 333, 999):
        exp, st = check_select(lib, orc, v.copy(), k)
        assert exp["count_eq"] == 1000 and exp["quota"] == k


@pytest.mark.parametrize("TF", [np.float32, np.float64])
def test_select_ties_across_chunks(lib, orc, TF):
    """Ties of one magnitude spread over many chunks; the quota boundary inside a chunk, exactly on a chunk boundary, in
    the first chunk and in the partial last chunk."""
    rng = np.random.default_rng(22)
    M = 4000
    c = chunk_of(lib, TF, M)
    ties = np.arange(100, 3990, 3)
    n_above = 50
    v = tie_vector(TF, M, ties, n_above, rng)
    last = (M - 1) // c
    cases = {
        "inside_a_chunk": int(np.searchsorted(ties, 2 * c + 40)),
        "on_a_chunk_boundary": int(np.searchsorted(ties, 3 * c)),
        "first_chunk": int(np.searchsorted(ties, c // 2)),
        "partial_last_chunk": int(np.searchsorted(ties, last * c + (M - last * c) // 2)),
    }
    assert M % c != 0
    for where, q in cases.items():
        exp, st = check_select(lib, orc, v.copy(), n_above + q)
        assert exp["quota"] == q and exp["need_ties"] == 1
        boundary = ties[q - 1] // c != ties[q] // c
        assert (st["cross"] == -1) == boundary, where
        assert boundary == (where == "on_a_chunk_boundary"), where
        if where == "first_chunk":
            assert st["cross"] == 0
        if where == "partial_last_chunk":
            assert st["cross"] == last


@pytest.mark.parametrize("TF", [np.float32, np.float64])
def test_select_signed_zeros_subnormals_inf(lib, orc, TF):
    """+-0, subnormals, +-inf; k above the number of non-zeros: the threshold magnitude is 0 and the zeros past the
    quota come back as +0.0 (x[sort_ind[k+1:end]] .= 0), the ones inside it keep their sign (sipb_project)."""
    rng = np.random.default_rng(23)
    M = 3001
    tiny = np.finfo(TF).smallest_subnormal
    v = np.zeros(M, dtype=TF)
    v[rng.random(M) < 0.5] = TF(-0.0)
    nz = rng.choice(M, 900, replace=False)
    v[nz[:300]] = (rng.integers(1, 50, 300) * tiny * rng.choice([-1, 1], 300)).astype(TF)
    v[nz[300:600]] = rng.standard_normal(300).astype(TF)
    v[nz[600:603]] = [np.inf, -np.inf, -np.inf]
    nnz = int(np.count_nonzero(v))
    for k in (2, 3, 100, 450, nnz - 1, nnz, nnz + 1, nnz + 700, M - 1):
        exp, st = check_select(lib, orc, v.copy(), k)
        if k > nnz:
            assert exp["key"] == 0 and exp["need_ties"] == 1


def test_select_large_f32(lib, orc):
    rng = np.random.default_rng(24)
    M = 30_000_001
    v = rng.standard_normal(M).astype(np.float32)
    v[rng.integers(0, M, M // 50)] = np.float32(2.5)                # a tie class around the threshold
    k = int(np.count_nonzero(np.abs(v) > 2.5)) + 150_000
    exp, st = check_select(lib, orc, v, k)
    assert exp["need_ties"] == 1 and st["chunk"] > 256


# ---------------------------------------------------------------------------------------------
# whole solves under the switches
# ---------------------------------------------------------------------------------------------
def solves_with_env(sip, var, value, specs):
    """Every spec solved in a fresh context created with var=value (the context reads the switch)."""
    import gc
    L = sip._lib
    os.environ[var] = value
    try:
        h = C.c_void_p()
        L.check(L.load().sipb_ctx_create(0, C.byref(h)))
    finally:
        os.environ.pop(var, None)
    old = L._ctx.get(0)
    L._ctx[0] = h
    try:
        res = []
        for spec, maxit in specs:
            opt = sip.PARSDMM_options()
            opt.maxit = maxit
            b = pr.build(sip, copy.deepcopy(spec), opt)
            res.append(sip.PARSDMM(spec["m"].copy(), b["AtA"], b["TD_OP"], b["set_Prop"], b["P_sub"], b["cg"], b["opt"]))
            del b
        return res
    finally:
        L._ctx[0] = old
        gc.collect()
        L.load().sipb_ctx_destroy(h)


LOG_ARRAYS = ("set_feasibility", "r_dual", "r_pri", "r_dual_total", "r_pri_total", "obj", "evol_x", "rho", "gamma", "cg_it",
              "cg_relres")


def assert_bit_identical(a, b):
    (xa, la, l_a, y_a), (xb, lb, l_b, y_b) = a, b
    assert np.array_equal(xa, xb)
    for name in LOG_ARRAYS:
        assert np.array_equal(np.asarray(getattr(la, name)), np.asarray(getattr(lb, name)), equal_nan=True), name
    assert len(l_a) == len(l_b) and all(np.array_equal(p, q) for p, q in zip(l_a + y_a, l_b + y_b))


def test_speculative_select_switch_bit_identical(sip):
    rng = np.random.default_rng(31)
    n2 = (96, 64)
    m2 = np.round(rng.standard_normal(int(np.prod(n2))) * 3).astype(np.float32)
    vec = dict(n=n2, d=(1.0, 1.0), TF=np.float32, m=m2, sets=[("cardinality", "identity", 0, int(0.3 * m2.size))], mode="matrix")
    specs = [(pr.spec_config3((24, 24, 24), np.float32), 60), (pr.spec_config3((24, 24, 24), np.float64), 60), (vec, 30)]
    on = solves_with_env(sip, "SIPB_SEL_SPEC", "1", specs)
    off = solves_with_env(sip, "SIPB_SEL_SPEC", "0", specs)
    for a, b in zip(on, off):
        assert_bit_identical(a, b)
    assert len(on[0][1].obj) > 20


def test_l1_skipv_switch_bit_identical(sip):
    """Config 2: the TV-l1 ball is active in the first iteration, inactive in the next few, active again later.  Pass 1
    stores v in every iteration (0), skips it after an inactive iteration (1, default) or never stores it (2)."""
    spec = pr.spec_config2((24, 20, 16), np.float32)
    runs = {v: solves_with_env(sip, "SIPB_L1_SKIPV", v, [(spec, 100)])[0] for v in ("0", "1", "2")}
    assert_bit_identical(runs["0"], runs["1"])
    assert_bit_identical(runs["0"], runs["2"])
    # pass 1 of the l1 set moves one v vector less in each iteration that skipped the store: with the default that is
    # every iteration after an inactive one, so some but not all iterations skip -> the ball was both active and inactive
    M = sum(int(np.prod([v - 1 if a == b else v for b, v in enumerate(spec["n"])])) for a in range(3))
    vbytes = M * 4
    iters = len(runs["0"][1].obj)
    pass1 = {k: r[1].timing["kernel_bytes"]["yl_update_pass1"] for k, r in runs.items()}
    assert round((pass1["0"] - pass1["2"]) / vbytes) == iters
    skipped = round((pass1["0"] - pass1["1"]) / vbytes)
    assert 1 <= skipped <= iters - 2, (skipped, iters)
