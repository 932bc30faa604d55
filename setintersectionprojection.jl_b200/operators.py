"""Transform-domain operators and compressed-diagonal (CDS) index work — host side.

Mirrors get_discrete_Grad.jl, get_TD_operator.jl and mat2CDS.jl of the reference.  The reference
materialises every operator as a SparseMatrixCSC through Kronecker products; here an operator is a
light `TDOperator` descriptor (kind, grid, spacing) that

  * is applied on the GPU matrix-free (`A @ x`, `A.T @ v` go through the C ABI, no CPU fallback),
  * can be materialised as a SciPy CSC matrix with exactly the reference's structure and values
    (`tosparse()`), and
  * yields `A'A` directly in CDS form (`ata_cds`) without a sparse-sparse product — bit-identical to
    `mat2CDS(A'*A)` (mat2CDS.jl:7-32, PARSDMM_precompute_distribute.jl:44-55).
"""
from __future__ import annotations

import copy
import ctypes as C

import numpy as np
import scipy.sparse as sp

from . import _lib

_KIND_CODE = {"identity": _lib.OP_IDENTITY, "D_x": _lib.OP_DX, "D_y": _lib.OP_DY, "D_z": _lib.OP_DZ,
              "TV": _lib.OP_TV, "D2D": _lib.OP_TV, "D3D": _lib.OP_TV, "D_xz": _lib.OP_DXZ}
SPECIAL_OPERATORS = ("DFT", "DCT", "wavelet", "curvelet")     # setup_constraints.jl:54 (JOLI; rejected)


def _is3d(n) -> bool:
    return len(n) == 3 and n[2] > 1          # get_TD_operator.jl:26


class TDOperator:
    """Matrix-free banded transform-domain operator on a 2-D/3-D grid (column-major vec(model))."""

    def __init__(self, kind: str, n, h, TF, block_mode: int = _lib.BLOCK_PLAIN):
        if kind not in _KIND_CODE:
            raise ValueError("provided an unknown transform domain operator %r" % kind)
        self.kind = "TV" if kind in ("D2D", "D3D") else kind
        self.TF = np.dtype(TF).type
        self.ndim = 3 if _is3d(n) else 2
        self.n = tuple(int(v) for v in n[: self.ndim])
        self.h = tuple(self.TF(v) for v in h[: self.ndim])       # h = TF(comp_grid.d[i])
        self.block_mode = block_mode
        self.op_kind = _KIND_CODE[kind]
        if self.kind == "D_y" and self.ndim == 2:
            raise ValueError("D_y needs a 3-D grid")
        if self.kind == "D_xz" and self.ndim == 3:
            raise ValueError("D_xz is only defined for 2-D grids (get_TD_operator.jl:69-73)")
        self.npts = int(np.prod(self.n))
        self._sparse = None

    # -- structure ---------------------------------------------------------------------------------
    def _axes(self):
        """Storage axes differenced by each row block, in row order (TV = vcat(D_z[,D_y],D_x))."""
        last = self.ndim - 1
        return {"D_x": [0], "D_y": [1], "D_z": [last], "TV": list(range(last, -1, -1))}.get(self.kind, [])

    def _block_rows(self, axis: int) -> int:
        return int(np.prod([v - 1 if a == axis else v for a, v in enumerate(self.n)]))

    @property
    def rows(self) -> int:
        if self.kind == "identity":
            return self.npts
        if self.kind == "D_xz":
            return (self.n[0] - 1) * (self.n[1] - 1)
        return sum(self._block_rows(a) for a in self._axes())

    @property
    def cols(self) -> int:
        return self.npts if self.block_mode == _lib.BLOCK_PLAIN else 2 * self.npts

    @property
    def shape(self):
        return (self.rows, self.cols)

    @property
    def dtype(self):
        return np.dtype(self.TF)

    def size(self, dim=None):
        return self.shape if dim is None else self.shape[dim - 1]

    def with_block(self, block_mode: int) -> "TDOperator":
        """[A 0], [0 A] or [A A] (PARSDMM_precompute_distribute_Minkowski.jl:78-88)."""
        return TDOperator(self.kind, self.n, self.h, self.TF, block_mode)

    def __repr__(self):
        return "TDOperator(%s, n=%s, %s, %dx%d)" % (self.kind, self.n, self.TF.__name__, *self.shape)

    # -- device application ------------------------------------------------------------------------
    def _apply(self, v, adjoint: bool):
        v = np.ascontiguousarray(v, dtype=self.TF).ravel()
        nin, nout = (self.rows, self.cols) if adjoint else (self.cols, self.rows)
        if v.size != nin:
            raise ValueError("dimension mismatch: operator is %dx%d, vector has %d" % (*self.shape, v.size))
        out = np.empty(nout, dtype=self.TF)
        n = (C.c_int64 * 3)(*(list(self.n) + [1] * (3 - self.ndim)))
        h = (C.c_double * 3)(*([float(x) for x in self.h] + [1.0] * (3 - self.ndim)))
        lib = _lib.load()
        _lib.check(lib.sipb_op_apply(_lib.ctx(), _lib.dtype_code(self.TF), self.ndim, n, h, self.op_kind,
                                     self.block_mode, 1 if adjoint else 0, v.ctypes.data, out.ctypes.data))
        return out

    def __matmul__(self, x):
        return self._apply(x, False)

    __mul__ = __matmul__          # Julia's A*x

    @property
    def T(self):
        return _Adjoint(self)

    # -- host materialisation (index work, bit-exact with the reference's Kronecker construction) ---
    def _diff_block(self, axis: int):
        """rows/cols/vals of kron(..., D, ...) for a forward difference along `axis`
        (get_discrete_Grad.jl:22-31,58-66): entries -1/h at (q, c) and +1/h at (q, c+stride)."""
        n = self.n
        dims = [v - 1 if a == axis else v for a, v in enumerate(n)]
        q = np.arange(int(np.prod(dims)), dtype=np.int64)
        if axis == 0:
            c = q + q // (n[0] - 1)
            stride = 1
        elif axis == 1:
            c = q + n[0] * (q // (n[0] * (n[1] - 1)))
            stride = n[0]
        else:
            c = q
            stride = n[0] * n[1]
        ih = self.TF(1) / self.h[axis]           # ones(TF,n-1)*1 ./ h
        nih = self.TF(-1) / self.h[axis]         # ones(TF,n-1)*-1 ./ h
        return q, c, stride, nih, ih

    def tosparse(self) -> sp.csc_matrix:
        if self._sparse is not None:
            return self._sparse
        TF = self.TF
        if self.kind == "identity":
            A = sp.identity(self.npts, dtype=TF, format="csc")
        elif self.kind == "D_xz":
            n0, n1 = self.n
            w = n0 - 1
            q = np.arange(w * (n1 - 1), dtype=np.int64)
            c = (q % w) + n0 * (q // w)
            a = (TF(1) / self.h[1]) * (TF(1) / self.h[0])     # D_z*D_x: each entry is one product
            rows = np.concatenate([q, q, q, q])
            cols = np.concatenate([c, c + 1, c + n0, c + n0 + 1])
            vals = np.concatenate([np.full(q.size, a, TF), np.full(q.size, -a, TF), np.full(q.size, -a, TF),
                                   np.full(q.size, a, TF)])
            A = sp.csc_matrix((vals, (rows, cols)), shape=(q.size, self.npts), dtype=TF)
        else:
            rows, cols, vals, r0 = [], [], [], 0
            for axis in self._axes():
                q, c, stride, nih, ih = self._diff_block(axis)
                rows += [q + r0, q + r0]
                cols += [c, c + stride]
                vals += [np.full(q.size, nih, TF), np.full(q.size, ih, TF)]
                r0 += q.size
            A = sp.csc_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))),
                              shape=(r0, self.npts), dtype=TF)
        if self.block_mode != _lib.BLOCK_PLAIN:
            Z = sp.csc_matrix(A.shape, dtype=TF)
            A = sp.hstack({_lib.BLOCK_LEFT: [A, Z], _lib.BLOCK_RIGHT: [Z, A], _lib.BLOCK_BOTH: [A, A]}[self.block_mode],
                          format="csc", dtype=TF)
        A.sort_indices()
        self._sparse = A
        return A

    # -- A'A in CDS form ---------------------------------------------------------------------------
    def ata_cds(self, zrange=None):
        """(R, offsets) == mat2CDS(A'*A): R is [cols x nd] Fortran-ordered, offsets ascending int64.
        `zrange=(k0,k1)` (3-D, un-blocked operators) returns only the rows of the planes [k0,k1) of the
        slowest axis — the slab a rank uploads in multi-GPU runs.

        For difference operators every off-diagonal entry of A'A is a single product (-1/h)(1/h) and the
        main diagonal is the left fold, in row order (z block, y block, x block), of the squares — the
        accumulation order of a sparse A'*A."""
        base = TDOperator(self.kind, self.n, self.h, self.TF) if self.block_mode != _lib.BLOCK_PLAIN else self
        if zrange is not None and (self.block_mode != _lib.BLOCK_PLAIN or self.ndim != 3 or self.kind == "D_xz"):
            raise ValueError("row slabs exist only for un-blocked 3-D operators")
        R, offs = base._ata_cds_plain(zrange)
        if self.block_mode == _lib.BLOCK_PLAIN:
            return R, offs
        return _minkowski_cds(R, offs, self.block_mode)

    # -- A'A as one row per stencil class (what the device keeps; no N x nd array is formed) ----------
    def ata_class_table(self):
        """(tab, offsets): offsets == ata_cds()[1]; tab[cls, j] = (A'A)[r, r + offsets[j]] for any row r of stencil
        class cls = ((half*3 + class(k))*3 + class(j))*3 + class(i), class = 0 first / 1 interior / 2 last index of
        the axis (54 classes; `half` = second Minkowski half).  None when the grid has an axis shorter than 3.

        Every A'A of get_TD_operator.jl holds one value per class and diagonal, so the table is read off the CDS form
        of the same operator on a 3 x 3 (x 3) grid, where row index and class coincide; a diagonal of the small
        matrix maps back through the balanced-ternary digits of its offset (strides 1, 3, 9 and the half size)."""
        if min(self.n) < 3:
            return None
        small = TDOperator(self.kind, (3,) * self.ndim, self.h, self.TF, self.block_mode)
        Rs, offs_s = small.ata_cds()
        ns = 3 ** self.ndim                                   # rows per half of the small problem
        strides_s = [1, 3, 9][: self.ndim] + [ns]
        strides = [1, self.n[0], self.n[0] * self.n[1]][: self.ndim] + [self.npts]
        offs = []
        for o in offs_s:
            rest, real = int(o), 0
            for st_s, st in zip(reversed(strides_s), reversed(strides)):      # most significant digit first
                d = int(np.rint(rest / st_s))
                if abs(d) > 1:
                    return None
                rest -= d * st_s
                real += d * st
            if rest != 0:
                return None
            offs.append(real)
        offs = np.array(offs, dtype=np.int64)
        order = np.argsort(offs, kind="stable")
        if np.unique(offs).size != offs.size:
            return None
        tab = np.zeros((54, offs.size), dtype=self.TF)
        nhalf = 1 if self.block_mode == _lib.BLOCK_PLAIN else 2
        for half in range(nhalf):
            for c in range(ns):
                digits = [(c // 3 ** a) % 3 for a in range(self.ndim)]         # (i, j[, k]) == per-axis classes
                ci, cj = digits[0], digits[1]
                ck = digits[2] if self.ndim == 3 else 0                        # 2-D: a single plane, class "first"
                if self.ndim == 2:
                    # the device decodes rows of a 2-D grid as (i, j, k) with n = (n0, n1, 1): j is the middle axis
                    cls = ((half * 3 + 0) * 3 + cj) * 3 + ci
                else:
                    cls = ((half * 3 + ck) * 3 + cj) * 3 + ci
                tab[cls, :] = Rs[half * ns + c, :][order]
        return np.ascontiguousarray(tab), offs[order]

    def _ata_cds_plain(self, zrange=None):
        TF, n = self.TF, self.n
        lo, hi = 0, self.npts
        if zrange is not None:
            plane = n[0] * n[1]
            lo, hi = plane * int(zrange[0]), plane * int(zrange[1])
        N = hi - lo
        if self.kind == "identity":
            return np.ones((N, 1), dtype=TF, order="F"), np.zeros(1, dtype=np.int64)
        if self.kind == "D_xz":
            A = self.tosparse()
            return mat2CDS(sp.csc_matrix(A.T) @ A)
        # Work on the grid shape instead of flat indices: every term touches a box of the (local) grid, so the
        # columns are filled through strided views of R (each column of the Fortran-ordered R is contiguous).
        # Same additions in the same order as a sparse A'*A: adding the skipped zeros would change nothing.
        k0, k1 = (0, n[-1]) if zrange is None else (int(zrange[0]), int(zrange[1]))
        shape = list(n)
        shape[-1] = k1 - k0
        strides = [1, n[0], n[0] * n[1]]
        axes = self._axes()
        offs = np.array(sorted([0] + [sgn * strides[a] for a in axes for sgn in (1, -1)]), dtype=np.int64)
        col = {int(o): j for j, o in enumerate(offs)}
        R = np.zeros((N, offs.size), dtype=TF, order="F")

        def view(j):
            return R[:, j].reshape(shape, order="F")

        def box(axis, start, stop):
            sl = [slice(None)] * self.ndim
            sl[axis] = slice(start, stop)
            return tuple(sl)

        diag = view(col[0])
        last = self.ndim - 1
        for axis in axes:
            ih = TF(1) / self.h[axis]
            nih = TF(-1) / self.h[axis]
            base = k0 if axis == last else 0                  # global coordinate of local index 0 along this axis
            ext = shape[axis]
            lo_box = box(axis, max(0, 1 - base), ext)                         # coord > 0: touched by row (coord-1), +1/h
            hi_box = box(axis, 0, max(0, min(ext, n[axis] - 1 - base)))       # coord < n-1: touched by row (coord), -1/h
            diag[lo_box] += ih * ih
            diag[hi_box] += nih * nih
            st = strides[axis]
            view(col[st])[hi_box] = nih * ih      # A'A[c, c+st] = A[k,c]*A[k,c+st], k = row(coord)
            view(col[-st])[lo_box] = ih * nih     # A'A[c, c-st] = A[k,c]*A[k,c-st], k = row(coord-1)
        return R, offs


class SparseOperator(TDOperator):
    """An explicit sparse transform-domain operator: `constraint.custom_TD_OP[1]` of the reference
    (setup_constraints.jl:70-72, examples/ConstraintSetupExamples.jl:125-146).  Held on the host as a SciPy CSC
    matrix (the SparseMatrixCSC of the reference); the device gets CSR and CSC copies and applies them with
    SparseArrays' fold order (ascending column inside a row, ascending row inside a column).
    Inside a generalized Minkowski set `with_block` gives [A 0], [0 A] or [A A]; the device applies the block form
    without forming it.  Single GPU, matrix/tensor mode."""

    def __init__(self, A, n, h, TF):
        self.kind = "custom"
        self.TF = np.dtype(TF).type
        self.ndim = 3 if _is3d(n) else 2
        self.n = tuple(int(v) for v in n[: self.ndim])
        self.h = tuple(self.TF(v) for v in h[: self.ndim])
        self.block_mode = _lib.BLOCK_PLAIN
        self.op_kind = _lib.OP_SPARSE
        self.npts = int(np.prod(self.n))
        A = sp.csc_matrix(A).astype(self.TF)
        A.sum_duplicates()
        A.sort_indices()
        if A.shape[1] != self.npts:
            raise ValueError("custom operator has %d columns, the grid has %d points" % (A.shape[1], self.npts))
        if A.shape[0] >= 2 ** 31 - 1 or A.nnz >= 2 ** 31 - 1:
            raise NotImplementedError("custom operator too large for 32-bit indices")
        self._sparse = A
        self._csr = None
        self._struct = None

    @property
    def rows(self) -> int:
        return self._sparse.shape[0]

    def with_block(self, block_mode):
        """[A 0], [0 A] or [A A] (PARSDMM_precompute_distribute_Minkowski.jl:78-88): a copy with 2N columns that
        shares A's host arrays; `tosparse()` of the copy is the hcat matrix."""
        B = copy.copy(self)
        B.block_mode = block_mode
        B._block = None
        return B

    def __repr__(self):
        return "SparseOperator(%dx%d, nnz=%d, %s)" % (*self.shape, self._sparse.nnz, self.TF.__name__)

    def tosparse(self) -> sp.csc_matrix:
        if self.block_mode == _lib.BLOCK_PLAIN:
            return self._sparse
        if getattr(self, "_block", None) is None:
            A = self._sparse
            Z = sp.csc_matrix(A.shape, dtype=self.TF)
            B = sp.hstack({_lib.BLOCK_LEFT: [A, Z], _lib.BLOCK_RIGHT: [Z, A], _lib.BLOCK_BOTH: [A, A]}[self.block_mode],
                          format="csc", dtype=self.TF)
            B.sort_indices()
            self._block = B
        return self._block

    def sparse_struct(self) -> _lib.Sparse:
        """ctypes view (sipb_sparse) of the CSR + CSC arrays; the arrays stay alive with this object."""
        if self._struct is None:
            A = self._sparse
            R = sp.csr_matrix(A)
            R.sort_indices()
            keep = dict(rowptr=np.ascontiguousarray(R.indptr, dtype=np.int64), colidx=np.ascontiguousarray(R.indices, dtype=np.int32),
                        val=np.ascontiguousarray(R.data, dtype=self.TF), colptr=np.ascontiguousarray(A.indptr, dtype=np.int64),
                        rowidx=np.ascontiguousarray(A.indices, dtype=np.int32), valt=np.ascontiguousarray(A.data, dtype=self.TF))
            st = _lib.Sparse()
            st.rows, st.cols, st.nnz = A.shape[0], A.shape[1], A.nnz
            for k, v in keep.items():
                setattr(st, k, v.ctypes.data)
            self._csr = keep
            self._struct = st
        return self._struct

    def _apply(self, v, adjoint: bool):
        v = np.ascontiguousarray(v, dtype=self.TF).ravel()
        nin, nout = (self.rows, self.cols) if adjoint else (self.cols, self.rows)
        if v.size != nin:
            raise ValueError("dimension mismatch: operator is %dx%d, vector has %d" % (*self.shape, v.size))
        out = np.empty(nout, dtype=self.TF)
        lib = _lib.load()
        if self.block_mode == _lib.BLOCK_PLAIN:
            _lib.check(lib.sipb_sparse_apply(_lib.ctx(), _lib.dtype_code(self.TF), C.byref(self.sparse_struct()),
                                             1 if adjoint else 0, v.ctypes.data, out.ctypes.data))
        else:
            _lib.check(lib.sipb_sparse_apply_block(_lib.ctx(), _lib.dtype_code(self.TF), C.byref(self.sparse_struct()),
                                                   self.block_mode, 1 if adjoint else 0, v.ctypes.data, out.ctypes.data))
        return out

    def ata_cds(self, zrange=None):
        """mat2CDS(A'*A) (PARSDMM_precompute_distribute.jl:47,52-55); for a block copy mat2CDS of the 2N x 2N block
        matrix [A'A 0;0 0], [0 0;0 A'A] or [A'A A'A;A'A A'A] (PARSDMM_precompute_distribute_Minkowski.jl:32-74)."""
        if zrange is not None:
            raise NotImplementedError("custom operators are single-GPU (no slab decomposition)")
        A = self._sparse
        AtA = sp.csc_matrix(sp.csc_matrix(A.T) @ A).astype(self.TF)
        AtA.sort_indices()
        R, offs = mat2CDS(AtA)
        if self.block_mode == _lib.BLOCK_PLAIN:
            return R, offs
        return _minkowski_cds(R, offs, self.block_mode)


class _Adjoint:
    def __init__(self, op: TDOperator):
        self.op = op
        self.shape = (op.cols, op.rows)
        self.dtype = op.dtype

    def __matmul__(self, v):
        return self.op._apply(v, True)

    __mul__ = __matmul__

    @property
    def T(self):
        return self.op


def _minkowski_cds(R, offs, block_mode):
    """CDS of [B 0;0 0], [0 0;0 B] or [B B;B B] (PARSDMM_precompute_distribute_Minkowski.jl:32-74) from
    the CDS of B, as mat2CDS of the 2N x 2N block matrix would return it."""
    N = R.shape[0]
    TF = R.dtype.type
    cols = {}

    def put(o, top, bottom):
        c = cols.setdefault(int(o), np.zeros(2 * N, dtype=TF))
        if top is not None:
            c[:N] += top
        if bottom is not None:
            c[N:] += bottom

    for j, o in enumerate(offs):
        col = R[:, j]
        if block_mode == _lib.BLOCK_LEFT:
            put(o, col, None)
        elif block_mode == _lib.BLOCK_RIGHT:
            put(o, None, col)
        else:
            put(o, col, col)          # diagonal blocks
            put(o + N, col, None)     # top-right block: A[r, N + r + o]
            put(o - N, None, col)     # bottom-left block: A[N + r, r + o]
    # only diagonals that hold at least one structural entry exist in mat2CDS output
    keep = sorted(cols)
    offs2 = np.array(keep, dtype=np.int64)
    R2 = np.zeros((2 * N, offs2.size), dtype=TF, order="F")
    for j, o in enumerate(keep):
        R2[:, j] = cols[o]
    return R2, offs2


# --------------------------------------------------------------------------------------------------
# reference-named constructors
# --------------------------------------------------------------------------------------------------
def get_discrete_Grad(*args) -> TDOperator:
    """get_discrete_Grad(n1,n2,h1,h2,TD_type) / (n1,n2,n3,h1,h2,h3,TD_type) — get_discrete_Grad.jl:16,51."""
    if len(args) == 5:
        n1, n2, h1, h2, kind = args
        return TDOperator(kind, (n1, n2), (h1, h2), type(h1) if isinstance(h1, np.floating) else np.float64)
    n1, n2, n3, h1, h2, h3, kind = args
    return TDOperator(kind, (n1, n2, n3), (h1, h2, h3), type(h1) if isinstance(h1, np.floating) else np.float64)


def get_TD_operator(comp_grid, TD_type: str, TF):
    """get_TD_operator.jl:12-95.  Returns (TD_OP, AtA_diag, dense, TD_n, banded)."""
    if TD_type in SPECIAL_OPERATORS:
        raise NotImplementedError("transform %r (JOLI) is outside the device CDS path and is rejected" % TD_type)
    n = tuple(int(v) for v in comp_grid.n)
    op = TDOperator(TD_type, n, comp_grid.d, TF)
    if op.ndim == 3:
        n1, n2, n3 = op.n
        TD_n = {"TV": (n1 - 1 + n1 + n1, n2 - 1 + n2 + n2, n3 - 1 + n3 + n3), "D_z": (n1, n2, n3 - 1),
                "D_x": (n1 - 1, n2, n3), "D_y": (n1, n2 - 1, n3), "identity": (n1, n2, n3)}[op.kind]
    else:
        n1, n2 = op.n
        TD_n = {"TV": ((n1 - 1) + n1, n2 + (n2 - 1)), "D_z": (n1, n2 - 1), "D_x": (n1 - 1, n2),
                "D_xz": (n1 - 1, n2 - 1), "identity": (n1, n2)}[op.kind]
    return op, op.kind == "identity", False, TD_n, True


def mat2CDS(A):
    """mat2CDS.jl:7-32 for a square sparse matrix: offsets = sorted unique (j - i) over the stored
    entries; R[r, k] = A[r, r + offsets[k]] (row aligned, zero padded)."""
    if isinstance(A, TDOperator):
        A = A.tosparse()
    A = sp.coo_matrix(A)
    m, n = A.shape
    if m != n:
        raise ValueError("mat2CDS expects a square matrix")
    d = A.col.astype(np.int64) - A.row.astype(np.int64)
    offs, inv = np.unique(d, return_inverse=True)
    R = np.zeros((m, offs.size), dtype=A.dtype, order="F")
    np.add.at(R, (A.row, inv), A.data)
    return R, offs.astype(np.int64)


def CDS_MVp(N, ndiags, R, offset, x, y):
    """y += A*x with A in CDS form, evaluated on the device (CDS_MVp.jl:9-28 / CDS_MVp_MT.jl:9-25)."""
    R = np.asfortranarray(R)
    x = np.ascontiguousarray(x, dtype=R.dtype)
    out = np.empty(N, dtype=R.dtype)
    offs = np.ascontiguousarray(offset, dtype=np.int64)
    lib = _lib.load()
    _lib.check(lib.sipb_cds_spmv(_lib.ctx(), _lib.dtype_code(R.dtype), N, ndiags, R.ctypes.data,
                                 offs.ctypes.data_as(C.POINTER(C.c_int64)), x.ctypes.data, out.ctypes.data))
    y += out
    return y


CDS_MVp_MT = CDS_MVp


def CDS_scaled_add(A, B, A_offsets, B_offsets, alpha):
    """A += alpha*B on matching diagonals, on the device (CDS_scaled_add!.jl:8-26).  Raises when a
    diagonal of B does not exist in A, like the reference."""
    assert A.flags.f_contiguous and A.dtype == B.dtype
    B = np.asfortranarray(B)
    ao = np.ascontiguousarray(A_offsets, dtype=np.int64)
    bo = np.ascontiguousarray(B_offsets, dtype=np.int64)
    lib = _lib.load()
    _lib.check(lib.sipb_cds_scaled_add(_lib.ctx(), _lib.dtype_code(A.dtype), A.shape[0], A.shape[1], A.ctypes.data,
                                       ao.ctypes.data_as(C.POINTER(C.c_int64)), B.shape[1], B.ctypes.data,
                                       bo.ctypes.data_as(C.POINTER(C.c_int64)), float(alpha)))
    return A


def cg(R, offsets, b, tol=1e-2, maxIter=100, x=None):
    """cg(A,b;tol,maxIter,x) with A in CDS form, on the device (cg.jl:44-128).
    Returns (x, flag, relres, iter)."""
    R = np.asfortranarray(R)
    TF = R.dtype.type
    b = np.ascontiguousarray(b, dtype=TF)
    x = np.zeros(b.size, dtype=TF) if x is None else np.ascontiguousarray(x, dtype=TF)
    offs = np.ascontiguousarray(offsets, dtype=np.int64)
    flag, it, relres = C.c_int(0), C.c_int(0), C.c_double(0)
    lib = _lib.load()
    _lib.check(lib.sipb_cds_cg(_lib.ctx(), _lib.dtype_code(TF), b.size, R.shape[1], R.ctypes.data,
                               offs.ctypes.data_as(C.POINTER(C.c_int64)), b.ctypes.data, x.ctypes.data, float(tol),
                               int(maxIter), C.byref(flag), C.byref(relres), C.byref(it)))
    return x, flag.value, TF(relres.value), it.value
