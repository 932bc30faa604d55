"""PARSDMM_precompute_distribute (+ Minkowski) — host side.

Mirrors PARSDMM_precompute_distribute.jl:6-77 and PARSDMM_precompute_distribute_Minkowski.jl:3-157:
appends the distance term, forms every A_i'A_i directly in compressed-diagonal storage and allocates
l, y.  "Distribute" here means: the returned AtA list is what `PARSDMM` uploads once to the GPU and
keeps resident (the device problem handle is cached on the list object).
"""
from __future__ import annotations

import copy

import numpy as np

from . import _lib
from . import distributed as dd
from .operators import SparseOperator, TDOperator


class CDSList(list):
    """Vector{Array{TF,2}} of CDS matrices; carries the cached device problem built from it.
    `slab` = (k0, k1) when the matrices hold only this rank's rows (multi-GPU slabs).

    Entries of stencil operators are LAZY: the device keeps one row per stencil class of every A'A
    (`TDOperator.ata_class_table`), so the N x nd array of the reference is only formed when the caller indexes the
    list (`AtA[i]`, iteration) — e.g. to inspect or modify it; once any entry has been formed the arrays are what
    gets uploaded (they may have been changed)."""
    _device = None
    slab = None

    def __init__(self):
        super().__init__()
        self._lazy = {}          # index -> (operator, zrange)

    def append_lazy(self, op, zrange):
        self._lazy[len(self)] = (op, zrange)
        super().append(None)

    def materialized(self) -> bool:
        """True when some lazy entry has been formed (or there are none): the arrays are then authoritative."""
        return any(super(CDSList, self).__getitem__(i) is not None for i in self._lazy)

    def is_lazy(self, i) -> bool:
        return i in self._lazy and super().__getitem__(i) is None

    def class_table(self, i):
        op, _ = self._lazy[i]
        return op.ata_class_table()

    def _form(self, i):
        v = super().__getitem__(i)
        if v is None and i in self._lazy:
            op, zr = self._lazy[i]
            v = op.ata_cds(zr)[0]
            super().__setitem__(i, v)
        return v

    def __getitem__(self, i):
        if isinstance(i, slice):
            return [self._form(k) for k in range(*i.indices(len(self)))]
        if i < 0:
            i += len(self)
        return self._form(i)

    def __iter__(self):
        return (self._form(i) for i in range(len(self)))


def _classes_enabled() -> bool:
    import os
    return os.environ.get("SIPB_Q_CLASSES", "1") != "0"


MAX_ATA_DIAGONALS = 999     # per A'A: the 999 x 99 offset table of PARSDMM_initialize.jl:217-221


def _require_device_operators(TD_OP):
    for A in TD_OP:
        if not isinstance(A, TDOperator):
            raise NotImplementedError("only the banded operators built by get_TD_operator are on the device path; "
                                      "got %r" % type(A))


def _require_banded_custom(set_Prop, i):
    # custom operator: the caller describes it through set_Prop (ConstraintSetupExamples.jl:114-117)
    if not set_Prop.banded[i] or set_Prop.dense[i]:
        raise NotImplementedError("custom operators must be flagged banded and not dense: the device path solves "
                                  "the x-subproblem in compressed-diagonal storage only")


def _require_width(offs):
    if offs.size > MAX_ATA_DIAGONALS:
        raise NotImplementedError("A'A of the custom operator has %d diagonals; the reference's offset table holds %d"
                                  % (offs.size, MAX_ATA_DIAGONALS))


def PARSDMM_precompute_distribute(TD_OP, set_Prop, comp_grid, options):
    """-> (TD_OP, AtA, l, y).  MUTATES TD_OP and set_Prop like the reference (push of the distance term,
    :17-26; AtA_offsets filled by mat2CDS, :52-59)."""
    if getattr(options, "parallel", False):
        raise NotImplementedError("options.parallel=true (one Julia worker per set) is replaced by slab domain "
                                  "decomposition on the device path and is rejected")
    _require_device_operators(TD_OP)
    TF = TD_OP[0].TF
    if not options.feasibility_only:
        TD_OP.append(TDOperator("identity", comp_grid.n, comp_grid.d, TF))
        set_Prop.TD_n.append(tuple(comp_grid.n))
        set_Prop.AtA_offsets.append(np.array([0], dtype=np.int64))
        set_Prop.banded.append(True)
        set_Prop.AtA_diag.append(True)
        set_Prop.ncvx.append(False)
        set_Prop.dense.append(False)
        set_Prop.tag.append(("distance squared", "identity", "matrix", ""))
    p = len(TD_OP)
    AtA = CDSList()
    zrange = None
    if dd.active() and TD_OP[0].ndim == 3:
        # "distribute": every rank builds and later uploads only the rows of its own z-slab
        zrange = dd.slab_range(TD_OP[0].n[2])
        AtA.slab = zrange
    for i in range(p):
        if isinstance(TD_OP[i], SparseOperator):
            _require_banded_custom(set_Prop, i)
            if set_Prop.AtA_diag[i]:          # :44-45: AtA = I when the caller says A'A is the identity
                R, offs = np.ones((TD_OP[i].cols, 1), dtype=TF, order="F"), np.array([0], dtype=np.int64)
            else:
                R, offs = TD_OP[i].ata_cds(zrange)
            _require_width(offs)
        else:
            ct = TD_OP[i].ata_class_table() if _classes_enabled() else None
            if ct is not None:       # == mat2CDS(TD_OP[i]'*TD_OP[i]), formed only when somebody indexes AtA[i]
                AtA.append_lazy(TD_OP[i], zrange)
                set_Prop.AtA_offsets[i] = ct[1]
                continue
            R, offs = TD_OP[i].ata_cds(zrange)    # == mat2CDS(TD_OP[i]'*TD_OP[i]) (identity when AtA_diag)
        AtA.append(R)
        set_Prop.AtA_offsets[i] = offs
    set_Prop.AtA_offsets = set_Prop.AtA_offsets[:p]
    if zrange is None:
        rows = [TD_OP[i].rows for i in range(p)]
    else:
        rows = [sum(b - a for a, b in dd.local_td_slices(TD_OP[i], *zrange)) for i in range(p)]
    y = [np.zeros(r, dtype=TF) for r in rows]
    l = [np.zeros(r, dtype=TF) for r in rows]
    return TD_OP, AtA, l, y


def PARSDMM_precompute_distribute_Minkowski(TD_OP_c1, TD_OP_c2, TD_OP_sum, set_Prop_c1, set_Prop_c2, set_Prop_sum,
                                            comp_grid, options):
    """-> (TD_OP, set_Prop, AtA, l, y) for a generalized Minkowski set (unknown [x1; x2]).
    Operators become [A 0], [0 A], [A A]; the distance term is [I I] (:78-101)."""
    if getattr(options, "parallel", False):
        raise NotImplementedError("options.parallel=true is rejected on the device path")
    for lst in (TD_OP_c1, TD_OP_c2, TD_OP_sum):
        _require_device_operators(lst)
    first = (TD_OP_c1 + TD_OP_c2 + TD_OP_sum)[0]
    TF = first.TF
    for i in range(len(TD_OP_c1)):
        TD_OP_c1[i] = TD_OP_c1[i].with_block(_lib.BLOCK_LEFT)
    for i in range(len(TD_OP_c2)):
        TD_OP_c2[i] = TD_OP_c2[i].with_block(_lib.BLOCK_RIGHT)
    for i in range(len(TD_OP_sum)):
        TD_OP_sum[i] = TD_OP_sum[i].with_block(_lib.BLOCK_BOTH)
    if not options.feasibility_only:
        TD_OP_sum.append(TDOperator("identity", comp_grid.n, comp_grid.d, TF, _lib.BLOCK_BOTH))
        set_Prop_sum.TD_n.append(tuple(comp_grid.n))
        set_Prop_sum.AtA_offsets.append(np.array([0], dtype=np.int64))
        set_Prop_sum.banded.append(True)
        set_Prop_sum.AtA_diag.append(False)
        set_Prop_sum.dense.append(False)
        set_Prop_sum.ncvx.append(False)
        set_Prop_sum.tag.append(("distance squared", "identity", "matrix", ""))
    set_Prop = copy.deepcopy(set_Prop_c1)
    for other in (set_Prop_c2, set_Prop_sum):
        for name in ("AtA_diag", "AtA_offsets", "TD_n", "banded", "dense", "ncvx", "tag"):
            getattr(set_Prop, name).extend(copy.deepcopy(getattr(other, name)))
    TD_OP = list(TD_OP_c1) + list(TD_OP_c2) + list(TD_OP_sum)
    s = len(TD_OP)
    AtA = CDSList()
    # stencil-class tables for every set or CDS arrays for every set: a custom operator has no table
    custom = any(isinstance(A, SparseOperator) for A in TD_OP)
    for i in range(s):
        ct = TD_OP[i].ata_class_table() if _classes_enabled() and not custom else None
        if ct is not None:
            AtA.append_lazy(TD_OP[i], None)
            set_Prop.AtA_offsets[i] = ct[1]
            continue
        if isinstance(TD_OP[i], SparseOperator):
            # mat2CDS of the block matrix of A'A (:32-74); its AtA_diag flag only matters for dense operators
            _require_banded_custom(set_Prop, i)
            R, offs = TD_OP[i].ata_cds()
            _require_width(offs)
            AtA.append(R)
            set_Prop.AtA_offsets[i] = offs
            continue
        R, offs = TD_OP[i].ata_cds()
        AtA.append(R)
        set_Prop.AtA_offsets[i] = offs
    set_Prop.AtA_offsets = set_Prop.AtA_offsets[:s]
    y = [np.zeros(TD_OP[i].rows, dtype=TF) for i in range(s)]
    l = [np.zeros(TD_OP[i].rows, dtype=TF) for i in range(s)]
    return TD_OP, set_Prop, AtA, l, y
