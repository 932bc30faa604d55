"""ctypes binding of the C ABI declared in include/sipb200.h.

The shared library is built in-tree by ``build.py`` (nvcc, sm_100a).  There is NO CPU fallback: if the
library is missing, or no CUDA device is present, every compute call raises.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libsipb200.so")

SIPB_OK = 0
SIPB_E_INVALID, SIPB_E_UNSUPPORTED, SIPB_E_CUDA, SIPB_E_NCCL, SIPB_E_STATE, SIPB_E_MISSING_DIAG = -1, -2, -3, -4, -5, -6
SIPB_F32, SIPB_F64 = 0, 1
(SET_BOUNDS_SCALAR, SET_BOUNDS_VECTOR, SET_L1, SET_L2, SET_ANNULUS, SET_CARDINALITY, SET_PROX_L1,
 SET_DISTANCE, SET_BOUNDS_FIBER, SET_CARD_FIBER, SET_CARD_SLICE, SET_HISTOGRAM) = range(12)
OP_IDENTITY, OP_DX, OP_DY, OP_DZ, OP_TV, OP_DXZ, OP_SPARSE = range(7)
BLOCK_PLAIN, BLOCK_LEFT, BLOCK_RIGHT, BLOCK_BOTH = range(4)
N_PHASES = 7
N_KERNEL_CLASSES = 24

PHASE_NAMES = ("initialization", "form rhs for linear system", "argmin x", "argmin y and l update",
               "stopping conditions check", "adjust rho and gamma", "Q-update")   # PARSDMM.jl:40,100,105,113,152,163,229


class SipbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("sipb200 error %d: %s" % (code, msg))
        self.code = code


class Sparse(C.Structure):
    """sipb_sparse: an explicit sparse operator in both orientations (host arrays, 0-based)."""
    _fields_ = [("rows", C.c_int64), ("cols", C.c_int64), ("nnz", C.c_int64),
                ("rowptr", C.c_void_p), ("colidx", C.c_void_p), ("val", C.c_void_p),
                ("colptr", C.c_void_p), ("rowidx", C.c_void_p), ("valt", C.c_void_p)]


class SetDesc(C.Structure):
    _fields_ = [("set_kind", C.c_int32), ("op_kind", C.c_int32), ("block_mode", C.c_int32), ("ncvx", C.c_int32),
                ("min", C.c_double), ("max", C.c_double), ("k", C.c_int64),
                ("min_vec", C.c_void_p), ("max_vec", C.c_void_p),
                ("fiber_axis", C.c_int32), ("reserved", C.c_int32), ("td_n", C.c_int64 * 3),
                ("sparse", C.POINTER(Sparse))]


class Options(C.Structure):
    _fields_ = [("maxit", C.c_int32), ("rho_update_frequency", C.c_int32), ("adjust_rho", C.c_int32),
                ("adjust_gamma", C.c_int32), ("adjust_feasibility_rho", C.c_int32), ("zero_ini_guess", C.c_int32),
                ("n_rho_ini", C.c_int32), ("profile_kernels", C.c_int32),
                ("evol_rel_tol", C.c_double), ("feas_tol", C.c_double), ("obj_tol", C.c_double),
                ("gamma_ini", C.c_double), ("rho_ini", C.POINTER(C.c_double)),
                ("fixed_iterations", C.c_int32), ("return_ly", C.c_int32), ("resident_io", C.c_int32),
                ("warm_resident", C.c_int32)]


class ResampleSeg(C.Structure):
    _fields_ = [("vec", C.c_int32), ("reserved", C.c_int32), ("src_off", C.c_int64), ("dst_off", C.c_int64),
                ("src_shape", C.c_int64 * 3), ("dst_shape", C.c_int64 * 3)]


class Log(C.Structure):
    _fields_ = [("iters", C.c_int32), ("feas_rows", C.c_int32), ("stopped_feasible", C.c_int32),
                ("p", C.c_int32), ("pp", C.c_int32),
                ("set_feasibility", C.POINTER(C.c_double)), ("r_dual", C.POINTER(C.c_double)),
                ("r_pri", C.POINTER(C.c_double)), ("r_dual_total", C.POINTER(C.c_double)),
                ("r_pri_total", C.POINTER(C.c_double)), ("obj", C.POINTER(C.c_double)),
                ("evol_x", C.POINTER(C.c_double)), ("rho", C.POINTER(C.c_double)), ("gamma", C.POINTER(C.c_double)),
                ("cg_it", C.POINTER(C.c_int32)), ("cg_relres", C.POINTER(C.c_double)),
                ("phase_seconds", C.c_double * N_PHASES), ("solve_seconds", C.c_double),
                ("device_seconds", C.c_double),
                ("kernel_launches", C.c_int64 * N_KERNEL_CLASSES), ("kernel_ms", C.c_double * N_KERNEL_CLASSES),
                ("kernel_bytes", C.c_double * N_KERNEL_CLASSES),
                ("total_launches", C.c_int64), ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64)]


# every symbol include/sipb200.h declares: (name, restype, argtypes)
_VP, _I, _I64, _D = C.c_void_p, C.c_int, C.c_int64, C.c_double
_PI64, _PD, _PI = C.POINTER(C.c_int64), C.POINTER(C.c_double), C.POINTER(C.c_int)
SYMBOLS = [
    ("sipb_abi_version", _I, []),
    ("sipb_last_error", C.c_char_p, []),
    ("sipb_kernel_class_name", C.c_char_p, [_I]),
    ("sipb_ctx_create", _I, [_I, C.POINTER(_VP)]),
    ("sipb_ctx_destroy", _I, [_VP]),
    ("sipb_ctx_num_sms", _I, [_VP, _PI]),
    ("sipb_comm_unique_id", _I, [_VP]),
    ("sipb_comm_init", _I, [_VP, _I, _I, _VP]),
    ("sipb_comm_info", _I, [_VP, _PI, _PI]),
    ("sipb_comm_peer_path", _I, [_VP, _PI]),
    ("sipb_slab_range", _I, [_I64, _I, _I, _PI64, _PI64]),
    ("sipb_problem_create", _I, [_VP, _I, _I, _PI64, _PD, _I, _I, C.POINTER(_VP)]),
    ("sipb_problem_add_set", _I, [_VP, C.POINTER(SetDesc)]),
    ("sipb_problem_set_ata", _I, [_VP, _I, _VP, _I64, _PI64, _I]),
    ("sipb_problem_set_ata_classes", _I, [_VP, _I, _VP, _PI64, _I]),
    ("sipb_problem_finalize", _I, [_VP]),
    ("sipb_problem_num_q_offsets", _I, [_VP, _PI]),
    ("sipb_problem_q_form", _I, [_VP, _PI]),
    ("sipb_problem_q_offsets", _I, [_VP, _PI64]),
    ("sipb_problem_destroy", _I, [_VP]),
    ("sipb_problem_warm_from", _I, [_VP, _VP, C.POINTER(ResampleSeg), _I]),
    ("sipb_solve", _I, [_VP, _VP, _VP, C.POINTER(_VP), C.POINTER(_VP), C.POINTER(Options), C.POINTER(Log)]),
    ("sipb_solve_batch", _I, [C.POINTER(_VP), _I, C.POINTER(_VP), C.POINTER(_VP), C.POINTER(C.POINTER(_VP)),
                              C.POINTER(C.POINTER(_VP)), C.POINTER(Options), C.POINTER(C.POINTER(Log)), _PI]),
    ("sipb_cds_spmv", _I, [_VP, _I, _I64, _I, _VP, _PI64, _VP, _VP]),
    ("sipb_cds_cg", _I, [_VP, _I, _I64, _I, _VP, _PI64, _VP, _VP, _D, _I, _PI, _PD, _PI]),
    ("sipb_project", _I, [_VP, _I, C.POINTER(SetDesc), _I64, _VP, _VP]),
    ("sipb_op_apply", _I, [_VP, _I, _I, _PI64, _PD, _I, _I, _I, _VP, _VP]),
    ("sipb_op_rows", _I, [_I, _PI64, _I, _PI64]),
    ("sipb_sparse_apply", _I, [_VP, _I, C.POINTER(Sparse), _I, _VP, _VP]),
    ("sipb_cds_scaled_add", _I, [_VP, _I, _I64, _I, _VP, _PI64, _I, _VP, _PI64, _D]),
    ("sipb_bench_spmv", _I, [_VP, _I, _I, _PI64, _I, _I, _I, _PD, _PI64]),
    ("sipb_bench_spmv2", _I, [_VP, _I, _I, _PI64, _I, _I, _I, _I, _I, _PD, _PI64]),
    ("sipb_cds_spmv_grid", _I, [_VP, _I, _PI64, _I, _VP, _PI64, _VP, _VP, _PI]),
    ("sipb_tile_probe", _I, [_VP, _I, _PI64, _I, _PI64, _VP, _VP, _VP, _VP, _I, _I, _VP, _VP, _VP, _VP, _PD, _PI]),
    ("sipb_select_probe", _I, [_VP, _I, _I64, _VP, _I64, C.c_uint64, _I, _VP, _PI64]),
    ("sipb_iter_probe", _I, [_VP, _I, _I, _VP, _VP, _VP, _PD, _PD, C.POINTER(_VP), C.POINTER(_VP), C.POINTER(_VP),
                             C.POINTER(_VP), _PI, _PD, C.POINTER(C.c_uint64), _VP, C.POINTER(_VP), _PD, _PD, _PI64,
                             _PI64, _PI]),
]

_lib = None
_lock = threading.Lock()


def load():
    """Load libsipb200.so (fails loudly when it has not been built)."""
    global _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise ImportError("%s is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                                  "(nvcc, sm_100a). There is no CPU fallback." % LIB_PATH)
            lib = C.CDLL(LIB_PATH)
            for name, res, args in SYMBOLS:
                fn = getattr(lib, name)          # AttributeError if the .so does not export a declared symbol
                fn.restype = res
                fn.argtypes = args
            _lib = lib
    return _lib


def check(rc: int) -> None:
    if rc != SIPB_OK:
        msg = load().sipb_last_error()
        raise SipbError(rc, msg.decode() if msg else "")


_ctx = {}


def ctx(device: int | None = None):
    """Per-process device context (one process drives one GPU)."""
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", "0")) if "LOCAL_RANK" in os.environ else 0
    if device not in _ctx:
        h = C.c_void_p()
        check(load().sipb_ctx_create(device, C.byref(h)))
        _ctx[device] = h
    return _ctx[device]


_batch_ctx = {}


def batch_ctx(device: int, index: int):
    """Extra contexts for batched projections: problem `index` of a batch gets its own stream / scratch."""
    key = (device, index)
    if key not in _batch_ctx:
        h = C.c_void_p()
        check(load().sipb_ctx_create(device, C.byref(h)))
        _batch_ctx[key] = h
    return _batch_ctx[key]


def dtype_code(dt) -> int:
    import numpy as np
    dt = np.dtype(dt)
    if dt == np.float32:
        return SIPB_F32
    if dt == np.float64:
        return SIPB_F64
    raise TypeError("only Float32/Float64 are supported, got %r" % (dt,))
