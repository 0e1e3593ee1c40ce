"""ctypes binding of libporeb200.so (include/poreb200.h).  No CPU fallback: importing the
binding without the built CUDA library, or computing without a GPU, raises."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
# POREB200_LIB: developer knob, path of an alternative build of the same library (A/B timing)
LIB_PATH = os.environ.get("POREB200_LIB") or os.path.join(HERE, "libporeb200.so")

PB_OK, PB_EINVAL, PB_ESINGULAR, PB_ECELLTYPE, PB_ECUDA, PB_ENOTIMPL = range(6)
BC_INTERIOR, BC_DIR, BC_NEU, BC_ROB = 0, 1, 2, 3
PAT_FACE_CELL, PAT_FACE_BFACE, PAT_CELL_CELL, PAT_CELL_BFACE = 0, 1, 2, 3

_i32p = C.POINTER(C.c_int32)
_i8p = C.POINTER(C.c_int8)
_u8p = C.POINTER(C.c_uint8)
_f64p = C.POINTER(C.c_double)
_i64p = C.POINTER(C.c_int64)
_f32p = C.POINTER(C.c_float)

_SIGNATURES = {
    "pb_last_error": (C.c_char_p, []),
    "pb_last_error_node": (C.c_int64, []),
    "pb_device_count": (C.c_int, []),
    "pb_set_device": (C.c_int, [C.c_int]),
    "pb_launch_count": (C.c_int64, []),
    "pb_device_pool_trim": (None, []),
    "pb_alloc_stats": (None, [_f64p]),
    "pb_csr_lanes_per_row": (C.c_int, [C.c_void_p]),
    "pb_fp64_peak": (C.c_int, [C.c_int, _f64p]),
    "pb_host_alloc": (C.c_int, [C.c_uint64, C.POINTER(C.c_void_p)]),
    "pb_host_free": (None, [C.c_void_p]),
    "pb_plan_create": (C.c_int, [C.c_int, C.c_int64, C.c_int64, C.c_int64, _i32p, _i32p, _i8p,
                                 _i32p, _i32p, C.POINTER(C.c_void_p)]),
    "pb_plan_destroy": (None, [C.c_void_p]),
    "pb_plan_sizes": (C.c_int, [C.c_void_p, _i64p, _i64p, _i64p, _i32p, _i32p]),
    "pb_plan_node_classes": (C.c_int, [C.c_void_p, C.c_int, C.c_int, _i32p, _u8p, _i64p, C.POINTER(C.c_int)]),
    "pb_solver_limits": (C.c_int, [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "pb_local_solve_batch": (C.c_int, [C.c_int, C.c_int, C.c_int64, C.c_int, C.c_int, _f64p, _f64p, _i32p]),
    "pb_plan_set_cell_map": (C.c_int, [C.c_void_p, _i64p, C.c_int64]),
    "pb_plan_set_active_nodes": (C.c_int, [C.c_void_p, _u8p]),
    "pb_plan_pattern_size": (C.c_int, [C.c_void_p, C.c_int, _i64p, _i64p]),
    "pb_plan_pattern_get": (C.c_int, [C.c_void_p, C.c_int, _i32p, _i32p]),
    "pb_plan_pattern_expanded": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, _i32p, _i32p]),
    "pb_plan_set_geometry": (C.c_int, [C.c_void_p] + [_f64p] * 6),
    "pb_mpfa_upload": (C.c_int, [C.c_void_p, _f64p, _u8p, _f64p, C.c_double]),
    "pb_mpfa_assemble": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, _f32p]),
    "pb_mpfa_download": (C.c_int, [C.c_void_p] + [_f64p] * 6),
    "pb_plan_take_output": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]),
    "pb_values_size": (C.c_int64, [C.c_void_p]),
    "pb_values_download": (C.c_int, [C.c_void_p, _f64p]),
    "pb_values_checksum": (C.c_int, [C.c_void_p, _f64p, _f64p]),
    "pb_values_destroy": (None, [C.c_void_p]),
    "pb_mpfa_system": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]),
    "pb_mpfa_rhs": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, _f64p, _f64p, _f64p]),
    "pb_mpsa_system": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]),
    "pb_mpsa_rhs": (C.c_int, [C.c_void_p, C.c_void_p, _f64p, _f64p, _f64p]),
    "pb_mpsa_upload": (C.c_int, [C.c_void_p, _f64p, _u8p, _f64p, C.c_double, C.c_int, _f64p]),
    "pb_mpsa_set_basis": (C.c_int, [C.c_void_p, _f64p]),
    "pb_mpsa_assemble": (C.c_int, [C.c_void_p, _f32p]),
    "pb_mpsa_download": (C.c_int, [C.c_void_p] + [_f64p] * 4),
    "pb_biot_download": (C.c_int, [C.c_void_p, C.c_int] + [_f64p] * 5),
    "pb_facegrid_create": (C.c_int, [C.c_int64, C.c_int64, _i32p, _i32p, _i8p, _f64p, _f64p, _f64p,
                                     C.POINTER(C.c_void_p)]),
    "pb_facegrid_destroy": (None, [C.c_void_p]),
    "pb_tpfa": (C.c_int, [C.c_void_p, _f64p, _u8p, _i32p, C.c_int] + [_f64p] * 6),
    "pb_tpfa_diff": (C.c_int, [C.c_void_p, _f64p, _i32p, _f64p, _f64p, _f64p]),
    "pb_upwind": (C.c_int, [C.c_void_p, _f64p, _u8p, _i32p, _f64p, _f64p]),
    "pb_upwind_coupling": (C.c_int, [C.c_int64, _f64p, _f64p, _f64p, _f64p]),
    "pb_compute_geometry_3d": (C.c_int, [C.c_int64, C.c_int64, C.c_int64, _i32p, _i32p, _i8p, _i32p, _i32p] + [_f64p] * 6
                               + [_f32p]),
    "pb_shard_create": (C.c_int, [C.c_int64, C.c_int64, C.c_int64, _i32p, _i32p, _f64p, _i32p, _i32p, _i64p, C.c_int64,
                                  C.POINTER(C.c_void_p)]),
    "pb_shard_sizes": (C.c_int, [C.c_void_p, _i64p]),
    "pb_shard_fill": (C.c_int, [C.c_void_p, _i64p, _i64p, _i64p, _u8p, _u8p, _u8p, _u8p, _i32p, _i32p, _f64p, _i32p, _i32p]),
    "pb_shard_destroy": (None, [C.c_void_p]),
    "pb_gather_columns": (C.c_int, [_f64p, C.c_int64, C.c_int64, _i64p, C.c_int64, _f64p]),
    "pb_csr_create": (C.c_int, [C.c_int64, C.c_int64, C.c_int64, _i32p, _i32p, _f64p,
                                C.POINTER(C.c_void_p)]),
    "pb_csr_destroy": (None, [C.c_void_p]),
    "pb_csr_shape": (C.c_int, [C.c_void_p, _i64p, _i64p, _i64p]),
    "pb_plan_output_csr": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "pb_csr_spgemm": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]),
    "pb_csr_axpby": (C.c_int, [C.c_double, C.c_void_p, C.c_double, C.c_void_p, C.POINTER(C.c_void_p)]),
    "pb_csr_scale_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]),
    "pb_csr_bmat": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_void_p), _i64p, _i64p, C.POINTER(C.c_void_p)]),
    "pb_csr_diagonal": (C.c_int, [C.c_void_p, _f64p]),
    "pb_csr_checksum": (C.c_int, [C.c_void_p, _f64p, _f64p]),
    "pb_csr_truncate_rows": (C.c_int, [C.c_void_p, C.c_int64]),
    "pb_csr_download": (C.c_int, [C.c_void_p, _i32p, _i32p, _f64p]),
    "pb_csr_spmv": (C.c_int, [C.c_void_p, _f64p, _f64p]),
    "pb_csr_spmv_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]),
    "pb_csr_spmv_dots_dev": (C.c_int, [C.c_void_p] * 7 + [C.c_uint64]),
    "pb_kry_init": (C.c_int, [C.c_int64] + [C.c_void_p] * 7 + [C.c_double, C.c_uint64]),
    "pb_kry_seed": (C.c_int, [C.c_void_p, C.c_uint64]),
    "pb_kry_p": (C.c_int, [C.c_int64] + [C.c_void_p] * 6 + [C.c_int, C.c_int, C.c_uint64]),
    "pb_kry_s": (C.c_int, [C.c_int64] + [C.c_void_p] * 6 + [C.c_int, C.c_int, C.c_uint64]),
    "pb_csr_block_diag_inv_dev": (C.c_int, [C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_uint64]),
    "pb_kry_xr": (C.c_int, [C.c_int64] + [C.c_void_p] * 8 + [C.c_int, C.c_int, C.c_uint64]),
    "pb_csr_spmv_bench": (C.c_int, [C.c_void_p, C.c_int, _f32p]),
    "pb_csr_local_block_inv_dev": (C.c_int, [C.c_void_p, C.c_int64] + [C.c_void_p] * 5 + [_i64p, C.c_void_p, C.c_void_p,
                                                                                         C.c_uint64]),
    "pb_local_block_apply_dev": (C.c_int, [C.c_int64] + [C.c_void_p] * 5 + [_i64p] + [C.c_void_p] * 4 + [C.c_uint64]),
    "pb_gm_dots": (C.c_int, [C.c_int64, C.c_void_p, C.c_int] + [C.c_void_p] * 3 + [C.c_uint64]),
    "pb_gm_orth": (C.c_int, [C.c_int64, C.c_void_p, C.c_int] + [C.c_void_p] * 4 + [C.c_uint64]),
    "pb_gm_givens": (C.c_int, [C.c_int, C.c_int] + [C.c_void_p] * 6 + [C.c_uint64]),
    "pb_gm_scale": (C.c_int, [C.c_int64, C.c_void_p, C.c_void_p, C.c_uint64]),
    "pb_gm_residual": (C.c_int, [C.c_int64] + [C.c_void_p] * 3 + [C.c_int, C.c_uint64]),
    "pb_gm_start": (C.c_int, [C.c_int, C.c_double] + [C.c_void_p] * 3 + [C.c_uint64]),
    "pb_gm_ysolve": (C.c_int, [C.c_int] + [C.c_void_p] * 4 + [C.c_uint64]),
    "pb_gm_combine": (C.c_int, [C.c_int64, C.c_void_p, C.c_int] + [C.c_void_p] * 3 + [C.c_int, C.c_uint64]),
    "pb_gm_axpy": (C.c_int, [C.c_int64, C.c_void_p, C.c_void_p, C.c_uint64]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


def load():
    """Load the CUDA library (built in-tree by porepy_b200/build.py).  Raises if missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not found: build it with `python -m porepy_b200.build` "
            "(porepy_b200 has no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int) -> None:
    """Map return codes to the reference's exceptions."""
    if rc == PB_OK:
        return
    lib = load()
    msg = lib.pb_last_error().decode(errors="replace")
    if rc == PB_ESINGULAR:
        # parity: numerics/linalg/matrix_operations.py:1487-1490
        raise ValueError(f"Error in inversion of local linear systems ({msg})")
    if rc == PB_ECELLTYPE:
        # parity: numerics/fv/_fvutils.py:735
        raise AssertionError(msg)
    if rc == PB_EINVAL:
        raise ValueError(msg)
    if rc == PB_ENOTIMPL:
        raise NotImplementedError(msg)
    raise RuntimeError(f"libporeb200: CUDA error: {msg}")


def ptr(a, typ):
    if a is None:
        return None
    return a.ctypes.data_as(typ)


def f64(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float64)


def require_gpu() -> None:
    lib = load()
    if lib.pb_device_count() < 1:
        raise RuntimeError("porepy_b200: no CUDA device visible and there is no CPU fallback")


# ------------------------------------------------------------------------------------------
# page-locked host buffers (pooled: cudaHostAlloc is slow, discretize() is called repeatedly)
# ------------------------------------------------------------------------------------------
import weakref  # noqa: E402

_POOL: dict = {}
_POOL_BYTES = [0]
_POOL_CAP = int(os.environ.get("POREB200_PINNED_POOL_BYTES", 64 << 30))


def _release(ptr: int, nbytes: int) -> None:
    if _lib is None:
        return
    if _POOL_BYTES[0] + nbytes <= _POOL_CAP:
        _POOL.setdefault(nbytes, []).append(ptr)
        _POOL_BYTES[0] += nbytes
    else:
        _lib.pb_host_free(C.c_void_p(ptr))


def pinned_empty(n: int, dtype=np.float64) -> np.ndarray:
    """Uninitialised 1-D array in page-locked host memory; returned to a pool when the array
    (and every view of it, e.g. a scipy matrix's ``data``) is garbage collected."""
    lib = load()
    nbytes = max(int(n) * np.dtype(dtype).itemsize, 8)
    free = _POOL.get(nbytes)
    if free:
        ptr = free.pop()
        _POOL_BYTES[0] -= nbytes
    else:
        out = C.c_void_p()
        check(lib.pb_host_alloc(nbytes, C.byref(out)))
        ptr = out.value
    buf = (C.c_char * nbytes).from_address(ptr)
    weakref.finalize(buf, _release, ptr, nbytes)
    return np.frombuffer(buf, dtype=dtype, count=int(n))
