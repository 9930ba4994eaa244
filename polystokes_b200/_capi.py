"""ctypes binding of the C ABI in ``include/polystokes_b200.h``.

The product library is ``libpolystokes_b200.so`` (CUDA, sm_100a).  There is no CPU fallback: if the
library is missing or no CUDA device is present the calls fail loudly.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
PRODUCT_LIB = os.path.join(_HERE, "libpolystokes_b200.so")

PS_UNSUPPORTED_SOLVER, PS_INCOMPLETE, PS_INVALID, PS_FAILED, PS_NOCONVERGE, PS_SUCCESS, PS_NOCHANGE = -4, -3, -2, -1, 0, 1, 2
PS_MEM_HOST, PS_MEM_DEVICE = 0, 1
PS_NUM_STAGES = 11
STAGE_NAMES = ["upload", "weights", "classify", "reduced", "indices", "region_matrices", "matrix_blocks", "assemble",
               "solve", "writeback", "download"]

CANCEL_CB = C.CFUNCTYPE(C.c_int, C.c_void_p)


class ps_params(C.Structure):
    _fields_ = [
        ("nx", C.c_int32), ("ny", C.c_int32), ("nz", C.c_int32),
        ("dx", C.c_double), ("dt", C.c_double), ("origin", C.c_double * 3),
        ("constantDensity", C.c_double), ("tolerance", C.c_double),
        ("maxSolverIterations", C.c_int32),
        ("activeLiquidBoundaryLayerSize", C.c_int32), ("activeSolidBoundaryLayerSize", C.c_int32),
        ("doReducedRegions", C.c_int32), ("doTile", C.c_int32), ("tileSize", C.c_int32), ("tilePadding", C.c_int32),
        ("exportMatrices", C.c_int32), ("exportComponentMatrices", C.c_int32), ("exportStats", C.c_int32),
        ("exportDataPrefix", C.c_char * 256),
        ("doSolve", C.c_int32), ("keepNonConvergedResults", C.c_int32), ("useWarmStart", C.c_int32),
        ("matrixSetup", C.c_int32), ("solverType", C.c_int32),
        ("useInputSurfaceWeights", C.c_int32), ("useInputCollisionWeights", C.c_int32),
        ("minDensity", C.c_double), ("maxDensity", C.c_double),
        ("device", C.c_int32), ("checkEvery", C.c_int32),
        ("cancel_cb", CANCEL_CB), ("cancel_ctx", C.c_void_p),
    ]


class ps_fields_in(C.Structure):
    _fields_ = [("memory", C.c_int32), ("surface", C.c_void_p), ("collision", C.c_void_p), ("viscosity", C.c_void_p),
                ("velocity", C.c_void_p * 3), ("collisionvel", C.c_void_p * 3)]


class ps_fields_out(C.Structure):
    _fields_ = [("memory", C.c_int32), ("velocity", C.c_void_p * 3), ("valid", C.c_void_p * 3)]


class ps_stats(C.Structure):
    _fields_ = [("dimData", C.c_double * 27), ("solveData", C.c_double * 6), ("result", C.c_int32), ("usedBiCGStab", C.c_int32),
                ("stage_ms", C.c_double * PS_NUM_STAGES), ("gpu_launches", C.c_int64)]


# every symbol include/polystokes_b200.h declares
SYMBOLS = ["ps_create", "ps_destroy", "ps_step", "ps_setup", "ps_solve", "ps_export", "ps_last_error", "ps_get_count", "ps_get_real",
           "ps_get_index_field", "ps_get_weight_field", "ps_get_csr", "ps_get_vector", "ps_apply", "ps_time_kernel", "ps_kernel_bytes", "ps_timer",
           "ps_comm_unique_id", "ps_comm_init", "ps_get_partition", "ps_create_multi", "ps_set_params", "ps_alloc_pinned", "ps_free_pinned",
           "ps_set_partition", "ps_rebalance"]

_cache = {}


def load(path=None):
    """Load the C-ABI library and declare its prototypes.  ``path`` defaults to the CUDA product library."""
    path = path or PRODUCT_LIB
    if path in _cache:
        return _cache[path]
    if not os.path.exists(path):
        raise RuntimeError(f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(nvcc, sm_100a).  polystokes_b200 has no CPU fallback.")
    L = C.CDLL(path)
    H = C.c_void_p
    L.ps_create.argtypes = [C.POINTER(ps_params), C.POINTER(H)]; L.ps_create.restype = C.c_int
    L.ps_create_multi.argtypes = [C.POINTER(ps_params), C.c_int, C.POINTER(C.c_int), C.POINTER(H)]; L.ps_create_multi.restype = C.c_int
    L.ps_destroy.argtypes = [H]; L.ps_destroy.restype = None
    L.ps_set_params.argtypes = [H, C.POINTER(ps_params)]; L.ps_set_params.restype = C.c_int
    L.ps_alloc_pinned.argtypes = [C.c_size_t]; L.ps_alloc_pinned.restype = C.c_void_p
    L.ps_free_pinned.argtypes = [C.c_void_p]; L.ps_free_pinned.restype = None
    L.ps_step.argtypes = [H, C.POINTER(ps_fields_in), C.POINTER(ps_fields_out), C.POINTER(ps_stats)]; L.ps_step.restype = C.c_int
    L.ps_setup.argtypes = [H, C.POINTER(ps_fields_in)]; L.ps_setup.restype = C.c_int
    L.ps_solve.argtypes = [H, C.POINTER(ps_fields_out), C.POINTER(ps_stats)]; L.ps_solve.restype = C.c_int
    L.ps_export.argtypes = [H, C.c_char_p, C.c_int]; L.ps_export.restype = C.c_int
    L.ps_last_error.argtypes = []; L.ps_last_error.restype = C.c_char_p
    L.ps_get_count.argtypes = [H, C.c_char_p]; L.ps_get_count.restype = C.c_int64
    L.ps_get_real.argtypes = [H, C.c_char_p]; L.ps_get_real.restype = C.c_double
    L.ps_get_index_field.argtypes = [H, C.c_int, C.c_int, C.c_void_p]; L.ps_get_index_field.restype = C.c_int64
    L.ps_get_weight_field.argtypes = [H, C.c_int, C.c_int, C.c_void_p]; L.ps_get_weight_field.restype = C.c_int64
    L.ps_get_csr.argtypes = [H, C.c_char_p] + [C.POINTER(C.c_int64)] * 3 + [C.c_void_p] * 3; L.ps_get_csr.restype = C.c_int
    L.ps_get_vector.argtypes = [H, C.c_char_p, C.c_void_p]; L.ps_get_vector.restype = C.c_int64
    L.ps_apply.argtypes = [H, C.c_void_p, C.c_void_p]; L.ps_apply.restype = C.c_int
    L.ps_time_kernel.argtypes = [H, C.c_char_p, C.c_int]; L.ps_time_kernel.restype = C.c_double
    L.ps_kernel_bytes.argtypes = [H, C.c_char_p]; L.ps_kernel_bytes.restype = C.c_double
    L.ps_timer.argtypes = [H, C.c_int]; L.ps_timer.restype = C.c_double
    L.ps_comm_unique_id.argtypes = [C.c_void_p]; L.ps_comm_unique_id.restype = C.c_int
    L.ps_comm_init.argtypes = [H, C.c_int, C.c_int, C.c_void_p]; L.ps_comm_init.restype = C.c_int
    L.ps_get_partition.argtypes = [H] + [C.POINTER(C.c_int32)] * 4; L.ps_get_partition.restype = C.c_int
    L.ps_set_partition.argtypes = [H, C.c_void_p]; L.ps_set_partition.restype = C.c_int
    L.ps_rebalance.argtypes = [H, C.c_void_p]; L.ps_rebalance.restype = C.c_int
    _cache[path] = L
    return L
