"""ctypes binding of libfea_b200.so (include/fea_b200.h).

The product path has no CPU fallback: if the CUDA library is missing or a call fails, a
``FeaError`` is raised.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libfea_b200.so")

# every symbol include/fea_b200.h declares (tests check the library exports all of them)
EXPORTS = [
    "fea_version", "fea_ctx_create", "fea_ctx_create_prio", "fea_ctx_destroy", "fea_last_error", "fea_host_alloc",
    "fea_host_free", "fea_device_alloc", "fea_device_free", "fea_device_upload", "fea_ctx_synchronize", "fea_ctx_event_record", "fea_ctx_event_elapsed_ms",
    "fea_ctx_wait_ctx", "fea_ctx_set_int", "fea_ctx_kernel_launches", "fea_batch_create",
    "fea_batch_create_from_conditions", "fea_batch_get_setup", "fea_batch_get_materials", "fea_batch_rasterize_regions",
    "fea_batch_classify", "fea_batch_stage_outputs", "fea_batch_staged_region_images", "fea_batch_fetch_outputs",
    "fea_batch_rasterize_cell_components", "fea_batch_assemble",
    "fea_batch_solve", "fea_batch_rasterize", "fea_batch_destroy", "fea_batch_download",
    "fea_batch_download_images", "fea_batch_rasterize_flags", "fea_batch_cell_strain_stress", "fea_batch_get_info", "fea_batch_get_solve_stats", "fea_batch_get_refine_rounds",
    "fea_batch_get_timed_launches",
    "fea_batch_sample_sizes", "fea_batch_get_conn", "fea_batch_get_element_stiffness",
    "fea_batch_get_csr", "fea_batch_spmv", "fea_rasterize_fields", "fea_solve_batch",
    "fea_batch_set_refinement", "fea_batch_get_mg_levels", "fea_batch_get_level_csr", "fea_batch_mg_apply",
]

STATUS_NAMES = {0: "OK", 1: "BAD_ARG", 2: "CUDA_ERROR", 3: "OUT_OF_MEMORY", 4: "BAD_STATE", 5: "MESH_ERROR"}
SAMPLE_NOT_RUN, SAMPLE_CONVERGED, SAMPLE_MAX_ITER, SAMPLE_BREAKDOWN, SAMPLE_EMPTY_ROW, SAMPLE_STAGNATED = -1, 0, 1, 2, 3, 4


class FeaError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libfea_b200: %s: %s" % (STATUS_NAMES.get(code, code), msg))
        self.code = code


class BatchDesc(C.Structure):
    _fields_ = [
        ("n_samples", C.c_int32), ("nodes_per_cell", C.c_int32),
        ("vtx_off", C.c_void_p), ("cell_off", C.c_void_p), ("reg_off", C.c_void_p),
        ("xy", C.c_void_p), ("conn", C.c_void_p), ("cell_region", C.c_void_p),
        ("D", C.c_void_p), ("fixed", C.c_void_p), ("rhs", C.c_void_p),
    ]


class ConditionsDesc(C.Structure):
    """fea_conditions_desc (include/fea_b200.h)."""
    _fields_ = [
        ("n_meshes", C.c_int32), ("n_samples", C.c_int32), ("nodes_per_cell", C.c_int32), ("reserved", C.c_int32),
        ("mesh_vtx_off", C.c_void_p), ("mesh_cell_off", C.c_void_p), ("xy", C.c_void_p), ("conn", C.c_void_p),
        ("sample_mesh", C.c_void_p),
        ("vforce_off", C.c_void_p), ("vforce_tag", C.c_void_p), ("vforce_mag", C.c_void_p),
        ("eforce_off", C.c_void_p), ("eforce_tag", C.c_void_p), ("eforce_mag", C.c_void_p),
        ("vfix_off", C.c_void_p), ("vfix_tag", C.c_void_p),
        ("efix_off", C.c_void_p), ("efix_tag", C.c_void_p),
        ("mat_off", C.c_void_p), ("mat_E_nu", C.c_void_p), ("mat_coord_off", C.c_void_p), ("mat_coords", C.c_void_p),
        ("default_E_nu", C.c_void_p),
    ]


class BatchInfo(C.Structure):
    _fields_ = [
        ("n_vertices", C.c_int64), ("n_cells", C.c_int64), ("n_active_dofs", C.c_int64),
        ("nnz", C.c_int64), ("block_rows", C.c_int64), ("sell_blocks", C.c_int64),
        ("n_flipped", C.c_int32), ("max_row_blocks", C.c_int32),
    ]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class SolveStats(C.Structure):
    _fields_ = [
        ("iterations", C.c_int32), ("n_converged", C.c_int32),
        ("spmv_launches_timed", C.c_int32), ("update_launches_timed", C.c_int32),
        ("spmv_ms_avg", C.c_float), ("update_ms_avg", C.c_float), ("solve_ms", C.c_float),
        ("kernel_launches", C.c_int64),
        ("cluster_systems", C.c_int32), ("cluster_count", C.c_int32), ("cluster_iterations", C.c_int64),
        ("cluster_ms", C.c_float), ("cluster_size", C.c_int32),
        ("refined_systems", C.c_int32), ("pad_", C.c_int32),
        ("cluster_block_reads_tmem", C.c_int64), ("cluster_block_reads_smem", C.c_int64), ("cluster_block_reads_l2", C.c_int64),
    ]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class MgLevel(C.Structure):
    """fea_mg_level (include/fea_b200.h)."""
    _fields_ = [
        ("n_vertices", C.c_int64), ("n_cells", C.c_int64), ("n_active_dofs", C.c_int64), ("nnz", C.c_int64),
        ("lambda_max", C.c_double), ("vcycle_ms", C.c_double),
    ]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


_lib: Optional[C.CDLL] = None


def load_library(path: Optional[str] = None) -> C.CDLL:
    """Load libfea_b200.so; raises if it has not been built (python __graft_entry__.py)."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    path = path or os.environ.get("FEA_B200_LIB", LIB_PATH)
    if not os.path.exists(path):
        raise FeaError(-1, "CUDA library not built: %s is missing (run `python __graft_entry__.py`); "
                           "there is no CPU fallback" % path)
    lib = C.CDLL(path)
    P, I32, I64, F64 = C.c_void_p, C.c_int32, C.c_int64, C.c_double
    sig = {
        "fea_version": (C.c_int, [P, P]),
        "fea_ctx_create": (C.c_int, [C.c_int, C.POINTER(P)]),
        "fea_ctx_create_prio": (C.c_int, [C.c_int, C.c_int, C.POINTER(P)]),
        "fea_ctx_destroy": (C.c_int, [P]),
        "fea_ctx_wait_ctx": (C.c_int, [P, P]),
        "fea_ctx_set_int": (C.c_int, [P, C.c_char_p, C.c_int64]),
        "fea_last_error": (C.c_char_p, [P]),
        "fea_host_alloc": (C.c_int, [P, C.c_size_t, C.POINTER(P)]),
        "fea_host_free": (C.c_int, [P, P]),
        "fea_ctx_synchronize": (C.c_int, [P]),
        "fea_device_alloc": (C.c_int, [P, C.c_size_t, C.POINTER(P)]),
        "fea_device_free": (C.c_int, [P, P]),
        "fea_device_upload": (C.c_int, [P, P, P, C.c_size_t]),
        "fea_ctx_event_record": (C.c_int, [P, I32]),
        "fea_ctx_event_elapsed_ms": (C.c_int, [P, I32, I32, P]),
        "fea_ctx_kernel_launches": (C.c_int, [P, P]),
        "fea_batch_create": (C.c_int, [P, C.POINTER(BatchDesc), C.POINTER(P)]),
        "fea_batch_create_from_conditions": (C.c_int, [P, C.POINTER(ConditionsDesc), C.POINTER(P)]),
        "fea_batch_get_setup": (C.c_int, [P, P, P, P, P, P]),
        "fea_batch_get_materials": (C.c_int, [P, P, P, P]),
        "fea_batch_rasterize_regions": (C.c_int, [P, P, P]),
        "fea_batch_classify": (C.c_int, [P, P, P]),
        "fea_batch_stage_outputs": (C.c_int, [P, P]),
        "fea_batch_staged_region_images": (C.c_int, [P, P]),
        "fea_batch_fetch_outputs": (C.c_int, [P, P, P, P, P, P, P, P, P, P, P]),
        "fea_batch_rasterize_cell_components": (C.c_int, [P, I32, I32, P, F64, P, P]),
        "fea_batch_assemble": (C.c_int, [P]),
        "fea_batch_solve": (C.c_int, [P, F64, I32]),
        "fea_batch_rasterize": (C.c_int, [P, I32, P, F64]),
        "fea_batch_destroy": (C.c_int, [P]),
        "fea_batch_download": (C.c_int, [P, P, P, P, P, P]),
        "fea_batch_download_images": (C.c_int, [P, P]),
        "fea_batch_get_info": (C.c_int, [P, C.POINTER(BatchInfo)]),
        "fea_batch_get_solve_stats": (C.c_int, [P, C.POINTER(SolveStats)]),
        "fea_batch_get_refine_rounds": (C.c_int, [P, P]),
        "fea_batch_get_timed_launches": (C.c_int, [P, I32, P, P, P]),
        "fea_batch_sample_sizes": (C.c_int, [P, P, P]),
        "fea_batch_get_conn": (C.c_int, [P, P, P]),
        "fea_batch_get_element_stiffness": (C.c_int, [P, P]),
        "fea_batch_get_csr": (C.c_int, [P, I32, P, P, P]),
        "fea_batch_spmv": (C.c_int, [P, I32, P, P]),
        "fea_batch_cell_strain_stress": (C.c_int, [P, I32, P, P]),
        "fea_batch_rasterize_flags": (C.c_int, [P, P, P, P]),
        "fea_rasterize_fields": (C.c_int, [P, P, C.c_int64, P, C.c_int64, I32, P, I32, I32, P, P, I32, P]),
        "fea_batch_set_refinement": (C.c_int, [P, I32]),
        "fea_batch_get_mg_levels": (C.c_int, [P, I32, C.POINTER(MgLevel), P]),
        "fea_batch_get_level_csr": (C.c_int, [P, I32, P, P, P]),
        "fea_batch_mg_apply": (C.c_int, [P, P, P]),
        "fea_solve_batch": (C.c_int, [P, C.POINTER(BatchDesc), F64, I32, I32, P, F64, P, P, P, P, P, P,
                                      C.POINTER(SolveStats)]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)
