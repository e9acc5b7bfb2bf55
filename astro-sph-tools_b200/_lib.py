"""ctypes binding of libastsph_b200.so (include/astro_sph_b200.h).

The library is built in-tree by ``__graft_entry__.build()`` (nvcc, sm_100a).  If it is missing, or no CUDA
device is visible, every compute entry point raises: there is no CPU fallback on the product path.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("ASTSPH_B200_LIB", os.path.join(_HERE, "csrc", "libastsph_b200.so"))

AST_OK, AST_EINVAL, AST_EWORKSPACE, AST_ECUDA, AST_EUNSUPPORTED = 0, 1, 2, 3, 4
FLAG_PERIODIC, FLAG_ACCUMULATE, FLAG_TIMING, FLAG_ORDER_AUTO, FLAG_ORDER_ALWAYS = 1, 2, 4, 8, 16
MAX_PROPS = 2
TILE = 32

KERNEL_IDS = {"cubic_spline_3d": 0, "wendland_c2_2d": 1, "wendland_c2_3d": 2, "cubic_spline_2d": 3}
KERNEL_TABLE = 4


class Project2DParams(C.Structure):
    _fields_ = [("n", C.c_int64), ("axis", C.c_int32), ("nx", C.c_int32), ("ny", C.c_int32), ("kernel_id", C.c_int32),
                ("n_prop", C.c_int32), ("flags", C.c_int32),
                ("x_min", C.c_double), ("x_max", C.c_double), ("y_min", C.c_double), ("y_max", C.c_double),
                ("box_a", C.c_double), ("box_b", C.c_double),
                ("small_max_px", C.c_int64), ("huge_min_tiles", C.c_int64),
                ("pair_capacity", C.c_int64), ("huge_capacity", C.c_int64),
                ("kernel_table", C.c_void_p), ("kernel_table_n", C.c_int32), ("kernel_dim", C.c_int32)]


class Project2DStats(C.Structure):
    _fields_ = [("n_pairs", C.c_int64), ("n_huge", C.c_int64), ("n_rounds", C.c_int64), ("n_launches", C.c_int64),
                ("stage_ms", C.c_float * 8), ("reordered", C.c_int32), ("reserved", C.c_int32)]


class Grid3DParams(C.Structure):
    _fields_ = [("n", C.c_int64), ("nx", C.c_int32), ("ny", C.c_int32), ("nz", C.c_int32), ("kernel_id", C.c_int32),
                ("flags", C.c_int32), ("reserved", C.c_int32),
                ("lo", C.c_double * 3), ("hi", C.c_double * 3), ("box", C.c_double * 3),
                ("small_max_vox", C.c_int64), ("huge_min_bricks", C.c_int64),
                ("pair_capacity", C.c_int64), ("huge_capacity", C.c_int64),
                ("kernel_table", C.c_void_p), ("kernel_table_n", C.c_int32), ("kernel_dim", C.c_int32),
                ("x_begin", C.c_int32), ("x_end", C.c_int32)]


class KnnParams(C.Structure):
    _fields_ = [("n", C.c_int64), ("k", C.c_int32), ("flags", C.c_int32), ("box", C.c_double),
                ("lo", C.c_double * 3), ("hi", C.c_double * 3), ("cell_target", C.c_double),
                ("q_begin", C.c_int64), ("q_count", C.c_int64)]


TABLE_MAX_DIM = 4
TABLE_POW10 = 1


class TableParams(C.Structure):
    _fields_ = [("ndim", C.c_int32), ("shape", C.c_int32 * TABLE_MAX_DIM), ("axes", C.c_void_p * TABLE_MAX_DIM),
                ("table", C.c_void_p), ("fill_value", C.c_double), ("fixed_dim", C.c_int32), ("flags", C.c_int32),
                ("fixed_value", C.c_double)]


ROUTE_MAX_WORLD = 32


class SlabRouteParams(C.Structure):
    _fields_ = [("n", C.c_int64), ("world", C.c_int32), ("periodic", C.c_int32), ("covers_all", C.c_int32), ("reserved", C.c_int32),
                ("length", C.c_double), ("w", C.c_double), ("bounds", C.c_double * (ROUTE_MAX_WORLD + 1))]


class GridRouteParams(C.Structure):
    _fields_ = [("n", C.c_int64), ("world", C.c_int32), ("periodic", C.c_int32),
                ("nx", C.c_int32), ("ny", C.c_int32), ("nz", C.c_int32), ("reserved", C.c_int32),
                ("lo", C.c_double * 3), ("hi", C.c_double * 3), ("box", C.c_double * 3),
                ("edges", C.c_int32 * (ROUTE_MAX_WORLD + 1))]


class WorkspaceError(RuntimeError):
    """AST_EWORKSPACE: a capacity or the workspace was too small (message says what is needed)."""


_lib = None

# every symbol include/astro_sph_b200.h declares (tests check that the built library exports all of them)
EXPORTS = ["ast_project2d_workspace_bytes", "ast_project2d", "ast_bin2d", "ast_contrib_count2d", "ast_kernel_eval",
           "ast_sort_workspace_bytes", "ast_radix_sort_u64", "ast_grid3d_workspace_bytes", "ast_grid3d", "ast_bin3d",
           "ast_knn_workspace_bytes", "ast_knn_h", "ast_knn_query", "ast_match_ids_workspace_bytes", "ast_match_ids", "ast_gather_rows", "ast_table_interp",
           "ast_slab_route_workspace_bytes", "ast_slab_route_count", "ast_slab_route_write",
           "ast_grid_route_workspace_bytes", "ast_grid_route_count", "ast_grid_route_write",
           "ast_last_error", "ast_abi_version", "ast_tile_size",
           "ast_device_sm_count"]


def load():
    """Load the shared library (no CUDA call is made here)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"CUDA library not built: {LIB_PATH} is missing. Run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). There is no CPU fallback.")
        lib = C.CDLL(LIB_PATH)
        lib.ast_last_error.restype = C.c_char_p
        for name in EXPORTS:
            if name != "ast_last_error":
                getattr(lib, name).restype = C.c_int
        _lib = lib
    return _lib


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("astro_sph_tools_b200 needs a CUDA device (built for sm_100a); there is no CPU fallback")
    return torch


def check(rc):
    if rc == AST_OK:
        return
    msg = load().ast_last_error().decode("utf-8", "replace")
    if rc == AST_EINVAL:
        raise ValueError(msg)
    if rc == AST_EWORKSPACE:
        raise WorkspaceError(msg)
    if rc == AST_EUNSUPPORTED:
        raise NotImplementedError(msg)
    raise RuntimeError(f"CUDA failure in libastsph_b200: {msg}")


def ptr(t):
    """raw device pointer of a torch tensor (or None)"""
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def stream_ptr(stream=None):
    import torch
    s = stream if stream is not None else torch.cuda.current_stream()
    return C.c_void_p(s.cuda_stream)
