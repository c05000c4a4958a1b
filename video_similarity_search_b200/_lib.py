"""ctypes binding of libslic_b200.so - the C ABI declared in include/slic_b200.h.

There is no CPU fallback: if the library is missing it is built with nvcc (sources are in-tree);
if that is impossible the import fails loudly.
"""
import ctypes
import os

from . import build as _build

_c = ctypes
_i32, _i64, _f32, _f64 = _c.c_int32, _c.c_int64, _c.c_float, _c.c_double
_ptr = _c.c_void_p

# name -> argument types (every function returns int status unless listed in _RESTYPES)
SIGNATURES = {
    "slic_abi_version": [],
    "slic_last_error": [],
    "slic_require_device": [],
    "slic_launch_count": [],
    "slic_profile_screen": [_i32],
    "slic_last_screen_time": [_ptr, _ptr],
    "slic_last_screen_exec_flop": [_ptr],
    "slic_screen_trace": [_i32, _ptr],
    "slic_normalize_rows": [_ptr, _i64, _i32, _i32, _ptr, _ptr, _ptr, _i32, _ptr],
    "slic_center_columns": [_ptr, _i64, _i32, _ptr, _ptr, _ptr],
    "slic_nn_exact_top1": [_ptr, _ptr, _i64, _ptr, _i64, _i32, _i32, _i64, _ptr, _ptr, _ptr],
    "slic_nn_top1": [_ptr, _ptr, _i64, _ptr, _ptr, _i64, _i32, _i32, _i32, _i64, _f32, _ptr, _ptr, _ptr, _ptr],
    "slic_sym_row_bests": [_ptr, _ptr, _i64, _i32, _i32, _i32, _i32, _ptr, _ptr],
    "slic_nn_top1_sym_part": [_ptr, _ptr, _i64, _i32, _i32, _i32, _i32, _ptr, _f32, _ptr, _ptr, _ptr],
    "slic_debug_sym_plan": [_i64, _i32, _i32, _i32, _i32, _i32, _ptr, _i64, _ptr],
    "slic_unpack_neighbor_keys": [_ptr, _i64, _ptr, _ptr, _ptr, _ptr],
    "slic_screen_scores_debug": [_ptr, _i64, _ptr, _i64, _i32, _ptr, _ptr],
    "slic_distance_matrix": [_ptr, _i64, _ptr, _i64, _i32, _i32, _i32, _i32, _ptr, _i64, _ptr],
    "slic_rows_topk": [_ptr, _i64, _i64, _i64, _i32, _i32, _ptr, _ptr, _ptr],
    "slic_topk_cosine": [_ptr, _i64, _ptr, _i64, _i32, _i32, _i32, _i64, _ptr, _ptr, _ptr],
    "slic_topk_cosine_tc": [_ptr, _ptr, _i64, _ptr, _ptr, _i64, _i32, _i32, _i32, _i32, _i64, _f32, _ptr, _ptr, _ptr, _ptr],
    "slic_hit_at_k": [_ptr, _i64, _i32, _ptr, _ptr, _ptr, _i32, _ptr, _ptr],
    "slic_finch_components": [_ptr, _i64, _i32, _f64, _ptr, _i32, _i32, _ptr, _ptr, _ptr, _ptr],
    "slic_finch_min_sim": [_ptr, _i64, _ptr, _i32, _i32, _ptr, _ptr, _ptr],
    "slic_finch_closest_link": [_ptr, _i64, _ptr, _i32, _i32, _ptr, _ptr, _ptr],
    "slic_compose_labels": [_ptr, _ptr, _i64, _ptr, _ptr],
    "slic_segmented_mean": [_ptr, _ptr, _i64, _i32, _i32, _ptr, _ptr],
    "slic_cluster_sums": [_ptr, _ptr, _i64, _i32, _i32, _ptr, _ptr, _ptr, _ptr],
    "slic_merge_cluster_sums": [_ptr, _ptr, _ptr, _i64, _i32, _i32, _ptr, _ptr, _ptr, _ptr],
    "slic_label_mask_u8": [_ptr, _i64, _ptr, _i64, _i32, _i32, _ptr, _ptr],
    "slic_label_mask_bits": [_ptr, _i64, _ptr, _i64, _i32, _ptr, _ptr],
    "slic_dense_labels": [_ptr, _i64, _ptr, _ptr, _ptr, _ptr],
    "slic_scatter_last_wins": [_ptr, _ptr, _i64, _i64, _i32, _ptr, _ptr, _ptr],
    "slic_cluster_metrics": [_ptr, _ptr, _i64, _i32, _i32, _i32, _ptr, _ptr],
    "slic_group_by_label": [_ptr, _i64, _i32, _ptr, _ptr, _ptr],
    "slic_first_neighbors_host": [_ptr, _i64, _i32, _i32, _ptr, _ptr],
    "slic_set_flann_threshold": [_i64],
    "slic_host_trace": [_i32, _ptr],
    "slic_set_upload_overlap": [_i32],
    "slic_copy_to_device": [_ptr, _ptr, _i64, _ptr],
    "slic_comm_create": [_ptr, _i32, _i64, _ptr],
    "slic_finch_multi": [_ptr, _ptr, _i64, _i32, _ptr, _i32, _i32, _ptr, _ptr, _ptr, _ptr, _ptr],
    "slic_comm_last_timeline": [_ptr, _ptr],
    "slic_comm_destroy": [_ptr],
    "slic_comm_window_create": [_i64, _ptr, _ptr],
    "slic_comm_connect": [_ptr, _i32, _i32, _ptr],
    "slic_comm_nn_top1": [_ptr, _ptr, _ptr, _i64, _i32, _i32, _ptr, _ptr, _ptr, _ptr],
    "slic_comm_finch": [_ptr, _ptr, _i64, _i32, _i32, _i32, _ptr, _ptr, _ptr, _ptr, _ptr, _ptr],
    "slic_finch": [_ptr, _i64, _i32, _ptr, _ptr, _ptr, _i32, _i32, _i32, _ptr, _ptr, _ptr, _ptr, _ptr, _ptr],
    "slic_finch_host": [_ptr, _i64, _i32, _ptr, _i32, _i32, _ptr, _ptr, _ptr, _ptr, _ptr],
    "slic_kmeans_plusplus": [_ptr, _i64, _i32, _i32, _i64, _ptr, _i32, _ptr, _ptr],
    "slic_spherical_kmeans": [_ptr, _i64, _i32, _i32, _ptr, _ptr, _ptr, _i32, _i32, _i32, _f64, _ptr, _ptr, _ptr, _ptr,
                              _ptr, _ptr],
}
_RESTYPES = {"slic_last_error": _c.c_char_p, "slic_launch_count": _c.c_int64}

SLIC_F32, SLIC_F64 = 0, 1
SLIC_METRIC_COSINE, SLIC_METRIC_EUCLIDEAN = 0, 1

_lib = None


class SlicError(RuntimeError):
    """A C-ABI call returned a negative status."""


def library_path():
    return _build.LIB_PATH


def load(build_if_missing=True):
    """Load (building first if necessary) libslic_b200.so and attach the prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.exists(path):
        if not build_if_missing:
            raise ImportError("libslic_b200.so is missing; run `python -m video_similarity_search_b200.build`")
        _build.build()
    lib = ctypes.CDLL(path)
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)           # AttributeError here = header / library out of sync: fail loudly
        fn.argtypes = argtypes
        fn.restype = _RESTYPES.get(name, _c.c_int)
    if lib.slic_abi_version() != 1:
        raise ImportError("libslic_b200.so ABI version mismatch")
    _lib = lib
    return lib


def check(status, what):
    if status != 0:
        msg = load().slic_last_error()
        raise SlicError("%s failed with status %d: %s" % (what, status, msg.decode() if msg else "?"))


def call(name, *args):
    lib = load()
    check(getattr(lib, name)(*args), name)
