"""ctypes binding of libvoxcarve.so — exactly the entry points include/voxcarve.h declares.

There is no fallback: if the library is missing or was built without its kernels, loading
raises, and every compute call needs a CUDA device (vc_create fails with VC_ERR_CUDA).
"""
import ctypes as C
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "lib", "libvoxcarve.so")

VC_OK, VC_ERR_ARG, VC_ERR_CUDA, VC_ERR_STATE, VC_ERR_CAPACITY, VC_ERR_COMM = 0, 1, 2, 3, 4, 5
VC_EXACT, VC_FAST_F32, VC_EXACT_FLAT = 0, 1, 2
VC_COLOR_CLOSEST, VC_COLOR_AVG = 1, 2
VC_MASK_BITS, VC_MASK_BGR8, VC_MASK_BGR8_RAW = 0, 1, 2
VC_MAX_TOTAL_VIEWS = 4096
VC_RAW_MAX_SIDE = 32766  # W and H of raw (distorted) input: cv::undistort refuses a side of 32767 or more


class GridDesc(C.Structure):
    _fields_ = [("X", C.c_int32), ("Y", C.c_int32), ("Z", C.c_int32), ("voxel_size", C.c_float),
                ("z_begin", C.c_int32), ("z_end", C.c_int32), ("device", C.c_int32)]


class Stats(C.Structure):
    _fields_ = [("last_carve_ms", C.c_double), ("last_classify_ms", C.c_double), ("nominal_voxel_views", C.c_uint64),
                ("executed_voxel_views", C.c_uint64), ("brick_corner_views", C.c_uint64),
                ("bricks_total", C.c_uint64), ("bricks_listed", C.c_uint64), ("flood_rounds", C.c_uint64), ("carve_launches", C.c_uint64),
                ("l2_persist_bytes", C.c_uint64), ("filter_rows", C.c_uint64), ("filter_slow_rows", C.c_uint64),
                ("filter_mismatches", C.c_uint64), ("subbrick_corner_views", C.c_uint64), ("volumes_compressible", C.c_uint64)]


# name -> (restype, argtypes); the single source of truth the symbol-export test checks against the header
_P = C.c_void_p
SIGNATURES = {
    "vc_create": (C.c_int, [C.POINTER(GridDesc), C.POINTER(_P)]),
    "vc_destroy": (None, [_P]),
    "vc_last_error": (C.c_char_p, [_P]),
    "vc_api_version": (C.c_int, []),
    "vc_set_stream": (C.c_int, [_P, _P]),
    "vc_synchronize": (C.c_int, [_P]),
    "vc_set_profiling": (C.c_int, [_P, C.c_int32]),
    "vc_set_views": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, _P, _P]),
    "vc_append_views": (C.c_int, [_P, C.c_int32, _P, _P, _P, C.c_int32, _P]),
    "vc_set_masks": (C.c_int, [_P, _P, C.c_int32]),
    "vc_set_images": (C.c_int, [_P, _P]),
    "vc_set_calibration": (C.c_int, [_P, _P, _P, C.c_int32]),
    "vc_set_images_raw": (C.c_int, [_P, _P]),
    "vc_download_masks": (C.c_int, [_P, _P]),
    "vc_download_images": (C.c_int, [_P, _P]),
    "vc_undistort_bgr": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P, C.c_int32, _P]),
    "vc_reset": (C.c_int, [_P]),
    "vc_carve": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.c_int32]),
    "vc_carve_download": (C.c_int, [_P, C.c_int32, _P, _P, C.c_uint64]),
    "vc_sparse_dims": (C.c_int, [_P, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    "vc_carve_download_sparse": (C.c_int, [_P, _P, C.c_uint64, _P, _P, C.c_uint64, C.POINTER(C.c_uint64)]),
    "vc_fast_carve": (C.c_int, [_P, C.c_int32]),
    "vc_color": (C.c_int, [_P, C.c_int32]),
    "vc_color_visible": (C.c_int, [_P, C.c_int32, C.c_float]),
    "vc_mc_classify": (C.c_int, [_P]),
    "vc_plan_slabs": (C.c_int, [_P, C.c_int32, C.POINTER(C.c_int32)]),
    "vc_set_slab": (C.c_int, [_P, C.c_int32, C.c_int32]),
    "vc_bind_volumes": (C.c_int, [_P, _P, _P]),
    "vc_device_volumes": (C.c_int, [_P, C.POINTER(_P), C.POINTER(_P)]),
    "vc_set_gathered": (C.c_int, [_P, C.c_int32]),
    "vc_alloc_full_volumes": (C.c_int, [_P]),
    "vc_halo_words": (C.c_int, [_P, C.POINTER(C.c_uint64)]),
    "vc_export_halo": (C.c_int, [_P, C.c_int32, C.POINTER(_P)]),
    "vc_import_halo": (C.c_int, [_P, C.c_int32, _P]),
    "vc_exchange_halos_peer": (C.c_int, [C.POINTER(_P), C.c_int32]),
    "vc_gather_peer": (C.c_int, [C.POINTER(_P), C.c_int32, C.c_int32]),
    "vc_comm_unique_id": (C.c_int, [_P]),
    "vc_comm_init": (C.c_int, [_P, C.c_int32, C.c_int32, _P]),
    "vc_comm_destroy": (C.c_int, [_P]),
    "vc_comm_info": (C.c_int, [_P, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "vc_exchange_halos": (C.c_int, [_P]),
    "vc_gather": (C.c_int, [_P, C.c_int32, C.POINTER(C.c_int32)]),
    "vc_comm_allreduce_u64": (C.c_int, [_P, _P, C.c_int32]),
    "vc_download_full": (C.c_int, [_P, C.c_int32, _P, C.c_uint64]),
    "vc_slab_words": (C.c_int, [_P, C.POINTER(C.c_uint64)]),
    "vc_upload_volumes": (C.c_int, [_P, _P, _P, C.c_uint64]),
    "vc_download_occupied": (C.c_int, [_P, _P, C.c_uint64]),
    "vc_download_seen": (C.c_int, [_P, _P, C.c_uint64]),
    "vc_count_occupied": (C.c_int, [_P, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "vc_surface_count": (C.c_int, [_P, C.POINTER(C.c_uint64)]),
    "vc_download_colors": (C.c_int, [_P, _P, _P, C.c_uint64]),
    "vc_download_mc": (C.c_int, [_P, _P, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "vc_get_stats": (C.c_int, [_P, C.POINTER(Stats)]),
    "vc_dense_upload": (C.c_int, [_P, _P]),
    "vc_dense_from_volumes": (C.c_int, [_P, C.c_int32, C.c_int32]),
    "vc_dense_apply_carved": (C.c_int, [_P]),
    "vc_dense_closure": (C.c_int, [_P, C.c_int32]),
    "vc_dense_download": (C.c_int, [_P, _P]),
    "vc_mc_mesh": (C.c_int, [_P, C.c_float, C.POINTER(C.c_uint64)]),
    "vc_download_mesh": (C.c_int, [_P, _P, _P, C.c_uint64]),
    "vc_mesh_from_volumes": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.c_float, C.POINTER(C.c_uint64)]),
    "vc_mesh_format_off": (C.c_int, [_P, C.c_float, C.c_float, C.c_float, C.c_float, C.POINTER(C.c_uint64)]),
    "vc_download_mesh_off": (C.c_int, [_P, C.c_uint64, _P, C.c_uint64]),
    "vc_format_g": (C.c_int, [C.c_int32, C.c_uint64, _P, _P, C.c_uint64, C.POINTER(C.c_uint64)]),
    "vc_selftest": (C.c_int, [C.c_int32, C.c_int32, C.c_uint64, C.c_uint64, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "vc_measure_peaks": (C.c_int, [C.c_int32, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
}

_lib = None


def load():
    """Load libvoxcarve.so (must have been built: python -m ar_voxel_project_b200.build)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} not built: run `python -m ar_voxel_project_b200.build` "
                               "(the engine has no CPU fallback)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the library lacks a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib
