"""ctypes binding of include/gsplat_b200.h.  Loading fails loudly when the library is missing; there is
no Python/CPU implementation of any entry point."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libgsplat_b200.so")

GS_OK, GS_ERR_INVALID, GS_ERR_CUDA, GS_ERR_OOM, GS_ERR_CAPACITY, GS_ERR_EMPTY = 0, -1, -2, -3, -4, -5
GS_FORMAT_RGBA8, GS_FORMAT_RGBA32F = 0, 1
GS_RENDER_OUT_DEVICE, GS_RENDER_REUSE_SORT, GS_RENDER_OUT_TILED, GS_RENDER_OUT_PEER = 1, 2, 4, 8
GS_RENDER_STATS, GS_RENDER_DEPTH_DEVICE = 16, 32


class GsStats(C.Structure):
    _fields_ = [
        ("n_splats", C.c_uint32), ("n_sorted", C.c_uint32), ("n_dropped", C.c_uint32), ("n_visible", C.c_uint32),
        ("n_instances", C.c_uint64), ("n_tiles", C.c_uint32), ("width", C.c_uint32), ("height", C.c_uint32),
        ("min_depth", C.c_double), ("max_depth", C.c_double),
        ("ms_sort", C.c_float), ("ms_project", C.c_float), ("ms_bin", C.c_float), ("ms_raster", C.c_float),
        ("ms_total", C.c_float), ("kernel_launches", C.c_uint32), ("n_instances_kept", C.c_uint32),
        ("n_tile_instances", C.c_uint64), ("n_records_streamed", C.c_uint64), ("n_pair_tests", C.c_uint64),
        ("n_pair_hits", C.c_uint64),
        ("n_slabs", C.c_uint32), ("n_slabs_run", C.c_uint32), ("n_slab_entries", C.c_uint64),
    ]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_ }


class GsRenderParams(C.Structure):
    _fields_ = [
        ("proj", C.c_float * 16), ("modelview", C.c_float * 16),
        ("width", C.c_uint32), ("height", C.c_uint32), ("focal", C.c_float),
        ("bg_rgba", C.c_float * 4), ("has_cutout", C.c_int32), ("cutout16", C.c_float * 16),
        ("out_format", C.c_int32), ("flags", C.c_uint32), ("depth_in", C.c_void_p),
    ]


# every symbol include/gsplat_b200.h declares: name -> (restype, argtypes)
_P = C.c_void_p
SYMBOLS = {
    "gs_create": (C.c_int, [C.c_int, C.POINTER(_P)]),
    "gs_destroy": (C.c_int, [_P]),
    "gs_last_error": (C.c_char_p, [_P]),
    "gs_version": (C.c_char_p, []),
    "gs_bin_size": (C.c_uint32, []),
    "gs_clear": (C.c_int, [_P]),
    "gs_push_splats": (C.c_int, [_P, _P, C.c_uint32]),
    "gs_reserve": (C.c_int, [_P, C.c_uint32]),
    "gs_push_packed": (C.c_int, [_P, _P, _P, _P, C.c_uint32]),
    "gs_num_splats": (C.c_int, [_P, C.POINTER(C.c_uint32)]),
    "gs_read_packed": (C.c_int, [_P, C.c_uint32, C.c_uint32, _P, _P, _P]),
    "gs_sort": (C.c_int, [_P, C.POINTER(C.c_float), C.POINTER(C.c_float), _P, C.POINTER(C.c_uint32)]),
    "gs_render": (C.c_int, [_P, C.POINTER(GsRenderParams), _P, C.POINTER(GsStats)]),
    "gs_render_async": (C.c_int, [_P, C.POINTER(GsRenderParams), _P, C.POINTER(C.c_uint64)]),
    "gs_wait": (C.c_int, [_P, C.c_uint64, C.POINTER(GsStats)]),
    "gs_render_stereo": (C.c_int, [_P, C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(GsRenderParams), C.POINTER(_P),
                                   C.POINTER(GsStats)]),
    "gs_read_projected": (C.c_int, [_P, C.c_uint32, C.c_uint32, _P]),
    "gs_get_stats": (C.c_int, [_P, C.POINTER(GsStats)]),
    "gs_set_shard": (C.c_int, [_P, C.c_uint32, C.c_uint32]),
    "gs_owned_tiles": (C.c_uint32, [C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32]),
    "gs_assemble_tiles": (C.c_int, [_P, _P, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int32, _P]),
    "gs_peer_export": (C.c_int, [_P, C.c_size_t, _P]),
    "gs_peer_import": (C.c_int, [_P, C.c_uint32, C.c_uint32, _P]),
    "gs_peer_frame": (C.c_int, [_P, C.c_uint64, C.POINTER(_P)]),
    "gs_device_alloc": (C.c_int, [_P, C.c_size_t, C.POINTER(_P)]),
    "gs_device_free": (C.c_int, [_P, _P]),
    "gs_host_alloc": (C.c_int, [_P, C.c_size_t, C.POINTER(_P)]),
    "gs_host_free": (C.c_int, [_P, _P]),
    "gs_memcpy_d2h": (C.c_int, [_P, _P, _P, C.c_size_t]),
    "gs_stream": (_P, [_P]),
    "gs_synchronize": (C.c_int, [_P]),
}

_lib = None


def load(path: str = LIB_PATH):
    """dlopen libgsplat_b200.so (the in-tree build unless `path` names another) and type every entry point.  Raises if
    the library was not built.  The first call decides which library the process uses."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(path):
        raise RuntimeError(
            f"{path} is missing: build it with __graft_entry__.build() "
            "(nvcc, sm_100a).  There is no CPU fallback for the splat path.")
    lib = C.CDLL(path)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the header and the library disagree
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
