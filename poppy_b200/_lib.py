"""ctypes loader of poppy_b200/libpoppy_cuda.so (include/poppy_cuda.h, include/poppy_host.h).

The library is built in-tree by poppy_b200/build.py (nvcc, sm_100a). There is no fallback of any kind: if the
shared object is missing or cannot be loaded this module raises, and every renderer entry point fails when no
CUDA device is present."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("POPPY_CUDA_LIB") or os.path.join(_HERE, "libpoppy_cuda.so")   # override: A/B builds only

_lib = None


class PoppyCudaError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"poppy_cuda error {code}: {msg}")
        self.code = code


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing - build it with `python -m poppy_b200.build` "
                          "(the morph renderer is native CUDA; there is no Python/CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    vp, i32, u64p = C.c_void_p, C.c_int, C.POINTER(C.c_uint64)
    sigs = {
        "poppy_cuda_device_count": (i32, []),
        "poppy_cuda_create": (i32, [C.POINTER(vp), i32, i32, i32, i32, i32, i32, i32]),
        "poppy_cuda_destroy": (None, [vp]),
        "poppy_cuda_get_info": (i32, [vp] + [C.POINTER(i32)] * 6),
        "poppy_cuda_set_keep_stages": (i32, [vp, i32]),
        # host stages (include/poppy_host.h)
        "poppy_host_morph_points": (i32, [vp, vp, i32, C.c_double, i32, i32, vp]),
        "poppy_host_triangulate": (i32, [vp, i32, i32, i32, vp, i32, C.POINTER(i32)]),
        "poppy_host_triangulate_next": (i32, [vp, i32, i32, i32, vp, i32, C.POINTER(i32)]),
        "poppy_host_chain_ratio": (C.c_double, [i32, i32]),
        "poppy_host_plan_create": (i32, [C.POINTER(vp), vp, vp, i32, i32, i32, i32, vp, i32, i32]),
        "poppy_host_plan_triangles": (i32, [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(i32)]),
        "poppy_host_plan_points": (i32, [vp, i32, C.POINTER(vp)]),
        "poppy_host_plan_destroy": (None, [vp]),
        "poppy_morph_images": (i32, [vp, vp, C.c_size_t, vp, C.c_size_t, vp, C.c_size_t, vp, vp, i32, C.c_double,
                               C.c_double, vp, C.c_size_t, vp]),
        "poppy_host_last_error": (C.c_char_p, []),
        "poppy_shim_morph_images": (i32, [i32, i32, i32, vp, C.c_size_t, vp, C.c_size_t, vp, C.c_size_t, vp, vp, i32, C.c_double, C.c_double,
                                    vp, C.c_size_t, vp]),
        "poppy_shim_morph_sequence": (i32, [i32, i32, i32, vp, C.c_size_t, vp, C.c_size_t, vp, C.c_size_t, vp, vp, i32, i32, vp, vp]),
        "poppy_shim_release": (None, []),
        "poppy_host_writer_create": (i32, [C.POINTER(vp), vp, i32, vp, vp, i32, vp]),
        "poppy_host_writer_create_i420": (i32, [C.POINTER(vp), vp, i32, vp, vp, i32, vp]),
        "poppy_host_writer_create_ffv1": (i32, [C.POINTER(vp), vp, i32, vp, vp]),
        "poppy_host_ffv1_config": (i32, [i32, i32, vp, C.c_size_t, C.POINTER(C.c_size_t)]),
        "poppy_host_mkv_open": (i32, [C.POINTER(vp), C.c_char_p, i32, i32, i32, i32]),
        "poppy_host_mkv_write": (i32, [vp, vp, C.c_size_t]),
        "poppy_host_mkv_close": (i32, [vp]),
        "poppy_host_writer_create_io": (i32, [C.POINTER(vp), vp, i32, i32, i32, i32]),
        "poppy_host_writer_submit": (i32, [vp, i32, i32, i32]),
        "poppy_host_writer_flush": (i32, [vp]),
        "poppy_host_writer_destroy": (None, [vp]),
        "poppy_host_writer_destroy_cuda": (None, [vp]),
        "poppy_cuda_set_chunk_frames": (i32, [vp, i32]),
        "poppy_cuda_set_stage_timing": (i32, [vp, i32]),
        "poppy_cuda_set_unsharp_mode": (i32, [vp, i32]),
        "poppy_cuda_unsharp_stats": (i32, [vp, u64p, u64p]),
        "poppy_cuda_set_tile_list_capacity": (i32, [vp, i32]),
        "poppy_cuda_set_pair": (i32, [vp, vp, C.c_size_t, vp, C.c_size_t, vp, C.c_size_t]),
        "poppy_cuda_set_image": (i32, [vp, i32, vp, C.c_size_t]),
        "poppy_cuda_set_source1_from_slot": (i32, [vp, i32]),
        "poppy_cuda_set_points": (i32, [vp, vp, vp, i32]),
        "poppy_cuda_render": (i32, [vp, i32, vp, vp, vp, vp, i32]),
        "poppy_cuda_render_range": (i32, [vp, i32, i32, vp, vp, vp, vp, i32]),
        "poppy_cuda_set_plan": (i32, [vp, vp, vp, i32]),
        "poppy_cuda_render_planned": (i32, [vp, i32, i32, i32, vp, vp, i32]),
        "poppy_cuda_set_segments": (i32, [vp, i32, i32]),
        "poppy_cuda_set_segment": (i32, [vp, i32, vp, C.c_size_t, vp, C.c_size_t, vp, C.c_size_t, vp, vp, i32]),
        "poppy_cuda_render_segments": (i32, [vp, i32, i32, vp, vp, vp, vp]),
        "poppy_cuda_get_segment_points": (i32, [vp, i32, i32, vp]),
        "poppy_shim_morph_segments": (i32, [i32, i32, i32, vp, i32, i32, vp, vp]),
        "poppy_shim_morph_segments_devices": (i32, [vp, i32, i32, i32, i32, vp, i32, i32, vp, vp]),
        "poppy_cuda_download": (i32, [vp, i32, i32, vp, C.c_size_t, C.c_size_t]),
        "poppy_cuda_download_async": (i32, [vp, i32, i32, vp, C.c_size_t, C.c_size_t, u64p]),
        "poppy_cuda_download_wait": (i32, [vp, C.c_uint64]),
        "poppy_cuda_download_i420": (i32, [vp, i32, i32, vp, C.c_size_t]),
        "poppy_cuda_download_i420_async": (i32, [vp, i32, i32, vp, C.c_size_t, u64p]),
        "poppy_cuda_download_ffv1": (i32, [vp, i32, i32, vp, C.c_size_t, C.POINTER(C.c_uint32)]),
        "poppy_cuda_alloc_pinned": (i32, [C.c_size_t, C.POINTER(vp)]),
        "poppy_cuda_free_pinned": (None, [vp]),
        "poppy_cuda_blur_margin": (i32, [i32, vp, C.c_size_t, i32, i32, i32, i32, vp, C.c_size_t]),
        "poppy_cuda_blur_margin_last_error": (C.c_char_p, []),
        "poppy_cuda_gabor_filter": (i32, [i32, vp, C.c_size_t, i32, i32, vp, C.c_size_t]),
        "poppy_cuda_denoise": (i32, [i32, vp, C.c_size_t, i32, i32, C.c_float, i32, i32, vp, C.c_size_t]),
        "poppy_cuda_get_morphed_points": (i32, [vp, i32, vp]),
        "poppy_cuda_frame_device_ptr": (i32, [vp, i32, C.POINTER(vp), C.POINTER(C.c_size_t)]),
        "poppy_cuda_checksum": (i32, [vp, i32, i32, u64p]),
        "poppy_cuda_sync": (i32, [vp]),
        "poppy_cuda_get_stream": (i32, [vp, C.POINTER(vp)]),
        "poppy_cuda_last_render_ms": (i32, [vp, C.POINTER(C.c_float)]),
        "poppy_cuda_launch_count": (i32, [vp, u64p]),
        "poppy_cuda_stage_times": (i32, [vp, C.POINTER(C.c_char_p), C.POINTER(C.c_float), u64p, i32]),
        "poppy_cuda_debug_read": (i32, [vp, i32, i32, vp, C.c_size_t]),
        "poppy_cuda_last_error": (C.c_char_p, [vp]),
        "poppy_cuda_version": (C.c_char_p, []),
    }
    for name, (res, args) in sigs.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


# every symbol include/poppy_cuda.h declares (checked by tests/test_abi.py)
CUDA_ABI_SYMBOLS = [
    "poppy_cuda_device_count", "poppy_cuda_create", "poppy_cuda_destroy", "poppy_cuda_set_keep_stages",
    "poppy_cuda_set_chunk_frames", "poppy_cuda_set_stage_timing", "poppy_cuda_set_pair", "poppy_cuda_set_points",
    "poppy_cuda_render", "poppy_cuda_render_range", "poppy_cuda_set_plan", "poppy_cuda_render_planned", "poppy_cuda_download", "poppy_cuda_get_morphed_points",
    "poppy_cuda_frame_device_ptr",
    "poppy_cuda_checksum", "poppy_cuda_sync", "poppy_cuda_get_stream", "poppy_cuda_last_render_ms",
    "poppy_cuda_launch_count", "poppy_cuda_stage_times", "poppy_cuda_debug_read", "poppy_cuda_last_error",
    "poppy_cuda_version", "poppy_cuda_get_info", "poppy_cuda_set_tile_list_capacity", "poppy_cuda_set_unsharp_mode",
    "poppy_cuda_unsharp_stats", "poppy_cuda_set_image", "poppy_cuda_set_source1_from_slot",
    "poppy_cuda_download_async", "poppy_cuda_download_wait", "poppy_cuda_download_i420", "poppy_cuda_download_i420_async",
    "poppy_cuda_download_ffv1",
    "poppy_cuda_alloc_pinned", "poppy_cuda_free_pinned",
    "poppy_cuda_blur_margin", "poppy_cuda_blur_margin_last_error", "poppy_cuda_gabor_filter",
    "poppy_cuda_denoise", "poppy_cuda_set_segments", "poppy_cuda_set_segment", "poppy_cuda_render_segments", "poppy_cuda_get_segment_points",
]
HOST_ABI_SYMBOLS = [
    "poppy_host_morph_points", "poppy_host_triangulate", "poppy_host_triangulate_next", "poppy_host_chain_ratio", "poppy_host_plan_create",
    "poppy_host_plan_triangles", "poppy_host_plan_points", "poppy_host_plan_destroy", "poppy_morph_images",
    "poppy_host_last_error", "poppy_host_writer_create", "poppy_host_writer_create_i420", "poppy_host_writer_create_ffv1",
    "poppy_host_ffv1_config", "poppy_host_mkv_open", "poppy_host_mkv_write", "poppy_host_mkv_close",
    "poppy_host_writer_create_io", "poppy_host_writer_submit",
    "poppy_host_writer_flush", "poppy_host_writer_destroy", "poppy_host_writer_destroy_cuda",
    "poppy_shim_morph_images", "poppy_shim_morph_sequence", "poppy_shim_morph_segments", "poppy_shim_morph_segments_devices",
    "poppy_shim_release",
]
