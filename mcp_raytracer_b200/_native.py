"""ctypes binding of the C-ABI library (include/rt_b200.h -> csrc/libmcprt_b200.so).

The library is the product.  If it is missing this module raises — there is no Python or
CPU fallback for the render path.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from typing import Optional

from .scene_data import rt_camera_info, rt_denoise_opts, rt_region, rt_render_opts, rt_scene_desc, rt_stats

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.environ.get("RT_B200_LIB") or os.path.join(CSRC, "libmcprt_b200.so")  # env: A/B-test another build

# every symbol include/rt_b200.h declares
EXPORTS = [
    "rt_camera_create", "rt_camera_destroy", "rt_camera_get_info", "rt_camera_set_stream",
    "rt_camera_render_region", "rt_camera_render", "rt_camera_render_region_device",
    "rt_camera_render_moments", "rt_camera_render_progressive", "rt_camera_trace_primary", "rt_last_error", "rt_device_count",
    "rt_abi_version", "rt_counts_events", "rt_block_owner", "rt_measure_fp32_peak", "rt_trim_device_cache", "rt_scene_validate",
    "rt_multi_create", "rt_multi_destroy", "rt_multi_get_info", "rt_multi_render_region",
    "rt_shared_buffer_create", "rt_shared_buffer_open", "rt_shared_buffer_release",
    "rt_debug_scatter", "rt_debug_get_ray", "rt_debug_light_pdf", "rt_debug_light_random_vec", "rt_debug_diffuse_bounce",
    "rt_camera_render_features", "rt_denoise", "rt_camera_render_denoised", "rt_multi_render_denoised",
    "rt_camera_render_progressive_denoised", "rt_multi_render_progressive", "rt_multi_render_progressive_denoised",
    "rt_progressive_caps",
]

STATUS_NAMES = {
    0: "RT_OK", 1: "RT_ERR_INVALID_ARGUMENT", 2: "RT_ERR_UNKNOWN_OBJECT_TYPE", 3: "RT_ERR_UNKNOWN_MATERIAL_TYPE",
    4: "RT_ERR_MATERIAL_NOT_FOUND", 5: "RT_ERR_NOT_DIELECTRIC", 6: "RT_ERR_BUFFER_TOO_SMALL", 7: "RT_ERR_NO_DEVICE",
    8: "RT_ERR_CUDA", 9: "RT_ERR_UNSUPPORTED",
}

_lib: Optional[C.CDLL] = None


class NativeLibraryMissing(RuntimeError):
    pass


def build(verbose: bool = False) -> str:
    """Compile csrc/ for sm_100a (nvcc cross-compiles without a GPU).  Returns the .so path."""
    out = None if verbose else subprocess.DEVNULL
    subprocess.check_call(["make", "-C", CSRC, "libmcprt_b200.so"], stdout=out)
    return LIB_PATH


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeLibraryMissing(
            f"{LIB_PATH} is not built. Run `python -c 'import __graft_entry__ as g; g.build()'` or `make -C {CSRC}`. "
            "There is no CPU fallback for the render path."
        )
    L = C.CDLL(LIB_PATH)
    vp = C.c_void_p
    L.rt_last_error.restype = C.c_char_p
    L.rt_device_count.restype = C.c_int32
    L.rt_abi_version.restype = C.c_int32
    L.rt_counts_events.restype = C.c_int32
    L.rt_block_owner.restype = C.c_int32
    L.rt_block_owner.argtypes = [C.c_int32] * 4
    L.rt_camera_create.argtypes = [C.POINTER(rt_scene_desc), C.POINTER(rt_render_opts), C.POINTER(vp)]
    L.rt_camera_destroy.argtypes = [vp]
    L.rt_camera_get_info.argtypes = [vp, C.POINTER(rt_camera_info)]
    L.rt_camera_set_stream.argtypes = [vp, vp]
    L.rt_camera_render_region.argtypes = [vp, C.POINTER(rt_region), vp, C.c_size_t, vp, C.POINTER(rt_stats)]
    L.rt_camera_render.argtypes = [vp, vp, C.c_size_t, vp, C.POINTER(rt_stats)]
    L.rt_camera_render_region_device.argtypes = [vp, C.POINTER(rt_region), vp, vp, vp, vp]
    L.rt_camera_render_moments.argtypes = [vp, C.POINTER(rt_region), vp, C.c_size_t, vp, vp, C.POINTER(rt_stats)]
    L.rt_camera_render_progressive.argtypes = [vp, C.POINTER(rt_region), vp, C.c_size_t, vp, C.c_int32, vp, vp, C.POINTER(rt_stats)]
    L.rt_camera_trace_primary.argtypes = [vp, C.POINTER(rt_region), vp, vp, vp, vp]
    L.rt_measure_fp32_peak.argtypes = [C.c_int32, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    L.rt_trim_device_cache.restype = C.c_uint64
    L.rt_scene_validate.argtypes = [C.POINTER(rt_scene_desc), C.POINTER(rt_render_opts), vp]
    i32 = C.c_int32
    L.rt_multi_create.argtypes = [C.POINTER(rt_scene_desc), C.POINTER(rt_render_opts), i32, vp, C.POINTER(vp)]
    L.rt_multi_destroy.argtypes = [vp]
    L.rt_multi_get_info.argtypes = [vp, C.POINTER(rt_camera_info), C.POINTER(i32), C.POINTER(i32)]
    L.rt_multi_render_region.argtypes = [vp, C.POINTER(rt_region), vp, C.c_size_t, vp, C.POINTER(rt_stats)]
    L.rt_shared_buffer_create.argtypes = [i32, C.c_size_t, C.POINTER(vp), vp]
    L.rt_shared_buffer_open.argtypes = [i32, vp, C.POINTER(vp)]
    L.rt_shared_buffer_release.argtypes = [i32, vp, i32]
    L.rt_debug_scatter.argtypes = [vp, i32, i32, vp, vp, vp]
    L.rt_debug_get_ray.argtypes = [vp, i32, vp, vp, vp, vp]
    L.rt_debug_light_pdf.argtypes = [vp, i32, i32, vp, vp, vp]
    L.rt_debug_light_random_vec.argtypes = [vp, i32, i32, vp, vp, vp]
    L.rt_debug_diffuse_bounce.argtypes = [vp, i32, vp, vp, vp, vp]
    L.rt_camera_render_features.argtypes = [vp, C.POINTER(rt_region), i32, vp, vp, vp]
    L.rt_denoise.argtypes = [i32, i32, i32, vp, vp, vp, vp, vp, C.POINTER(rt_denoise_opts), vp]
    L.rt_camera_render_denoised.argtypes = [vp, C.POINTER(rt_region), vp, C.c_size_t, vp, C.POINTER(rt_denoise_opts), C.POINTER(rt_stats)]
    L.rt_multi_render_denoised.argtypes = [vp, C.POINTER(rt_region), vp, C.c_size_t, vp, C.POINTER(rt_denoise_opts), C.POINTER(rt_stats)]
    L.rt_camera_render_progressive_denoised.argtypes = [vp, C.POINTER(rt_region), vp, C.c_size_t, vp, vp, i32, C.POINTER(rt_denoise_opts),
                                                        vp, vp, C.POINTER(rt_stats)]
    L.rt_multi_render_progressive.argtypes = [vp, C.POINTER(rt_region), vp, C.c_size_t, vp, i32, vp, vp, C.POINTER(rt_stats)]
    L.rt_multi_render_progressive_denoised.argtypes = [vp, C.POINTER(rt_region), vp, C.c_size_t, vp, vp, i32, C.POINTER(rt_denoise_opts),
                                                       vp, vp, C.POINTER(rt_stats)]
    L.rt_progressive_caps.restype = i32
    L.rt_progressive_caps.argtypes = [i32, i32, i32, vp]
    _lib = L
    return L


def last_error() -> str:
    return (lib().rt_last_error() or b"").decode("utf-8", "replace")
