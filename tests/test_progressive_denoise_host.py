"""CPU-side checks of the progressive denoised render (rt_camera_render_progressive_denoised): argument errors without a
device, the binding, and the moments output validator."""
import ctypes as C

import numpy as np
import pytest

from mcp_raytracer_b200.scene_data import rt_denoise_opts, rt_region, rt_stats


def test_null_camera_is_an_invalid_argument():
    from mcp_raytracer_b200 import _native

    L = _native.lib()
    buf = np.zeros(12, np.uint8)
    reg = rt_region(0, 0, 2, 2)
    opts = rt_denoise_opts(5, 0, 0, 0)
    st = rt_stats()
    assert L.rt_camera_render_progressive_denoised(None, C.byref(reg), buf.ctypes.data, buf.nbytes, None, None, 4, C.byref(opts),
                                                   None, None, C.byref(st)) == 1
    assert "null camera" in _native.last_error()
    assert L.rt_camera_render_progressive_denoised(None, None, None, 0, None, None, 1, None, None, None, None) == 1


def test_progressive_denoised_is_bound():
    from mcp_raytracer_b200 import Camera, _native

    assert "rt_camera_render_progressive_denoised" in _native.EXPORTS
    fn = _native.lib().rt_camera_render_progressive_denoised
    assert fn.argtypes is not None and len(fn.argtypes) == 11
    assert fn.argtypes[6] is C.c_int32  # n_passes
    assert callable(getattr(Camera, "renderProgressiveDenoised"))


def test_moments_output_is_checked_before_the_library_writes_it():
    """The library writes the moments through their base pointer as a C-contiguous float32 [H][W][8] array."""
    from mcp_raytracer_b200 import RaytracerError
    from mcp_raytracer_b200.camera import _moments_output

    W, H = 5, 4
    m = np.zeros((H, W, 8), np.float32)
    assert _moments_output(m, W, H) == m.ctypes.data
    assert _moments_output(None, W, H) is None
    with pytest.raises(RaytracerError, match="moments buffer"):
        _moments_output(m.astype(np.float64), W, H)
    with pytest.raises(RaytracerError, match="moments buffer"):
        _moments_output(m[:-1], W, H)
    with pytest.raises(RaytracerError, match="moments buffer"):  # a view with strides: writing it as contiguous corrupts it
        _moments_output(np.zeros((H, 2 * W, 8), np.float32)[:, ::2], W, H)
    with pytest.raises(RaytracerError, match="moments buffer"):
        _moments_output(np.zeros((W, H, 8), np.float32).transpose(1, 0, 2), W, H)
