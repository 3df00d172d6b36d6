"""CPU-side checks of the denoiser: the C-ABI mirror of rt_denoise_opts, argument errors reported before any device
check, and the properties of the filter's numpy specification (tests/denoise_reference.py)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import denoise_reference as dref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_denoise_opts_layout_matches_the_header():
    from mcp_raytracer_b200 import scene_data as sd

    src = r'''
    #include <stdio.h>
    #include "rt_b200.h"
    int main(void){ printf("%zu\n", sizeof(rt_denoise_opts)); return 0; }'''
    exe = os.path.join("/tmp", f"rt_dn_sizes_{os.getpid()}")
    subprocess.run(["gcc", "-x", "c", "-", "-I", os.path.join(ROOT, "include"), "-o", exe], input=src.encode(), check=True)
    size = int(subprocess.check_output([exe]))
    os.remove(exe)
    assert size == C.sizeof(sd.rt_denoise_opts)


def _inputs(H=6, W=5):
    color = np.full((H, W, 3), 0.5, np.float32)
    albedo = np.full((H, W, 3), 0.5, np.float32)
    normal = np.zeros((H, W, 3), np.float32)
    normal[..., 2] = 1
    depth = np.ones((H, W), np.float32)
    moments = np.zeros((H, W, 8), np.float32)
    moments[..., 6] = 4
    return color, albedo, normal, depth, moments


def test_argument_errors_come_before_the_device_check():
    from mcp_raytracer_b200 import _native
    from mcp_raytracer_b200.scene_data import rt_denoise_opts, rt_region, rt_stats

    L = _native.lib()
    color, albedo, normal, depth, moments = _inputs()
    out = np.zeros_like(color)
    ptr = lambda a: a.ctypes.data  # noqa: E731
    args = [ptr(color), ptr(albedo), ptr(normal), ptr(depth), ptr(moments)]
    H, W = color.shape[:2]

    def dn(w, h, arrays, opts, o):
        return L.rt_denoise(-1, w, h, *arrays, C.byref(opts) if opts is not None else None, o)

    good = rt_denoise_opts(5, 0, 0, 0)
    for k in range(5):  # each required input missing
        a = list(args)
        a[k] = None
        assert dn(W, H, a, good, ptr(out)) == 1
    assert dn(W, H, args, good, None) == 1
    assert dn(0, H, args, good, ptr(out)) == 1
    assert dn(W, -1, args, good, ptr(out)) == 1
    for bad in (rt_denoise_opts(9, 0, 0, 0), rt_denoise_opts(-1, 0, 0, 0), rt_denoise_opts(5, -1, 0, 0), rt_denoise_opts(5, 0, -2, 0),
                rt_denoise_opts(5, 0, 0, -0.5), rt_denoise_opts(5, float("nan"), 0, 0)):
        assert dn(W, H, args, bad, ptr(out)) == 1
        assert b"denoise" in L.rt_last_error()
    # valid arguments: no CPU fallback
    expected = 0 if L.rt_device_count() > 0 else 7
    assert dn(W, H, args, good, ptr(out)) == expected
    assert dn(W, H, args, None, ptr(out)) == expected
    reg = rt_region(0, 0, W, H)
    assert L.rt_camera_render_features(None, C.byref(reg), 1, ptr(albedo), ptr(normal), ptr(depth)) == 1
    rgb = np.zeros(H * W * 3, np.uint8)
    st = rt_stats()
    assert L.rt_camera_render_denoised(None, C.byref(reg), ptr(rgb), rgb.nbytes, None, C.byref(good), C.byref(st)) == 1


def test_python_denoise_refuses_bad_shapes_and_options():
    from mcp_raytracer_b200 import RaytracerError, denoise

    color, albedo, normal, depth, moments = _inputs()
    with pytest.raises(RaytracerError, match="moments"):
        denoise(color, albedo, normal, depth, moments[..., :7])
    with pytest.raises(RaytracerError, match="unknown denoise options"):
        denoise(color, albedo, normal, depth, moments, {"sigma": 1})
    with pytest.raises(RaytracerError, match="INVALID_ARGUMENT"):
        denoise(color, albedo, normal, depth, moments, {"iterations": 9})


def _noisy_scene(H=24, W=20, seed=3):
    rng = np.random.default_rng(seed)
    color = (0.4 + 0.2 * rng.standard_normal((H, W, 3))).astype(np.float32)
    albedo = np.full((H, W, 3), 0.6, np.float32)
    normal = np.zeros((H, W, 3), np.float32)
    normal[..., 2] = 1
    depth = np.full((H, W), 2.0, np.float32)
    moments = np.zeros((H, W, 8), np.float32)
    moments[..., 0:3] = color * 16
    moments[..., 3:6] = 0.04 * 15 * 16
    moments[..., 6] = 16
    return color, albedo, normal, depth, moments


def test_reference_returns_a_constant_image_unchanged():
    color, albedo, normal, depth, moments = _inputs(12, 10)
    out = dref.denoise(color, albedo, normal, depth, moments)
    np.testing.assert_allclose(out, color, rtol=1e-12)


def test_reference_iterations_zero_is_the_identity():
    color, albedo, normal, depth, moments = _noisy_scene()
    out = dref.denoise(color, albedo, normal, depth, moments, {"iterations": 0})
    np.testing.assert_allclose(out, color, rtol=1e-12)
    assert not np.allclose(dref.denoise(color, albedo, normal, depth, moments), color)  # the default filter does smooth


def test_reference_keeps_a_step_edge_between_two_albedos():
    H, W = 16, 16
    color, albedo, normal, depth, moments = _noisy_scene(H, W)
    albedo[:, : W // 2] = (0.8, 0.2, 0.1)
    albedo[:, W // 2:] = (0.1, 0.3, 0.9)
    color[:] = albedo * 0.7  # one irradiance, two albedos
    out = dref.denoise(color, albedo, normal, depth, moments)
    assert np.abs(out - color).max() <= 1e-6


def test_reference_keeps_a_step_edge_between_two_normals():
    H, W = 16, 16
    color, albedo, normal, depth, moments = _noisy_scene(H, W)
    normal[:] = 0
    normal[:, : W // 2, 0] = 1
    normal[:, W // 2:, 1] = 1
    color[:, : W // 2] = 0.9
    color[:, W // 2:] = 0.1
    moments[..., 3:6] = 1.0  # noisy enough that the luminance stop alone would let the edge blur
    out = dref.denoise(color, albedo, normal, depth, moments)
    assert np.abs(out - color).max() <= 1e-6


def test_reference_non_finite_pixel_leaves_its_neighbours_finite():
    color, albedo, normal, depth, moments = _noisy_scene()
    color[10, 7] = (np.nan, 0.3, np.inf)
    color[3, 3, 1] = np.inf
    out = dref.denoise(color, albedo, normal, depth, moments)
    bad = ~np.isfinite(color).all(-1)
    assert np.isfinite(out[~bad]).all()
    np.testing.assert_array_equal(out[bad], color[bad].astype(np.float64))  # passed through unchanged
    assert np.array_equal(dref.gamma_rgb8(out)[10, 7], [0, 140, 255])


def test_reference_unknown_variance_lets_the_features_decide():
    color, albedo, normal, depth, moments = _noisy_scene()
    moments[..., 6] = 1  # one sample: no variance estimate, luminance weights are 1
    out = dref.denoise(color, albedo, normal, depth, moments)
    assert np.isfinite(out).all() and out.std() < 0.5 * color.std()
