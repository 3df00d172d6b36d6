"""CPU-side checks of the denoiser: the C-ABI mirror of rt_denoise_opts, argument errors reported before any device
check, and the properties of the filter's numpy specification (tests/denoise_reference.py)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import denoise_cases as dc
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


# ---- the edge-case generator of the GPU parity test (tests/denoise_cases.py) and the spec properties it relies on ----
def _recount(args):
    """The claims of a case, counted from its arrays alone."""
    c, a, n, z, m = args
    with np.errstate(all="ignore"):
        demod = c / np.maximum(a, np.float32(dref.ALBEDO_MIN))  # FP32, as the filter stores it
    fin = lambda x: np.isfinite(x).all(-1)  # noqa: E731
    valid = fin(c) & fin(a) & fin(n) & np.isfinite(z) & fin(demod)
    miss = valid & (z == -1) & (n == 0).all(-1) & (a == 1).all(-1)
    return {"misses": int(miss.sum()), "invalid": int((~valid).sum()), "few_samples": int((m[..., 6] < 2).sum()),
            "negative_m2": int((m[..., 3:6] < 0).any(-1).sum()), "zero_albedo": int((a == 0).any(-1).sum())}, valid, miss


@pytest.mark.parametrize("kind", dc.KINDS)
def test_case_generator_produces_what_each_case_claims(kind):
    for H, W in dc.SHAPES:
        args, claims = dc.make_case(kind, H, W)
        assert all(x.dtype == np.float32 for x in args)
        assert [x.shape for x in args] == [(H, W, 3), (H, W, 3), (H, W, 3), (H, W), (H, W, 8)]
        counts, valid, miss = _recount(args)
        assert counts == claims, (H, W)
        assert np.array_equal(dref.prepare(*args)["valid"], valid), (H, W)  # the spec sees the same invalid pixels
        if kind in dc.DEFINES:
            assert claims[dc.DEFINES[kind]] > 0, (H, W)
        if kind.startswith("miss_") and H * W > 1:
            assert (valid & ~miss).any(), (H, W)  # misses next to hits
        c, a, n, z, m = args
        hit = valid & (z >= 0)
        assert np.all(np.abs(np.linalg.norm(n[hit], axis=-1) - 1) <= 1e-6)  # unit normals, as the features write them
        assert np.all(hit | miss | ~valid)
        if kind in ("n0", "n1", "n2", "n64"):
            assert np.all(m[..., 6] == float(kind[1:]))
        if kind == "m2_zero":
            assert np.all(m[..., 3:6] == 0)


def test_parity_sets_cover_every_case_shape_iteration_count_and_option():
    sets = dc.parity_sets()
    assert len({s[0] for s in sets}) == len(sets)
    assert {s[1] for s in sets} == set(dc.KINDS)
    assert {s[2] for s in sets} == set(dc.SHAPES)
    assert {s[3]["iterations"] for s in sets} == set(range(9))
    for _, opts in dc.OPTIONS:
        assert any({k: v for k, v in s[3].items() if k != "iterations"} == opts for s in sets)


@pytest.mark.parametrize("kind", [k for k in dc.KINDS if k.startswith("nonfinite_")] + ["demod_overflow"])
def test_reference_passes_invalid_pixels_through_bit_for_bit(kind):
    for H, W in dc.SHAPES:
        args, claims = dc.make_case(kind, H, W)
        _, valid, _ = _recount(args)
        out = dref.denoise(*args)
        assert np.array_equal(out[~valid], args[0][~valid].astype(np.float64), equal_nan=True)
        assert np.isfinite(out[valid]).all()


@pytest.mark.parametrize("kind", ["miss_single", "n0", "n1", "n64", "m2_zero", "albedo_edges", "depth_tiny", "depth_huge"])
def test_reference_leaves_a_1x1_image_unchanged(kind):
    args, _ = dc.make_case(kind, 1, 1)
    for it in range(9):
        out = dref.denoise(*args, {"iterations": it})
        np.testing.assert_allclose(out, args[0], rtol=1e-15, atol=0)  # demodulate, divide by the one weight, remodulate


@pytest.mark.parametrize("shape", [(16, 16), (17, 33), (33, 17), (7, 300)])
def test_reference_miss_block_ignores_the_colours_of_hits(shape):
    args, _ = dc.make_case("miss_block", *shape)
    _, _, miss = _recount(args)
    other = list(args)
    other[0] = args[0].copy()
    other[0][~miss] = np.random.default_rng(1).uniform(0, 5, (int((~miss).sum()), 3)).astype(np.float32)
    # a hit is no miss' tap.  Only the hits' variance reaches a miss, through the 3x3 blur; it is the render's until the
    # first pass, after which it depends on the hits' colours (their luminance weights), so the property is one pass's.
    a = dref.denoise(*args, {"iterations": 1})
    b = dref.denoise(*other, {"iterations": 1})
    assert np.array_equal(a[miss], b[miss])
    assert not np.array_equal(a[~miss], b[~miss])


@pytest.mark.parametrize("kind", ["miss_block", "n_mixed", "depth_ramps", "facets", "albedo_edges"])
def test_reference_step_beyond_the_image_is_the_centre_tap(kind):
    for H, W in dc.SHAPES:
        args, _ = dc.make_case(kind, H, W)
        P = dref.prepare(*args)
        o = dref.options()
        for step in (max(H, W), 2 * max(H, W) + 1, 128):
            if step < max(H, W):
                continue
            i, v = dref.atrous_pass(P, P["i"], P["var"], step, o)
            np.testing.assert_allclose(i, P["i"], rtol=1e-15, atol=0)
            np.testing.assert_allclose(v, P["var"], rtol=1e-15, atol=0)
