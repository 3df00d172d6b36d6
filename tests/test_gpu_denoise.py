"""GPU checks of the opt-in denoiser: feature buffers against the primary-visibility hook, the FP32 filter against its numpy
specification (tests/denoise_reference.py), region / determinism / option plumbing, and image quality against a
high-sample render with another seed.  Run on a B200 with `-m gpu`."""
import numpy as np
import pytest

import denoise_reference as dref
from mcp_raytracer_b200 import (
    Camera, RaytracerError, createCameraFromSceneData, denoise, generateCornellSceneData,
    generateImageBuffer, generateLayeredMixedSceneData, generateRainSceneData, generateSceneData, generateSpheresSceneData,
    generateWeekendFinalSceneData,
)
from mcp_raytracer_b200.raytracer import applySceneCameraOptions
from mcp_raytracer_b200.scene_data import FlatScene

pytestmark = pytest.mark.gpu

SCENES = {
    "C1-spheres": lambda: generateSpheresSceneData({"count": 100, "seed": 12345}),
    "C2-cornell": generateCornellSceneData,
    "C3-weekend": generateWeekendFinalSceneData,
    "C4-rain": lambda: generateRainSceneData({"count": 20000, "seed": 1, "sphereRadius": 0.01}),
    "C5-layered": generateLayeredMixedSceneData,
}
MAT_LAMBERT, MAT_METAL, MAT_GLASS, MAT_LIGHT, MAT_MIXED, MAT_LAYERED = range(6)


def feature_albedo(flat: FlatScene):
    """The scene compiler's feature albedo per material node, restated: FP32 storage, FP64 evaluation (rt_scene.cpp H3)."""
    f32 = lambda x: np.asarray(x, np.float64).astype(np.float32).astype(np.float64)  # noqa: E731
    out = []
    for k, ty in enumerate(np.asarray(flat.mat_type_a)):
        c0, c1 = (int(x) for x in np.asarray(flat.mat_child_a).reshape(-1, 2)[k])
        if ty in (MAT_LAMBERT, MAT_METAL):
            a = f32(np.asarray(flat.mat_color_a, np.float64).reshape(-1, 3)[k])
        elif ty == MAT_MIXED:
            w = min(1.0, max(0.0, float(np.asarray(flat.mat_param_a)[k])))  # mixedMaterial.ts:29
            a = f32(f32(out[c0] * w) + f32(out[c1] * (1.0 - w)))
        elif ty == MAT_LAYERED:
            a = out[c0]  # layeredMaterial.ts:61-63
        else:  # glass, light
            a = np.ones(3)
        out.append(a)
    return np.array(out, np.float32)


def object_albedo(sd, ids):
    flat = FlatScene(sd)
    mats = feature_albedo(flat)
    a = np.ones(ids.shape + (3,), np.float32)
    hit = ids >= 0
    a[hit] = mats[flat.obj_material[ids[hit]]]
    return a


def camera_dir_norm(cam):
    """|d| of the pixel-centre camera rays with the reference's FP32 rounding (camera.ts:176-196)."""
    W, H = cam.imageWidth, cam.imageHeight
    i = np.arange(W, dtype=np.float32)[None, :, None]
    j = np.arange(H, dtype=np.float32)[:, None, None]
    pc = (cam.pixel00Loc + cam.pixelDeltaU * i).astype(np.float32) + (cam.pixelDeltaV * j).astype(np.float32)
    d = (pc.astype(np.float32) - cam.center).astype(np.float64)
    return np.sqrt((d * d).sum(-1))


@pytest.mark.parametrize("name", list(SCENES))
@pytest.mark.parametrize("bvh", ["reference", "sah", "list"])
def test_features_at_one_sample_equal_the_primary_hits(gpu, name, bvh):
    sd = SCENES[name]()
    if bvh == "list" and len(sd["objects"]) > 128:
        pytest.skip("LIST trees hold at most 128 objects")
    # aperture 0: the primary-visibility hook traces pixel centres without defocus
    with Camera(sd, {"aperture": 0}, {"width": 160, "samples": 1, "bvh": bvh, "seed": 4}) as cam:
        ids, t, nrm, _ = cam.tracePrimary()
        f = cam.renderFeatures(1)
        dnorm = camera_dir_norm(cam)
    hit = ids >= 0
    assert np.array_equal(f["normal"], nrm)
    assert np.all(f["depth"][~hit] == -1)
    ref = t[hit].astype(np.float64) * dnorm[hit]
    assert np.all(np.abs(f["depth"][hit] - ref) <= 1e-6 * ref)
    assert np.array_equal(f["albedo"], object_albedo(sd, ids))


def _uniform_3x3(ids):
    H, W = ids.shape
    same = np.zeros((H, W), bool)
    same[1:-1, 1:-1] = True
    for dy in (-1, 0, 1):
        for dx in (-1, 0, 1):
            same[1:-1, 1:-1] &= ids[1 + dy:H - 1 + dy, 1 + dx:W - 1 + dx] == ids[1:-1, 1:-1]
    return same & (ids >= 0)


@pytest.mark.parametrize("name", ["C2-cornell", "C5-layered"])
def test_features_over_jittered_samples(gpu, name):
    sd = SCENES[name]()
    with createCameraFromSceneData(sd, {"width": 128, "samples": 8, "seed": 2}) as cam:
        ids, _, nrm, _ = cam.tracePrimary()
        f1 = cam.renderFeatures(8)
        f2 = cam.renderFeatures(8)
    for k in f1:
        assert np.array_equal(f1[k], f2[k]), k
    flat = FlatScene(sd)
    planar = np.asarray(flat.obj_type) != 0
    sel = _uniform_3x3(ids)
    sel[sel] &= planar[ids[sel]]
    assert sel.sum() > 1000
    assert np.abs(f1["normal"][sel] - nrm[sel]).max() <= 2e-6
    assert np.abs(f1["albedo"][sel] - object_albedo(sd, ids)[sel]).max() <= 2e-6
    assert np.all(f1["depth"][sel] > 0)


def _crop_inputs(seed=5):
    sd = generateCornellSceneData()
    with createCameraFromSceneData(sd, {"width": 128, "samples": 8, "aTolerance": 0, "seed": seed}) as cam:
        W, H = cam.imageWidth, cam.imageHeight
        lin = np.zeros((H, W, 3), np.float32)
        mom = np.zeros((H, W, 8), np.float32)
        cam.renderRegion(None, None, lin, mom)
        f = cam.renderFeatures(8)
    ys, xs = slice(40, 88), slice(30, 94)  # 64 x 48
    return lin[ys, xs], f["albedo"][ys, xs], f["normal"][ys, xs], f["depth"][ys, xs], mom[ys, xs]


@pytest.mark.parametrize("iterations", [0, 1, 5])
def test_filter_matches_the_numpy_specification(gpu, iterations):
    args = _crop_inputs()
    got = denoise(*args, options={"iterations": iterations})
    ref = dref.denoise(*args, {"iterations": iterations})
    err = np.abs(got - ref)
    assert np.all(err <= 1e-4 * np.abs(ref) + 1e-7), float((err / (np.abs(ref) + 1e-7)).max())
    if iterations:
        assert np.abs(got - args[0]).max() > 1e-3  # it filtered


def test_region_writes_only_region_pixels_and_equals_denoise_of_the_crop(gpu):
    sd = generateCornellSceneData()
    region = {"x": 20, "y": 12, "width": 70, "height": 50}
    with createCameraFromSceneData(sd, {"width": 128, "samples": 16, "aTolerance": 0, "seed": 8}) as cam:
        W, H = cam.imageWidth, cam.imageHeight
        rgb = np.full(W * H * 3, 7, np.uint8)
        lin = np.full((H, W, 3), -5.0, np.float32)
        st = cam.renderDenoised(rgb, lin, region)
        lin0 = np.zeros((H, W, 3), np.float32)
        mom = np.zeros((H, W, 8), np.float32)
        cam.renderRegion(None, region, lin0, mom)
        f = cam.renderFeatures(8, region)
    ys, xs = slice(12, 62), slice(20, 90)
    inside = np.zeros((H, W), bool)
    inside[ys, xs] = True
    rgb = rgb.reshape(H, W, 3)
    assert np.all(rgb[~inside] == 7) and np.all(lin[~inside] == -5.0)
    assert st.pixels == 70 * 50 and st.kernelLaunches >= 1 + 1 + 5 + 2
    crop = denoise(lin0[ys, xs], f["albedo"][ys, xs], f["normal"][ys, xs], f["depth"][ys, xs], mom[ys, xs])
    np.testing.assert_allclose(lin[ys, xs], crop, rtol=1e-6, atol=1e-7)


def test_denoised_render_is_deterministic_and_rgb8_follows_the_gamma_rule(gpu):
    sd = generateLayeredMixedSceneData()
    out = []
    for _ in range(2):
        with createCameraFromSceneData(sd, {"width": 96, "samples": 8, "seed": 3}) as cam:
            rgb = np.zeros(cam.imageWidth * cam.imageHeight * 3, np.uint8)
            lin = np.zeros((cam.imageHeight, cam.imageWidth, 3), np.float32)
            cam.renderDenoised(rgb, lin)
        out.append((rgb, lin))
    assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][1], out[1][1])
    assert np.array_equal(out[0][0].reshape(lin.shape), dref.gamma_rgb8(out[0][1]))


def rel_mse(x, r, mask=None):
    e = (x.astype(np.float64) - r) ** 2 / (r.astype(np.float64) ** 2 + 0.01)
    return float(e[mask].mean() if mask is not None else e.mean())


def _edge_pixels(ids, radius=2):
    H, W = ids.shape
    p = np.pad(ids, radius, mode="edge")
    edge = np.zeros((H, W), bool)
    for dy in range(-radius, radius + 1):
        for dx in range(-radius, radius + 1):
            edge |= p[radius + dy:radius + dy + H, radius + dx:radius + dx + W] != ids
    return edge


def _render_linear(sd, opts, denoised=False, options=None):
    with createCameraFromSceneData(sd, opts) as cam:
        lin = np.zeros((cam.imageHeight, cam.imageWidth, 3), np.float32)
        if denoised:
            cam.renderDenoised(None, lin, options=options)
        else:
            cam.renderRegion(None, None, lin)
        ids = cam.tracePrimary()[0]
    return lin, ids


@pytest.mark.parametrize("name", ["C2-cornell", "C5-layered"])
def test_denoised_quality_against_a_converged_render(gpu, name):
    sd = SCENES[name]()
    base = {"width": 256, "aspect": 1.0, "aTolerance": 0}
    ref, ids = _render_linear(sd, {**base, "samples": 8192, "seed": 1234})
    noisy, _ = _render_linear(sd, {**base, "samples": 16, "seed": 7})
    den, _ = _render_linear(sd, {**base, "samples": 16, "seed": 7}, denoised=True)
    e_noisy, e_den = rel_mse(noisy, ref), rel_mse(den, ref)
    edge = _edge_pixels(ids)
    e_noisy_edge, e_den_edge = rel_mse(noisy, ref, edge), rel_mse(den, ref, edge)
    print(f"{name}: relMSE noisy {e_noisy:.5f} denoised {e_den:.5f}; edges {e_noisy_edge:.5f} / {e_den_edge:.5f}")
    assert e_den <= 0.4 * e_noisy
    assert e_den_edge <= e_noisy_edge
    m_den, m_ref = den.mean(axis=(0, 1)), ref.mean(axis=(0, 1))
    assert np.all(np.abs(m_den - m_ref) <= 0.01 * m_ref), (m_den, m_ref)


@pytest.mark.xfail(strict=True, reason="bar missed, measured on a B200 (1000 W): Cornell 128x128 @4096 spp, RMS(denoised - undenoised) "
                   "1.54e-2 = 1.11 x the RMS sigma of the pixel mean (1.38e-2) against a bar of 0.25; the luminance stop scales "
                   "with sigma, so the filter does not fade out as the noise does (profiles/README.md section 9)")
def test_filter_fades_out_as_noise_does(gpu):
    sd = generateCornellSceneData()
    opts = {"width": 128, "aspect": 1.0, "aTolerance": 0, "samples": 4096, "seed": 21}
    with createCameraFromSceneData(sd, opts) as cam:
        W, H = cam.imageWidth, cam.imageHeight
        lin = np.zeros((H, W, 3), np.float32)
        mom = np.zeros((H, W, 8), np.float32)
        cam.renderRegion(None, None, lin, mom)
        den = np.zeros((H, W, 3), np.float32)
        cam.renderDenoised(None, den)
    n = mom[..., 6:7].astype(np.float64)
    sigma_mean = np.sqrt(mom[..., 3:6] / (n - 1) / n)
    rms_diff = float(np.sqrt(((den.astype(np.float64) - lin) ** 2).mean()))
    rms_sigma = float(np.sqrt((sigma_mean ** 2).mean()))
    print(f"4096 spp: RMS(denoised - undenoised) {rms_diff:.3e}, RMS sigma of the mean {rms_sigma:.3e}")
    assert rms_diff <= 0.25 * rms_sigma


@pytest.mark.parametrize("opts", [{}, {"lightSampling": "shadowRays", "aTolerance": 0, "samples": 16}])
def test_reference_defaults_and_shadow_rays_through_render_denoised(gpu, opts):
    sd = generateCornellSceneData()
    base = {"width": 128, "aspect": 1.0}
    ref, _ = _render_linear(sd, {**base, "samples": 4096, "aTolerance": 0, "seed": 77})
    den, _ = _render_linear(sd, {**base, **opts, "seed": 5}, denoised=True)
    m_den, m_ref = den.mean(axis=(0, 1)), ref.mean(axis=(0, 1))
    assert np.all(np.abs(m_den - m_ref) <= 0.01 * m_ref), (m_den, m_ref)


def test_partitioned_cameras_and_other_modes_are_refused(gpu):
    sd = generateCornellSceneData()
    for opts in ({"partCount": 2, "partIndex": 0}, {"mode": "bounces"}, {"mode": "samples"}):
        with createCameraFromSceneData(sd, {"width": 32, "samples": 2, **opts}) as cam:
            with pytest.raises(RaytracerError, match="RT_ERR_UNSUPPORTED"):
                cam.renderDenoised(np.zeros(cam.imageWidth * cam.imageHeight * 3, np.uint8))


def test_scene_option_renders_denoised_on_one_gpu(gpu):
    cfg = {"type": "cornell", "render": {"width": 96, "samples": 8, "seed": 3}}
    img = generateImageBuffer(cfg, {"denoise": True, "parallel": True, "raw": True})
    sd = applySceneCameraOptions(generateSceneData(cfg), cfg.get("camera"))
    with createCameraFromSceneData(sd, cfg["render"]) as cam:
        rgb = np.zeros(cam.imageWidth * cam.imageHeight * 3, np.uint8)
        cam.renderDenoised(rgb)
    assert np.array_equal(img.reshape(-1), rgb)
    img2 = generateImageBuffer(cfg, {"denoise": {"iterations": 2, "sigmaLuminance": 2.0}, "raw": True})
    assert img2.shape == img.shape and not np.array_equal(img2, img)
