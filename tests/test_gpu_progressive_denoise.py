"""GPU checks of the progressive denoised render (rt_camera_render_progressive_denoised / Camera.renderProgressiveDenoised):
the last pass is renderDenoised's image, with renderRegion's moments and the one-shot stats, over scenes, kernels, options,
pass counts and regions; every earlier pass is the filter of the render with that pass's sample cap; each preview is
cleaner than its noisy image; early stops, callback errors and argument errors.  Run on a B200 with `-m gpu`."""
import numpy as np
import pytest

import denoise_reference as dref
from mcp_raytracer_b200 import (
    RaytracerError, createCameraFromSceneData, denoise, generateCornellSceneData, generateDefaultSceneData,
    generateLayeredMixedSceneData, generateRainSceneData, generateSpheresSceneData,
)

pytestmark = pytest.mark.gpu

SCENES = {
    "C1-spheres": lambda: generateSpheresSceneData({"count": 100, "seed": 12345}),
    "C2-cornell": generateCornellSceneData,
    "C4-rain": lambda: generateRainSceneData({"count": 20000, "seed": 1, "sphereRadius": 0.01}),
    "C5-layered": generateLayeredMixedSceneData,
    "default": generateDefaultSceneData,
}
# (scene, render options, denoise options); the pixel-stream kernel each one runs
CASES = {
    "cornell-fixed": ("C2-cornell", {"width": 96, "samples": 16, "aTolerance": 0, "seed": 5}, None),  # k_render_stream<LIST>
    "C1-adaptive": ("C1-spheres", {"width": 120, "samples": 100, "aTolerance": 0.05, "aBatch": 10, "seed": 3}, None),  # <SAH>
    "C2-adaptive": ("C2-cornell", {"width": 96, "samples": 64, "aTolerance": 0.05, "aBatch": 8, "seed": 23}, None),
    "C4-rain-adaptive": ("C4-rain", {"width": 96, "samples": 30, "aTolerance": 0.1, "aBatch": 10, "seed": 23}, None),  # _trav
    "C5-layered": ("C5-layered", {"width": 96, "samples": 12, "aTolerance": 0, "seed": 2}, None),
    "default-reference-tree": ("default", {"width": 96, "samples": 8, "aTolerance": 0, "seed": 9, "bvh": "reference"}, None),
    "shadow-rays": ("C2-cornell", {"width": 80, "samples": 12, "aTolerance": 0, "seed": 4, "lightSampling": "shadowRays"}, None),
    "zero-samples": ("C2-cornell", {"width": 64, "samples": 0, "seed": 4}, None),
    "iterations-0": ("C2-cornell", {"width": 80, "samples": 8, "aTolerance": 0, "seed": 6}, {"iterations": 0}),
    "iterations-1": ("default", {"width": 80, "samples": 8, "aTolerance": 0, "seed": 6}, {"iterations": 1, "sigmaLuminance": 2.5}),
    "iterations-8": ("C2-cornell", {"width": 80, "samples": 8, "aTolerance": 0, "seed": 6},
                     {"iterations": 8, "sigmaLuminance": 6.0, "sigmaNormal": 64.0, "sigmaDepth": 0.5}),
}


def _regions(W, H):
    return {
        "whole": None,
        "ragged": {"x": 7, "y": 5, "width": W // 2 + 3, "height": H // 2 + 1},
        "right-bottom": {"x": W - 29, "y": H - 17, "width": 40, "height": 40},  # clipped at the image
        "row": {"x": 3, "y": H // 2, "width": W - 5, "height": 1},
        "column": {"x": W // 3, "y": 0, "width": 1, "height": H},
    }


def _bounds(W, H, region):
    if region is None:
        return 0, 0, W, H
    x0, y0 = region["x"], region["y"]
    return x0, y0, min(W, x0 + region["width"]), min(H, y0 + region["height"])


def _inside(W, H, region):
    x0, y0, x1, y1 = _bounds(W, H, region)
    m = np.zeros((H, W), bool)
    m[y0:y1, x0:x1] = True
    return m


def _buffers(W, H):
    return np.full((H, W, 3), 77, np.uint8), np.full((H, W, 3), -3.0, np.float32), np.full((H, W, 8), -5.0, np.float32)


def _same(a, b):
    """Bit-identical arrays (NaN pixels of a zero-sample render included)."""
    return a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def _stat_key(st):
    return (st.pixels, st.samples["total"], st.samples["min"], st.samples["max"], st.bounces["total"], st.bounces["min"],
            st.bounces["max"], st.rays)


def _one_shot(cam, region, dn):
    """renderDenoised's rgb8 / linear / stats and renderRegion's moments, on the buffers the progressive call gets."""
    W, H = cam.imageWidth, cam.imageHeight
    rgb, lin, mom = _buffers(W, H)
    st = cam.renderDenoised(rgb, lin, region, dn)
    cam.renderRegion(None, region, None, mom)
    return rgb, lin, mom, st


def _progressive(cam, passes, region, dn, keep=False, stop_after=None):
    """renderProgressiveDenoised with fresh buffers; `keep`: copies of every preview, as onPass sees them."""
    W, H = cam.imageWidth, cam.imageHeight
    rgb, lin, mom = _buffers(W, H)
    seen = []

    def on_pass(k, n, cap, so_far):
        seen.append({"pass": k, "cap": cap, "stats": _stat_key(so_far),
                     **({"rgb": rgb.copy(), "lin": lin.copy(), "mom": mom.copy()} if keep else {})})
        return stop_after is not None and len(seen) == stop_after

    st = cam.renderProgressiveDenoised(rgb, passes, on_pass, region=region, linear=lin, moments=mom, options=dn)
    return rgb, lin, mom, st, seen


# ---- 1. the last pass is the one-shot call ----
@pytest.mark.parametrize("case", list(CASES))
def test_last_pass_equals_render_denoised(gpu, case):
    name, opts, dn = CASES[case]
    sd = SCENES[name]()
    S = opts["samples"]
    with createCameraFromSceneData(sd, opts) as cam:
        W, H = cam.imageWidth, cam.imageHeight
        if name == "C4-rain":
            assert cam.info.n_bvh_nodes >= 16384 and cam.info.bvh_kind == 2  # deep tree: k_render_stream_trav
        for rname, region in _regions(W, H).items():
            want = _one_shot(cam, region, dn)
            out = ~_inside(W, H, region)
            for passes in (1, 3, 7, S + 3):
                rgb, lin, mom, st, seen = _progressive(cam, passes, region, dn)
                what = (case, rname, passes)
                assert _same(rgb, want[0]) and _same(lin, want[1]) and _same(mom, want[2]), what
                assert _stat_key(st) == _stat_key(want[3]), (what, _stat_key(st), _stat_key(want[3]))
                assert st.deviceMs > 0 and st.kernelLaunches >= want[3].kernelLaunches, what
                assert np.all(rgb[out] == 77) and np.all(lin[out] == -3.0) and np.all(mom[out] == -5.0), what
                caps = [s["cap"] for s in seen]
                assert caps == sorted(set(caps)) and caps[-1] == S and len(seen) <= passes, what


# ---- 2. every pass is the filter of the render with that pass's cap ----
PASS_CASES = {
    "cornell-fixed": ("C2-cornell", {"width": 96, "samples": 24, "aTolerance": 0, "seed": 5}, 5, None),
    "C1-adaptive": ("C1-spheres", {"width": 120, "samples": 100, "aTolerance": 0.05, "aBatch": 10, "seed": 3}, 6, None),
    "C4-rain-adaptive": ("C4-rain", {"width": 96, "samples": 30, "aTolerance": 0.1, "aBatch": 10, "seed": 23}, 3, {"iterations": 3}),
}


@pytest.mark.parametrize("case", list(PASS_CASES))
def test_every_pass_is_the_filter_of_that_passs_render(gpu, case):
    """Streams are keyed by (pixel, sample) and a pixel stopped by convergence stops at the same batch, so the moments
    after a pass with cap C are those of a camera with samples = C; the preview is the filter of that render's colour
    and moments with the features of the full camera (min(samples, 8) rays)."""
    name, opts, passes, dn = PASS_CASES[case]
    sd = SCENES[name]()
    S = opts["samples"]
    with createCameraFromSceneData(sd, opts) as cam:
        W, H = cam.imageWidth, cam.imageHeight
        regions = {"whole": None, "ragged": {"x": 7, "y": 5, "width": W // 2 + 3, "height": H // 2 + 1}}
        runs = {rname: _progressive(cam, passes, region, dn, keep=True)[4] for rname, region in regions.items()}
        again = _progressive(cam, passes, None, dn, keep=True)[4]  # every check below relies on bit-deterministic renders
        assert [p["cap"] for p in again] == [p["cap"] for p in runs["whole"]]
        for p, q in zip(runs["whole"], again):
            assert all(_same(p[k], q[k]) for k in ("rgb", "lin", "mom")), ("a repeated call differs", case, p["pass"])
        feats = {rname: cam.renderFeatures(min(S, 8), region) for rname, region in regions.items()}
    checked = 0
    for rname, region in regions.items():
        x0, y0, x1, y1 = _bounds(W, H, region)
        ys, xs = slice(y0, y1), slice(x0, x1)
        f = feats[rname]
        for p in runs[rname]:
            cap = p["cap"]
            if cap < 2:  # one sample: no jitter, so not the first sample of the full camera
                continue
            with createCameraFromSceneData(sd, {**opts, "samples": cap}) as c:
                lin0 = np.zeros((H, W, 3), np.float32)
                mom0 = np.full((H, W, 8), -5.0, np.float32)
                c.renderRegion(None, region, lin0, mom0)
            what = (case, rname, p["pass"], cap)
            assert _same(p["mom"], mom0), ("moments differ from the one-shot render with samples = cap", what)
            if region is None:
                want = denoise(lin0, f["albedo"], f["normal"], f["depth"], mom0, dn)
                assert _same(p["lin"], want), ("preview differs from rt_denoise of that render", what)
            else:
                args = (lin0[ys, xs], f["albedo"][ys, xs], f["normal"][ys, xs], f["depth"][ys, xs], mom0[ys, xs])
                _check_against_spec(p["lin"][ys, xs], args, dn, what)
            assert np.array_equal(p["rgb"][ys, xs], dref.gamma_rgb8(p["lin"][ys, xs])), ("rgb8 is not gamma_rgb8(linear)", what)
            checked += 1
    assert checked >= 2 * (passes - 1), checked


def _check_against_spec(got, args, opts, what):
    """The filter's bars against denoise_reference: 1e-4 relative (+1e-7) where the spec is finite, non-finite exactly
    where it is, and pass-through pixels bit-equal to the input colour."""
    ref = dref.denoise(*args, opts)
    fin = np.isfinite(ref)
    assert np.array_equal(np.isfinite(got), fin), ("finite pixels differ from the spec's", what)
    with np.errstate(invalid="ignore"):
        err = np.abs(got.astype(np.float64) - ref)
    assert np.all((err <= 1e-4 * np.abs(ref) + 1e-7)[fin]), ("off the spec", what, float((err[fin] / (np.abs(ref[fin]) + 1e-7)).max()))
    passed = ~dref.prepare(*args)["valid"]
    color = np.asarray(args[0], np.float32)
    assert np.array_equal(got[passed].view(np.uint32), color[passed].view(np.uint32)), ("pass-through pixels changed", what)


# ---- 3. each preview is cleaner than its noisy image ----
def _rel_mse(x, r):
    return float(((x.astype(np.float64) - r) ** 2 / (r.astype(np.float64) ** 2 + 0.01)).mean())


def test_every_preview_meets_the_quality_bar(gpu):
    sd = SCENES["C2-cornell"]()
    base = {"width": 128, "aspect": 1.0, "aTolerance": 0}
    with createCameraFromSceneData(sd, {**base, "samples": 8192, "seed": 1234}) as cam:
        ref = np.zeros((cam.imageHeight, cam.imageWidth, 3), np.float32)
        cam.renderRegion(None, None, ref)
    with createCameraFromSceneData(sd, {**base, "samples": 32, "seed": 7}) as cam:
        seen = _progressive(cam, 4, None, None, keep=True)[4]
    assert [p["cap"] for p in seen] == [8, 16, 24, 32]
    for p in seen:
        with createCameraFromSceneData(sd, {**base, "samples": p["cap"], "seed": 7}) as cam:
            noisy = np.zeros_like(ref)
            cam.renderRegion(None, None, noisy)
        e_noisy, e_den = _rel_mse(noisy, ref), _rel_mse(p["lin"], ref)
        print(f"pass {p['pass']} ({p['cap']} spp): relMSE noisy {e_noisy:.5f} denoised {e_den:.5f}")
        assert e_den <= 0.4 * e_noisy, (p["cap"], e_noisy, e_den)


# ---- 4. early stop, callback errors, reuse and argument errors ----
def test_early_stop_errors_and_reuse(gpu):
    sd = SCENES["C2-cornell"]()
    opts = {"width": 64, "samples": 40, "aTolerance": 0.05, "aBatch": 4, "seed": 2}
    region = {"x": 3, "y": 5, "width": 50, "height": 30}
    with createCameraFromSceneData(sd, opts) as cam:
        W, H = cam.imageWidth, cam.imageHeight
        want = _one_shot(cam, region, None)
        full = _progressive(cam, 8, region, None, keep=True)[4]
        rgb, lin, mom, st, seen = _progressive(cam, 8, region, None, stop_after=3)
        assert len(seen) == 3
        p = full[2]
        assert _same(rgb, p["rgb"]) and _same(lin, p["lin"]) and _same(mom, p["mom"])
        assert _stat_key(st) == p["stats"] == seen[-1]["stats"] and st.samples["total"] < want[3].samples["total"]
        with pytest.raises(RuntimeError, match="boom"):
            cam.renderProgressiveDenoised(np.zeros((H, W, 3), np.uint8), 4, lambda *a: (_ for _ in ()).throw(RuntimeError("boom")))
        got = _one_shot(cam, region, None)  # the camera still renders the one-shot bytes
        assert all(_same(a, b) for a, b in zip(got[:3], want[:3]))
        buf = np.zeros(W * H * 3, np.uint8)
        for bad in ({"iterations": 9}, {"iterations": -1}, {"sigmaLuminance": -1.0}, {"sigmaDepth": float("nan")},
                    {"sigmaNormal": float("inf")}):
            with pytest.raises(RaytracerError, match="RT_ERR_INVALID_ARGUMENT"):
                cam.renderProgressiveDenoised(buf, 2, options=bad)
        for n in (0, -1):
            with pytest.raises(RaytracerError, match="RT_ERR_INVALID_ARGUMENT"):
                cam.renderProgressiveDenoised(buf, n)
        with pytest.raises(RaytracerError, match="RT_ERR_BUFFER_TOO_SMALL"):
            cam.renderProgressiveDenoised(buf[:-1], 2)
    for bad in ({"partIndex": 0, "partCount": 2}, {"mode": "bounces"}, {"mode": "samples"}):
        with createCameraFromSceneData(sd, {**opts, **bad}) as cam:
            with pytest.raises(RaytracerError, match="RT_ERR_UNSUPPORTED"):
                cam.renderProgressiveDenoised(np.zeros(cam.imageWidth * cam.imageHeight * 3, np.uint8), 2)
