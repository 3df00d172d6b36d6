"""GPU checks of the progressive renders on every device (rt_multi_render_progressive / _denoised, MultiCamera.renderProgressive
and renderProgressiveDenoised): pass by pass, the caps, the bytes in the caller's buffers and the stats so far equal one
Camera's renderProgressive / renderProgressiveDenoised, on 1 and every visible GPU, with 2, 3 and 8 parts on one GPU
(RT_B200_MULTI_PARTS), and on both the peer-write and host-merge paths; pixels outside the region keep their sentinels;
one pass is the one-shot multi call; reuse, early stops, callback errors and argument errors.  Run on a B200 with `-m gpu`."""
import numpy as np
import pytest

from mcp_raytracer_b200 import (
    MultiCamera, RaytracerError, createCameraFromSceneData, generateCornellSceneData, generateLayeredMixedSceneData,
    generateRainSceneData, generateSpheresSceneData,
)
from mcp_raytracer_b200 import _native
from test_gpu_progressive_denoise import CASES as DN_CASES, SCENES as DN_SCENES, _one_shot as dn_one_shot

pytestmark = pytest.mark.gpu

SCENES = {
    "C1-spheres": lambda: generateSpheresSceneData({"count": 100, "seed": 12345}),
    "C2-cornell": generateCornellSceneData,
    "C4-rain": lambda: generateRainSceneData({"count": 20000, "seed": 1, "sphereRadius": 0.01}),
    "C4-rain-100k": lambda: generateRainSceneData({"count": 100000, "seed": 1, "sphereRadius": 0.01}),
    "C5-layered": generateLayeredMixedSceneData,
}
# the kernels of test_progressive_render_ends_in_the_one_shot_image, with partitions
PLAIN_CASES = {
    "cornell-fixed": ("C2-cornell", {"width": 96, "samples": 50}),                                        # k_render_pool<LIST>
    "C5-sorted": ("C5-layered", {"width": 80, "samples": 24}),                                            # k_render_sorted
    "rain-20k-fixed": ("C4-rain", {"width": 96, "samples": 9}),                                           # k_render_trav
    "rain-100k-fixed": ("C4-rain-100k", {"width": 96, "samples": 6}),                                     # k_render_trav
    "C1-adaptive": ("C1-spheres", {"width": 120, "samples": 100, "aTolerance": 0.05, "aBatch": 10}),      # k_render_stream<SAH>
    "cornell-adaptive": ("C2-cornell", {"width": 96, "samples": 64, "aTolerance": 0.05, "aBatch": 8}),    # k_render_stream<LIST>
    "rain-adaptive": ("C4-rain", {"width": 96, "samples": 30, "aTolerance": 0.1, "aBatch": 10}),          # k_render_stream_trav
    "C1-bounces": ("C1-spheres", {"width": 96, "samples": 12, "mode": "bounces"}),                        # a render mode
}


def _configs():
    """(devices, parts or None, host merge): every device count, 2 / 3 / 8 parts on one GPU, both paths."""
    n = _native.lib().rt_device_count()
    base = [(1, None)] + ([(n, None)] if n > 1 else []) + [(1, p) for p in (2, 3, 8)]
    return [(d, p, h) for d, p in base for h in (False, True)]


def _multi(monkeypatch, sd, opts, devices, parts, host_merge):
    if parts:
        monkeypatch.setenv("RT_B200_MULTI_PARTS", str(parts))
    else:
        monkeypatch.delenv("RT_B200_MULTI_PARTS", raising=False)
    if host_merge:
        monkeypatch.setenv("RT_B200_MULTI_NO_P2P", "1")
    else:
        monkeypatch.delenv("RT_B200_MULTI_NO_P2P", raising=False)
    mc = MultiCamera(sd, opts, nDevices=devices)
    monkeypatch.delenv("RT_B200_MULTI_PARTS", raising=False)
    monkeypatch.delenv("RT_B200_MULTI_NO_P2P", raising=False)
    assert mc.nDevices == (parts or devices)
    if parts:
        assert mc.peerWrites == (not host_merge)  # parts on device 0 itself need no peer mapping
    return mc


def _regions(W, H):
    return {
        "whole": None,
        "ragged": {"x": 7, "y": 5, "width": W // 2 + 3, "height": H // 2 + 1},
        "right-bottom": {"x": W - 29, "y": H - 17, "width": 40, "height": 40},  # clipped at the image
        "row": {"x": 3, "y": H // 2, "width": W - 5, "height": 1},
        "column": {"x": W // 3, "y": 0, "width": 1, "height": H},
        "few-rows": {"x": 2, "y": 9, "width": W - 4, "height": 2},  # fewer rows than parts
    }


def _inside(W, H, region):
    m = np.zeros((H, W), bool)
    if region is None:
        m[:] = True
    else:
        m[region["y"]:region["y"] + region["height"], region["x"]:region["x"] + region["width"]] = True
    return m


def _same(a, b):
    """Bit-identical arrays (NaN pixels of a zero-sample render included)."""
    return a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def _stat_key(st):
    return (st.pixels, st.samples["total"], st.samples["min"], st.samples["max"], st.bounces["total"], st.bounces["min"],
            st.bounces["max"], st.rays)


def _run(cam, passes, region, dn=False, options=None, stop_after=None):
    """renderProgressive (dn: renderProgressiveDenoised with moments) on sentinel buffers; every pass's bytes as onPass
    sees them.  Returns (final buffers, stats, passes)."""
    W, H = cam.imageWidth, cam.imageHeight
    rgb = np.full((H, W, 3), 77, np.uint8)
    lin = np.full((H, W, 3), -3.0, np.float32)
    mom = np.full((H, W, 8), -5.0, np.float32) if dn else None
    seen = []

    def on_pass(k, n, cap, so_far):
        seen.append({"pass": k, "n": n, "cap": cap, "stats": _stat_key(so_far), "rgb": rgb.copy(), "lin": lin.copy(),
                     "mom": mom.copy() if dn else None, "ms": so_far.deviceMs, "launches": so_far.kernelLaunches})
        return stop_after is not None and len(seen) == stop_after

    if dn:
        st = cam.renderProgressiveDenoised(rgb, passes, on_pass, region=region, linear=lin, moments=mom, options=options)
    else:
        st = cam.renderProgressive(rgb, passes, on_pass, region=region, linear=lin)
    return (rgb, lin, mom), st, seen


def _assert_passes(got, want, W, H, region, what):
    (rgb, lin, mom), st, seen = got
    (wrgb, wlin, wmom), wst, wseen = want
    assert [(p["pass"], p["n"], p["cap"]) for p in seen] == [(p["pass"], p["n"], p["cap"]) for p in wseen], what
    for p, q in zip(seen, wseen):
        w = (what, p["pass"])
        assert _same(p["rgb"], q["rgb"]) and _same(p["lin"], q["lin"]), w
        assert q["mom"] is None or _same(p["mom"], q["mom"]), w
        assert p["stats"] == q["stats"], (w, p["stats"], q["stats"])
        assert p["ms"] > 0 or not p["stats"][1], w
    assert _same(rgb, wrgb) and _same(lin, wlin) and (wmom is None or _same(mom, wmom)), what
    assert _stat_key(st) == _stat_key(wst), what
    out = ~_inside(W, H, region)
    assert np.all(rgb[out] == 77) and np.all(lin[out] == -3.0) and (mom is None or np.all(mom[out] == -5.0)), what


def _one_shot(cam, region, dn, options=None):
    """One Camera's one-shot call on the sentinel buffers: renderRegion, or renderDenoised with renderRegion's moments."""
    if dn:
        return dn_one_shot(cam, region, options)
    W, H = cam.imageWidth, cam.imageHeight
    rgb = np.full((H, W, 3), 77, np.uint8)
    lin = np.full((H, W, 3), -3.0, np.float32)
    st = cam.renderRegion(rgb, region, lin)
    return rgb, lin, None, st


def _check_against_one_camera(monkeypatch, sd, opts, dn, options=None):
    """Every pass against one Camera's progressive call, and the last pass against one Camera's one-shot call."""
    S = opts["samples"]
    with createCameraFromSceneData(sd, opts) as cam:
        W, H = cam.imageWidth, cam.imageHeight
        regions = _regions(W, H)
        want = {(r, n): _run(cam, n, region, dn, options) for r, region in regions.items() for n in (1, 3, 7, S + 3)}
        shot = {r: _one_shot(cam, region, dn, options) for r, region in regions.items()}
    for devices, parts, host_merge in _configs():
        with _multi(monkeypatch, sd, opts, devices, parts, host_merge) as mc:
            for (r, n), w in want.items():
                what = (devices, parts, host_merge, r, n)
                got = _run(mc, n, regions[r], dn, options)
                _assert_passes(got, w, W, H, regions[r], what)
                (rgb, lin, mom), st, _ = got
                srgb, slin, smom, sst = shot[r]
                assert _same(rgb, srgb) and _same(lin, slin) and (smom is None or _same(mom, smom)), ("not the one-shot image", what)
                # The bounce extremes are left out: one-shot adaptive renders (k_render_adaptive) take them only from
                # lanes that folded a pixel, so in sparse regions (a 1-pixel row or column) they can miss a path's bounces.
                assert _stat_key(st)[:5] + _stat_key(st)[7:] == _stat_key(sst)[:5] + _stat_key(sst)[7:], ("not the one-shot stats", what)


# ---- 1. plain form, pass by pass ----
@pytest.mark.parametrize("case", list(PLAIN_CASES))
def test_multi_progressive_equals_one_camera(gpu, case, monkeypatch):
    name, opts = PLAIN_CASES[case]
    _check_against_one_camera(monkeypatch, SCENES[name](), {"aTolerance": 0, "seed": 23, **opts}, dn=False)


# ---- 2. denoised form, pass by pass ----
@pytest.mark.parametrize("case", list(DN_CASES))
def test_multi_progressive_denoised_equals_one_camera(gpu, case, monkeypatch):
    name, opts, options = DN_CASES[case]
    _check_against_one_camera(monkeypatch, DN_SCENES[name](), opts, dn=True, options=options)


TALL = ("C2-cornell", {"width": 48, "aspect": 48 / 400, "samples": 12, "aTolerance": 0.1, "aBatch": 4, "seed": 8})  # 48 x 400


def test_bands_on_one_gpu_equal_one_camera(gpu, monkeypatch):
    """RT_B200_DENOISE_BANDS cuts the rows into 3 or more-than-rows bands, dealt to the parts, their buffers NaN-filled
    first; at 8 iterations the 510-row halo exceeds every band of this 400-row image."""
    name, opts = TALL
    sd = SCENES[name]()
    with createCameraFromSceneData(sd, opts) as cam:
        W, H = cam.imageWidth, cam.imageHeight
        assert (W, H) == (48, 400)
        want = {k: _run(cam, 3, None, True, {"iterations": k}) for k in range(9)}
    for bands in (3, H + 5):
        for parts, host_merge in ((None, False), (2, False), (2, True)):
            monkeypatch.setenv("RT_B200_DENOISE_BANDS", str(bands))
            with _multi(monkeypatch, sd, opts, 1, parts, host_merge) as mc:
                for k in range(9):
                    _assert_passes(_run(mc, 3, None, True, {"iterations": k}), want[k], W, H, None, (bands, parts, host_merge, k))
    monkeypatch.delenv("RT_B200_DENOISE_BANDS")


# ---- 3. one pass is the one-shot multi call ----
def test_one_pass_equals_the_one_shot_multi_call(gpu, monkeypatch):
    for name, opts in (("C2-cornell", {"width": 96, "samples": 16, "aTolerance": 0, "seed": 5}),
                       ("C1-spheres", {"width": 120, "samples": 40, "aTolerance": 0.05, "aBatch": 8, "seed": 3})):
        sd = SCENES[name]()
        region = {"x": 7, "y": 5, "width": 61, "height": 37}
        for devices, parts, host_merge in _configs():
            with _multi(monkeypatch, sd, opts, devices, parts, host_merge) as mc:
                W, H = mc.imageWidth, mc.imageHeight
                for dn in (False, True):
                    rgb = np.full((H, W, 3), 77, np.uint8)
                    lin = np.full((H, W, 3), -3.0, np.float32)
                    st = mc.renderDenoised(rgb, lin, region) if dn else mc.renderRegion(rgb, region, lin)
                    (prgb, plin, _), pst, seen = _run(mc, 1, region, dn)
                    what = (name, devices, parts, host_merge, dn)
                    assert len(seen) == 1 and seen[0]["cap"] == opts["samples"], what
                    assert _same(prgb, rgb) and _same(plin, lin), what
                    assert _stat_key(pst) == _stat_key(st) and pst.kernelLaunches == st.kernelLaunches, what


# ---- 4. determinism across reuse ----
def test_reuse_is_deterministic(gpu, monkeypatch):
    """State that leaks between calls (PixelStats, fixed-point sums, device 0's colour, the features) changes the bytes."""
    sd = SCENES["C2-cornell"]()
    opts = {"width": 96, "samples": 40, "aTolerance": 0.05, "aBatch": 4, "seed": 2}
    region = {"x": 3, "y": 5, "width": 70, "height": 50}
    for devices, parts, host_merge in _configs():
        with _multi(monkeypatch, sd, opts, devices, parts, host_merge) as mc:
            W, H = mc.imageWidth, mc.imageHeight
            for dn in (False, True):
                what = (devices, parts, host_merge, dn)
                a = _run(mc, 5, region, dn)
                _assert_passes(_run(mc, 5, region, dn), a, W, H, region, what)
                _run(mc, 3, None, dn, {"iterations": 2} if dn else None)  # another region, other options
                _assert_passes(_run(mc, 5, region, dn), a, W, H, region, what)
                _run(mc, 7, {"x": 0, "y": 0, "width": 40, "height": 90}, not dn, stop_after=2)  # an early stop of the other form
                _assert_passes(_run(mc, 5, region, dn), a, W, H, region, what)


# ---- 5. early stop, callback errors, argument errors ----
def test_early_stop_errors(gpu, monkeypatch):
    sd = SCENES["C2-cornell"]()
    opts = {"width": 64, "samples": 40, "aTolerance": 0.05, "aBatch": 4, "seed": 2}
    region = {"x": 3, "y": 5, "width": 50, "height": 30}
    for devices, parts, host_merge in _configs():
        with _multi(monkeypatch, sd, opts, devices, parts, host_merge) as mc:
            W, H = mc.imageWidth, mc.imageHeight
            for dn in (False, True):
                what = (devices, parts, host_merge, dn)
                full = _run(mc, 8, region, dn)
                (rgb, lin, mom), st, seen = _run(mc, 8, region, dn, stop_after=3)
                p = full[2][2]
                assert len(seen) == 3 and seen[-1]["cap"] == p["cap"], what
                assert _same(rgb, p["rgb"]) and _same(lin, p["lin"]) and (mom is None or _same(mom, p["mom"])), what
                assert _stat_key(st) == p["stats"] == seen[-1]["stats"], what
                assert st.samples["total"] < _stat_key(full[1])[1], what
                boom = lambda *a: (_ for _ in ()).throw(RuntimeError("boom"))  # noqa: E731
                with pytest.raises(RuntimeError, match="boom"):
                    if dn:
                        mc.renderProgressiveDenoised(np.zeros((H, W, 3), np.uint8), 4, boom)
                    else:
                        mc.renderProgressive(np.zeros((H, W, 3), np.uint8), 4, boom)
                one = _run(mc, 1, region, dn)  # still the one-shot bytes
                rgb1 = np.full((H, W, 3), 77, np.uint8)
                lin1 = np.full((H, W, 3), -3.0, np.float32)
                mc.renderDenoised(rgb1, lin1, region) if dn else mc.renderRegion(rgb1, region, lin1)
                assert _same(one[0][0], rgb1) and _same(one[0][1], lin1), what
            buf = np.zeros(W * H * 3, np.uint8)
            for n in (0, -1):
                with pytest.raises(RaytracerError, match="RT_ERR_INVALID_ARGUMENT"):
                    mc.renderProgressive(buf, n)
                with pytest.raises(RaytracerError, match="RT_ERR_INVALID_ARGUMENT"):
                    mc.renderProgressiveDenoised(buf, n)
            with pytest.raises(RaytracerError, match="RT_ERR_BUFFER_TOO_SMALL"):
                mc.renderProgressive(buf[:-1], 2)
            with pytest.raises(RaytracerError, match="RT_ERR_BUFFER_TOO_SMALL"):
                mc.renderProgressiveDenoised(buf[:-1], 2)
            for bad in ({"iterations": 9}, {"iterations": -1}, {"sigmaLuminance": -1.0}, {"sigmaDepth": float("nan")},
                        {"sigmaNormal": float("inf")}):
                with pytest.raises(RaytracerError, match="RT_ERR_INVALID_ARGUMENT"):
                    mc.renderProgressiveDenoised(buf, 2, options=bad)
            for call in (mc.renderProgressive, mc.renderProgressiveDenoised):
                with pytest.raises(RaytracerError, match="negative region"):
                    call(buf, 2, region={"x": -1, "y": 0, "width": 4, "height": 4})
    for mode in ("bounces", "samples"):
        with _multi(monkeypatch, sd, {**opts, "mode": mode}, 1, 2, False) as mc:
            buf = np.zeros(mc.imageWidth * mc.imageHeight * 3, np.uint8)
            with pytest.raises(RaytracerError, match="RT_ERR_UNSUPPORTED"):
                mc.renderProgressiveDenoised(buf, 2)
            mc.renderProgressive(buf, 2)  # the plain form renders every mode
