"""GPU checks of the denoiser on every device (rt_multi_render_denoised / MultiCamera.renderDenoised): the filtered image is
bit-identical to one Camera's renderDenoised for every device count, on the peer-write path and the host-merge path, over
scenes, options and regions; pixels outside the region are untouched; stats equal the one-camera stats.  The band and
halo logic also runs on one GPU: RT_B200_DENOISE_BANDS=n filters n bands one after another, their buffers filled with NaN
first.  Run on a B200 with `-m gpu`."""
import numpy as np
import pytest

from mcp_raytracer_b200 import (
    MultiCamera, RaytracerError, createCameraFromSceneData, generateCornellSceneData, generateDefaultSceneData,
    generateLayeredMixedSceneData, generateSceneData, generateSpheresSceneData, renderScene,
)
from mcp_raytracer_b200 import _native
from mcp_raytracer_b200.raytracer import applySceneCameraOptions

pytestmark = pytest.mark.gpu

SCENES = {
    "C1-spheres": lambda: generateSpheresSceneData({"count": 100, "seed": 12345}),
    "C2-cornell": generateCornellSceneData,
    "C5-layered": generateLayeredMixedSceneData,
    "default": generateDefaultSceneData,
}
# (scene, render options, denoise options)
CASES = {
    "cornell-fixed": ("C2-cornell", {"width": 96, "samples": 16, "aTolerance": 0, "seed": 5}, None),
    "C1-adaptive": ("C1-spheres", {"width": 120, "samples": 40, "seed": 3}, None),  # the reference's adaptive defaults
    "C5-mixed-layered": ("C5-layered", {"width": 96, "samples": 12, "aTolerance": 0, "seed": 2}, None),
    "default-defocus": ("default", {"width": 120, "samples": 8, "aTolerance": 0, "seed": 9}, None),
    "shadow-rays": ("C2-cornell", {"width": 80, "samples": 12, "aTolerance": 0, "seed": 4, "lightSampling": "shadowRays"}, None),
    "iterations-0": ("C2-cornell", {"width": 80, "samples": 8, "aTolerance": 0, "seed": 6}, {"iterations": 0}),
    "iterations-1": ("default", {"width": 80, "samples": 8, "aTolerance": 0, "seed": 6}, {"iterations": 1, "sigmaLuminance": 2.5}),
    "iterations-8": ("C2-cornell", {"width": 80, "samples": 8, "aTolerance": 0, "seed": 6},
                     {"iterations": 8, "sigmaLuminance": 6.0, "sigmaNormal": 64.0, "sigmaDepth": 0.5}),
}


def _devices():
    n = _native.lib().rt_device_count()
    return [1] + ([n] if n > 1 else [])


def _regions(W, H, n):
    return {
        "whole": None,
        "ragged": {"x": 7, "y": 5, "width": W // 2 + 3, "height": H // 2 + 1},
        "right-bottom": {"x": W - 29, "y": H - 17, "width": 40, "height": 40},  # clipped at the image
        "row": {"x": 3, "y": H // 2, "width": W - 5, "height": 1},
        "column": {"x": W // 3, "y": 0, "width": 1, "height": H},
        "few-rows": {"x": 2, "y": 9, "width": W - 4, "height": max(1, min(3, n - 1))},  # fewer rows than devices (n > 1)
    }


def _inside(W, H, region):
    m = np.zeros((H, W), bool)
    if region is None:
        m[:] = True
    else:
        m[region["y"]:region["y"] + region["height"], region["x"]:region["x"] + region["width"]] = True
    return m


def _render(cam, region, dn):
    W, H = cam.imageWidth, cam.imageHeight
    rgb = np.full((H, W, 3), 77, np.uint8)
    lin = np.full((H, W, 3), -3.0, np.float32)
    st = cam.renderDenoised(rgb, lin, region, dn)
    return rgb, lin, st


def _single(sd, opts, regions, dn):
    with createCameraFromSceneData(sd, opts) as cam:
        return {k: _render(cam, r, dn) for k, r in regions.items()}


def _set_path(monkeypatch, no_p2p):
    if no_p2p:
        monkeypatch.setenv("RT_B200_MULTI_NO_P2P", "1")
    else:
        monkeypatch.delenv("RT_B200_MULTI_NO_P2P", raising=False)


def _assert_same(got, want, W, H, region, what):
    rgb, lin, st = got
    wrgb, wlin, wst = want
    assert np.array_equal(rgb, wrgb) and np.array_equal(lin, wlin), what
    out = ~_inside(W, H, region)
    assert np.all(rgb[out] == 77) and np.all(lin[out] == -3.0), what
    assert (st.pixels, st.samples["total"], st.samples["min"], st.samples["max"], st.bounces["total"], st.rays) == \
           (wst.pixels, wst.samples["total"], wst.samples["min"], wst.samples["max"], wst.bounces["total"], wst.rays), what


@pytest.mark.parametrize("case", list(CASES))
def test_multi_denoised_equals_one_camera(gpu, case, monkeypatch):
    name, opts, dn = CASES[case]
    sd = SCENES[name]()
    ndev = _native.lib().rt_device_count()
    with createCameraFromSceneData(sd, opts) as cam:
        W, H = cam.imageWidth, cam.imageHeight
    regions = _regions(W, H, ndev)
    want = _single(sd, opts, regions, dn)
    for n in _devices():
        for no_p2p in (False, True):
            _set_path(monkeypatch, no_p2p)
            with MultiCamera(sd, opts, nDevices=n) as mc:
                assert mc.nDevices == n and (mc.imageWidth, mc.imageHeight) == (W, H)
                for rname, region in regions.items():
                    got = _render(mc, region, dn)
                    _assert_same(got, want[rname], W, H, region, (case, n, no_p2p, rname))
                    assert got[2].deviceMs > 0 and got[2].kernelLaunches >= want[rname][2].kernelLaunches
    monkeypatch.delenv("RT_B200_MULTI_NO_P2P", raising=False)


def test_repeated_calls_are_deterministic(gpu, monkeypatch):
    """The buffers of one call (device 0's colour, every device's scratch) are reused by the next: same bytes again."""
    monkeypatch.delenv("RT_B200_MULTI_NO_P2P", raising=False)
    sd = SCENES["default"]()
    opts = {"width": 96, "samples": 8, "aTolerance": 0, "seed": 1}
    n = _devices()[-1]
    with MultiCamera(sd, opts, nDevices=n) as mc:
        a = _render(mc, None, None)
        _render(mc, {"x": 4, "y": 4, "width": 30, "height": 20}, {"iterations": 3})
        b = _render(mc, None, None)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


# ---- bands on one GPU: RT_B200_DENOISE_BANDS deals n bands to the devices, each band's buffers NaN-filled first ----
TALL = ("C2-cornell", {"width": 48, "aspect": 48 / 400, "samples": 8, "aTolerance": 0, "seed": 8})  # 48 x 400


@pytest.mark.parametrize("region", [None, {"x": 5, "y": 37, "width": 30, "height": 301}], ids=["whole", "ragged"])
def test_bands_on_one_gpu_equal_one_camera(gpu, region, monkeypatch):
    """At K = 8 the 510-row prepare halo exceeds every band of this 400-row image; 7 bands of a 301-row region are 43 rows;
    more bands than rows leave most of them empty."""
    monkeypatch.delenv("RT_B200_MULTI_NO_P2P", raising=False)
    name, opts = TALL
    sd = SCENES[name]()
    with createCameraFromSceneData(sd, opts) as cam:
        W, H = cam.imageWidth, cam.imageHeight
        assert (W, H) == (48, 400)
        want = {k: _render(cam, region, {"iterations": k}) for k in range(9)}
    rows = H if region is None else region["height"]
    for bands in (2, 3, 7, rows + 5):
        monkeypatch.setenv("RT_B200_DENOISE_BANDS", str(bands))
        with MultiCamera(sd, opts, nDevices=1) as mc:
            for k in range(9):
                _assert_same(_render(mc, region, {"iterations": k}), want[k], W, H, region, (bands, k))
    monkeypatch.delenv("RT_B200_DENOISE_BANDS")


def test_bands_on_the_host_merge_path(gpu, monkeypatch):
    """Host merge on every device, the region cut into bands on device 0."""
    name, opts = TALL
    sd = SCENES[name]()
    region = {"x": 0, "y": 11, "width": 48, "height": 250}
    with createCameraFromSceneData(sd, opts) as cam:
        want = {k: _render(cam, region, {"iterations": k}) for k in (0, 4, 8)}
    monkeypatch.setenv("RT_B200_MULTI_NO_P2P", "1")
    monkeypatch.setenv("RT_B200_DENOISE_BANDS", "5")
    with MultiCamera(sd, opts, nDevices=_devices()[-1]) as mc:
        for k in want:
            _assert_same(_render(mc, region, {"iterations": k}), want[k], 48, 400, region, k)
    monkeypatch.delenv("RT_B200_DENOISE_BANDS")
    monkeypatch.delenv("RT_B200_MULTI_NO_P2P")


def test_multi_denoised_errors(gpu):
    sd = SCENES["C2-cornell"]()
    for mode in ("bounces", "samples"):
        with MultiCamera(sd, {"width": 32, "samples": 4, "mode": mode}, nDevices=_devices()[-1]) as mc:
            with pytest.raises(RaytracerError, match="RT_ERR_UNSUPPORTED"):
                mc.renderDenoised(np.zeros(mc.imageWidth * mc.imageHeight * 3, np.uint8))
    with MultiCamera(sd, {"width": 32, "samples": 4}, nDevices=_devices()[-1]) as mc:
        buf = np.zeros(mc.imageWidth * mc.imageHeight * 3, np.uint8)
        for bad in ({"iterations": 9}, {"iterations": -1}, {"sigmaLuminance": -1.0}, {"sigmaDepth": float("nan")},
                    {"sigmaNormal": float("inf")}):
            with pytest.raises(RaytracerError, match="RT_ERR_INVALID_ARGUMENT"):
                mc.renderDenoised(buf, options=bad)
        with pytest.raises(RaytracerError, match="RT_ERR_BUFFER_TOO_SMALL"):
            mc.renderDenoised(buf[:-1])
        with pytest.raises(RaytracerError, match="negative region"):
            mc.renderDenoised(buf, region={"x": -1, "y": 0, "width": 4, "height": 4})


def test_render_scene_denoise_parallel_uses_every_gpu(gpu, monkeypatch):
    calls = []
    orig = MultiCamera.renderDenoised

    def counted(self, *a, **k):
        calls.append(self.nDevices)
        return orig(self, *a, **k)

    monkeypatch.setattr(MultiCamera, "renderDenoised", counted)
    cfg = {"type": "cornell", "render": {"width": 96, "samples": 8, "aTolerance": 0, "seed": 3}}
    dn = {"iterations": 4, "sigmaLuminance": 3.0}
    img, st = renderScene(cfg, {"denoise": dn, "parallel": True})
    ndev = _native.lib().rt_device_count()
    assert calls == ([ndev] if ndev > 1 else [])
    sd = applySceneCameraOptions(generateSceneData(cfg), cfg.get("camera"))
    with createCameraFromSceneData(sd, cfg["render"]) as cam:
        rgb = np.zeros((cam.imageHeight, cam.imageWidth, 3), np.uint8)
        one = cam.renderDenoised(rgb, options=dn)
    assert np.array_equal(img, rgb) and st.rays == one.rays and st.samples == one.samples
