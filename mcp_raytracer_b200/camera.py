"""Host-side mirror of the reference's `Camera` (src/camera.ts) over the C ABI.

Same names and argument meaning as the reference so callers and tests read alike:

* `Camera(world, cameraOptions, renderData)`      <- src/camera.ts:107-166 (world = SceneData here)
* `camera.render(pixelData) -> RenderStats`       <- src/camera.ts:439-446
* `camera.renderRegion(buffer, region)`           <- src/camera.ts:388-431
* `RenderStats`, `RenderStats.merge`              <- src/render-utils/renderStats.ts:6-64
* `RenderMode`                                    <- src/camera.ts:13-17
* `createCameraFromSceneData`, `generateScene`    <- src/scenes/scenes.ts:52-104

All arithmetic happens in the CUDA library; this file only marshals.  `pixelData` is a
numpy uint8 array of imageWidth*imageHeight*3 bytes (the Uint8ClampedArray of the reference).
"""
from __future__ import annotations

import ctypes as C
import enum
import math
from typing import Any, Dict, List, Optional

import numpy as np

from . import _native
from .scene_data import (
    FlatScene, RaytracerError, denoise_opts_struct, merge_render_options, render_opts_struct, rt_camera_info, rt_region, rt_stats,
)
from .scenes import generateSceneData


class RenderMode(str, enum.Enum):
    Default = "default"
    Bounces = "bounces"
    Samples = "samples"


class RenderStats:
    """src/render-utils/renderStats.ts:6-64"""

    def __init__(self) -> None:
        self.pixels = 0
        self.samples = {"total": 0, "min": math.inf, "max": 0, "avg": 0}
        self.bounces = {"total": 0, "min": math.inf, "max": 0, "avg": 0}
        # measurement extras (not in the reference)
        self.rays = 0
        self.deviceMs = 0.0
        self.kernelLaunches = 0
        self.nodeVisits = 0
        self.primTests = 0

    @staticmethod
    def from_struct(s: rt_stats) -> "RenderStats":
        r = RenderStats()
        r.pixels = int(s.pixels)
        r.samples["total"] = int(s.samples_total)
        r.bounces["total"] = int(s.bounces_total)
        if r.pixels > 0:
            r.samples["min"] = int(s.samples_min)
            r.samples["max"] = int(s.samples_max)
            r.bounces["min"] = int(s.bounces_min)
            r.bounces["max"] = int(s.bounces_max)
            r.samples["avg"] = r.samples["total"] / r.pixels
        if r.samples["total"] > 0:
            r.bounces["avg"] = r.bounces["total"] / r.samples["total"]
        r.rays = int(s.rays)
        r.deviceMs = float(s.device_ms)
        r.kernelLaunches = int(s.kernel_launches)
        r.nodeVisits = int(s.node_visits)   # instrumented build only (rt_counts_events)
        r.primTests = int(s.prim_tests)
        return r

    @staticmethod
    def merge(stats: List["RenderStats"]) -> "RenderStats":
        m = RenderStats()
        for s in stats:
            m.pixels += s.pixels
            m.samples["total"] += s.samples["total"]
            m.samples["min"] = min(m.samples["min"], s.samples["min"])
            m.samples["max"] = max(m.samples["max"], s.samples["max"])
            m.bounces["total"] += s.bounces["total"]
            m.bounces["min"] = min(m.bounces["min"], s.bounces["min"])
            m.bounces["max"] = max(m.bounces["max"], s.bounces["max"])
            m.rays += s.rays
            m.deviceMs = max(m.deviceMs, s.deviceMs)
            m.kernelLaunches += s.kernelLaunches
            m.nodeVisits += getattr(s, "nodeVisits", 0)
            m.primTests += getattr(s, "primTests", 0)
        if m.pixels > 0:
            m.samples["avg"] = m.samples["total"] / m.pixels
        if m.samples["total"] > 0:
            m.bounces["avg"] = m.bounces["total"] / m.samples["total"]
        return m


def _check(st: int) -> None:
    """Raise RaytracerError for a failed library call (a non-zero rt_status), with the library's message."""
    if st != 0:
        raise RaytracerError(f"{_native.last_error()} [{_native.STATUS_NAMES.get(st, st)}]")


def _image_outputs(rgb8: Optional[np.ndarray], linear: Optional[np.ndarray], W: int, H: int):
    """Check the RGB8 and linear output arrays of a render of a W x H image (None = not wanted): the library writes them
    through their base pointers as C-contiguous [H][W][3] arrays.  Returns (rgb8 pointer, rgb8 bytes, linear pointer)."""
    if rgb8 is not None and (rgb8.dtype != np.uint8 or not rgb8.flags["C_CONTIGUOUS"]):
        raise RaytracerError("pixel buffer must be a C-contiguous uint8 array")
    if linear is not None and (linear.dtype != np.float32 or linear.size < W * H * 3 or not linear.flags["C_CONTIGUOUS"]):
        raise RaytracerError("linear buffer must be float32 [H][W][3]")
    return (rgb8.ctypes.data if rgb8 is not None else None, rgb8.nbytes if rgb8 is not None else 0,
            linear.ctypes.data if linear is not None else None)


def _moments_output(moments: Optional[np.ndarray], W: int, H: int):
    """Check the moments output array of a render of a W x H image (None = not wanted): the library writes it through its
    base pointer as a C-contiguous [H][W][8] float32 array.  Returns its pointer."""
    if moments is None:
        return None
    if moments.dtype != np.float32 or moments.size < W * H * 8 or not moments.flags["C_CONTIGUOUS"]:
        raise RaytracerError("moments buffer must be a C-contiguous float32 [H][W][8] array")
    return moments.ctypes.data


def _progressive(onPass, call) -> None:
    """Run the progressive library call `call(fn)` with `fn` the rt_progress_fn that calls
    onPass(pass, passes, samplesCap, RenderStats) after each pass (None = no callback); a true result stops the render.  An
    exception in onPass stops the render too, and is raised once the library has returned: it never unwinds through the C
    frame."""
    errors: List[BaseException] = []

    @C.CFUNCTYPE(C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.POINTER(rt_stats))
    def cb(_user, k, n, cap, so_far):
        if onPass is None:
            return 0
        try:
            return 1 if onPass(int(k), int(n), int(cap), RenderStats.from_struct(so_far.contents)) else 0
        except BaseException as e:  # noqa: BLE001
            errors.append(e)
            return 1

    _check(call(C.cast(cb, C.c_void_p)))
    if errors:
        raise errors[0]


def _region_struct(region: Optional[Dict[str, int]], W: int, H: int) -> rt_region:
    if region is None:
        return rt_region(0, 0, W, H)
    return rt_region(int(region["x"]), int(region["y"]), int(region["width"]), int(region["height"]))


class Camera:
    channels = 3

    def __init__(self, world: Dict[str, Any], cameraOptions: Optional[Dict[str, Any]] = None,
                 renderData: Optional[Dict[str, Any]] = None):
        sceneData = world
        if cameraOptions:
            sceneData = dict(world)
            cam = dict(world.get("camera") or {})
            cam.update({k: v for k, v in cameraOptions.items() if v is not None})
            sceneData["camera"] = cam
        self._flat = FlatScene(sceneData)
        self.options = merge_render_options(sceneData.get("render"), renderData)
        self._opts = render_opts_struct(self.options)
        L = _native.lib()
        h = C.c_void_p()
        _check(L.rt_camera_create(C.byref(self._flat.desc), C.byref(self._opts), C.byref(h)))
        self._h = h
        info = rt_camera_info()
        L.rt_camera_get_info(self._h, C.byref(info))
        self.info = info
        self.imageWidth = info.image_width
        self.imageHeight = info.image_height
        v = lambda a: np.array(list(a), dtype=np.float32)  # noqa: E731
        self.center, self.pixel00Loc = v(info.center), v(info.pixel00_loc)
        self.pixelDeltaU, self.pixelDeltaV = v(info.pixel_delta_u), v(info.pixel_delta_v)
        self.u, self.v, self.w = v(info.u), v(info.v), v(info.w)
        self.defocusDiskU, self.defocusDiskV = v(info.defocus_disk_u), v(info.defocus_disk_v)
        self.focusDistance = info.focus_distance
        self.aperture = float(self._flat.camera.aperture)
        self.background = {"type": "gradient", "top": list(self._flat.camera.background_top),
                           "bottom": list(self._flat.camera.background_bottom)}
        self.useAdaptiveSampling = bool(info.use_adaptive_sampling)
        self.nLights = info.n_lights

    # -- lifecycle --
    def close(self) -> None:
        if getattr(self, "_h", None):
            _native.lib().rt_camera_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def setStream(self, cuda_stream: int) -> None:
        _check(_native.lib().rt_camera_set_stream(self._h, C.c_void_p(cuda_stream)))

    # -- the hot path --
    def renderRegion(self, buffer: np.ndarray, region: Optional[Dict[str, int]], linear: Optional[np.ndarray] = None,
                     moments: Optional[np.ndarray] = None) -> RenderStats:
        W, H = self.imageWidth, self.imageHeight
        bp, bl, lp = _image_outputs(buffer, linear, W, H)
        reg = _region_struct(region, W, H)
        st = rt_stats()
        L = _native.lib()
        if moments is not None:
            if moments.dtype != np.float32 or moments.size < W * H * 8:
                raise RaytracerError("moments buffer must be float32 [H][W][8]")
            _check(L.rt_camera_render_moments(self._h, C.byref(reg), bp, bl, lp, moments.ctypes.data, C.byref(st)))
        else:
            _check(L.rt_camera_render_region(self._h, C.byref(reg), bp, bl, lp, C.byref(st)))
        return RenderStats.from_struct(st)

    def render(self, pixelData: np.ndarray, linear: Optional[np.ndarray] = None) -> RenderStats:
        return self.renderRegion(pixelData, None, linear)

    def renderProgressive(self, pixelData: np.ndarray, passes: int, onPass=None, region: Optional[Dict[str, int]] = None,
                          linear: Optional[np.ndarray] = None) -> RenderStats:
        """The image of `render`, delivered in `passes` growing prefixes of the samples (rt_camera_render_progressive).
        onPass(pass, passes, samplesCap, RenderStats) is called after each pass with `pixelData` refreshed; return True to
        stop early.  The reference has no preview surface (SURVEY.md section 8f row 2)."""
        W, H = self.imageWidth, self.imageHeight
        bp, bl, lp = _image_outputs(pixelData, linear, W, H)
        reg = _region_struct(region, W, H)
        st = rt_stats()
        _progressive(onPass, lambda fn: _native.lib().rt_camera_render_progressive(self._h, C.byref(reg), bp, bl, lp, int(passes), fn,
                                                                                   None, C.byref(st)))
        return RenderStats.from_struct(st)

    def renderRegionDevice(self, region, rgb8_ptr: int = 0, linear_ptr: int = 0, moments_ptr: int = 0, stats_ptr: int = 0) -> None:
        """Enqueue on the camera's stream; device pointers; no synchronisation."""
        reg = _region_struct(region, self.imageWidth, self.imageHeight)
        vp = lambda p: C.c_void_p(p) if p else None  # noqa: E731
        _check(_native.lib().rt_camera_render_region_device(self._h, C.byref(reg), vp(rgb8_ptr), vp(linear_ptr),
                                                                 vp(moments_ptr), vp(stats_ptr)))

    # -- parity hook --
    def tracePrimary(self, region: Optional[Dict[str, int]] = None):
        W, H = self.imageWidth, self.imageHeight
        reg = _region_struct(region, W, H)
        ids = np.full((H, W), -2, np.int32)
        t = np.zeros((H, W), np.float32)
        nrm = np.zeros((H, W, 3), np.float32)
        ff = np.zeros((H, W), np.uint8)
        _check(_native.lib().rt_camera_trace_primary(self._h, C.byref(reg), ids.ctypes.data, t.ctypes.data,
                                                          nrm.ctypes.data, ff.ctypes.data))
        return ids, t, nrm, ff

    # -- opt-in denoiser (not in the reference) --
    def renderFeatures(self, nSamples: int, region: Optional[Dict[str, int]] = None) -> Dict[str, np.ndarray]:
        """First-hit features averaged over the camera rays of samples 0..nSamples-1 (rt_camera_render_features):
        albedo [H,W,3], normal [H,W,3], depth [H,W] (-1 where no ray hit).  Pixels outside `region` are 0."""
        W, H = self.imageWidth, self.imageHeight
        reg = _region_struct(region, W, H)
        alb = np.zeros((H, W, 3), np.float32)
        nrm = np.zeros((H, W, 3), np.float32)
        dep = np.zeros((H, W), np.float32)
        _check(_native.lib().rt_camera_render_features(self._h, C.byref(reg), int(nSamples), alb.ctypes.data, nrm.ctypes.data,
                                                            dep.ctypes.data))
        return {"albedo": alb, "normal": nrm, "depth": dep}

    def renderDenoised(self, pixelData: Optional[np.ndarray], linear: Optional[np.ndarray] = None, region: Optional[Dict[str, int]] = None,
                       options: Optional[Dict[str, Any]] = None) -> RenderStats:
        """Render, then denoise on the device (rt_camera_render_denoised): `pixelData` / `linear` receive the filtered image.
        options: {iterations, sigmaLuminance, sigmaNormal, sigmaDepth}; absent = defaults."""
        W, H = self.imageWidth, self.imageHeight
        bp, bl, lp = _image_outputs(pixelData, linear, W, H)
        reg = _region_struct(region, W, H)
        opts = denoise_opts_struct(options)
        st = rt_stats()
        _check(_native.lib().rt_camera_render_denoised(self._h, C.byref(reg), bp, bl, lp, C.byref(opts), C.byref(st)))
        return RenderStats.from_struct(st)

    def renderProgressiveDenoised(self, pixelData: Optional[np.ndarray], passes: int, onPass=None, region: Optional[Dict[str, int]] = None,
                                  linear: Optional[np.ndarray] = None, moments: Optional[np.ndarray] = None,
                                  options: Optional[Dict[str, Any]] = None) -> RenderStats:
        """`renderProgressive` with a denoised preview (rt_camera_render_progressive_denoised): after each pass `pixelData` /
        `linear` hold the filtered image of the samples so far and `moments` ([H][W][8], optional) the render's moments,
        then onPass runs as in `renderProgressive`.  The last pass gives the bytes of `renderDenoised`.  options as there."""
        W, H = self.imageWidth, self.imageHeight
        bp, bl, lp = _image_outputs(pixelData, linear, W, H)
        mp = _moments_output(moments, W, H)
        reg = _region_struct(region, W, H)
        opts = denoise_opts_struct(options)
        st = rt_stats()
        _progressive(onPass, lambda fn: _native.lib().rt_camera_render_progressive_denoised(
            self._h, C.byref(reg), bp, bl, lp, mp, int(passes), C.byref(opts), fn, None, C.byref(st)))
        return RenderStats.from_struct(st)

    # -- per-function parity hooks (rt_debug_*): one device function of the render path on explicit inputs --
    DEBUG_UNIFORMS = 16

    def _uniforms(self, uniforms, n: int) -> np.ndarray:
        u = np.full((n, self.DEBUG_UNIFORMS), 0.5, np.float64)
        a = np.asarray(uniforms, np.float64).reshape(n, -1) if n else np.zeros((0, 0))
        u[:, :a.shape[1]] = a[:, :self.DEBUG_UNIFORMS]
        return np.ascontiguousarray(u)

    def debugScatter(self, objectIndex: int, rayOrigin, rayDir, p, normal, frontFace, uniforms):
        """material.scatter + material.emitted of objects[objectIndex].material at n synthetic hits.
        Returns dict of arrays: kind (0 null, 1 scattered ray, 2 pdf), used, attenuation, dir, emitted."""
        ro, rd, pp, nn = (np.ascontiguousarray(np.atleast_2d(x), np.float64) for x in (rayOrigin, rayDir, p, normal))
        n = ro.shape[0]
        hits = np.zeros((n, 13), np.float64)  # rt_debug_hit: 12 doubles + two int32
        hits[:, 0:3], hits[:, 3:6], hits[:, 6:9], hits[:, 9:12] = ro, rd, pp, nn
        ff = np.zeros((n, 2), np.int32)
        ff[:, 0] = np.asarray(frontFace, np.int32).reshape(n)
        hits[:, 12] = ff.view(np.float64).reshape(n)
        u = self._uniforms(uniforms, n)
        out = np.zeros((n, 11), np.float32)  # rt_debug_scatter_out: 2 int32 + 9 float
        _check(_native.lib().rt_debug_scatter(self._h, int(objectIndex), n, hits.ctypes.data, u.ctypes.data, out.ctypes.data))
        ints = out[:, 0:2].copy().view(np.int32)
        return {"kind": ints[:, 0], "used": ints[:, 1], "attenuation": out[:, 2:5], "dir": out[:, 5:8], "emitted": out[:, 8:11]}

    def debugGetRay(self, ij, uniforms):
        """Camera.getRay(i, j) for n pixels: (origin [n,3], direction [n,3], uniforms used [n])."""
        a = np.ascontiguousarray(np.atleast_2d(ij), np.int32)
        n = a.shape[0]
        u = self._uniforms(uniforms, n)
        out = np.zeros((n, 6), np.float32)
        used = np.zeros(n, np.int32)
        _check(_native.lib().rt_debug_get_ray(self._h, n, a.ctypes.data, u.ctypes.data, out.ctypes.data, used.ctypes.data))
        return out[:, 0:3], out[:, 3:6], used

    def debugLightPdf(self, lightIndex: int, origin, direction) -> np.ndarray:
        o, d = (np.ascontiguousarray(np.atleast_2d(x), np.float64) for x in (origin, direction))
        out = np.zeros(o.shape[0], np.float32)
        _check(_native.lib().rt_debug_light_pdf(self._h, int(lightIndex), o.shape[0], o.ctypes.data, d.ctypes.data, out.ctypes.data))
        return out

    def debugLightRandomVec(self, lightIndex: int, origin, uniforms) -> np.ndarray:
        o = np.ascontiguousarray(np.atleast_2d(origin), np.float64)
        u = self._uniforms(uniforms, o.shape[0])
        out = np.zeros((o.shape[0], 3), np.float32)
        _check(_native.lib().rt_debug_light_random_vec(self._h, int(lightIndex), o.shape[0], o.ctypes.data, u.ctypes.data, out.ctypes.data))
        return out

    def debugDiffuseBounce(self, p, normal, uniforms) -> np.ndarray:
        """camera.ts:285-308 at n hit points: [n,6] = direction, mixture pdf value, scatter pdf value, continues."""
        pp, nn = (np.ascontiguousarray(np.atleast_2d(x), np.float64) for x in (p, normal))
        u = self._uniforms(uniforms, pp.shape[0])
        out = np.zeros((pp.shape[0], 6), np.float32)
        _check(_native.lib().rt_debug_diffuse_bounce(self._h, pp.shape[0], pp.ctypes.data, nn.ctypes.data, u.ctypes.data, out.ctypes.data))
        return out


class MultiCamera:
    """One process, N GPUs (rt_multi_*): the native stand-in for the reference's worker pool (src/raytracer.ts:60-90).
    Same `render` / `renderRegion` as `Camera`; device k renders the 8x4 blocks it owns and writes them straight into
    device 0's framebuffer over NVLink peer mappings."""

    channels = 3

    def __init__(self, sceneData: Dict[str, Any], renderData: Optional[Dict[str, Any]] = None, devices: Optional[List[int]] = None,
                 nDevices: int = 0):
        self._flat = FlatScene(sceneData)
        self.options = merge_render_options(sceneData.get("render"), renderData)
        self._opts = render_opts_struct(self.options)
        L = _native.lib()
        h = C.c_void_p()
        dev = (C.c_int32 * len(devices))(*devices) if devices else None
        _check(L.rt_multi_create(C.byref(self._flat.desc), C.byref(self._opts), len(devices) if devices else int(nDevices), dev, C.byref(h)))
        self._h = h
        info, n, p2p = rt_camera_info(), C.c_int32(), C.c_int32()
        L.rt_multi_get_info(self._h, C.byref(info), C.byref(n), C.byref(p2p))
        self.info = info
        self.imageWidth, self.imageHeight = info.image_width, info.image_height
        self.nDevices, self.peerWrites = n.value, bool(p2p.value)

    def close(self) -> None:
        if getattr(self, "_h", None):
            _native.lib().rt_multi_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def renderRegion(self, buffer: np.ndarray, region: Optional[Dict[str, int]], linear: Optional[np.ndarray] = None) -> RenderStats:
        W, H = self.imageWidth, self.imageHeight
        bp, bl, lp = _image_outputs(buffer, linear, W, H)
        reg = _region_struct(region, W, H)
        st = rt_stats()
        _check(_native.lib().rt_multi_render_region(self._h, C.byref(reg), bp, bl, lp, C.byref(st)))
        return RenderStats.from_struct(st)

    def render(self, pixelData: np.ndarray, linear: Optional[np.ndarray] = None) -> RenderStats:
        return self.renderRegion(pixelData, None, linear)

    def renderDenoised(self, pixelData: Optional[np.ndarray], linear: Optional[np.ndarray] = None, region: Optional[Dict[str, int]] = None,
                       options: Optional[Dict[str, Any]] = None) -> RenderStats:
        """`Camera.renderDenoised` on every device (rt_multi_render_denoised): the same bytes as one Camera's.  Each device
        filters a band of the region's rows after every device has rendered."""
        W, H = self.imageWidth, self.imageHeight
        bp, bl, lp = _image_outputs(pixelData, linear, W, H)
        reg = _region_struct(region, W, H)
        opts = denoise_opts_struct(options)
        st = rt_stats()
        _check(_native.lib().rt_multi_render_denoised(self._h, C.byref(reg), bp, bl, lp, C.byref(opts), C.byref(st)))
        return RenderStats.from_struct(st)

    def renderProgressive(self, pixelData: np.ndarray, passes: int, onPass=None, region: Optional[Dict[str, int]] = None,
                          linear: Optional[np.ndarray] = None) -> RenderStats:
        """`Camera.renderProgressive` on every device (rt_multi_render_progressive): the same caps, and after each pass the
        same bytes as one Camera's.  onPass runs once per pass, after every device's part of it has landed."""
        W, H = self.imageWidth, self.imageHeight
        bp, bl, lp = _image_outputs(pixelData, linear, W, H)
        reg = _region_struct(region, W, H)
        st = rt_stats()
        _progressive(onPass, lambda fn: _native.lib().rt_multi_render_progressive(self._h, C.byref(reg), bp, bl, lp, int(passes), fn,
                                                                                  None, C.byref(st)))
        return RenderStats.from_struct(st)

    def renderProgressiveDenoised(self, pixelData: Optional[np.ndarray], passes: int, onPass=None, region: Optional[Dict[str, int]] = None,
                                  linear: Optional[np.ndarray] = None, moments: Optional[np.ndarray] = None,
                                  options: Optional[Dict[str, Any]] = None) -> RenderStats:
        """`Camera.renderProgressiveDenoised` on every device (rt_multi_render_progressive_denoised): after each pass the same
        bytes as one Camera's; each device filters a band of the region's rows, as in `renderDenoised`."""
        W, H = self.imageWidth, self.imageHeight
        bp, bl, lp = _image_outputs(pixelData, linear, W, H)
        mp = _moments_output(moments, W, H)
        reg = _region_struct(region, W, H)
        opts = denoise_opts_struct(options)
        st = rt_stats()
        _progressive(onPass, lambda fn: _native.lib().rt_multi_render_progressive_denoised(
            self._h, C.byref(reg), bp, bl, lp, mp, int(passes), C.byref(opts), fn, None, C.byref(st)))
        return RenderStats.from_struct(st)


def createCameraFromSceneData(sceneData: Dict[str, Any], renderOptions: Optional[Dict[str, Any]] = None) -> Camera:
    """src/scenes/scenes.ts:60-104"""
    return Camera(sceneData, None, renderOptions)


def generateScene(sceneConfig: Dict[str, Any]) -> Camera:
    """src/scenes/scenes.ts:52-55"""
    return createCameraFromSceneData(generateSceneData(sceneConfig), sceneConfig.get("render"))


def denoise(color, albedo, normal, depth, moments, options: Optional[Dict[str, Any]] = None, device: int = -1) -> np.ndarray:
    """The denoiser on explicit arrays (rt_denoise): color/albedo/normal [H,W,3], depth [H,W], moments [H,W,8] as
    `Camera.renderRegion(..., moments=)` and `Camera.renderFeatures` return them.  Returns the filtered colour [H,W,3]."""
    c = np.ascontiguousarray(color, np.float32)
    if c.ndim != 3 or c.shape[2] != 3:
        raise RaytracerError("color must be [H][W][3]")
    H, W = c.shape[:2]
    shapes = {"albedo": (H, W, 3), "normal": (H, W, 3), "depth": (H, W), "moments": (H, W, 8)}
    arrs = {}
    for name, a in (("albedo", albedo), ("normal", normal), ("depth", depth), ("moments", moments)):
        arrs[name] = np.ascontiguousarray(a, np.float32)
        if arrs[name].shape != shapes[name]:
            raise RaytracerError(f"{name} must have shape {shapes[name]}, not {arrs[name].shape}")
    opts = denoise_opts_struct(options)
    out = np.zeros((H, W, 3), np.float32)
    _check(_native.lib().rt_denoise(int(device), W, H, c.ctypes.data, arrs["albedo"].ctypes.data, arrs["normal"].ctypes.data,
                                    arrs["depth"].ctypes.data, arrs["moments"].ctypes.data, C.byref(opts), out.ctypes.data))
    return out


def measureFp32Peak(device: int = -1):
    t, mhz = C.c_double(), C.c_double()
    _check(_native.lib().rt_measure_fp32_peak(device, C.byref(t), C.byref(mhz)))
    return t.value, mhz.value


class _SceneReport(C.Structure):  # rt_scene_report (include/rt_b200.h)
    _fields_ = [(n, C.c_int32) for n in ("bvh_kind", "n_slots", "n_prefix", "n_node_slots", "n_leaves", "max_leaf_size",
                                         "max_depth", "n_lights", "errors")] + [("reserved", C.c_int32 * 3)]


def validateScene(sceneData: Dict[str, Any], renderOptions: Optional[Dict[str, Any]] = None) -> Dict[str, int]:
    """Host-only (no GPU): run the scene compiler of `createCameraFromSceneData` and check the structure the
    kernels walk (rt_scene_validate).  Raises the reference's errors for a bad scene; `errors` must be 0."""
    flat = FlatScene(sceneData)
    opts = render_opts_struct(merge_render_options(flat.render, renderOptions))
    rep = _SceneReport()
    _check(_native.lib().rt_scene_validate(C.byref(flat.desc), C.byref(opts), C.byref(rep)))
    return {n: int(getattr(rep, n)) for n, _ in _SceneReport._fields_ if n != "reserved"}


def trimDeviceCache() -> int:
    """Return the device buffers kept from destroyed cameras to the driver (rt_trim_device_cache); bytes released."""
    return int(_native.lib().rt_trim_device_cache())
