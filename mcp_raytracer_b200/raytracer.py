"""Render orchestration — mirror of `src/raytracer.ts` with the parallel renderer replaced
by native dispatch (the seam SURVEY.md §8b names).

* `generateImageBuffer(sceneConfig, options)`  <- src/raytracer.ts:39-113
    options.parallel=False : `camera.render(pixelData)`            (raytracer.ts:56-59)
    options.denoise=True or {iterations, sigma*}: `camera.renderDenoised(pixelData)` (not in the reference); with
                             parallel=True on more than one GPU `MultiCamera.renderDenoised`: every device renders its
                             blocks and filters a band of rows, the same bytes as on one GPU
    options.parallel=True  : the image is split over GPUs instead of worker threads
                             (raytracer.ts:60-90): `MultiCamera` (rt_multi_* of the C ABI) compiles
                             the scene once, every visible device renders its interleaved set of 8x4
                             blocks and stores them straight into device 0's framebuffer, stats merged
                             like RenderStats.merge — the roles `divideIntoRegions` + workers +
                             SharedArrayBuffer play in the reference.
  Returns PNG bytes like the reference (PIL instead of sharp; PNG encoding is outside the
  hot path) or, with `options.raw=True`, the RGB8 array itself.
* `ImagePipeline`                               for a stream of requests: image k is deflated on a host thread
  while image k + 1 renders (the post step of src/raytracer.ts:102-110 taken off the GPU's critical path)
* `divideIntoRegions`                           <- src/raytracer.ts:185-205 (kept for callers
  that want the reference's row-strip partition, e.g. the CPU-baseline harness)
"""
from __future__ import annotations

import io
import math
import sys
from typing import Any, Dict, List, Optional

import numpy as np

from . import _native
from .camera import Camera, MultiCamera, RenderStats, createCameraFromSceneData
from .scenes import generateSceneData


def divideIntoRegions(imageWidth: int, imageHeight: int, count: int) -> List[Dict[str, int]]:
    regionHeight = math.ceil(imageHeight / count)
    regions = []
    for i in range(count):
        startY = i * regionHeight
        height = min(regionHeight, imageHeight - startY)
        if height <= 0:
            break
        regions.append({"x": 0, "y": startY, "width": imageWidth, "height": height})
    return regions


def applySceneCameraOptions(sceneData: Dict[str, Any], camera: Optional[Dict[str, Any]]) -> Dict[str, Any]:
    """`scene.camera` of the MCP `raytrace` tool (cameraOptionsSchema, src/mcp.ts:132-142) is accepted by the reference and then
    dropped: generateScene reads only scene.type / options / render (src/scenes/scenes.ts:52-55).  This maps it onto the fields
    the renderer does read, so the tool's documented camera options take effect (TypeScript twin: ts/nativeCamera.ts)."""
    if not camera:
        return sceneData
    cam = dict(sceneData.get("camera") or {})
    render = dict(sceneData.get("render") or {})
    for src, dst in (("vfov", "vfov"), ("lookFrom", "from"), ("lookAt", "at"), ("vUp", "up")):
        if camera.get(src) is not None:
            cam[dst] = camera[src]
    for src, dst in (("imageWidth", "width"), ("aspectRatio", "aspect"), ("samples", "samples"), ("adaptiveTolerance", "aTolerance"),
                     ("adaptiveBatchSize", "aBatch")):
        if camera.get(src) is not None:
            render[dst] = camera[src]
    return {**sceneData, "camera": cam, "render": render}


def renderScene(sceneConfig: Dict[str, Any], options: Optional[Dict[str, Any]] = None):
    """Everything `generateImageBuffer` does before PNG encoding: returns (rgb8[H,W,3], RenderStats)."""
    options = options or {}
    parallel = options.get("parallel", False)
    verbose = options.get("verbose", False)
    sceneData = applySceneCameraOptions(generateSceneData(sceneConfig), sceneConfig.get("camera"))
    render = sceneConfig.get("render")
    ndev = _native.lib().rt_device_count()
    threads = options.get("threads") or ndev  # "threads" = number of GPUs here
    dn = options.get("denoise")
    if dn and parallel and min(threads, ndev) > 1:
        threads = min(threads, ndev)
        if verbose:
            print(f"Denoising: rendering and filtering on {threads} GPUs", file=sys.stderr)
        # every device renders its blocks, then filters a band of rows: the bytes of the one-GPU denoiser
        with MultiCamera(sceneData, render, nDevices=threads) as camera:
            W, H = camera.imageWidth, camera.imageHeight
            pixelData = np.zeros(W * H * 3, np.uint8)
            stats = camera.renderDenoised(pixelData, options=None if dn is True else dn)
    elif dn:
        if verbose:
            print("Denoising: rendering on one GPU", file=sys.stderr)
        with createCameraFromSceneData(sceneData, render) as camera:
            W, H = camera.imageWidth, camera.imageHeight
            pixelData = np.zeros(W * H * 3, np.uint8)
            stats = camera.renderDenoised(pixelData, options=None if dn is True else dn)
    elif not parallel or threads <= 1:
        with createCameraFromSceneData(sceneData, render) as camera:
            pixelData = np.zeros(camera.imageWidth * camera.imageHeight * camera.channels, np.uint8)
            stats = camera.render(pixelData)
            W, H = camera.imageWidth, camera.imageHeight
    else:
        threads = min(threads, max(ndev, 1))
        if verbose:
            print(f"Starting parallel render on {threads} GPUs", file=sys.stderr)
        # one process, `threads` GPUs, inside the C ABI (rt_multi_*): scene compiled once, every device writes the
        # blocks it owns into device 0's framebuffer, stats merged like RenderStats.merge (raytracer.ts:71-89)
        with MultiCamera(sceneData, render, nDevices=threads) as camera:
            W, H = camera.imageWidth, camera.imageHeight
            pixelData = np.zeros(W * H * 3, np.uint8)  # the SharedArrayBuffer of raytracer.ts:71-72
            stats = camera.render(pixelData)
    if verbose:
        print(f"Adaptive sampling stats: avg={stats.samples['avg']:.2f}, min={stats.samples['min']}, max={stats.samples['max']}", file=sys.stderr)
        print(f"Ray bounce stats: avg={stats.bounces['avg']:.2f}, min={stats.bounces['min']}, max={stats.bounces['max']}", file=sys.stderr)
    return pixelData.reshape(H, W, 3), stats


def encodePng(rgb: np.ndarray, compressLevel: int = 6) -> bytes:
    """RGB8 [H, W, 3] -> PNG bytes (sharp / libvips in the reference, src/raytracer.ts:102-110; PIL + zlib here).  zlib
    releases the GIL, so several images deflate in parallel on host threads."""
    from PIL import Image

    buf = io.BytesIO()
    Image.fromarray(rgb, "RGB").save(buf, format="PNG", compress_level=compressLevel)
    return buf.getvalue()


def generateImageBuffer(sceneConfig: Optional[Dict[str, Any]] = None, options: Optional[Dict[str, Any]] = None):
    sceneConfig = sceneConfig or {"type": "default"}
    options = options or {}
    rgb, _stats = renderScene(sceneConfig, options)
    if rgb.size == 0:
        raise RuntimeError("Generated pixelData buffer is empty before calling sharp.")  # raytracer.ts:97-99
    if options.get("raw"):
        return rgb
    return encodePng(rgb)


class ImagePipeline:
    """`generateImageBuffer` for a stream of requests (the MCP server's situation), with the post-processing OFF the GPU's
    critical path (SURVEY.md section 8f row 3).  At GPU speed the PNG deflate of an image takes longer than rendering it
    (Cornell 1024x1024 @64 spp: ~8 ms of render, ~50 ms of zlib), so a server that encodes before it accepts the next
    request leaves the GPU idle most of the time.  Here request k's image is deflated on a host thread while request
    k + 1 renders: renders are serialised (one at a time per GPU set), encodes run concurrently on `encoders` threads.

        pipe = ImagePipeline(encoders=4)
        futures = [pipe.submit(cfg, {"parallel": True}) for cfg in requests]
        pngs = [f.result() for f in futures]
    """

    def __init__(self, encoders: int = 4, compressLevel: int = 6):
        import concurrent.futures
        import threading

        self._render_lock = threading.Lock()
        self._pool = concurrent.futures.ThreadPoolExecutor(max_workers=max(1, encoders) + 1, thread_name_prefix="rt-png")
        self._level = compressLevel

    def submit(self, sceneConfig: Optional[Dict[str, Any]] = None, options: Optional[Dict[str, Any]] = None):
        cfg = sceneConfig or {"type": "default"}
        opts = options or {}

        def job():
            with self._render_lock:                      # the GPU does one render at a time ...
                rgb, _stats = renderScene(cfg, opts)
            if rgb.size == 0:
                raise RuntimeError("Generated pixelData buffer is empty before calling sharp.")
            return rgb if opts.get("raw") else encodePng(rgb, self._level)   # ... and is free again while this image deflates

        return self._pool.submit(job)

    def close(self) -> None:
        self._pool.shutdown(wait=True)

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()
