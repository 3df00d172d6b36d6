"""mcp_raytracer_b200 — B200-native drop-in for the path-tracing hot path of df07/mcp-raytracer.

Only what the path needs lives here: `csrc/` (CUDA kernels for sm_100a + the C ABI of
include/rt_b200.h) and the host-side mirror of the reference interface for this path
(scene generators, SceneData flattening, Camera, render orchestration).
"""
from .camera import Camera, MultiCamera, RenderMode, RenderStats, createCameraFromSceneData, denoise, generateScene, measureFp32Peak, trimDeviceCache, validateScene  # noqa: F401
from .raytracer import ImagePipeline, divideIntoRegions, encodePng, generateImageBuffer, renderScene  # noqa: F401
from .scene_data import FlatScene, RaytracerError  # noqa: F401
from .scenes import (  # noqa: F401
    SeededRandom, generateCornellSceneData, generateDefaultSceneData, generateLayeredMixedSceneData,
    generateRainSceneData, generateSceneData, generateSpheresSceneData, generateWeekendFinalSceneData,
)
