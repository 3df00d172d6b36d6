/* nativeCamera.ts — drop-in replacement for the hot path of src/camera.ts.
 *
 * UNVERIFIED HERE (no node/tsc in the build image).  Mirrors, line for line, the Python host code
 * that IS exercised by the test-suite: mcp_raytracer_b200/scene_data.py (flattening) and
 * mcp_raytracer_b200/camera.py (Camera over the C ABI).
 *
 * NOT COMPILED HERE (no tsc); the N-API shim it loads is syntax-checked against a stub header (ts/addon/rt_napi.c).
 *
 * Usage inside the reference: in src/scenes/scenes.ts `createCameraFromSceneData` return
 * `new NativeCamera(sceneData, renderOptions)` instead of building Hittables + BVHNode + Camera;
 * `camera.render(pixelData)` / `camera.renderRegion(pixelData, region)` keep their signatures
 * (src/camera.ts:388,439), so src/raytracer.ts and src/render-utils/renderWorker.ts are unchanged.
 */
import { createRequire } from 'module';
import type { SceneData, MaterialData, SceneObject } from '../src/scenes/sceneData.js';
import type { RenderOptions, RenderRegion } from '../src/camera.js';
import { RenderStats } from '../src/render-utils/renderStats.js';

const addon = createRequire(import.meta.url)('./addon/build/Release/rt_b200.node');

const OBJ = { sphere: 0, plane: 1, quad: 2 } as const;
const MODE = { default: 0, bounces: 1, samples: 2 } as const;
const enum Mat { Lambert, Metal, Glass, Light, Mixed, Layered }

/** SceneData -> SoA typed arrays (rt_scene_desc).  Same traversal and error text as
 *  createSceneObject / createMaterial / createDielectric, src/scenes/scenes.ts:109-199. */
export function flattenScene(sceneData: SceneData) {
  const byId: Record<string, MaterialData> = {};
  sceneData.materials?.forEach(({ id, material }) => { byId[id] = material; });
  const matType: number[] = [], matColor: number[] = [], matParam: number[] = [], matChild: number[] = [];
  const memo = new Map<string, number>();
  const node = (type: number, color = [0, 0, 0], param = 0, child = [-1, -1]) => {
    matType.push(type); matColor.push(...color); matParam.push(param); matChild.push(...child); return matType.length - 1;
  };
  const material = (ref: string | MaterialData): number => {
    if (typeof ref === 'string' && memo.has(ref)) return memo.get(ref)!;
    const data = typeof ref === 'string' ? byId[ref] : ref;
    if (!data) throw new Error(`Material not found: ${ref}`);
    let idx: number;
    switch (data.type) {
      case 'lambert': idx = node(Mat.Lambert, data.color); break;
      case 'metal': idx = node(Mat.Metal, data.color, data.fuzz); break;
      case 'glass': idx = node(Mat.Glass, undefined, data.ior); break;
      case 'light': idx = node(Mat.Light, data.emit); break;
      case 'mixed': { const a = material(data.diff), b = material(data.spec); idx = node(Mat.Mixed, undefined, data.weight, [a, b]); break; }
      case 'layered': {
        const outer = typeof data.outer === 'string' ? byId[data.outer] : data.outer;
        if (!outer) throw new Error(`Material not found: ${data.outer}`);
        if (outer.type !== 'glass') throw new Error(`Material is not a dielectric: ${data.outer}`);
        const o = material(data.outer), i = material(data.inner); idx = node(Mat.Layered, undefined, 0, [i, o]); break;
      }
      default: throw new Error(`Unknown material type: ${(data as any).type}`);
    }
    if (typeof ref === 'string') memo.set(ref, idx);
    return idx;
  };
  const n = sceneData.objects.length;
  const objType = new Uint8Array(n), objPos = new Float64Array(3 * n), objU = new Float64Array(3 * n), objV = new Float64Array(3 * n);
  const objR = new Float64Array(n), objMaterial = new Int32Array(n), objLight = new Uint8Array(n);
  sceneData.objects.forEach((o: SceneObject, i) => {
    objMaterial[i] = material(o.material);
    if (!(o.type in OBJ)) throw new Error(`Unknown object type: ${(o as any).type}`);
    objType[i] = OBJ[o.type]; objPos.set(o.pos, 3 * i); objLight[i] = o.light ? 1 : 0;
    if (o.type === 'sphere') objR[i] = o.r; else { objU.set(o.u, 3 * i); objV.set(o.v, 3 * i); }
  });
  const c = sceneData.camera, bg = c.background ?? { top: [1, 1, 1], bottom: [0.5, 0.7, 1.0] };
  return {
    objType, objPos, objU, objV, objR, objMaterial, objLight,
    matType: Uint8Array.from(matType), matColor: Float64Array.from(matColor), matParam: Float64Array.from(matParam), matChild: Int32Array.from(matChild),
    camera: { vfov: c.vfov ?? 90, aperture: c.aperture ?? 0, focus: c.focus ?? 1.0,
      from: Float64Array.from(c.from ?? [0, 0, 0]), at: Float64Array.from(c.at ?? [0, 0, -1]), up: Float64Array.from(c.up ?? [0, 1, 0]),
      backgroundTop: Float64Array.from(bg.top), backgroundBottom: Float64Array.from(bg.bottom) },
  };
}

/** `scene.camera` of the MCP `raytrace` tool (cameraOptionsSchema, src/mcp.ts:132-142) is accepted by the reference and then
 *  DROPPED: generateScene only reads scene.type / options / render (src/scenes/scenes.ts:52-55).  This maps it onto the fields
 *  the renderer does read, so the tool's documented camera options take effect (SURVEY.md §8f row 4).  Python mirror:
 *  mcp_raytracer_b200/raytracer.py applySceneCameraOptions. */
export function applySceneCameraOptions(sceneData: SceneData, cam?: Record<string, any>): SceneData {
  if (!cam) return sceneData;
  const camera = { ...sceneData.camera }, render: Record<string, any> = { ...(sceneData.render ?? {}) };
  if (cam.vfov !== undefined) camera.vfov = cam.vfov;
  if (cam.lookFrom !== undefined) camera.from = cam.lookFrom;
  if (cam.lookAt !== undefined) camera.at = cam.lookAt;
  if (cam.vUp !== undefined) camera.up = cam.vUp;
  if (cam.imageWidth !== undefined) render.width = cam.imageWidth;
  if (cam.aspectRatio !== undefined) render.aspect = cam.aspectRatio;
  if (cam.samples !== undefined) render.samples = cam.samples;
  if (cam.adaptiveTolerance !== undefined) render.aTolerance = cam.adaptiveTolerance;
  if (cam.adaptiveBatchSize !== undefined) render.aBatch = cam.adaptiveBatchSize;
  return { ...sceneData, camera, render };
}

type NativeOpts = { seed?: number, device?: number, partIndex?: number, partCount?: number, nDevices?: number,
                    lightSampling?: 'mixture' | 'shadowRays' };   // RT_LIGHTS_*: shadowRays = next-event estimation (not the reference's estimator)
/** rt_denoise_opts: iterations 0..8 (default 5); a sigma of 0 or absent selects its default. */
export type DenoiseOptions = { iterations?: number, sigmaLuminance?: number, sigmaNormal?: number, sigmaDepth?: number };

/** One GPU (`multi` false) or every visible GPU inside one call (`multi` true: rt_multi_*, the native stand-in for the
 *  worker pool of src/raytracer.ts:60-90).  Same `render` / `renderRegion` signatures as src/camera.ts:388,439. */
export class NativeCamera {
  readonly imageWidth: number; readonly imageHeight: number; readonly channels = 3;
  private handle: unknown; private flat: ReturnType<typeof flattenScene>;
  constructor(sceneData: SceneData, renderOptions: RenderOptions = {}, native: NativeOpts = {}, multi = false) {
    const o = { width: 400, aspect: 16 / 9, samples: 100, aTolerance: 0.05, aBatch: 10, mode: 'default', depth: 100, roulette: true, rouletteDepth: 3,
                ...sceneData.render, ...renderOptions };   // src/camera.ts:73-83,116 ; src/scenes/scenes.ts:97-100
    this.flat = flattenScene(sceneData);
    const opts = { ...o, roulette: o.roulette ? 1 : 0, mode: MODE[o.mode as keyof typeof MODE],
      seed: native.seed ?? 0, device: native.device ?? -1, partIndex: native.partIndex ?? 0, partCount: native.partCount ?? 1,
      lightSampling: native.lightSampling === 'shadowRays' ? 1 : 0 };
    this.handle = multi ? addon.createMulti(this.flat, opts, native.nDevices ?? 0) : addon.createCamera(this.flat, opts);
    const info = addon.cameraInfo(this.handle);
    this.imageWidth = info.imageWidth; this.imageHeight = info.imageHeight;
  }
  private static stats(s: any): RenderStats {
    const r = new RenderStats();
    r.pixels = s.pixels; r.samples.total = s.samplesTotal; r.bounces.total = s.bouncesTotal;
    if (s.pixels > 0) { r.samples.min = s.samplesMin; r.samples.max = s.samplesMax; r.bounces.min = s.bouncesMin; r.bounces.max = s.bouncesMax; r.samples.avg = s.samplesTotal / s.pixels; }
    if (s.samplesTotal > 0) r.bounces.avg = s.bouncesTotal / s.samplesTotal;
    return r;
  }
  renderRegion(buffer: Uint8ClampedArray, region: RenderRegion): RenderStats {
    return NativeCamera.stats(addon.renderRegion(this.handle, region, buffer));
  }
  render(pixelData: Uint8ClampedArray): RenderStats {
    return this.renderRegion(pixelData, { x: 0, y: 0, width: this.imageWidth, height: this.imageHeight });
  }
  /** The render on a libuv worker (napi_async_work): generateImageBuffer stays `async` without blocking the event loop. */
  async renderAsync(pixelData: Uint8ClampedArray): Promise<RenderStats> {
    return NativeCamera.stats(await addon.renderRegionAsync(this.handle, { x: 0, y: 0, width: this.imageWidth, height: this.imageHeight }, pixelData));
  }
  /** Render, then denoise on the device (rt_camera_render_denoised; `multi`: rt_multi_render_denoised, every GPU renders its
   *  blocks and filters a band of rows, the same bytes as on one GPU).  Not in the reference. */
  renderDenoised(pixelData: Uint8ClampedArray, region?: RenderRegion, options: DenoiseOptions = {}): RenderStats {
    return NativeCamera.stats(addon.renderDenoised(this.handle, region ?? { x: 0, y: 0, width: this.imageWidth, height: this.imageHeight },
                                                   pixelData, options));
  }
  /** Release the GPU memory now (the reference builds a camera per request: do not wait for the GC). */
  destroy(): void { addon.destroyCamera(this.handle); }
}
