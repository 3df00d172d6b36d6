/*
 * rt_b200.h — C ABI of the B200-native path-tracing hot path.
 *
 * This is the drop-in boundary for ONE path of df07/mcp-raytracer: the per-pixel
 * path tracer behind `Camera.render` / `Camera.renderRegion`
 * (reference: src/camera.ts:388-446) and everything it calls.  The reference has no
 * FFI of its own; the seam is the TypeScript method pair the orchestration layer calls
 * (src/raytracer.ts:59 serial, src/render-utils/renderWorker.ts:26 per worker).  What
 * crosses that seam in the reference is plain JSON `SceneData` + `RenderOptions`
 * (src/render-utils/renderWorker.ts:8-14), so that is what this ABI carries — flattened
 * into SoA arrays by the host language (TypeScript in the reference; Python here, see
 * mcp_raytracer_b200/scene_data.py and INTEGRATION.md for the N-API binding).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no C++/torch types, no exceptions across the ABI.
 *   - every function returns an rt_status; rt_last_error() gives a thread-local message.
 *   - the caller owns every host buffer for the duration of the call; the library owns
 *     device memory behind the opaque rt_camera handle.
 *   - scalars the reference keeps as JS numbers (radius, fuzz, ior, weight, vfov, aperture,
 *     focus, aspect, aTolerance) travel as double; vectors the reference stores in gl-matrix
 *     Float32Array (src/geometry/vec3.ts:21) also travel as double and are rounded to FP32
 *     by the consumer exactly where `Vec3.create` would round them (src/geometry/vec3.ts:263).
 *
 * The same rt_scene_desc / rt_render_opts structs are consumed by the CPU oracle under
 * oracle/ (test infrastructure only) so that both sides see bit-identical inputs.
 */
#ifndef RT_B200_H
#define RT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RT_B200_ABI_VERSION 2

typedef enum rt_status {
  RT_OK = 0,
  RT_ERR_INVALID_ARGUMENT = 1, /* null pointer, bad size, bad region; object geometry that is not finite in FP32 */
  RT_ERR_UNKNOWN_OBJECT_TYPE = 2, /* reference: `Unknown object type` src/scenes/scenes.ts:137 */
  RT_ERR_UNKNOWN_MATERIAL_TYPE = 3, /* reference: `Unknown material type` src/scenes/scenes.ts:178 */
  RT_ERR_MATERIAL_NOT_FOUND = 4, /* reference: `Material not found` src/scenes/scenes.ts:154,191 */
  RT_ERR_NOT_DIELECTRIC = 5, /* reference: `Material is not a dielectric` src/scenes/scenes.ts:195 */
  RT_ERR_BUFFER_TOO_SMALL = 6, /* reference: empty pixelData src/raytracer.ts:97-99 */
  RT_ERR_NO_DEVICE = 7, /* no CUDA device: there is NO CPU fallback */
  RT_ERR_CUDA = 8, /* a CUDA runtime call failed; message in rt_last_error() */
  RT_ERR_UNSUPPORTED = 9
} rt_status;

/* SceneObject.type — src/scenes/sceneData.ts:40-70 */
enum { RT_OBJ_SPHERE = 0, RT_OBJ_PLANE = 1, RT_OBJ_QUAD = 2 };

/* MaterialData.type — src/scenes/sceneData.ts:76-110 */
enum {
  RT_MAT_LAMBERT = 0, /* color = albedo */
  RT_MAT_METAL = 1,   /* color = albedo, param = fuzz */
  RT_MAT_GLASS = 2,   /* param = ior */
  RT_MAT_LIGHT = 3,   /* color = emit */
  RT_MAT_MIXED = 4,   /* child[0] = diff, child[1] = spec, param = weight */
  RT_MAT_LAYERED = 5  /* child[0] = inner, child[1] = outer (must be RT_MAT_GLASS) */
};

/* RenderMode — src/camera.ts:13-17 */
enum { RT_MODE_DEFAULT = 0, RT_MODE_BOUNCES = 1, RT_MODE_SAMPLES = 2 };

/* BVH the device traverses.  REFERENCE = the reference's own median-split topology
 * (src/geometry/bvh.ts:34-102) walked left-then-right, bit-faithful to its quirks
 * (inverted boxes of negative-radius spheres, infinite plane boxes, first-visited wins
 * on equal t).  SAH = binned-SAH tree with near-first ordering: same nearest hits except
 * for those quirks.  LIST = no hierarchy, every object tested (<= 128 objects; what the
 * reference's BVH degenerates to on Cornell).  AUTO picks REFERENCE when the scene has a
 * negative-radius sphere, LIST for <= 16 objects (<= 64 in a room: five or more quads/planes;
 * both crossovers measured), SAH otherwise. */
enum { RT_BVH_AUTO = 0, RT_BVH_REFERENCE = 1, RT_BVH_SAH = 2, RT_BVH_LIST = 3 };

/* Device integrator layout.  MEGAKERNEL = register-resident paths with per-lane path
 * regeneration; WAVEFRONT = ray-gen / traverse / per-material shade kernels over path
 * queues in HBM; SORTED = the megakernel with a CTA-wide sort of the hits by material class
 * between tracing and shading (shared memory; kernels without a sorted variant run as
 * MEGAKERNEL).  Same estimator, same RNG streams, bit-identical image.  AUTO = SORTED when the
 * scene has Mixed/Layered materials, else MEGAKERNEL. */
enum { RT_INTEGRATOR_AUTO = 0, RT_INTEGRATOR_MEGAKERNEL = 1, RT_INTEGRATOR_WAVEFRONT = 2, RT_INTEGRATOR_SORTED = 3 };

/* How the direct light of the listed lights (SceneObject.light, src/scenes/scenes.ts:74-79) is estimated at a diffuse
 * bounce.  MIXTURE = the reference's estimator: ONE scattered ray drawn from 0.5 cosine + 0.5 light pdf
 * (src/camera.ts:285-315, src/geometry/pdf.ts:57-99); the parity configuration and the default.
 * SHADOW_RAYS = next-event estimation: a shadow ray towards a point drawn on a listed light carries that light's
 * emission (weighted by cos / (pi * light pdf), visibility = the closest hit along it is a listed light), the path
 * continues on a cosine-distributed ray, and a listed light met by that ray adds no emission (it was counted by the
 * shadow ray).  Same expectation per pixel — the converged image is the reference's — at lower variance per sample
 * when lights are small; NOT the same sample values, so same-seed comparisons with the reference estimator do not
 * apply.  Runs in the pixel-stream kernels for every tree kind, adaptive or fixed spp, all modes. */
enum { RT_LIGHTS_MIXTURE = 0, RT_LIGHTS_SHADOW_RAYS = 1 };

/* CameraData — src/scenes/sceneData.ts:22-37; defaults src/camera.ts:62-71 */
typedef struct rt_camera_desc {
  double vfov;
  double from[3];
  double at[3];
  double up[3];
  double aperture;
  double focus; /* 0 => |from - at| (src/camera.ts:129) */
  double background_top[3];
  double background_bottom[3];
} rt_camera_desc;

/* SceneData flattened to SoA — src/scenes/sceneData.ts:8-20.  Object order is
 * SceneData.objects order (it decides BVH tie-breaks and light order). */
typedef struct rt_scene_desc {
  uint32_t n_objects;
  const uint8_t* obj_type;     /* [n_objects] RT_OBJ_* */
  const double* obj_pos;       /* [n_objects][3] sphere centre | plane/quad corner */
  const double* obj_u;         /* [n_objects][3] plane/quad u (ignored for spheres) */
  const double* obj_v;         /* [n_objects][3] plane/quad v */
  const double* obj_r;         /* [n_objects] sphere radius (may be negative) */
  const int32_t* obj_material; /* [n_objects] index of the root material node */
  const uint8_t* obj_light;    /* [n_objects] SceneObject.light flag */
  uint32_t n_materials;
  const uint8_t* mat_type;     /* [n_materials] RT_MAT_* */
  const double* mat_color;     /* [n_materials][3] */
  const double* mat_param;     /* [n_materials] */
  const int32_t* mat_child;    /* [n_materials][2], -1 when unused */
  rt_camera_desc camera;
} rt_scene_desc;

/* RenderOptions after the reference's three-layer merge (Camera.defaultRenderData <-
 * sceneData.render <- caller; src/camera.ts:73-83, src/scenes/scenes.ts:97-100) plus the
 * knobs that exist only on this side of the boundary. */
typedef struct rt_render_opts {
  int32_t width;
  double aspect;
  int32_t samples;
  int32_t depth;
  double a_tolerance;
  int32_t a_batch;
  int32_t roulette;       /* bool */
  int32_t roulette_depth;
  int32_t mode;           /* RT_MODE_* */
  /* --- not in the reference --- */
  uint64_t seed;          /* Philox seed; the reference's Math.random is unseedable */
  int32_t bvh;            /* RT_BVH_* */
  int32_t integrator;     /* RT_INTEGRATOR_* */
  int32_t device;         /* CUDA device ordinal, -1 = current */
  /* image-space partition for one-process-per-GPU runs (and, internally, rt_multi_*): the unit is the 8x4
   * pixel block; every run of part_count consecutive blocks (row-major over the whole image) gives each part
   * one block, in an order rotated by a hash of the run's index (block_owner, csrc/rt_types.h; Python mirror
   * mcp_raytracer_b200/distributed.py).  Only owned pixels are rendered / written. */
  int32_t part_index;     /* 0 <= part_index < part_count */
  int32_t part_count;     /* <= 1 means the whole region */
  int32_t light_sampling; /* RT_LIGHTS_* */
} rt_render_opts;

/* RenderRegion — src/camera.ts:54-59 */
typedef struct rt_region {
  int32_t x, y, width, height;
} rt_region;

/* RenderStats — src/render-utils/renderStats.ts:6-19.  min fields are +Infinity in the
 * reference when no pixel was rendered; here they are INT32_MAX in that case. */
typedef struct rt_stats {
  uint64_t pixels;
  uint64_t samples_total;
  int32_t samples_min;
  int32_t samples_max;
  uint64_t bounces_total;
  int32_t bounces_min;
  int32_t bounces_max;
  /* --- measurement extras --- */
  uint64_t rays;        /* closest-hit queries = world.hit calls (src/camera.ts:249) */
  double device_ms;     /* CUDA-event time of the render kernels on the camera's stream */
  int32_t kernel_launches; /* kernels of this library launched by the call */
  int32_t reserved;
  /* executed traversal work, filled ONLY by the instrumented build of the library (libmcprt_b200_count.so,
   * -DRT_COUNT_EVENTS; rt_counts_events() == 1), 0 otherwise: the roofline's "executed" figure for tree scenes */
  uint64_t node_visits;  /* wide-node visits (four child-box tests each) */
  uint64_t prim_tests;   /* primitive tests (always-tested prefix + leaves; LIST: every slot for every ray) */
} rt_stats;

/* Derived camera state, for host-side mirrors of the reference's public Camera fields
 * (src/camera.ts:85-105). */
typedef struct rt_camera_info {
  int32_t image_width, image_height, channels;
  int32_t n_objects, n_lights, n_bvh_nodes, bvh_kind, integrator_kind;
  float center[3], pixel00_loc[3], pixel_delta_u[3], pixel_delta_v[3];
  float u[3], v[3], w[3], defocus_disk_u[3], defocus_disk_v[3];
  double focus_distance;
  int32_t use_adaptive_sampling;
  int32_t device;
  double build_ms; /* host flatten + BVH build + upload */
} rt_camera_info;

typedef struct rt_camera rt_camera; /* opaque: scene + BVH + options resident on one GPU */

/* ---- lifecycle: replaces createCameraFromSceneData + new Camera(...)
 *      (src/scenes/scenes.ts:60-104, src/camera.ts:107-166) ---- */
rt_status rt_camera_create(const rt_scene_desc* scene, const rt_render_opts* opts, rt_camera** out);
rt_status rt_camera_destroy(rt_camera* cam);
rt_status rt_camera_get_info(const rt_camera* cam, rt_camera_info* out);

/* Launch on this CUDA stream (a cudaStream_t passed as void*; NULL = the legacy default
 * stream).  Lets the host framework time the render with its own events. */
rt_status rt_camera_set_stream(rt_camera* cam, void* cuda_stream);

/* ---- the hot path: replaces Camera.renderRegion (src/camera.ts:388-431) ----
 * rgb8: HOST buffer of image_width*image_height*3 bytes, row-major, full-image stride
 * (offset=(j*W+i)*3, src/camera.ts:461); only pixels inside `region` (and owned by this
 * part) are written.  linear_rgb: optional HOST float buffer [H][W][3] receiving the
 * pre-gamma pixel colour (finalColor, src/camera.ts:326-340), or NULL.  Synchronous. */
rt_status rt_camera_render_region(rt_camera* cam, const rt_region* region, uint8_t* rgb8,
                                  size_t rgb8_len, float* linear_rgb, rt_stats* stats);

/* replaces Camera.render (src/camera.ts:439-446): the full image. */
rt_status rt_camera_render(rt_camera* cam, uint8_t* rgb8, size_t rgb8_len, float* linear_rgb,
                           rt_stats* stats);

/* Same as rt_camera_render_region but rgb8 / linear_rgb / moments are DEVICE pointers on
 * the camera's device and nothing is copied or synchronised: the call returns once the
 * kernels are enqueued on the camera's stream.  `moments` (optional, device,
 * [H][W][8] float) receives per pixel: sum r,g,b; the sum of squared deviations of r,g,b from the
 * pixel mean (Welford: variance = that / (samples - 1)); samples; bounces.
 * `stats_dev` (optional, device, sizeof(rt_stats)) receives the reduced statistics
 * except device_ms.  Exception: RT_INTEGRATOR_WAVEFRONT drives its kernels from the host (queue counts are
 * read back between the stages of a bounce), so with that integrator the call blocks until the render is done. */
rt_status rt_camera_render_region_device(rt_camera* cam, const rt_region* region, uint8_t* rgb8_dev,
                                         float* linear_rgb_dev, float* moments_dev,
                                         rt_stats* stats_dev);

/* Host-buffer render that also returns the per-pixel moments (parity tests). */
rt_status rt_camera_render_moments(rt_camera* cam, const rt_region* region, uint8_t* rgb8,
                                   size_t rgb8_len, float* linear_rgb, float* moments,
                                   rt_stats* stats);

/* ---- progressive output (SURVEY.md section 8f row 2) ----
 * The reference renders every pixel to completion before anything is visible (src/camera.ts:400-423) and has no preview
 * surface.  This call delivers the SAME image as rt_camera_render_region in n_passes steps: after pass k every pixel holds
 * its first ceil(samples * k / n_passes) samples (adaptive sampling: rounded up to a multiple of aBatch, pixels that have
 * converged stop for good, exactly where the one-shot render stops them), the host buffers are refreshed, and `on_pass` is
 * called with the statistics so far; a non-zero return ends the render early.  Fixed-spp passes add sample windows to the
 * exact fixed-point sums, the pixel-stream kernels keep each pixel's PixelStats on the device between passes, and the
 * random streams are keyed by (pixel, sample): the final image is bit-identical to the one-shot render.  Synchronous. */
typedef int32_t (*rt_progress_fn)(void* user, int32_t pass, int32_t n_passes, int32_t samples_per_pixel_cap, const rt_stats* so_far);
rt_status rt_camera_render_progressive(rt_camera* cam, const rt_region* region, uint8_t* rgb8, size_t rgb8_len,
                                       float* linear_rgb, int32_t n_passes, rt_progress_fn on_pass, void* user,
                                       rt_stats* stats);
/* Host-only: the sample cap of each of the n_passes passes of every progressive call, for a camera of `samples` per pixel
 * and `batch` = aBatch when it samples adaptively, 1 otherwise.  caps[k - 1] = the cap passed to on_pass after pass k, or
 * -1 for a pass with no new samples, which the calls skip (more passes than samples).  Returns the number of passes that
 * run, or -1 for samples < 0, batch < 1, n_passes < 1 or a null `caps`. */
int32_t rt_progressive_caps(int32_t samples, int32_t batch, int32_t n_passes, int32_t* caps);

/* ---- parity hook: primary visibility through pixel centres (getRay with no jitter and
 * no defocus, src/camera.ts:176-196) + closest hit over (0.001, inf) (src/camera.ts:249).
 * HOST outputs, each optional: obj_id [H][W] (index into SceneData.objects, -1 = miss),
 * t [H][W], normal [H][W][3] (the reference's face-forwarded rec.normal), front_face. */
rt_status rt_camera_trace_primary(rt_camera* cam, const rt_region* region, int32_t* obj_id,
                                  float* t, float* normal, uint8_t* front_face);

/* ---- opt-in denoiser (not in the reference) ----
 * The spatial filter of SVGF (Schied et al., HPG 2017) without its temporal part, guided by first-hit feature buffers: the
 * colour is demodulated by the feature albedo, filtered by `iterations` a-trous passes (step 2^k, 5x5 B3-spline taps) whose
 * weights stop at normal, depth and luminance edges (the luminance stop scaled by the per-pixel variance of the render's
 * moments), and remodulated.  FP32; the filter reads only pixels inside the region.  tests/denoise_reference.py is its
 * specification.  rt_denoise_opts: iterations 0..8 are taken as given (0 = demodulate and remodulate only); a sigma of 0
 * selects its default (luminance 4, normal 128, depth 1); opts == NULL = all defaults (5 iterations). */
typedef struct rt_denoise_opts {
  int32_t iterations;
  float sigma_luminance, sigma_normal, sigma_depth;
} rt_denoise_opts;

/* First-hit features averaged over the camera rays of samples 0..n_samples-1 (n_samples >= 1) — the rays the render kernels
 * draw for those samples (jitter when samples > 1, defocus when the aperture is open).  HOST outputs, each optional, only
 * region pixels written: albedo [H][W][3] (the root material's feature albedo: Lambert / Metal colour, 1 for Glass and
 * Light, Mixed = weighted mean of its children, Layered = its inner material; 1 on a miss), normal [H][W][3] (mean of the
 * face-forwarded normals, renormalised when more than one ray hit; 0 when none did), depth [H][W] (mean Euclidean hit
 * distance over the rays that hit, -1 when none did).  Synchronous. */
rt_status rt_camera_render_features(rt_camera* cam, const rt_region* region, int32_t n_samples,
                                    float* albedo, float* normal, float* depth);
/* The filter on explicit HOST inputs [H][W][...] of one whole image (width x height): colour [3], albedo [3], normal [3],
 * depth [1] as rt_camera_render_features writes them, moments [8] as rt_camera_render_moments writes them; out [H][W][3]
 * must not alias an input.  A pixel whose inputs are not finite, or whose colour over max(albedo, 1e-3) overflows FP32, is
 * passed through unchanged and is no neighbour's tap.  Any width and height > 0.  device -1 = current.  Synchronous. */
rt_status rt_denoise(int32_t device, int32_t width, int32_t height, const float* color, const float* albedo, const float* normal,
                     const float* depth, const float* moments, const rt_denoise_opts* opts, float* out);
/* Render with moments, features of the first min(samples, 8) samples, and the filter, all on the device; one copy back.
 * rgb8 / linear_rgb as rt_camera_render_region (the filtered image).  stats = the render's, except device_ms and
 * kernel_launches, which cover every kernel of the call.  RT_ERR_UNSUPPORTED for partitioned cameras (part_count > 1) and
 * render modes other than RT_MODE_DEFAULT.  Synchronous. */
rt_status rt_camera_render_denoised(rt_camera* cam, const rt_region* region, uint8_t* rgb8, size_t rgb8_len, float* linear_rgb,
                                    const rt_denoise_opts* opts, rt_stats* stats);
/* rt_camera_render_progressive with a denoised preview: passes, caps, on_pass and stats as that call.  After each pass
 * rgb8 / linear_rgb hold the region's filtered image of the samples so far, and `moments` (optional HOST [H][W][8], the
 * layout of rt_camera_render_moments) the render's moments.  The features are computed once, in the first pass, from the
 * first min(samples, 8) samples; the filter reads the noisy colour, which stays on the device.  The last pass is
 * bit-identical to rt_camera_render_denoised (rgb8, linear_rgb, stats except device_ms and kernel_launches) and its moments
 * to rt_camera_render_moments.  Errors as rt_camera_render_denoised, and RT_ERR_INVALID_ARGUMENT for n_passes < 1.
 * Synchronous. */
rt_status rt_camera_render_progressive_denoised(rt_camera* cam, const rt_region* region, uint8_t* rgb8, size_t rgb8_len,
                                                float* linear_rgb, float* moments, int32_t n_passes,
                                                const rt_denoise_opts* opts, rt_progress_fn on_pass, void* user,
                                                rt_stats* stats);

/* ---- one process, N GPUs: replaces the worker pool of generateImageBuffer(parallel: true)
 *      (src/raytracer.ts:60-90: N worker_threads over row strips of a SharedArrayBuffer, RenderStats.merge) ----
 * The scene is compiled once and uploaded to `n_devices` GPUs (devices == NULL: ordinals 0..n-1; n_devices <= 0:
 * every visible GPU).  Device k renders the 8x4 blocks it owns and its kernels store the finished pixels directly
 * into device[0]'s framebuffer over NVLink peer mappings — no gather step, no collective; where peer access is
 * not available each device renders into its own buffer and the owned blocks are merged on the host.  The image
 * is bit-identical to rt_camera_render_region's for every n_devices.  opts->device / part_* are ignored. */
typedef struct rt_multi rt_multi;
rt_status rt_multi_create(const rt_scene_desc* scene, const rt_render_opts* opts, int32_t n_devices,
                          const int32_t* devices, rt_multi** out);
rt_status rt_multi_destroy(rt_multi* multi);
/* info (optional): the camera block of device[0]; n_devices / peer_writes (optional): GPUs in use, 1 = the
 * peer-write path is active. */
rt_status rt_multi_get_info(const rt_multi* multi, rt_camera_info* info, int32_t* n_devices, int32_t* peer_writes);
/* Camera.renderRegion over all the GPUs: HOST buffers as rt_camera_render_region; stats merged like
 * RenderStats.merge (src/render-utils/renderStats.ts:42-64), device_ms = the slowest device.  Synchronous. */
rt_status rt_multi_render_region(rt_multi* multi, const rt_region* region, uint8_t* rgb8, size_t rgb8_len,
                                 float* linear_rgb, rt_stats* stats);
/* rt_camera_render_denoised on every device of the rt_multi: rgb8 / linear_rgb are bit-identical to that call's on one
 * camera with the same scene, options and region, for every n_devices and on both paths.  Device k renders its blocks'
 * colour and moments into device[0]'s memory; after every device's render, each device filters a contiguous band of the
 * region's rows, recomputing the rows its passes read beyond the band (up to 2^(iterations+1) - 1 rows each side, clipped
 * to the region) and reading the colour over the peer mapping; the bands land in device[0]'s framebuffer.  Without peer
 * access the colour and moments are merged on the host and device[0] filters the whole region.  Each device holds
 * whole-image feature and filter buffers (84 bytes per pixel); device[0] also holds the colour and moments (44 bytes per
 * pixel).  Errors as rt_camera_render_denoised (RT_ERR_UNSUPPORTED for render modes other than RT_MODE_DEFAULT).
 * stats: merged as rt_multi_render_region merges them; device_ms = device[0]'s span from the start of its render to the
 * end of the call's last kernel (waiting for the other devices included); kernel_launches = the sum over the devices.
 * Synchronous. */
rt_status rt_multi_render_denoised(rt_multi* multi, const rt_region* region, uint8_t* rgb8, size_t rgb8_len,
                                   float* linear_rgb, const rt_denoise_opts* opts, rt_stats* stats);
/* Progressive renders on every device.  Pass by pass, each call delivers what its one-camera counterpart
 * (rt_camera_render_progressive, rt_camera_render_progressive_denoised) delivers on a camera with the same scene, options
 * and region, for every n_devices and on both paths: the same caps passed to `on_pass`, bit-identical rgb8 / linear_rgb
 * (/ moments) in the caller's buffers after each pass, and the same `so_far` stats except device_ms and kernel_launches.
 * Pixels outside the region are never written.  Each pass renders like rt_multi_render_region (the denoised form: like
 * rt_multi_render_denoised, with the features computed in the first pass only); every device keeps its pixels' state
 * between the passes.  `on_pass` runs on the calling thread, once per pass, after every device's part of that pass has
 * landed in the caller's buffers; a non-zero return stops every device after that pass.  The call returns only when no
 * work of it is left queued on any device.  With n_passes == 1 the result equals rt_multi_render_region /
 * rt_multi_render_denoised (rgb8, linear_rgb, stats).  Errors as the one-camera calls: RT_ERR_INVALID_ARGUMENT for a null
 * multi, n_passes < 1 or bad denoise options, RT_ERR_BUFFER_TOO_SMALL, and RT_ERR_UNSUPPORTED from the denoised form for
 * render modes other than RT_MODE_DEFAULT (the plain form renders every mode).  stats: device_ms = the sum over the
 * passes of each pass's time as the one-shot multi call counts it (the plain form: the slowest device's render; the
 * denoised form: device[0]'s span from its render to the last band); kernel_launches = the sum over devices and passes.
 * Synchronous. */
rt_status rt_multi_render_progressive(rt_multi* multi, const rt_region* region, uint8_t* rgb8, size_t rgb8_len,
                                      float* linear_rgb, int32_t n_passes, rt_progress_fn on_pass, void* user,
                                      rt_stats* stats);
rt_status rt_multi_render_progressive_denoised(rt_multi* multi, const rt_region* region, uint8_t* rgb8, size_t rgb8_len,
                                               float* linear_rgb, float* moments, int32_t n_passes,
                                               const rt_denoise_opts* opts, rt_progress_fn on_pass, void* user,
                                               rt_stats* stats);

/* ---- one process PER GPU (torch.distributed ranks of one node): a device buffer every rank can write ----
 * Rank 0 creates the framebuffer and hands the 64-byte CUDA IPC handle to the other ranks (any transport);
 * they open it and pass the pointer as rgb8_dev to rt_camera_render_region_device: their kernels then write
 * the pixels they own straight into rank 0's memory (the SharedArrayBuffer of src/raytracer.ts:71-72). */
rt_status rt_shared_buffer_create(int32_t device, size_t bytes, void** dev_ptr, uint8_t handle[64]);
rt_status rt_shared_buffer_open(int32_t device, const uint8_t handle[64], void** dev_ptr);
rt_status rt_shared_buffer_release(int32_t device, void* dev_ptr, int32_t opened /* 1: from _open, 0: from _create */);

/* ---- per-function parity hooks ----------------------------------------------------------------
 * Each call runs ONE device function of the render path (the same code the render kernels inline) on
 * `n` explicit records, with the uniforms `Math.random()` would return given by the caller: RT_DEBUG_UNIFORMS
 * doubles per record, consumed in the reference's draw order, each rounded to FP32 (give k / 2^24 values to
 * feed the CPU oracle bit-identical numbers); draws past the end read 0.5.  Host pointers; synchronous.
 * Used by tests/test_gpu_functions.py against the reference's own Jest vectors; not on the render path. */
#define RT_DEBUG_UNIFORMS 16
typedef struct rt_debug_hit { /* rIn + HitRecord — src/geometry/hittable.ts:9-18 */
  double ray_origin[3], ray_dir[3];
  double p[3], normal[3];  /* rec.p, rec.normal (face-forwarded unit normal) */
  int32_t front_face;      /* rec.frontFace */
  int32_t reserved;
} rt_debug_hit;
typedef struct rt_debug_scatter_out { /* ScatterResult | null — src/materials/material.ts:14-23 */
  int32_t kind;            /* 0 = null (absorbed, or a light), 1 = `scattered` ray (specular), 2 = `pdf` (cosine pdf about rec.normal) */
  int32_t uniforms_used;
  float attenuation[3];
  float dir[3];            /* kind 1: scattered.direction */
  float emitted[3];        /* material.emitted(rec) */
} rt_debug_scatter_out;
/* material.scatter + material.emitted of SceneData.objects[object_index].material at each hit
 * (src/materials/{lambertian,metal,dielectric,diffuseLight,layeredMaterial,mixedMaterial}.ts) */
rt_status rt_debug_scatter(rt_camera* cam, int32_t object_index, int32_t n, const rt_debug_hit* hits,
                           const double* uniforms, rt_debug_scatter_out* out);
/* Camera.getRay(i, j) — src/camera.ts:176-210.  ij [n][2]; ray_out [n][6] = origin.xyz, direction.xyz
 * (direction NOT normalised, like the reference); used [n] = uniforms consumed (optional). */
rt_status rt_debug_get_ray(rt_camera* cam, int32_t n, const int32_t* ij, const double* uniforms,
                           float* ray_out, int32_t* used);
/* lights[light_index].pdfValue(origin, direction) — src/entities/quad.ts:123-140, sphere.ts:106-131.
 * light_index counts the scene's lights in SceneData.objects order (src/scenes/scenes.ts:74-79). */
rt_status rt_debug_light_pdf(rt_camera* cam, int32_t light_index, int32_t n, const double* origin,
                             const double* direction, float* value);
/* lights[light_index].pdfRandomVec(origin) — src/entities/quad.ts:148-158, sphere.ts:140-147 +
 * src/geometry/vec3.ts:345-351; two uniforms per record.  out [n][3]. */
rt_status rt_debug_light_random_vec(rt_camera* cam, int32_t light_index, int32_t n, const double* origin,
                                    const double* uniforms, float* out);
/* The diffuse branch of rayColor — src/camera.ts:285-308 with MixturePDF (src/geometry/pdf.ts:57-99), CosinePDF
 * (:32-51) and ONBasis (src/geometry/onbasis.ts:18-51): three uniforms per record (component select, r1, r2).
 * out [n][6] = direction.xyz, mixture pdf value, scatter pdf value, continues (pdf value > 0.0001). */
rt_status rt_debug_diffuse_bounce(rt_camera* cam, int32_t n, const double* p, const double* normal,
                                  const double* uniforms, float* out);

/* ---- misc ---- */
const char* rt_last_error(void);
int32_t rt_device_count(void);
int32_t rt_abi_version(void);
int32_t rt_counts_events(void); /* 1 = instrumented build: node visits / primitive tests are counted into the stats (slower) */
/* which part (0 <= part < part_count) renders pixel (x, y) of an image `image_width` wide: the partition rule of
 * rt_render_opts.part_index / rt_multi_*, for host code that assembles or checks partitioned renders. */
int32_t rt_block_owner(int32_t x, int32_t y, int32_t image_width, int32_t part_count);
/* measured FP32 FMA throughput of `device` in TFLOP/s (dependent-chain FFMA microbenchmark),
 * the roofline denominator for this path. */
rt_status rt_measure_fp32_peak(int32_t device, double* tflops, double* sm_clock_mhz);
/* Device buffers of destroyed cameras are kept for the next rt_camera_create (the reference builds
 * its scene per request, src/render-utils/renderWorker.ts:20; cudaMalloc/cudaFree per image cost
 * more than the scene build).  This returns them to the driver; result = bytes released. */
uint64_t rt_trim_device_cache(void);

/* Host-only diagnostic (no GPU needed): runs the scene compiler of rt_camera_create — validation of
 * createSceneObject/createMaterial (src/scenes/scenes.ts:109-199), acceleration-structure choice and build —
 * and checks the result: every object in exactly one slot, every leaf primitive inside its child box, every
 * child box inside its parent's, stack depth.  `errors` = number of violated invariants (0 = sound). */
typedef struct rt_scene_report {
  int32_t bvh_kind;      /* RT_BVH_* actually chosen */
  int32_t n_slots;       /* primitive slots = objects */
  int32_t n_prefix;      /* always-tested slots (all of them for RT_BVH_LIST) */
  int32_t n_node_slots;  /* 64-byte node slots (a 4-wide SAH node takes two) */
  int32_t n_leaves;
  int32_t max_leaf_size;
  int32_t max_depth;
  int32_t n_lights;
  int32_t errors;
  int32_t reserved[3];
} rt_scene_report;
rt_status rt_scene_validate(const rt_scene_desc* scene, const rt_render_opts* opts, rt_scene_report* report);

#ifdef __cplusplus
}
#endif
#endif /* RT_B200_H */
