/*
 * rt_napi.c — N-API shim over the C ABI of include/rt_b200.h.
 *
 * NOT BUILT IN THIS REPOSITORY'S IMAGE: there is no node toolchain and no real node_api.h here (SURVEY.md §0).  The
 * file is syntax- and type-checked against a stub of the Node-API header (ts/addon/stub/node_api.h,
 * tests/test_host_and_abi.py::test_napi_shim_compiles_against_the_stub_header); the C ABI entry points it calls are
 * exercised end to end from Python ctypes by the test-suite.  A maintainer of df07/mcp-raytracer builds it with
 * node-gyp (binding.gyp).
 *
 * Exports:
 *   createCamera(flat, opts) -> handle                          rt_camera_create   (one GPU)
 *   createMulti(flat, opts, nDevices) -> handle                 rt_multi_create    (all GPUs: generateImageBuffer's parallel:true)
 *   renderRegion(handle, region, pixelData) -> stats            rt_camera_render_region / rt_multi_render_region, synchronous
 *   renderRegionAsync(handle, region, pixelData) -> Promise     same on a libuv worker (napi_async_work): keeps the event loop
 *                                                               free, like the reference's worker threads (src/raytracer.ts:60-90)
 *   renderDenoised(handle, region, pixelData, options?) -> stats rt_camera_render_denoised / rt_multi_render_denoised, synchronous;
 *                                                               options {iterations, sigmaLuminance, sigmaNormal, sigmaDepth}
 *   cameraInfo(handle) -> { imageWidth, imageHeight, ... }      rt_camera_get_info / rt_multi_get_info
 *   destroyCamera(handle)                                       rt_camera_destroy / rt_multi_destroy — releases the GPU memory NOW
 *   deviceCount(), trimDeviceCache()
 * A non-zero rt_status becomes a thrown JS Error (or a rejected Promise) carrying rt_last_error(), so upstream error
 * behaviour (src/scenes/scenes.ts:137,154,178,191,195; src/raytracer.ts:162-173) is unchanged.
 *
 * Ownership: the JS handle is an external around a small box {camera | multi}.  destroyCamera() destroys the native object
 * and clears the box; the GC finalizer only frees what is still there.  V8 is told about the device memory behind a handle
 * (napi_adjust_external_memory) so that a long-lived MCP server that forgets destroyCamera() still collects in time.
 */
#include <node_api.h>
#include <stdlib.h>
#include <string.h>

#include "../../include/rt_b200.h"

#define CHECK(env, call) do { if ((call) != napi_ok) { napi_throw_error((env), NULL, "N-API call failed: " #call); return NULL; } } while (0)

typedef struct cam_box {
  rt_camera* cam;   /* exactly one of cam / multi is set */
  rt_multi* multi;
  int64_t external_bytes;
  int busy;         /* an async render is in flight: destroy waits for its completion callback */
  int destroy_requested;
} cam_box;

static napi_value throw_msg(napi_env env, const char* msg) { napi_throw_error(env, NULL, msg); return NULL; }
static napi_value throw_rt(napi_env env) { return throw_msg(env, rt_last_error()); }

static void box_release(napi_env env, cam_box* b) {
  if (b->cam) rt_camera_destroy(b->cam);
  if (b->multi) rt_multi_destroy(b->multi);
  b->cam = NULL; b->multi = NULL;
  if (b->external_bytes) { int64_t now; napi_adjust_external_memory(env, -b->external_bytes, &now); b->external_bytes = 0; }
}
static void finalize_box(napi_env env, void* data, void* hint) { (void)hint; cam_box* b = (cam_box*)data; box_release(env, b); free(b); }

/* typed-array field of an object -> raw pointer + element count; NULL when absent or of the wrong element type */
static void* ta_field(napi_env env, napi_value obj, const char* name, napi_typedarray_type want, size_t* len) {
  napi_value v; napi_typedarray_type ty; void* data = NULL; napi_value ab; size_t off; bool has = false;
  *len = 0;
  if (napi_has_named_property(env, obj, name, &has) != napi_ok || !has) return NULL;
  if (napi_get_named_property(env, obj, name, &v) != napi_ok) return NULL;
  if (napi_get_typedarray_info(env, v, &ty, len, &data, &ab, &off) != napi_ok || ty != want) { *len = 0; return NULL; }
  return data;
}
static double num_field(napi_env env, napi_value obj, const char* name, double dflt) {
  napi_value v; double d = dflt; bool has = false; napi_valuetype t;
  if (napi_has_named_property(env, obj, name, &has) != napi_ok || !has) return dflt;
  if (napi_get_named_property(env, obj, name, &v) != napi_ok || napi_typeof(env, v, &t) != napi_ok || t != napi_number) return dflt;
  napi_get_value_double(env, v, &d);
  return d;
}
static int vec3_field(napi_env env, napi_value obj, const char* name, double out[3]) {
  size_t n; double* p = (double*)ta_field(env, obj, name, napi_float64_array, &n);
  if (!p || n < 3) return 0;
  memcpy(out, p, 3 * sizeof(double));
  return 1;
}

/* FlatScene (ts/nativeCamera.ts flattenScene) -> rt_scene_desc, every array length checked against n_objects / n_materials:
 * a short array must be a JS error, never an out-of-bounds read in the scene compiler */
static const char* read_scene(napi_env env, napi_value flat, rt_scene_desc* s) {
  size_t n = 0, m = 0, k = 0;
  napi_value cam;
  memset(s, 0, sizeof(*s));
  s->obj_type = (const uint8_t*)ta_field(env, flat, "objType", napi_uint8_array, &n);
  if (!s->obj_type || n == 0 || n > 0xffffffffu) return "flat.objType must be a non-empty Uint8Array";
  s->n_objects = (uint32_t)n;
  s->obj_pos = (const double*)ta_field(env, flat, "objPos", napi_float64_array, &k); if (k != 3 * n) return "flat.objPos must be a Float64Array of 3 * objects";
  s->obj_u = (const double*)ta_field(env, flat, "objU", napi_float64_array, &k);     if (k != 3 * n) return "flat.objU must be a Float64Array of 3 * objects";
  s->obj_v = (const double*)ta_field(env, flat, "objV", napi_float64_array, &k);     if (k != 3 * n) return "flat.objV must be a Float64Array of 3 * objects";
  s->obj_r = (const double*)ta_field(env, flat, "objR", napi_float64_array, &k);     if (k != n) return "flat.objR must be a Float64Array of one entry per object";
  s->obj_material = (const int32_t*)ta_field(env, flat, "objMaterial", napi_int32_array, &k); if (k != n) return "flat.objMaterial must be an Int32Array of one entry per object";
  s->obj_light = (const uint8_t*)ta_field(env, flat, "objLight", napi_uint8_array, &k);       if (k != n) return "flat.objLight must be a Uint8Array of one entry per object";
  s->mat_type = (const uint8_t*)ta_field(env, flat, "matType", napi_uint8_array, &m);
  if (!s->mat_type || m == 0 || m > 0xffffffffu) return "flat.matType must be a non-empty Uint8Array";
  s->n_materials = (uint32_t)m;
  s->mat_color = (const double*)ta_field(env, flat, "matColor", napi_float64_array, &k); if (k != 3 * m) return "flat.matColor must be a Float64Array of 3 * materials";
  s->mat_param = (const double*)ta_field(env, flat, "matParam", napi_float64_array, &k); if (k != m) return "flat.matParam must be a Float64Array of one entry per material";
  s->mat_child = (const int32_t*)ta_field(env, flat, "matChild", napi_int32_array, &k);  if (k != 2 * m) return "flat.matChild must be an Int32Array of 2 * materials";
  if (napi_get_named_property(env, flat, "camera", &cam) != napi_ok) return "flat.camera missing";
  s->camera.vfov = num_field(env, cam, "vfov", 90); s->camera.aperture = num_field(env, cam, "aperture", 0); s->camera.focus = num_field(env, cam, "focus", 1.0);
  if (!vec3_field(env, cam, "from", s->camera.from) || !vec3_field(env, cam, "at", s->camera.at) || !vec3_field(env, cam, "up", s->camera.up) ||
      !vec3_field(env, cam, "backgroundTop", s->camera.background_top) || !vec3_field(env, cam, "backgroundBottom", s->camera.background_bottom))
    return "flat.camera.{from,at,up,backgroundTop,backgroundBottom} must be Float64Array(3)";
  return NULL;
}
static void read_opts(napi_env env, napi_value o, rt_render_opts* r) { /* defaults: Camera.defaultRenderData, src/camera.ts:73-83 */
  memset(r, 0, sizeof(*r));
  r->width = (int32_t)num_field(env, o, "width", 400); r->aspect = num_field(env, o, "aspect", 16.0 / 9.0);
  r->samples = (int32_t)num_field(env, o, "samples", 100); r->depth = (int32_t)num_field(env, o, "depth", 100);
  r->a_tolerance = num_field(env, o, "aTolerance", 0.05); r->a_batch = (int32_t)num_field(env, o, "aBatch", 10);
  r->roulette = (int32_t)num_field(env, o, "roulette", 1); r->roulette_depth = (int32_t)num_field(env, o, "rouletteDepth", 3);
  r->mode = (int32_t)num_field(env, o, "mode", RT_MODE_DEFAULT); r->seed = (uint64_t)num_field(env, o, "seed", 0);
  r->bvh = RT_BVH_AUTO; r->integrator = RT_INTEGRATOR_AUTO; r->device = (int32_t)num_field(env, o, "device", -1);
  r->part_index = (int32_t)num_field(env, o, "partIndex", 0); r->part_count = (int32_t)num_field(env, o, "partCount", 1);
  r->light_sampling = (int32_t)num_field(env, o, "lightSampling", RT_LIGHTS_MIXTURE);
}
/* what V8 should know about: framebuffer + fixed-point accumulator + queue per pixel, plus the scene arrays */
static int64_t device_bytes(const rt_camera_info* ci, const rt_scene_desc* s, int n_devices) {
  const int64_t px = (int64_t)ci->image_width * ci->image_height;
  return n_devices * (px * (3 + 32 + 1) + (int64_t)s->n_objects * 250 + (int64_t)s->n_materials * 48);
}

static napi_value make_handle(napi_env env, rt_camera* cam, rt_multi* multi, const rt_scene_desc* s) {
  cam_box* b = (cam_box*)calloc(1, sizeof(cam_box));
  napi_value ext;
  rt_camera_info ci; int32_t nd = 1;
  if (!b) { if (cam) rt_camera_destroy(cam); if (multi) rt_multi_destroy(multi); return throw_msg(env, "out of memory"); }
  b->cam = cam; b->multi = multi;
  memset(&ci, 0, sizeof(ci));
  if (cam) rt_camera_get_info(cam, &ci); else rt_multi_get_info(multi, &ci, &nd, NULL);
  b->external_bytes = device_bytes(&ci, s, nd);
  { int64_t now; napi_adjust_external_memory(env, b->external_bytes, &now); }
  if (napi_create_external(env, b, finalize_box, NULL, &ext) != napi_ok) { box_release(env, b); free(b); return throw_msg(env, "napi_create_external failed"); }
  return ext;
}

static napi_value CreateCamera(napi_env env, napi_callback_info info) {
  size_t argc = 2; napi_value argv[2];
  rt_scene_desc s; rt_render_opts r; rt_camera* h = NULL; const char* err;
  CHECK(env, napi_get_cb_info(env, info, &argc, argv, NULL, NULL));
  if (argc < 2) return throw_msg(env, "createCamera(flat, opts)");
  if ((err = read_scene(env, argv[0], &s)) != NULL) return throw_msg(env, err);
  read_opts(env, argv[1], &r);
  if (rt_camera_create(&s, &r, &h) != RT_OK) return throw_rt(env);
  return make_handle(env, h, NULL, &s);
}

static napi_value CreateMulti(napi_env env, napi_callback_info info) {
  size_t argc = 3; napi_value argv[3];
  rt_scene_desc s; rt_render_opts r; rt_multi* h = NULL; const char* err; double nd = 0;
  CHECK(env, napi_get_cb_info(env, info, &argc, argv, NULL, NULL));
  if (argc < 2) return throw_msg(env, "createMulti(flat, opts, nDevices?)");
  if ((err = read_scene(env, argv[0], &s)) != NULL) return throw_msg(env, err);
  read_opts(env, argv[1], &r);
  if (argc >= 3) napi_get_value_double(env, argv[2], &nd);
  if (rt_multi_create(&s, &r, (int32_t)nd, NULL, &h) != RT_OK) return throw_rt(env);
  return make_handle(env, NULL, h, &s);
}

static cam_box* get_box(napi_env env, napi_value v) {
  cam_box* b = NULL;
  if (napi_get_value_external(env, v, (void**)&b) != napi_ok || !b || (!b->cam && !b->multi)) { napi_throw_error(env, NULL, "camera handle is invalid or destroyed"); return NULL; }
  return b;
}
static int read_region(napi_env env, napi_value v, rt_region* reg) {
  reg->x = (int32_t)num_field(env, v, "x", 0); reg->y = (int32_t)num_field(env, v, "y", 0);
  reg->width = (int32_t)num_field(env, v, "width", -1); reg->height = (int32_t)num_field(env, v, "height", -1);
  return reg->width >= 0 && reg->height >= 0;
}
static rt_status render_box(cam_box* b, const rt_region* reg, uint8_t* data, size_t len, rt_stats* st) {
  return b->cam ? rt_camera_render_region(b->cam, reg, data, len, NULL, st) : rt_multi_render_region(b->multi, reg, data, len, NULL, st);
}
static napi_value stats_object(napi_env env, const rt_stats* st) {
  napi_value out, v;
  if (napi_create_object(env, &out) != napi_ok) return NULL;
#define SETD(name, val) do { napi_create_double(env, (double)(val), &v); napi_set_named_property(env, out, name, v); } while (0)
  SETD("pixels", st->pixels); SETD("samplesTotal", st->samples_total); SETD("samplesMin", st->samples_min); SETD("samplesMax", st->samples_max);
  SETD("bouncesTotal", st->bounces_total); SETD("bouncesMin", st->bounces_min); SETD("bouncesMax", st->bounces_max);
  SETD("rays", st->rays); SETD("deviceMs", st->device_ms);
  return out;
}

static napi_value RenderRegion(napi_env env, napi_callback_info info) {
  size_t argc = 3; napi_value argv[3];
  napi_typedarray_type ty; size_t len; void* data; napi_value ab; size_t off;
  rt_region reg; rt_stats st; cam_box* b;
  CHECK(env, napi_get_cb_info(env, info, &argc, argv, NULL, NULL));
  if (argc < 3) return throw_msg(env, "renderRegion(handle, region, pixelData)");
  if (!(b = get_box(env, argv[0]))) return NULL;
  if (b->busy) return throw_msg(env, "an asynchronous render is in flight on this camera");
  if (!read_region(env, argv[1], &reg)) return throw_msg(env, "region must be {x, y, width, height}");
  CHECK(env, napi_get_typedarray_info(env, argv[2], &ty, &len, &data, &ab, &off)); /* Uint8ClampedArray, also over a SharedArrayBuffer */
  if (ty != napi_uint8_clamped_array && ty != napi_uint8_array) return throw_msg(env, "pixelData must be a Uint8ClampedArray");
  if (render_box(b, &reg, (uint8_t*)data, len, &st) != RT_OK) return throw_rt(env);
  return stats_object(env, &st);
}

/* render + denoise on the device (not in the reference) */
static napi_value RenderDenoised(napi_env env, napi_callback_info info) {
  size_t argc = 4; napi_value argv[4];
  napi_typedarray_type ty; size_t len; void* data; napi_value ab; size_t off;
  napi_valuetype vt = napi_undefined;
  rt_region reg; rt_stats st; cam_box* b;
  rt_denoise_opts o = {5, 0.f, 0.f, 0.f};
  CHECK(env, napi_get_cb_info(env, info, &argc, argv, NULL, NULL));
  if (argc < 3) return throw_msg(env, "renderDenoised(handle, region, pixelData, options?)");
  if (!(b = get_box(env, argv[0]))) return NULL;
  if (b->busy) return throw_msg(env, "an asynchronous render is in flight on this camera");
  if (!read_region(env, argv[1], &reg)) return throw_msg(env, "region must be {x, y, width, height}");
  CHECK(env, napi_get_typedarray_info(env, argv[2], &ty, &len, &data, &ab, &off));
  if (ty != napi_uint8_clamped_array && ty != napi_uint8_array) return throw_msg(env, "pixelData must be a Uint8ClampedArray");
  if (argc > 3) CHECK(env, napi_typeof(env, argv[3], &vt));
  if (vt == napi_object) {
    o.iterations = (int32_t)num_field(env, argv[3], "iterations", 5);
    o.sigma_luminance = (float)num_field(env, argv[3], "sigmaLuminance", 0);
    o.sigma_normal = (float)num_field(env, argv[3], "sigmaNormal", 0);
    o.sigma_depth = (float)num_field(env, argv[3], "sigmaDepth", 0);
  }
  if ((b->cam ? rt_camera_render_denoised(b->cam, &reg, (uint8_t*)data, len, NULL, &o, &st)
              : rt_multi_render_denoised(b->multi, &reg, (uint8_t*)data, len, NULL, &o, &st)) != RT_OK)
    return throw_rt(env);
  return stats_object(env, &st);
}

/* ---- the same call on a libuv worker thread ---- */
typedef struct render_job {
  cam_box* box; rt_region reg; uint8_t* data; size_t len; rt_stats st; rt_status rc; char err[512];
  napi_deferred deferred; napi_async_work work; napi_ref keep_pixels, keep_handle; /* keep the buffer and the handle alive */
} render_job;
static void job_execute(napi_env env, void* p) { /* worker thread: no N-API calls here */
  render_job* j = (render_job*)p; (void)env;
  j->rc = render_box(j->box, &j->reg, j->data, j->len, &j->st);
  if (j->rc != RT_OK) { strncpy(j->err, rt_last_error(), sizeof(j->err) - 1); j->err[sizeof(j->err) - 1] = 0; } /* thread-local message: copy it here */
}
static void job_complete(napi_env env, napi_status status, void* p) {
  render_job* j = (render_job*)p;
  j->box->busy = 0;
  if (status == napi_ok && j->rc == RT_OK) {
    napi_value v = stats_object(env, &j->st);
    napi_resolve_deferred(env, j->deferred, v);
  } else {
    napi_value msg, e;
    napi_create_string_utf8(env, status == napi_ok ? j->err : "render cancelled", NAPI_AUTO_LENGTH, &msg);
    napi_create_error(env, NULL, msg, &e);
    napi_reject_deferred(env, j->deferred, e);
  }
  if (j->box->destroy_requested) box_release(env, j->box);
  napi_delete_reference(env, j->keep_pixels); napi_delete_reference(env, j->keep_handle);
  napi_delete_async_work(env, j->work);
  free(j);
}
static napi_value RenderRegionAsync(napi_env env, napi_callback_info info) {
  size_t argc = 3; napi_value argv[3], promise, name;
  napi_typedarray_type ty; size_t len; void* data; napi_value ab; size_t off;
  cam_box* b; render_job* j;
  CHECK(env, napi_get_cb_info(env, info, &argc, argv, NULL, NULL));
  if (argc < 3) return throw_msg(env, "renderRegionAsync(handle, region, pixelData)");
  if (!(b = get_box(env, argv[0]))) return NULL;
  if (b->busy) return throw_msg(env, "an asynchronous render is already in flight on this camera"); /* one render at a time per camera (rt_b200.h) */
  CHECK(env, napi_get_typedarray_info(env, argv[2], &ty, &len, &data, &ab, &off));
  if (ty != napi_uint8_clamped_array && ty != napi_uint8_array) return throw_msg(env, "pixelData must be a Uint8ClampedArray");
  if (!(j = (render_job*)calloc(1, sizeof(render_job)))) return throw_msg(env, "out of memory");
  if (!read_region(env, argv[1], &j->reg)) { free(j); return throw_msg(env, "region must be {x, y, width, height}"); }
  j->box = b; j->data = (uint8_t*)data; j->len = len;
  if (napi_create_promise(env, &j->deferred, &promise) != napi_ok || napi_create_reference(env, argv[2], 1, &j->keep_pixels) != napi_ok ||
      napi_create_reference(env, argv[0], 1, &j->keep_handle) != napi_ok ||
      napi_create_string_utf8(env, "rt_b200.renderRegion", NAPI_AUTO_LENGTH, &name) != napi_ok ||
      napi_create_async_work(env, NULL, name, job_execute, job_complete, j, &j->work) != napi_ok) { free(j); return throw_msg(env, "could not create the async render job"); }
  b->busy = 1;
  if (napi_queue_async_work(env, j->work) != napi_ok) { b->busy = 0; napi_delete_async_work(env, j->work); free(j); return throw_msg(env, "could not queue the async render job"); }
  return promise;
}

static napi_value CameraInfo(napi_env env, napi_callback_info info) {
  size_t argc = 1; napi_value argv[1], out, v;
  rt_camera_info ci; int32_t nd = 1, p2p = 0; cam_box* b; rt_status rc;
  CHECK(env, napi_get_cb_info(env, info, &argc, argv, NULL, NULL));
  if (argc < 1 || !(b = get_box(env, argv[0]))) return argc < 1 ? throw_msg(env, "cameraInfo(handle)") : NULL;
  rc = b->cam ? rt_camera_get_info(b->cam, &ci) : rt_multi_get_info(b->multi, &ci, &nd, &p2p);
  if (rc != RT_OK) return throw_rt(env);
  CHECK(env, napi_create_object(env, &out));
  SETD("imageWidth", ci.image_width); SETD("imageHeight", ci.image_height); SETD("channels", ci.channels);
  SETD("nLights", ci.n_lights); SETD("focusDistance", ci.focus_distance); SETD("useAdaptiveSampling", ci.use_adaptive_sampling);
  SETD("nDevices", nd); SETD("peerWrites", p2p); SETD("buildMs", ci.build_ms);
  return out;
}

static napi_value DestroyCamera(napi_env env, napi_callback_info info) {
  size_t argc = 1; napi_value argv[1], u; cam_box* b = NULL;
  CHECK(env, napi_get_cb_info(env, info, &argc, argv, NULL, NULL));
  if (argc >= 1 && napi_get_value_external(env, argv[0], (void**)&b) == napi_ok && b) {
    if (b->busy) b->destroy_requested = 1; /* released by the completion callback of the render in flight */
    else box_release(env, b);              /* GPU memory goes back now; the finalizer finds an empty box */
  }
  napi_get_undefined(env, &u);
  return u;
}
static napi_value DeviceCount(napi_env env, napi_callback_info info) { napi_value v; (void)info; napi_create_int32(env, rt_device_count(), &v); return v; }
/* device buffers of destroyed cameras are cached for the next createCamera; a long-lived MCP server can hand them back */
static napi_value TrimDeviceCache(napi_env env, napi_callback_info info) { napi_value v; (void)info; napi_create_double(env, (double)rt_trim_device_cache(), &v); return v; }

static napi_value Init(napi_env env, napi_value exports) {
  napi_property_descriptor d[] = {
    {"createCamera", 0, CreateCamera, 0, 0, 0, napi_default, 0}, {"createMulti", 0, CreateMulti, 0, 0, 0, napi_default, 0},
    {"renderRegion", 0, RenderRegion, 0, 0, 0, napi_default, 0}, {"renderRegionAsync", 0, RenderRegionAsync, 0, 0, 0, napi_default, 0},
    {"renderDenoised", 0, RenderDenoised, 0, 0, 0, napi_default, 0},
    {"cameraInfo", 0, CameraInfo, 0, 0, 0, napi_default, 0}, {"destroyCamera", 0, DestroyCamera, 0, 0, 0, napi_default, 0},
    {"deviceCount", 0, DeviceCount, 0, 0, 0, napi_default, 0}, {"trimDeviceCache", 0, TrimDeviceCache, 0, 0, 0, napi_default, 0},
  };
  napi_define_properties(env, exports, sizeof(d) / sizeof(d[0]), d);
  return exports;
}
NAPI_MODULE(NODE_GYP_MODULE_NAME, Init)
