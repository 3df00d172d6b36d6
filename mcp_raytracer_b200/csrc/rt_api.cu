// rt_api.cu — the C ABI of include/rt_b200.h on top of the CUDA kernels.
//
// There is NO CPU fallback: without a CUDA device every entry point that would compute
// returns RT_ERR_NO_DEVICE.
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <functional>
#include <map>
#include <memory>
#include <thread>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/rt_b200.h"
#include "rt_scene.h"
#include "rt_types.h"

namespace rt {
cudaError_t launch_render_mega(const DevScene& S, const RenderParams& R, int sms, cudaStream_t st);
void render_tile_grid(const RenderParams& R, int* tiles_x, int* tiles_y);
bool render_needs_full(const DevScene& S, const RenderParams& R);
int render_adaptive_blocks(const DevScene& S, const RenderParams& R, int sms, int* warps);
cudaError_t launch_trace_primary(const DevScene& S, const RenderParams& R, int* obj_id, float* t, float* normal,
                                 uint8_t* front, cudaStream_t st);
cudaError_t launch_fp32_peak(float* out, int blocks, int iters, cudaStream_t st);
cudaError_t launch_render_features(const DevScene& S, const RenderParams& R, int n_samples, float* albedo, float* normal, float* depth,
                                   cudaStream_t st);
cudaError_t launch_denoise(const DenoiseParams& D, int b0, int b1, cudaStream_t st, int* launches);
cudaError_t launch_render_wavefront(const DevScene& S, const RenderParams& R, WfHost& H, int sms, cudaStream_t st, int* launches);
cudaError_t launch_finalize_stats(const unsigned long long* raw, rt_stats* out, int launches, cudaStream_t st);
// per-function parity hooks (rt_debug.cuh)
cudaError_t launch_debug_scatter(const DevScene& S, int root, int n, const void* hits, const float* uniforms, void* out, cudaStream_t st);
cudaError_t launch_debug_get_ray(const DevScene& S, int n, const int* ij, const float* uniforms, float* out, int* used, cudaStream_t st);
cudaError_t launch_debug_light_pdf(const DevScene& S, int light, int n, const float* origin, const float* dir, float* value, cudaStream_t st);
cudaError_t launch_debug_light_random(const DevScene& S, int light, int n, const float* origin, const float* uniforms, float* out, cudaStream_t st);
cudaError_t launch_debug_diffuse(const DevScene& S, int n, const float* p, const float* nrm, const float* uniforms, float* out, cudaStream_t st);
} // namespace rt

using namespace rt;

static thread_local std::string g_err;
static rt_status fail(rt_status st, const std::string& msg) {
  g_err = msg;
  return st;
}
// No C++ exception crosses the ABI (include/rt_b200.h): every extern "C" body that allocates host memory sits between these.
#define RT_GUARD_BEGIN try {
#define RT_GUARD_END                                                                                   \
  } catch (const std::bad_alloc&) { return fail(RT_ERR_INVALID_ARGUMENT, "out of host memory"); }      \
  catch (const std::exception& e) { return fail(RT_ERR_INVALID_ARGUMENT, std::string("internal error: ") + e.what()); }
#define CU(call)                                                                                      \
  do {                                                                                                \
    cudaError_t e_ = (call);                                                                          \
    if (e_ != cudaSuccess) return fail(RT_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
  } while (0)

// ---------------------------------------------------------------------------------------------
// Device memory cache.  The reference builds its scene objects per request and per worker
// (renderWorker.ts:20), so a drop-in creates and destroys a camera per image; cudaMalloc/cudaFree
// of the image-sized buffers then cost more than compiling the scene (cudaFree of the 32 MB
// accumulator was measured at 100-170 ms every other call).  Freed blocks stay in a per-device
// size-class list (8 classes per octave, <= 12.5 % slack) and are handed out again;
// rt_trim_device_cache() gives them back to the driver.  Blocks are only reused after the stream of
// the camera that owned them was synchronised (free_camera does that).
// ---------------------------------------------------------------------------------------------
namespace {
struct DevCache {
  std::mutex mu;
  std::multimap<std::pair<int, size_t>, void*> free_blocks; // (device, class size) -> block
  std::unordered_map<void*, std::pair<int, size_t>> live;   // block -> (device, class size)
  size_t cached_bytes = 0;
};
DevCache& dev_cache() {
  static DevCache* c = new DevCache(); // never destroyed: cameras may outlive static destructors
  return *c;
}
const size_t kDevCacheMax = (size_t)4 << 30;
size_t dev_class_size(size_t n) {
  if (n <= 512) return 512;
  int lg = 63 - __builtin_clzll((unsigned long long)(n - 1)); // 2^lg < n <= 2^(lg+1)
  size_t step = (size_t)1 << (lg - 3);                        // 8 classes per octave (lg >= 9 here)
  return (n + step - 1) / step * step;
}
size_t dev_trim_locked(DevCache& C) {
  size_t freed = 0;
  for (auto& kv : C.free_blocks) {
    int prev = -1;
    cudaGetDevice(&prev);
    if (prev != kv.first.first) cudaSetDevice(kv.first.first);
    cudaFree(kv.second);
    if (prev >= 0 && prev != kv.first.first) cudaSetDevice(prev);
    freed += kv.first.second;
  }
  C.free_blocks.clear();
  C.cached_bytes = 0;
  return freed;
}
template <class T>
cudaError_t dev_alloc(T** out, size_t n) {
  *out = nullptr;
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  const size_t cls = dev_class_size(n);
  DevCache& C = dev_cache();
  std::lock_guard<std::mutex> lk(C.mu);
  auto it = C.free_blocks.find({dev, cls});
  void* p = nullptr;
  if (it != C.free_blocks.end()) {
    p = it->second;
    C.free_blocks.erase(it);
    C.cached_bytes -= cls;
  } else {
    e = cudaMalloc(&p, cls);
    if (e != cudaSuccess) { // give the cached blocks back and try once more
      cudaGetLastError();
      dev_trim_locked(C);
      e = cudaMalloc(&p, cls);
      if (e != cudaSuccess) return e;
    }
  }
  C.live[p] = {dev, cls};
  *out = (T*)p;
  return cudaSuccess;
}
void dev_free(void* p) {
  if (!p) return;
  DevCache& C = dev_cache();
  std::lock_guard<std::mutex> lk(C.mu);
  auto it = C.live.find(p);
  if (it == C.live.end()) { cudaFree(p); return; }
  const std::pair<int, size_t> key = it->second;
  C.live.erase(it);
  if (C.cached_bytes + key.second > kDevCacheMax) { cudaFree(p); return; }
  C.free_blocks.insert({key, p});
  C.cached_bytes += key.second;
}
} // namespace

struct DeviceGuard { // switch to the camera's device for the duration of a call
  int prev = -1;
  bool ok = true;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
    if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
  }
  ~DeviceGuard() {
    int cur = -1;
    if (prev >= 0 && cudaGetDevice(&cur) == cudaSuccess && cur != prev) cudaSetDevice(prev);
  }
};

struct rt_camera {
  std::shared_ptr<HostScene> hs; // compiled scene; shared by the cameras of an rt_multi (one per GPU)
  DevScene ds{};
  rt_render_opts opts{};
  int device = 0;
  int integrator = RT_INTEGRATOR_MEGAKERNEL;
  cudaStream_t stream = nullptr;
  bool owns_stream = false; // rt_multi gives each device its own stream
  double build_ms = 0;
  // scene buffers
  std::vector<void*> allocs;
  // image-sized scratch (lazily allocated, reused across renders)
  uint8_t* d_rgb8 = nullptr;
  float* d_linear = nullptr;
  float* d_moments = nullptr;
  int32_t* d_ids = nullptr;
  float* d_t = nullptr;
  float* d_normal = nullptr;
  uint8_t* d_front = nullptr;
  float* d_falb = nullptr;   // feature buffers (rt_camera_render_features)
  float* d_fnrm = nullptr;
  float* d_fdepth = nullptr;
  float* d_dn = nullptr;     // denoiser scratch: dn_floats_per_pixel floats per pixel
  float* d_dnout = nullptr;  // progressive denoised renders: the filtered [H][W][3] image (d_linear keeps the noisy colour)
  unsigned long long* d_stats = nullptr;
  // work queue of the render kernel: [0] = next item, [1..] = finished chunks per tile
  int* d_queue = nullptr;
  size_t queue_ints = 0;
  unsigned long long* d_scratch = nullptr; // fixed-point radiance sums [H][W][4]
  PixState* d_pixstate = nullptr;          // progressive renders of the pixel-stream kernels: PixelStats between passes
  AdRecord* d_adrec = nullptr;             // k_render_adaptive: per-warp sample records of the batch in flight
  size_t adrec_elems = 0;
  size_t scratch_elems = 0;
  int sms = 0;
  int chunks = 1;
  WfHost wf{};          // wavefront integrator: path pool + queues (allocated on first use)
  bool wf_ready = false;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
};

template <class T>
static rt_status upload(rt_camera* c, const std::vector<T>& v, const T** out) {
  *out = nullptr;
  if (v.empty()) return RT_OK;
  void* p = nullptr;
  CU(dev_alloc(&p, v.size() * sizeof(T)));
  c->allocs.push_back(p);
  CU(cudaMemcpy(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
  *out = (const T*)p;
  return RT_OK;
}

// Path pool and queues of the wavefront integrator; also the clean-up of a pool whose allocation failed half way
// (every pointer is null until allocated: rt_camera value-initialises WfHost).
static void wf_release(rt_camera* c) {
  WfBuffers& W = c->wf.W;
  dev_free(W.ray_o); dev_free(W.ray_d); dev_free(W.tp); dev_free(W.rad); dev_free(W.pix);
  for (int k = 0; k < WF_TAGS; ++k) dev_free(W.q_shade[k]);
  dev_free(c->wf.q_extend[0]); dev_free(c->wf.q_extend[1]); dev_free(c->wf.q_free[0]); dev_free(c->wf.q_free[1]);
  dev_free(W.counters); dev_free(c->wf.owned_blocks);
  if (c->wf.h_counters) cudaFreeHost(c->wf.h_counters);
  std::memset(&c->wf, 0, sizeof(c->wf));
  c->wf_ready = false;
}

static void free_camera(rt_camera* c) {
  if (!c) return;
  DeviceGuard g(c->device);
  cudaStreamSynchronize(c->stream); // the blocks go back to the cache: nothing of this camera may still be in flight
  for (void* p : c->allocs) dev_free(p);
  dev_free(c->d_rgb8); dev_free(c->d_linear); dev_free(c->d_moments); dev_free(c->d_ids);
  dev_free(c->d_t); dev_free(c->d_normal); dev_free(c->d_front); dev_free(c->d_falb); dev_free(c->d_fnrm); dev_free(c->d_fdepth);
  dev_free(c->d_dn); dev_free(c->d_dnout); dev_free(c->d_stats); dev_free(c->d_queue); dev_free(c->d_scratch); dev_free(c->d_pixstate); dev_free(c->d_adrec);
  wf_release(c);
  if (c->ev0) cudaEventDestroy(c->ev0);
  if (c->ev1) cudaEventDestroy(c->ev1);
  if (c->owns_stream && c->stream) cudaStreamDestroy(c->stream);
  delete c;
}

static rt_status clip_region(const rt_camera* c, const rt_region* r, RenderParams& P) {
  const int W = c->hs->image_width, H = c->hs->image_height;
  rt_region full{0, 0, W, H};
  if (!r) r = &full;
  if (r->x < 0 || r->y < 0 || r->width < 0 || r->height < 0) return fail(RT_ERR_INVALID_ARGUMENT, "negative region");
  std::memset(&P, 0, sizeof(P));
  P.x0 = r->x < W ? r->x : W;
  P.y0 = r->y < H ? r->y : H;
  long long x1 = (long long)r->x + r->width, y1 = (long long)r->y + r->height; // camera.ts:390-391
  P.x1 = (int)(x1 < W ? x1 : W);
  P.y1 = (int)(y1 < H ? y1 : H);
  P.part_index = c->opts.part_index;
  P.part_count = c->opts.part_count;
  return RT_OK;
}

static const unsigned long long kStatsInit[kStatCount] = {0, 0, 0, 0, 0x7fffffffull, 0, 0x7fffffffull, 0, 0, 0};

// Raw counters -> rt_stats without timing or launches.  unpack_stats(kStatsInit) is the identity of merge_stats.
static rt_stats unpack_stats(const unsigned long long* raw) {
  rt_stats s;
  std::memset(&s, 0, sizeof(s));
  s.pixels = raw[kStatPixels];
  s.samples_total = raw[kStatSamples];
  s.bounces_total = raw[kStatBounces];
  s.rays = raw[kStatRays];
  s.samples_min = (int32_t)raw[kStatSamplesMin];
  s.samples_max = (int32_t)raw[kStatSamplesMax];
  s.bounces_min = (int32_t)raw[kStatBouncesMin];
  s.bounces_max = (int32_t)raw[kStatBouncesMax];
  s.node_visits = raw[kStatNodeVisits];
  s.prim_tests = raw[kStatPrimTests];
  return s;
}

// RenderStats.merge: work and kernel launches add up, extremes combine.  device_ms is each caller's own rule.
static void merge_stats(rt_stats* total, const rt_stats& s) {
  total->pixels += s.pixels; total->samples_total += s.samples_total; total->bounces_total += s.bounces_total; total->rays += s.rays;
  total->node_visits += s.node_visits; total->prim_tests += s.prim_tests;
  total->samples_min = std::min(total->samples_min, s.samples_min); total->samples_max = std::max(total->samples_max, s.samples_max);
  total->bounces_min = std::min(total->bounces_min, s.bounces_min); total->bounces_max = std::max(total->bounces_max, s.bounces_max);
  total->kernel_launches += s.kernel_launches;
}

// Copy the region of P out of (or into) an [H][W] image of `k` bytes per pixel: `dst` and `src` have that same layout.
static cudaError_t copy_region(void* dst, const void* src, size_t k, const RenderParams& P, int W, cudaMemcpyKind kind, cudaStream_t st) {
  if (P.x1 <= P.x0 || P.y1 <= P.y0) return cudaSuccess;
  const size_t off = ((size_t)P.y0 * W + P.x0) * k, pitch = (size_t)W * k;
  return cudaMemcpy2DAsync((char*)dst + off, pitch, (const char*)src + off, pitch, (size_t)(P.x1 - P.x0) * k, P.y1 - P.y0, kind, st);
}

// Grow-only device buffer of the camera: at least `need` elements.  Work in flight may still use the old block, so the
// camera's stream is drained before it goes back to the cache.
template <class T, class N>
static rt_status grow(rt_camera* c, T*& buf, N& capacity, size_t need) {
  if (need <= (size_t)capacity) return RT_OK;
  CU(cudaStreamSynchronize(c->stream));
  dev_free(buf);
  buf = nullptr;
  capacity = 0;
  CU(dev_alloc(&buf, need * sizeof(T)));
  capacity = (N)need;
  return RT_OK;
}

extern "C" {

const char* rt_last_error(void) { return g_err.c_str(); }
int32_t rt_abi_version(void) { return RT_B200_ABI_VERSION; }
int32_t rt_counts_events(void) {
#ifdef RT_COUNT_EVENTS
  return 1;
#else
  return 0;
#endif
}
int32_t rt_block_owner(int32_t x, int32_t y, int32_t image_width, int32_t part_count) {
  if (part_count <= 1 || x < 0 || y < 0 || image_width <= 0) return 0;
  return block_owner(x / 8, y / 4, (image_width + 7) / 8, part_count);
}
uint64_t rt_trim_device_cache(void) {
  DevCache& C = dev_cache();
  std::lock_guard<std::mutex> lk(C.mu);
  return (uint64_t)dev_trim_locked(C);
}

// Host-only: compile the scene like rt_camera_create and check the structure the kernels will walk.
rt_status rt_scene_validate(const rt_scene_desc* scene, const rt_render_opts* opts, rt_scene_report* rep) {
  RT_GUARD_BEGIN
  if (!scene || !opts || !rep) return fail(RT_ERR_INVALID_ARGUMENT, "null argument");
  HostScene hs;
  std::string err;
  rt_status st = compile_scene(scene, opts, hs, err);
  if (st != RT_OK) return fail(st, err);
  std::memset(rep, 0, sizeof(*rep));
  const int n = (int)hs.p0.size();
  rep->bvh_kind = hs.bvh_kind;
  rep->n_slots = n;
  rep->n_prefix = hs.n_unbounded;
  rep->n_node_slots = (int)hs.nodes.size();
  rep->max_depth = hs.max_depth;
  rep->n_lights = (int)hs.lights.size();
  int errors = 0;
  // every object sits in exactly one slot
  std::vector<int> seen_obj(hs.n_objects, 0), seen_slot(n, 0);
  if (n != hs.n_objects) ++errors;
  for (int s = 0; s < n; ++s) {
    const int obj = hs.slot_info[s].y & 0x3fffffff;
    if (obj < 0 || obj >= hs.n_objects || seen_obj[obj]++) ++errors;
  }
  for (int s = 0; s < hs.n_unbounded && s < n; ++s) seen_slot[s]++;
  struct B { float mn[3], mx[3]; };
  auto inside = [](const B& in, const B& out) { // with the slack of the FP32 roundings that made the boxes
    for (int a = 0; a < 3; ++a) {
      const float tol = 1e-5f * std::max(1.f, std::max(std::fabs(in.mn[a]), std::fabs(in.mx[a])));
      if (in.mn[a] < out.mn[a] - tol || in.mx[a] > out.mx[a] + tol) return false;
    }
    return true;
  };
  auto inverted = [](const B& b) { return b.mn[0] > b.mx[0] || b.mn[1] > b.mx[1] || b.mn[2] > b.mx[2]; };
  auto prim_box = [&](int s, B& b) { // false: unbounded (plane)
    const ExactPrim& e = hs.exact[s];
    if (e.type == OBJ_SPHERE) {
      const float r = std::fabs((float)e.r);
      for (int a = 0; a < 3; ++a) { b.mn[a] = e.q[a] - r; b.mx[a] = e.q[a] + r; }
      return true;
    }
    if (e.type == OBJ_QUAD) {
      for (int a = 0; a < 3; ++a) {
        const float c[4] = {e.q[a], e.q[a] + e.u[a], e.q[a] + e.v[a], e.q[a] + e.u[a] + e.v[a]};
        b.mn[a] = std::min(std::min(c[0], c[1]), std::min(c[2], c[3]));
        b.mx[a] = std::max(std::max(c[0], c[1]), std::max(c[2], c[3]));
      }
      return true;
    }
    return false;
  };
  auto check_leaf = [&](int ref, const B& box) {
    const int v = ~ref, first = v >> 6, count = ((v >> 4) & 3) + 1, mask = v & 15;
    ++rep->n_leaves;
    rep->max_leaf_size = std::max(rep->max_leaf_size, count);
    for (int k = 0; k < count; ++k) {
      const int s = first + k;
      if (s < 0 || s >= n) { ++errors; continue; }
      seen_slot[s]++;
      if (((mask >> k) & 1) != (hs.exact[s].type != OBJ_SPHERE)) ++errors; // planar mask matches the slot's type
      B pb;
      if (prim_box(s, pb) && !inverted(box) && !(hs.exact[s].r < 0) && !inside(pb, box)) ++errors;
    }
  };
  if (hs.bvh_kind == BVH_SAH && !hs.nodes.empty()) {
    const WideNode* W = reinterpret_cast<const WideNode*>(hs.nodes.data());
    const int nw = (int)hs.nodes.size() / 2;
    std::vector<int> visited(nw, 0);
    std::vector<std::pair<int, B>> todo; // (wide node, the box its parent holds for it)
    B all;
    for (int a = 0; a < 3; ++a) { all.mn[a] = -INFINITY; all.mx[a] = INFINITY; }
    todo.push_back({0, all});
    while (!todo.empty()) {
      const int idx = todo.back().first;
      const B pbox = todo.back().second;
      todo.pop_back();
      if (idx < 0 || idx >= nw || visited[idx]++) { ++errors; continue; }
      for (int k = 0; k < 4; ++k) {
        const int ref = W[idx].ref[k];
        if (ref == kEmptyRef) continue;
        B cb;
        for (int a = 0; a < 3; ++a) { cb.mn[a] = W[idx].box[k][a] - W[idx].box[k][3 + a]; cb.mx[a] = W[idx].box[k][a] + W[idx].box[k][3 + a]; } // (centre, half-extent)
        if (!inside(cb, pbox)) ++errors;
        if (ref < 0) check_leaf(ref, cb);
        else todo.push_back({ref, cb});
      }
    }
    for (int v : visited) if (v != 1) ++errors;
  } else if (hs.bvh_kind == BVH_REFERENCE && !hs.nodes.empty()) {
    std::vector<int> visited(hs.nodes.size(), 0);
    std::vector<int> todo{0};
    while (!todo.empty()) {
      const int idx = todo.back();
      todo.pop_back();
      if (idx < 0 || idx >= (int)hs.nodes.size() || visited[idx]++) { ++errors; continue; }
      const Node& nd = hs.nodes[idx];
      const int refs[2] = {nd.left, nd.right};
      for (int k = 0; k < 2; ++k) {
        if (refs[k] == kEmptyRef) continue;
        B cb;
        for (int a = 0; a < 3; ++a) { cb.mn[a] = k ? nd.rmin[a] : nd.lmin[a]; cb.mx[a] = k ? nd.rmax[a] : nd.lmax[a]; }
        if (refs[k] < 0) check_leaf(refs[k], cb);
        else todo.push_back(refs[k]);
      }
    }
  }
  for (int s = 0; s < n; ++s) if (seen_slot[s] != 1) ++errors;
  rep->errors = errors;
  return RT_OK;
  RT_GUARD_END
}
int32_t rt_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

// Upload a compiled scene to `opts->device` and make the camera (everything of rt_camera_create after the scene compiler).
static rt_status camera_from_host(std::shared_ptr<HostScene> hs, const rt_render_opts* opts, rt_camera** out, double compile_ms) {
  *out = nullptr;
  rt_camera* c = nullptr;
  try {
  auto t0 = std::chrono::steady_clock::now();
  c = new rt_camera();
  c->hs = hs;
  if (opts->part_count > 1 && (opts->part_index < 0 || opts->part_index >= opts->part_count)) {
    delete c;
    return fail(RT_ERR_INVALID_ARGUMENT, "part_index out of range");
  }
  c->opts = *opts;
  c->integrator = opts->integrator == RT_INTEGRATOR_WAVEFRONT || opts->integrator == RT_INTEGRATOR_SORTED ? opts->integrator
                                                                                                          : RT_INTEGRATOR_MEGAKERNEL;
  if (opts->integrator == RT_INTEGRATOR_AUTO) {
    // composite materials (Mixed / Layered) make neighbouring lanes run different shading code: sorting the
    // CTA's hits by material class pays there (+8 % on the 49-sphere layered/mixed scene), not on Cornell (-8 %)
    for (const I4& m : c->hs->matB)
      if (m.x == MAT_MIXED || m.x == MAT_LAYERED) { c->integrator = RT_INTEGRATOR_SORTED; break; }
  }
  int ndev = rt_device_count();
  if (ndev <= 0) { delete c; return fail(RT_ERR_NO_DEVICE, "no CUDA device visible; this library has no CPU fallback"); }
  int dev = opts->device;
  if (dev < 0) { if (cudaGetDevice(&dev) != cudaSuccess) dev = 0; }
  if (dev >= ndev) { delete c; return fail(RT_ERR_INVALID_ARGUMENT, "device ordinal out of range"); }
  c->device = dev;
  DeviceGuard g(dev);
  if (!g.ok) { delete c; return fail(RT_ERR_CUDA, "cudaSetDevice failed"); }
  DevScene& d = c->ds;
  d.cam = c->hs->cam;
  const Node* nodes = nullptr;
#define UP(vec, ptr)                                   \
  do {                                                 \
    rt_status s_ = upload(c, vec, ptr);                \
    if (s_ != RT_OK) { free_camera(c); return s_; }    \
  } while (0)
  UP(c->hs->nodes, &nodes);
  d.nodes = reinterpret_cast<const F4*>(nodes);
  UP(c->hs->p0, &d.p0); UP(c->hs->p1, &d.p1); UP(c->hs->p2, &d.p2); UP(c->hs->p3, &d.p3);
  UP(c->hs->slot_info, &d.slot_info); UP(c->hs->exact, &d.exact);
  UP(c->hs->matA, &d.matA); UP(c->hs->matB, &d.matB); UP(c->hs->matE, &d.matE);
  UP(c->hs->lights, &d.lights); UP(c->hs->matF, &d.matF);
#undef UP
  d.n_nodes = (int)c->hs->nodes.size();
  d.n_slots = (int)c->hs->p0.size();
  d.n_unbounded = c->hs->n_unbounded;
  d.n_mats = (int)c->hs->matA.size();
  d.n_lights = (int)c->hs->lights.size();
  d.bvh_kind = c->hs->bvh_kind;
  d.planar_any = c->hs->planar_any;
  for (int k = 0; k < 6; ++k) d.list_n[k] = c->hs->list_n[k];
  d.sph_cmax = c->hs->sph_cmax;
  d.sph_r2max = c->hs->sph_r2max;
  d.seed_lo = (uint32_t)opts->seed;
  d.seed_hi = (uint32_t)(opts->seed >> 32);
  if (dev_alloc(&c->d_stats, sizeof(kStatsInit)) != cudaSuccess || cudaEventCreate(&c->ev0) != cudaSuccess ||
      cudaEventCreate(&c->ev1) != cudaSuccess) {
    std::string m = cudaGetErrorString(cudaGetLastError());
    free_camera(c);
    return fail(RT_ERR_CUDA, "allocating stats/events: " + m);
  }
  cudaDeviceGetAttribute(&c->sms, cudaDevAttrMultiProcessorCount, dev);
  {
    c->chunks = 0; // 0 = chosen per launch (enqueue_render)
    if (const char* e = getenv("RT_B200_CHUNKS")) { // development override
      int v = atoi(e);
      if (v >= 1 && v <= 64) c->chunks = v;
    }
  }
  const double upload_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  c->build_ms = compile_ms + upload_ms;
  if (getenv("RT_B200_BUILD_TRACE")) std::fprintf(stderr, "[rt_b200 build] %-12s %8.2f ms (device %d)\n[rt_b200 build] %-12s %8.2f ms\n", "upload", upload_ms, dev, "compile", compile_ms);
  *out = c;
  return RT_OK;
  } catch (const std::exception& e) { // std::bad_alloc on a huge scene: nothing half-built stays behind
    if (c) free_camera(c);
    return fail(RT_ERR_INVALID_ARGUMENT, std::string("rt_camera_create: ") + e.what());
  }
}

// validate + compile: scene errors are reported even on a box without a GPU, exactly like the reference throws
// before rendering anything
static rt_status compile_shared(const rt_scene_desc* scene, const rt_render_opts* opts, std::shared_ptr<HostScene>& hs, double& ms) {
  try {
    auto t0 = std::chrono::steady_clock::now();
    hs = std::make_shared<HostScene>();
    std::string err;
    rt_status st = compile_scene(scene, opts, *hs, err);
    ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (st != RT_OK) return fail(st, err);
    return RT_OK;
  } catch (const std::exception& e) {
    return fail(RT_ERR_INVALID_ARGUMENT, std::string("scene compiler: ") + e.what());
  }
}

rt_status rt_camera_create(const rt_scene_desc* scene, const rt_render_opts* opts, rt_camera** out) {
  if (!scene || !opts || !out) return fail(RT_ERR_INVALID_ARGUMENT, "null argument");
  *out = nullptr;
  std::shared_ptr<HostScene> hs;
  double ms = 0;
  rt_status st = compile_shared(scene, opts, hs, ms);
  if (st != RT_OK) return st;
  return camera_from_host(hs, opts, out, ms);
}

rt_status rt_camera_destroy(rt_camera* cam) {
  free_camera(cam);
  return RT_OK;
}

rt_status rt_camera_get_info(const rt_camera* c, rt_camera_info* o) {
  if (!c || !o) return fail(RT_ERR_INVALID_ARGUMENT, "null argument");
  std::memset(o, 0, sizeof(*o));
  const DevCamera& k = c->hs->cam;
  o->image_width = c->hs->image_width; o->image_height = c->hs->image_height; o->channels = 3;
  o->n_objects = c->hs->n_objects; o->n_lights = (int)c->hs->lights.size(); o->n_bvh_nodes = (int)c->hs->nodes.size();
  o->bvh_kind = c->hs->bvh_kind; o->integrator_kind = c->integrator;
  std::memcpy(o->center, k.center, 12); std::memcpy(o->pixel00_loc, k.p00, 12);
  std::memcpy(o->pixel_delta_u, k.du, 12); std::memcpy(o->pixel_delta_v, k.dv, 12);
  std::memcpy(o->u, c->hs->cam_u, 12); std::memcpy(o->v, c->hs->cam_v, 12); std::memcpy(o->w, c->hs->cam_w, 12);
  std::memcpy(o->defocus_disk_u, k.ddu, 12); std::memcpy(o->defocus_disk_v, k.ddv, 12);
  o->focus_distance = c->hs->focus_distance;
  o->use_adaptive_sampling = k.adaptive;
  o->device = c->device;
  o->build_ms = c->build_ms;
  return RT_OK;
}

rt_status rt_camera_set_stream(rt_camera* c, void* s) {
  if (!c) return fail(RT_ERR_INVALID_ARGUMENT, "null camera");
  if (c->stream != (cudaStream_t)s) {
    // work already enqueued on the old stream uses this camera's buffers; destroy/realloc only wait for the current one
    DeviceGuard g(c->device);
    CU(cudaStreamSynchronize(c->stream));
  }
  c->stream = (cudaStream_t)s;
  return RT_OK;
}

// Wavefront integrator: allocate the path pool once, list the 8x4 blocks this GPU owns in the region.
static rt_status wf_prepare(rt_camera* c, const RenderParams& P) {
  WfHost& H = c->wf;
  const int blocks_x = P.tiles_x * 2, blocks_y = P.tiles_y * 4;
  std::vector<int> owned;
  owned.reserve((size_t)blocks_x * blocks_y);
  for (int by = 0; by < blocks_y; ++by)
    for (int bx = 0; bx < blocks_x; ++bx) {
      if (P.part_count > 1 && block_owner((P.x0 / 16) * 2 + bx, (P.y0 / 16) * 4 + by, (c->hs->image_width + 7) / 8, P.part_count) != P.part_index) continue;
      const int px0 = (P.x0 / 16) * 16 + bx * 8, py0 = (P.y0 / 16) * 16 + by * 4;
      if (px0 >= P.x1 || py0 >= P.y1 || px0 + 8 <= P.x0 || py0 + 4 <= P.y0) continue;
      owned.push_back(by * blocks_x + bx);
    }
  if (!c->wf_ready) {
    std::memset(&H, 0, sizeof(H));
    static const int slots_env = getenv("RT_B200_WF_SLOTS") ? atoi(getenv("RT_B200_WF_SLOTS")) : 0;
    const int n = slots_env > 0 ? slots_env : (1 << 22); // 4 Mi paths in flight, 80 B each
    WfBuffers& W = H.W;
    W.n_slots = n;
    auto alloc_pool = [&]() -> cudaError_t {
      cudaError_t e;
      if ((e = dev_alloc(&W.ray_o, (size_t)n * sizeof(F4))) != cudaSuccess) return e;
      if ((e = dev_alloc(&W.ray_d, (size_t)n * sizeof(F4))) != cudaSuccess) return e;
      if ((e = dev_alloc(&W.tp, (size_t)n * sizeof(F4))) != cudaSuccess) return e;
      if ((e = dev_alloc(&W.rad, (size_t)n * sizeof(F4))) != cudaSuccess) return e;
      if ((e = dev_alloc(&W.pix, (size_t)n * sizeof(U2))) != cudaSuccess) return e;
      for (int k = 0; k < WF_TAGS; ++k)
        if ((e = dev_alloc(&W.q_shade[k], (size_t)n * sizeof(int))) != cudaSuccess) return e;
      for (int k = 0; k < 2; ++k) {
        if ((e = dev_alloc(&H.q_extend[k], (size_t)n * sizeof(int))) != cudaSuccess) return e;
        if ((e = dev_alloc(&H.q_free[k], (size_t)n * sizeof(int))) != cudaSuccess) return e;
      }
      if ((e = dev_alloc(&W.counters, WFC_COUNT * sizeof(int))) != cudaSuccess) return e;
      return cudaMallocHost(&H.h_counters, WFC_COUNT * sizeof(int));
    };
    const cudaError_t pe = alloc_pool();
    if (pe != cudaSuccess) { // nothing half-built stays behind: the next render may try again
      cudaGetLastError();
      wf_release(c);
      return fail(RT_ERR_CUDA, std::string("wavefront path pool: ") + cudaGetErrorString(pe));
    }
    c->wf_ready = true;
  }
  rt_status st = grow(c, H.owned_blocks, H.owned_capacity, owned.size());
  if (st != RT_OK) return st;
  if (!owned.empty()) { // on the camera's stream (a user stream may be non-blocking: the legacy default stream does not order with it)
    CU(cudaMemcpyAsync(H.owned_blocks, owned.data(), owned.size() * sizeof(int), cudaMemcpyHostToDevice, c->stream));
    CU(cudaStreamSynchronize(c->stream)); // `owned` is a pageable local
  }
  H.n_owned = (int)owned.size();
  H.blocks_x = blocks_x;
  H.W.total_pairs = (unsigned long long)owned.size() * 32ull * (unsigned long long)std::max(0, c->hs->cam.samples);
  return RT_OK;
}

// One pass of a progressive render (rt_camera_render_progressive); null = the whole render in one launch.
struct ProgPass {
  int s0, s1;   // fixed spp: samples [s0, s1) of every pixel; pixel stream: s0 = the previous cap, s1 = this pass's cap
  bool first;   // first pass: the accumulators start from zero
};
// enqueue: stats init, render kernel, optional stats finalisation.  No synchronisation.
static rt_status enqueue_render(rt_camera* c, RenderParams& P, rt_stats* stats_dev, int* launches, const ProgPass* pass = nullptr) {
  CU(cudaMemcpyAsync(c->d_stats, kStatsInit, sizeof(kStatsInit), cudaMemcpyHostToDevice, c->stream));
  P.stats = c->d_stats;
  *launches = 0;
  if (P.x1 > P.x0 && P.y1 > P.y0) {
    render_tile_grid(P, &P.tiles_x, &P.tiles_y);
    if (P.part_count > 1) { // runs of part_count consecutive blocks (whole-image numbering) that overlap the region's block rows
      const long long bpr = (c->hs->image_width + 7) / 8;
      const long long i0 = (long long)(P.y0 / 4) * bpr, i1 = (long long)((P.y1 - 1) / 4 + 1) * bpr;
      P.run0 = (int)(i0 / P.part_count);
      P.n_runs = (int)((i1 - 1) / P.part_count) - P.run0 + 1;
    }
    if (render_needs_full(c->ds, P)) P.chunks = 1;
    else if (c->chunks > 0) P.chunks = std::min(c->chunks, std::max(1, c->hs->cam.samples)); // never an empty chunk (k_render_sorted skips them)
    else {
      // Sample chunks per pixel: enough (8x4 block, chunk) warp items that the blocks this GPU owns
      // keep it busy for >= 20 rounds of resident warps (3 CTAs x 8 warps per SM), so the tail of the render stays ~1/40 of it
      // whether the GPU renders the whole image or 1/8 of it.  Sums are exact fixed point, so the
      // image does not depend on this choice.  A chunk stays <= 2048 samples (limb accumulators).
      const long long owned = std::max(1LL, (long long)P.tiles_x * P.tiles_y * 8 / std::max(1, P.part_count));
      const long long target = 20LL * c->sms * 3 * 8; // (Cornell 1024^2 @1024, one GPU: chunks 1 / 2 / 3 / 4 / 8 = 114.8 / 108.5 / 107.7 / 108.0 / 109.5 ms)
      long long k = (target + owned - 1) / owned;
      k = std::min<long long>(k, std::max(1, c->hs->cam.samples / 16));
      P.chunks = (int)std::min<long long>(std::max<long long>(k, 1), 64);
    }
    if (P.chunks > 1 || !render_needs_full(c->ds, P)) P.chunks = std::max(P.chunks, (c->hs->cam.samples + 2047) / 2048);
    if (pass) {
      if (render_needs_full(c->ds, P)) { // pixel stream: PixelStats wait in d_pixstate between the passes
        P.s0 = pass->s0;
        P.pass_cap = pass->s1;
        if (!c->d_pixstate) CU(dev_alloc(&c->d_pixstate, (size_t)c->hs->image_width * c->hs->image_height * sizeof(PixState)));
        P.pixstate = c->d_pixstate;
      } else { // fixed spp: a window of every pixel's samples on top of the fixed-point sums of the earlier passes
        P.s0 = pass->s0;
        P.s_cnt = pass->s1 - pass->s0;
        P.div_samples = pass->s1;
        P.keep_accum = 1;
        P.chunks = std::max(1, std::min(P.chunks, P.s_cnt));
      }
    }
    {
      // plain adaptive renders: batch-parallel kernel (k_render_adaptive); PixelStats between batches reuse the pass buffer
      int warps = 0;
      const int gb = pass ? 0 : render_adaptive_blocks(c->ds, P, c->sms, &warps);
      if (gb > 0) {
        if (!c->d_pixstate) CU(dev_alloc(&c->d_pixstate, (size_t)c->hs->image_width * c->hs->image_height * sizeof(PixState)));
        rt_status st = grow(c, c->d_adrec, c->adrec_elems, (size_t)warps * gb * 32 * (size_t)c->hs->cam.a_batch);
        if (st != RT_OK) return st;
        P.adstate = c->d_pixstate;
        P.adrec = c->d_adrec;
        P.ad_blocks = gb;
      }
    }
    const size_t need_q = 1 + std::max((size_t)P.tiles_x * P.tiles_y * 8, (size_t)P.n_runs); // queue head + one completion counter per 8x4 block / run
    rt_status st = grow(c, c->d_queue, c->queue_ints, need_q);
    if (st != RT_OK) return st;
    // fixed-point radiance sums [H][W][4] u64, only when a pixel's samples are split over CTAs
    const bool wavefront = c->integrator == RT_INTEGRATOR_WAVEFRONT && !render_needs_full(c->ds, P) && !pass; // passes: megakernel layouts only
    const size_t need_s = (P.chunks > 1 || wavefront || P.keep_accum) ? (size_t)4 * c->hs->image_width * c->hs->image_height : 0;
    if ((st = grow(c, c->d_scratch, c->scratch_elems, need_s)) != RT_OK) return st;
    CU(cudaMemsetAsync(c->d_queue, 0, need_q * sizeof(int), c->stream));
    if (need_s && !(pass && !pass->first)) {
      // only the rows of the region are touched
      const size_t row = (size_t)4 * c->hs->image_width;
      CU(cudaMemsetAsync(c->d_scratch + row * P.y0, 0, row * (size_t)(P.y1 - P.y0) * sizeof(unsigned long long), c->stream));
    }
    {
      static const int trav_env = getenv("RT_B200_TRAV_MIN") ? atoi(getenv("RT_B200_TRAV_MIN")) : -1; // development override
      static const int burst_env = getenv("RT_B200_TRAV_BURST") ? atoi(getenv("RT_B200_TRAV_BURST")) : -1; // development override
      // swept on the 100k-sphere scene with the 4-wide tree (8 spp, ms): burst 4: min 4/8/10/12/16/20 = 118/116/116/118/124/133;
      // burst 6: 123/119/119/120/124/131; burst 2 and 8 are worse at every setting.  After the pair queue moved behind the shading
      // (k_render_trav) and the sampler change: burst 3/4/5/6/8 at min 8: 86.8/86.9/87.8/90.7/93.4, at min 12: 86.6/86.4/87.1/89.9/92.3
      // (profiles/r02c_trav_burst_sweep.log) — flat around the settings below
      P.trav_min_lanes = trav_env >= 0 ? trav_env : 8;
      P.trav_burst = burst_env >= 1 ? burst_env : 4;
    }
    P.sorted = c->integrator == RT_INTEGRATOR_SORTED;
    P.queue = c->d_queue;
    P.tile_done = c->d_queue + 1;
    P.accum = c->d_scratch;
    if (wavefront) {
      rt_status ws = wf_prepare(c, P);
      if (ws != RT_OK) return ws;
      CU(launch_render_wavefront(c->ds, P, c->wf, c->sms, c->stream, launches));
    } else {
      CU(launch_render_mega(c->ds, P, c->sms, c->stream));
      *launches = 1;
    }
  }
  if (stats_dev) {
    CU(launch_finalize_stats(c->d_stats, stats_dev, *launches + 1, c->stream));
    *launches += 1;
  }
  return RT_OK;
}

rt_status rt_camera_render_region_device(rt_camera* c, const rt_region* region, uint8_t* rgb8_dev, float* linear_dev,
                                         float* moments_dev, rt_stats* stats_dev) {
  RT_GUARD_BEGIN
  if (!c) return fail(RT_ERR_INVALID_ARGUMENT, "null camera");
  DeviceGuard g(c->device);
  RenderParams P;
  rt_status st = clip_region(c, region, P);
  if (st != RT_OK) return st;
  P.rgb8 = rgb8_dev; P.linear = linear_dev; P.moments = moments_dev;
  int launches = 0;
  return enqueue_render(c, P, stats_dev, &launches);
  RT_GUARD_END
}

// ev0, enqueue_render, the optional step `post` (more work on the camera's stream, its launches counted), `end`, then the
// raw counters to `raw` (kStatCount values of host memory).  No synchronisation.
static rt_status timed_render(rt_camera* c, RenderParams& P, cudaEvent_t end, unsigned long long* raw, int* launches,
                              const ProgPass* pass = nullptr, const std::function<rt_status(int*)>& post = {}) {
  CU(cudaEventRecord(c->ev0, c->stream));
  rt_status st = enqueue_render(c, P, nullptr, launches, pass);
  if (st != RT_OK) return st;
  if (post) {
    int l = 0;
    if ((st = post(&l)) != RT_OK) return st;
    *launches += l;
  }
  CU(cudaEventRecord(end, c->stream));
  CU(cudaMemcpyAsync(raw, c->d_stats, sizeof(unsigned long long) * kStatCount, cudaMemcpyDeviceToHost, c->stream));
  return RT_OK;
}

static rt_status denoise_band(rt_camera* c, const RenderParams& P, int b0, int b1, const DenoiseParams& opts, const float* color,
                              const float* moments, float* out, uint8_t* rgb8, bool poison, int* launches);
static rt_status denoise_features(rt_camera* c, const RenderParams& P, int b0, int b1, int iterations, bool poison, int* launches);
static rt_status denoise_filter(rt_camera* c, const RenderParams& P, int b0, int b1, const DenoiseParams& opts, const float* color,
                                const float* moments, float* out, uint8_t* rgb8, int* launches);

// Partitioned camera: copy the 8x4 blocks it owns in the region of P from its rgb8 / linear / moments buffers (each
// optional) into the caller's [H][W] arrays, through host staging of the region's rows.  Synchronises the camera's stream.
static rt_status copy_owned_blocks(rt_camera* c, const RenderParams& P, uint8_t* rgb8, float* linear, float* moments) {
  const int W = c->hs->image_width, rh = P.y1 - P.y0;
  std::vector<uint8_t> hr;
  std::vector<float> hl, hm;
  const size_t row0 = (size_t)P.y0 * W;
  if (rgb8) { hr.resize((size_t)rh * W * 3); CU(cudaMemcpyAsync(hr.data(), c->d_rgb8 + row0 * 3, hr.size(), cudaMemcpyDeviceToHost, c->stream)); }
  if (linear) { hl.resize((size_t)rh * W * 3); CU(cudaMemcpyAsync(hl.data(), c->d_linear + row0 * 3, hl.size() * 4, cudaMemcpyDeviceToHost, c->stream)); }
  if (moments) { hm.resize((size_t)rh * W * 8); CU(cudaMemcpyAsync(hm.data(), c->d_moments + row0 * 8, hm.size() * 4, cudaMemcpyDeviceToHost, c->stream)); }
  CU(cudaStreamSynchronize(c->stream));
  const int bpr = (W + 7) / 8;
  for (int y = P.y0; y < P.y1; ++y) {
    for (int x = P.x0; x < P.x1;) {
      const int bx = x / 8;
      const int xe = std::min(P.x1, (bx + 1) * 8);
      if (block_owner(bx, y / 4, bpr, c->opts.part_count) == c->opts.part_index) {
        const size_t dst = (size_t)y * W + x, src = (size_t)(y - P.y0) * W + x;
        const size_t n = (size_t)(xe - x);
        if (rgb8) std::memcpy(rgb8 + dst * 3, hr.data() + src * 3, n * 3);
        if (linear) std::memcpy(linear + dst * 3, hl.data() + src * 3, n * 12);
        if (moments) std::memcpy(moments + dst * 8, hm.data() + src * 8, n * 32);
      }
      x = xe;
    }
  }
  return RT_OK;
}

// Render the region and copy it to the caller's [H][W] arrays.  With `dn`, the colour and moments stay on the device and
// are filtered in place before ev1 (one band covering the region); RGB8 is written from the filtered image.  `pass`: one
// pass of a progressive render (the host-merge path of rt_multi_render_progressive*).
static rt_status render_host(rt_camera* c, const rt_region* region, uint8_t* rgb8, size_t rgb8_len, float* linear,
                             float* moments, rt_stats* stats, const DenoiseParams* dn = nullptr, const ProgPass* pass = nullptr) {
  RT_GUARD_BEGIN
  if (!c) return fail(RT_ERR_INVALID_ARGUMENT, "null camera");
  const int W = c->hs->image_width, H = c->hs->image_height;
  const size_t npx = (size_t)W * H;
  if (rgb8 && rgb8_len < npx * 3) return fail(RT_ERR_BUFFER_TOO_SMALL, "rgb8 buffer smaller than width*height*3");
  DeviceGuard g(c->device);
  RenderParams P;
  rt_status st = clip_region(c, region, P);
  if (st != RT_OK) return st;
  if (rgb8 && !c->d_rgb8) CU(dev_alloc(&c->d_rgb8, npx * 3));
  if ((linear || dn) && !c->d_linear) CU(dev_alloc(&c->d_linear, npx * 3 * sizeof(float)));
  if ((moments || dn) && !c->d_moments) CU(dev_alloc(&c->d_moments, npx * 8 * sizeof(float)));
  P.rgb8 = rgb8 && !dn ? c->d_rgb8 : nullptr;
  P.linear = linear || dn ? c->d_linear : nullptr;
  P.moments = moments || dn ? c->d_moments : nullptr;
  std::function<rt_status(int*)> denoise;
  if (dn)
    denoise = [&](int* l) { return denoise_band(c, P, P.y0, P.y1, *dn, P.linear, P.moments, P.linear, rgb8 ? c->d_rgb8 : nullptr, false, l); };
  int launches = 0;
  unsigned long long raw[kStatCount];
  if ((st = timed_render(c, P, c->ev1, raw, &launches, pass, denoise)) != RT_OK) return st;
  const bool whole_tiles = c->opts.part_count <= 1;
  const int rw = P.x1 - P.x0, rh = P.y1 - P.y0;
  if (rw > 0 && rh > 0) {
    if (whole_tiles) {
      // only the region's pixels are written (camera.ts:400-401): pitched copies of the sub-rectangle
      if (rgb8) CU(copy_region(rgb8, c->d_rgb8, 3, P, W, cudaMemcpyDeviceToHost, c->stream));
      if (linear) CU(copy_region(linear, c->d_linear, 12, P, W, cudaMemcpyDeviceToHost, c->stream));
      if (moments) CU(copy_region(moments, c->d_moments, 32, P, W, cudaMemcpyDeviceToHost, c->stream));
      CU(cudaStreamSynchronize(c->stream));
    } else {
      // partitioned render: only the blocks this part owns
      if ((st = copy_owned_blocks(c, P, rgb8, linear, moments)) != RT_OK) return st;
    }
  } else {
    CU(cudaStreamSynchronize(c->stream));
  }
  if (stats) {
    *stats = unpack_stats(raw);
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
    stats->device_ms = ms;
    stats->kernel_launches = launches;
  }
  return RT_OK;
  RT_GUARD_END
}

rt_status rt_camera_render_region(rt_camera* cam, const rt_region* region, uint8_t* rgb8, size_t rgb8_len,
                                  float* linear_rgb, rt_stats* stats) {
  return render_host(cam, region, rgb8, rgb8_len, linear_rgb, nullptr, stats);
}
rt_status rt_camera_render(rt_camera* cam, uint8_t* rgb8, size_t rgb8_len, float* linear_rgb, rt_stats* stats) {
  return render_host(cam, nullptr, rgb8, rgb8_len, linear_rgb, nullptr, stats);
}
rt_status rt_camera_render_moments(rt_camera* cam, const rt_region* region, uint8_t* rgb8, size_t rgb8_len,
                                   float* linear_rgb, float* moments, rt_stats* stats) {
  return render_host(cam, region, rgb8, rgb8_len, linear_rgb, moments, stats);
}

// The sample cap after each of the n_passes passes of a progressive render of S samples per pixel: ceil(S k / n_passes),
// rounded up to a multiple of `batch` before the last pass, which ends at S.  The pixel stream stops on batch boundaries
// only (the convergence check of camera.ts:348-368 runs there, so a pixel's decisions are those of the one-shot render):
// `batch` is aBatch for adaptive cameras, 1 otherwise.  -1 = a pass with no new samples (more passes than samples), which
// is skipped; with S = 0 only the last pass runs.
static std::vector<int> pass_caps(int S, int batch, int n_passes) {
  std::vector<int> caps((size_t)n_passes, -1);
  int prev = 0;
  for (int k = 1; k <= n_passes; ++k) {
    long long cap = ((long long)S * k + n_passes - 1) / n_passes;
    if (k < n_passes) cap = std::min<long long>(S, (cap + batch - 1) / batch * batch);
    else cap = S;
    if ((int)cap <= prev && !(S <= 0 && k == n_passes)) continue;
    caps[(size_t)k - 1] = prev = (int)cap;
  }
  return caps;
}
static std::vector<int> camera_pass_caps(const rt_camera* c, int n_passes) {
  const DevCamera& cam = c->hs->cam;
  return pass_caps(cam.samples, cam.adaptive ? std::max(1, cam.a_batch) : 1, n_passes);
}

// Fold the stats of one pass (`ms` of device time) into the running total of a progressive render: work, launches and
// device_ms add up.  The pixel stream (`stream`) counts a pixel in the pass that completes it; at fixed spp every pass
// touches every pixel, and all of them have `cap` samples now.
static void fold_pass_stats(rt_stats* total, const rt_stats& ps, double ms, bool stream, int cap) {
  const int32_t samples_min = total->samples_min;
  merge_stats(total, ps);
  total->device_ms += ms;
  if (!stream) {
    total->pixels = ps.pixels;
    total->samples_min = ps.pixels ? (int32_t)cap : samples_min;
    total->samples_max = ps.pixels ? (int32_t)cap : 0;
  }
}

// Progressive render: the same image as rt_camera_render_region, delivered in n_passes growing prefixes of the samples.
// With `dn`, every pass also renders the moments and filters the region into d_dnout (see rt_camera_render_progressive_denoised);
// `moments` (host, optional) receives them after each pass.
static rt_status progressive_host(rt_camera* c, const rt_region* region, uint8_t* rgb8, size_t rgb8_len, float* linear, float* moments,
                                  int32_t n_passes, rt_progress_fn on_pass, void* user, rt_stats* stats, const DenoiseParams* dn = nullptr) {
  RT_GUARD_BEGIN
  if (!c) return fail(RT_ERR_INVALID_ARGUMENT, "null camera");
  if (n_passes < 1) return fail(RT_ERR_INVALID_ARGUMENT, "n_passes must be >= 1");
  if (c->opts.part_count > 1) return fail(RT_ERR_UNSUPPORTED, "progressive renders are not partitioned");
  const int W = c->hs->image_width, H = c->hs->image_height;
  const size_t npx = (size_t)W * H;
  if (rgb8 && rgb8_len < npx * 3) return fail(RT_ERR_BUFFER_TOO_SMALL, "rgb8 buffer smaller than width*height*3");
  DeviceGuard g(c->device);
  RenderParams P0;
  rt_status st = clip_region(c, region, P0);
  if (st != RT_OK) return st;
  const bool with_moments = moments || dn;
  if (rgb8 && !c->d_rgb8) CU(dev_alloc(&c->d_rgb8, npx * 3));
  if ((linear || dn) && !c->d_linear) CU(dev_alloc(&c->d_linear, npx * 3 * sizeof(float)));
  if (with_moments && !c->d_moments) CU(dev_alloc(&c->d_moments, npx * 8 * sizeof(float)));
  if (dn && !c->d_dnout) CU(dev_alloc(&c->d_dnout, npx * 3 * sizeof(float)));
  const int S = c->hs->cam.samples;
  // moments run the pixel stream at fixed spp too (render_needs_full), which counts a pixel in the pass that completes it.
  // At fixed spp both rules give the same totals (no pixel completes before the last pass), so no test can tell them apart.
  const bool stream = c->hs->cam.adaptive || c->hs->cam.mode != 0 || with_moments;
  const std::vector<int> caps = camera_pass_caps(c, n_passes);
  rt_stats total = unpack_stats(kStatsInit);
  int prev = 0, passes_run = 0;
  for (int k = 1; k <= n_passes; ++k) {
    const int cap = caps[(size_t)k - 1];
    if (cap < 0) continue;
    RenderParams P = P0;
    P.rgb8 = rgb8 && !dn ? c->d_rgb8 : nullptr;
    P.linear = linear || dn ? c->d_linear : nullptr;
    P.moments = with_moments ? c->d_moments : nullptr;
    // The filter writes d_dnout, never the noisy colour in d_linear: a pixel that converged in an earlier pass is not
    // rendered again, and the next pass's filter must read its noisy colour.  The features are a function of (pixel,
    // sample) only: the first pass computes them, with the sample count of the one-shot call, for every later pass.
    std::function<rt_status(int*)> denoise;
    const bool first = passes_run == 0;
    if (dn)
      denoise = [&](int* l) {
        int lf = 0;
        if (first) {
          rt_status s = denoise_features(c, P, P.y0, P.y1, dn->iterations, false, &lf);
          if (s != RT_OK) return s;
        }
        rt_status s = denoise_filter(c, P, P.y0, P.y1, *dn, P.linear, P.moments, c->d_dnout, rgb8 ? c->d_rgb8 : nullptr, l);
        *l += lf;
        return s;
      };
    const ProgPass pass{prev, cap, first};
    int launches = 0;
    unsigned long long raw[kStatCount];
    st = timed_render(c, P, c->ev1, raw, &launches, (S > 0 && n_passes > 1) ? &pass : nullptr, denoise);
    if (st != RT_OK) return st;
    if (rgb8) CU(copy_region(rgb8, c->d_rgb8, 3, P0, W, cudaMemcpyDeviceToHost, c->stream));
    if (linear) CU(copy_region(linear, dn ? c->d_dnout : c->d_linear, 12, P0, W, cudaMemcpyDeviceToHost, c->stream));
    if (moments) CU(copy_region(moments, c->d_moments, 32, P0, W, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    rt_stats ps = unpack_stats(raw);
    ps.kernel_launches = launches;
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
    fold_pass_stats(&total, ps, ms, stream, cap);
    prev = cap;
    ++passes_run;
    if (on_pass && on_pass(user, k, n_passes, (int32_t)cap, &total) != 0) break; // the caller has seen enough
  }
  if (stats) *stats = total;
  return RT_OK;
  RT_GUARD_END
}

rt_status rt_camera_render_progressive(rt_camera* c, const rt_region* region, uint8_t* rgb8, size_t rgb8_len, float* linear, int32_t n_passes,
                                       rt_progress_fn on_pass, void* user, rt_stats* stats) {
  return progressive_host(c, region, rgb8, rgb8_len, linear, nullptr, n_passes, on_pass, user, stats);
}

rt_status rt_camera_trace_primary(rt_camera* c, const rt_region* region, int32_t* obj_id, float* t, float* normal,
                                  uint8_t* front_face) {
  RT_GUARD_BEGIN
  if (!c) return fail(RT_ERR_INVALID_ARGUMENT, "null camera");
  DeviceGuard g(c->device);
  const int W = c->hs->image_width, H = c->hs->image_height;
  const size_t npx = (size_t)W * H;
  RenderParams P;
  rt_status st = clip_region(c, region, P);
  if (st != RT_OK) return st;
  if (!c->d_ids) CU(dev_alloc(&c->d_ids, npx * 4));
  if (!c->d_t) CU(dev_alloc(&c->d_t, npx * 4));
  if (!c->d_normal) CU(dev_alloc(&c->d_normal, npx * 12));
  if (!c->d_front) CU(dev_alloc(&c->d_front, npx));
  CU(launch_trace_primary(c->ds, P, c->d_ids, c->d_t, c->d_normal, c->d_front, c->stream));
  if (obj_id) CU(copy_region(obj_id, c->d_ids, 4, P, W, cudaMemcpyDeviceToHost, c->stream));
  if (t) CU(copy_region(t, c->d_t, 4, P, W, cudaMemcpyDeviceToHost, c->stream));
  if (normal) CU(copy_region(normal, c->d_normal, 12, P, W, cudaMemcpyDeviceToHost, c->stream));
  if (front_face) CU(copy_region(front_face, c->d_front, 1, P, W, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return RT_OK;
  RT_GUARD_END
}

// ---- denoiser (rt_denoise.cuh) ----
// Scratch of the filter per pixel: two (colour, variance) ping-pong float4, the (normal, depth) float4, the depth gradient.
static const size_t kDnFloatsPerPixel = 14;
static void dn_scratch(DenoiseParams& D, float* base, size_t npx) {
  D.buf[0] = reinterpret_cast<F4*>(base);
  D.buf[1] = reinterpret_cast<F4*>(base + npx * 4);
  D.feat = reinterpret_cast<F4*>(base + npx * 8);
  D.grad = base + npx * 12;
}
// rt_denoise_opts -> filter constants (NULL = all defaults; a zero sigma = its default; iterations are taken as given)
static rt_status dn_options(const rt_denoise_opts* o, DenoiseParams& D) {
  const rt_denoise_opts defaults{5, 0.f, 0.f, 0.f};
  if (!o) o = &defaults;
  if (o->iterations < 0 || o->iterations > 8) return fail(RT_ERR_INVALID_ARGUMENT, "denoise iterations must be 0..8");
  if (!(o->sigma_luminance >= 0.f) || !(o->sigma_normal >= 0.f) || !(o->sigma_depth >= 0.f) || !std::isfinite(o->sigma_luminance) ||
      !std::isfinite(o->sigma_normal) || !std::isfinite(o->sigma_depth))
    return fail(RT_ERR_INVALID_ARGUMENT, "denoise sigmas must be finite and >= 0");
  D.iterations = o->iterations;
  D.sigma_l = o->sigma_luminance > 0.f ? o->sigma_luminance : 4.f;
  D.sigma_n = o->sigma_normal > 0.f ? o->sigma_normal : 128.f;
  D.sigma_z = o->sigma_depth > 0.f ? o->sigma_depth : 1.f;
  return RT_OK;
}

static rt_status features_prepare(rt_camera* c, size_t npx) {
  if (!c->d_falb) CU(dev_alloc(&c->d_falb, npx * 12));
  if (!c->d_fnrm) CU(dev_alloc(&c->d_fnrm, npx * 12));
  if (!c->d_fdepth) CU(dev_alloc(&c->d_fdepth, npx * 4));
  return RT_OK;
}

// Features and filter of the rows [b0, b1) of the region of P, on camera c's device and stream.  `color` / `moments` are
// [H][W] buffers this device can read, written by a render of the region; `out` / `rgb8` receive the band's rows.  The
// camera's whole-image feature and scratch buffers hold what the band's stages compute: the band plus the rows its passes
// read (dn_halo), clipped to the region.  `out` may alias `color` only when one band covers the region.  `poison` first
// fills those buffers with NaN, so that a read outside the computed rows changes the image.
static rt_status denoise_band(rt_camera* c, const RenderParams& P, int b0, int b1, const DenoiseParams& opts, const float* color,
                              const float* moments, float* out, uint8_t* rgb8, bool poison, int* launches) {
  int lf = 0;
  rt_status st = denoise_features(c, P, b0, b1, opts.iterations, poison, &lf);
  if (st != RT_OK) return st;
  st = denoise_filter(c, P, b0, b1, opts, color, moments, out, rgb8, launches);
  *launches += lf;
  return st;
}

// Feature step of denoise_band: the first-hit features of the rows a band's filter with `iterations` passes reads, over the
// one-shot render's first min(samples, 8) camera rays per pixel.
static rt_status denoise_features(rt_camera* c, const RenderParams& P, int b0, int b1, int iterations, bool poison, int* launches) {
  *launches = 0;
  if (P.x1 <= P.x0 || b1 <= b0) return RT_OK;
  const size_t npx = (size_t)c->hs->image_width * c->hs->image_height;
  rt_status st = features_prepare(c, npx);
  if (st != RT_OK) return st;
  if (!c->d_dn) CU(dev_alloc(&c->d_dn, npx * kDnFloatsPerPixel * sizeof(float)));
  if (poison) {
    CU(cudaMemsetAsync(c->d_falb, 0xff, npx * 12, c->stream));
    CU(cudaMemsetAsync(c->d_fnrm, 0xff, npx * 12, c->stream));
    CU(cudaMemsetAsync(c->d_fdepth, 0xff, npx * 4, c->stream));
    CU(cudaMemsetAsync(c->d_dn, 0xff, npx * kDnFloatsPerPixel * sizeof(float), c->stream));
  }
  RenderParams F = P; // the feature rows: one beyond what prepare computes
  const int hf = dn_halo(iterations, -1) + 1;
  F.y0 = std::max(P.y0, b0 - hf);
  F.y1 = std::min(P.y1, b1 + hf);
  const int n_feat = std::max(1, std::min(c->hs->cam.samples, 8));
  CU(launch_render_features(c->ds, F, n_feat, c->d_falb, c->d_fnrm, c->d_fdepth, c->stream));
  *launches = 1;
  return RT_OK;
}

// Filter step of denoise_band: prepare, the a-trous passes and finish of the band, on the features denoise_features left.
static rt_status denoise_filter(rt_camera* c, const RenderParams& P, int b0, int b1, const DenoiseParams& opts, const float* color,
                                const float* moments, float* out, uint8_t* rgb8, int* launches) {
  *launches = 0;
  if (P.x1 <= P.x0 || b1 <= b0) return RT_OK;
  const int W = c->hs->image_width;
  const size_t npx = (size_t)W * c->hs->image_height;
  if (!c->d_dn) CU(dev_alloc(&c->d_dn, npx * kDnFloatsPerPixel * sizeof(float)));
  DenoiseParams D = opts;
  D.width = W;
  D.x0 = P.x0; D.y0 = P.y0; D.x1 = P.x1; D.y1 = P.y1;
  D.color = color; D.albedo = c->d_falb; D.normal = c->d_fnrm; D.depth = c->d_fdepth; D.moments = moments;
  dn_scratch(D, c->d_dn, npx);
  D.out = out;
  D.rgb8 = rgb8;
  CU(launch_denoise(D, b0, b1, c->stream, launches));
  return RT_OK;
}

rt_status rt_camera_render_features(rt_camera* c, const rt_region* region, int32_t n_samples, float* albedo, float* normal, float* depth) {
  RT_GUARD_BEGIN
  if (!c) return fail(RT_ERR_INVALID_ARGUMENT, "null camera");
  if (n_samples < 1) return fail(RT_ERR_INVALID_ARGUMENT, "n_samples must be >= 1");
  DeviceGuard g(c->device);
  const int W = c->hs->image_width, H = c->hs->image_height;
  const size_t npx = (size_t)W * H;
  RenderParams P;
  rt_status st = clip_region(c, region, P);
  if (st != RT_OK) return st;
  if ((st = features_prepare(c, npx)) != RT_OK) return st;
  CU(launch_render_features(c->ds, P, n_samples, c->d_falb, c->d_fnrm, c->d_fdepth, c->stream));
  if (albedo) CU(copy_region(albedo, c->d_falb, 12, P, W, cudaMemcpyDeviceToHost, c->stream));
  if (normal) CU(copy_region(normal, c->d_fnrm, 12, P, W, cudaMemcpyDeviceToHost, c->stream));
  if (depth) CU(copy_region(depth, c->d_fdepth, 4, P, W, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return RT_OK;
  RT_GUARD_END
}

rt_status rt_denoise(int32_t device, int32_t width, int32_t height, const float* color, const float* albedo, const float* normal,
                     const float* depth, const float* moments, const rt_denoise_opts* opts, float* out) {
  RT_GUARD_BEGIN
  if (!color || !albedo || !normal || !depth || !moments || !out) return fail(RT_ERR_INVALID_ARGUMENT, "null argument");
  if (width <= 0 || height <= 0) return fail(RT_ERR_INVALID_ARGUMENT, "width and height must be > 0");
  DenoiseParams D{};
  rt_status st = dn_options(opts, D);
  if (st != RT_OK) return st;
  const int ndev = rt_device_count();
  if (ndev <= 0) return fail(RT_ERR_NO_DEVICE, "no CUDA device visible; this library has no CPU fallback");
  if (device < 0) { if (cudaGetDevice(&device) != cudaSuccess) device = 0; }
  if (device >= ndev) return fail(RT_ERR_INVALID_ARGUMENT, "device ordinal out of range");
  DeviceGuard g(device);
  if (!g.ok) return fail(RT_ERR_CUDA, "cudaSetDevice failed");
  const size_t npx = (size_t)width * height;
  struct Blocks { // back to the device cache once nothing of this call is in flight
    float* in = nullptr;
    float* scratch = nullptr;
    ~Blocks() { cudaStreamSynchronize(0); dev_free(in); dev_free(scratch); }
  } b;
  CU(dev_alloc(&b.in, npx * 18 * sizeof(float)));
  CU(dev_alloc(&b.scratch, npx * kDnFloatsPerPixel * sizeof(float)));
  float* d_col = b.in;
  float* d_alb = b.in + npx * 3;
  float* d_nrm = b.in + npx * 6;
  float* d_mom = b.in + npx * 9;
  float* d_dep = b.in + npx * 17;
  CU(cudaMemcpyAsync(d_col, color, npx * 12, cudaMemcpyHostToDevice, 0));
  CU(cudaMemcpyAsync(d_alb, albedo, npx * 12, cudaMemcpyHostToDevice, 0));
  CU(cudaMemcpyAsync(d_nrm, normal, npx * 12, cudaMemcpyHostToDevice, 0));
  CU(cudaMemcpyAsync(d_mom, moments, npx * 32, cudaMemcpyHostToDevice, 0));
  CU(cudaMemcpyAsync(d_dep, depth, npx * 4, cudaMemcpyHostToDevice, 0));
  D.width = width;
  D.x0 = 0; D.y0 = 0; D.x1 = width; D.y1 = height;
  D.color = d_col; D.albedo = d_alb; D.normal = d_nrm; D.depth = d_dep; D.moments = d_mom;
  dn_scratch(D, b.scratch, npx);
  D.out = d_col;
  D.rgb8 = nullptr;
  int launches = 0;
  CU(launch_denoise(D, 0, height, 0, &launches));
  CU(cudaMemcpyAsync(out, d_col, npx * 12, cudaMemcpyDeviceToHost, 0));
  CU(cudaStreamSynchronize(0));
  return RT_OK;
  RT_GUARD_END
}

rt_status rt_camera_render_denoised(rt_camera* c, const rt_region* region, uint8_t* rgb8, size_t rgb8_len, float* linear,
                                    const rt_denoise_opts* opts, rt_stats* stats) {
  RT_GUARD_BEGIN
  if (!c) return fail(RT_ERR_INVALID_ARGUMENT, "null camera");
  DenoiseParams D{};
  rt_status st = dn_options(opts, D);
  if (st != RT_OK) return st;
  if (rgb8 && rgb8_len < (size_t)c->hs->image_width * c->hs->image_height * 3)
    return fail(RT_ERR_BUFFER_TOO_SMALL, "rgb8 buffer smaller than width*height*3");
  // the filter reads the neighbours of a pixel, which other parts render; modes other than default are not radiance
  if (c->opts.part_count > 1) return fail(RT_ERR_UNSUPPORTED, "denoised renders are not partitioned");
  if (c->hs->cam.mode != RT_MODE_DEFAULT) return fail(RT_ERR_UNSUPPORTED, "denoised renders need the default render mode");
  return render_host(c, region, rgb8, rgb8_len, linear, nullptr, stats, &D);
  RT_GUARD_END
}

// Progressive render with a denoised preview after every pass; the last pass is rt_camera_render_denoised's image.
rt_status rt_camera_render_progressive_denoised(rt_camera* c, const rt_region* region, uint8_t* rgb8, size_t rgb8_len, float* linear,
                                                float* moments, int32_t n_passes, const rt_denoise_opts* opts, rt_progress_fn on_pass,
                                                void* user, rt_stats* stats) {
  RT_GUARD_BEGIN
  if (!c) return fail(RT_ERR_INVALID_ARGUMENT, "null camera");
  if (n_passes < 1) return fail(RT_ERR_INVALID_ARGUMENT, "n_passes must be >= 1");
  DenoiseParams D{};
  rt_status st = dn_options(opts, D);
  if (st != RT_OK) return st;
  if (rgb8 && rgb8_len < (size_t)c->hs->image_width * c->hs->image_height * 3)
    return fail(RT_ERR_BUFFER_TOO_SMALL, "rgb8 buffer smaller than width*height*3");
  if (c->opts.part_count > 1) return fail(RT_ERR_UNSUPPORTED, "denoised renders are not partitioned");
  if (c->hs->cam.mode != RT_MODE_DEFAULT) return fail(RT_ERR_UNSUPPORTED, "denoised renders need the default render mode");
  return progressive_host(c, region, rgb8, rgb8_len, linear, moments, n_passes, on_pass, user, stats, &D);
  RT_GUARD_END
}

rt_status rt_measure_fp32_peak(int32_t device, double* tflops, double* sm_clock_mhz) {
  if (!tflops) return fail(RT_ERR_INVALID_ARGUMENT, "null argument");
  int ndev = rt_device_count();
  if (ndev <= 0) return fail(RT_ERR_NO_DEVICE, "no CUDA device visible");
  if (device < 0) { if (cudaGetDevice(&device) != cudaSuccess) device = 0; }
  DeviceGuard g(device);
  int sms = 0, khz = 0;
  CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
  CU(cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, device));
  const int blocks = sms * 16, iters = 2048;
  float* d = nullptr;
  CU(dev_alloc(&d, (size_t)blocks * 256 * sizeof(float)));
  cudaEvent_t a = nullptr, b = nullptr;
  cudaError_t e = cudaEventCreate(&a);
  if (e == cudaSuccess) e = cudaEventCreate(&b);
  double best = 0;
  for (int rep = 0; rep < 5 && e == cudaSuccess; ++rep) {
    float ms = 0;
    if ((e = cudaEventRecord(a, 0)) != cudaSuccess) break;
    if ((e = launch_fp32_peak(d, blocks, iters, 0)) != cudaSuccess) break;
    if ((e = cudaEventRecord(b, 0)) != cudaSuccess) break;
    if ((e = cudaEventSynchronize(b)) != cudaSuccess) break;
    if ((e = cudaEventElapsedTime(&ms, a, b)) != cudaSuccess) break;
    double flops = (double)blocks * 256.0 * iters * 16.0 * 8.0 * 2.0;
    double tf = flops / (ms * 1e-3) / 1e12;
    if (rep > 0 && tf > best) best = tf;
  }
  if (a) cudaEventDestroy(a);
  if (b) cudaEventDestroy(b);
  dev_free(d);
  if (e != cudaSuccess) return fail(RT_ERR_CUDA, std::string("FP32 peak measurement: ") + cudaGetErrorString(e));
  *tflops = best;
  if (sm_clock_mhz) *sm_clock_mhz = khz / 1000.0;
  return RT_OK;
}

} // extern "C"

// ---------------------------------------------------------------------------------------------
// rt_multi: ONE process drives N GPUs — the native replacement of the reference's worker pool
// (src/raytracer.ts:60-90: N worker_threads, row strips, SharedArrayBuffer).  The scene is compiled once
// and uploaded to every device; device k renders the 8x4 blocks it owns (block_owner, rt_types.h) and
// its kernels store the finished pixels STRAIGHT INTO device 0's framebuffer over NVLink peer mappings
// (3 bytes per pixel, written once): there is no gather step, no staging copy and no collective —
// device 0's stream waits on one event per peer and copies the image to the caller's buffer.
// Without peer access between the devices every camera renders into its own buffer and the owned
// blocks are merged on the host (render_host's partition path), one host thread per device.
// ---------------------------------------------------------------------------------------------
struct rt_multi {
  std::vector<rt_camera*> cams; // part k on devices[k]
  std::vector<int> devices;
  bool p2p = false;
  uint8_t* d_rgb8 = nullptr;    // on devices[0]
  float* d_linear = nullptr;
  float* d_color = nullptr;     // on devices[0], rt_multi_render_denoised: the render's colour [H][W][3] and moments [H][W][8]
  float* d_moments = nullptr;
  std::vector<cudaEvent_t> done;
  std::vector<cudaEvent_t> rendered; // rt_multi_render_denoised: device k's render has landed in device 0's memory
  unsigned long long* h_stats = nullptr; // pinned [n][kStatCount]
};

// One host thread per device runs job(k); returns the first failing device's status, with its message.
static rt_status on_every_device(int n, const std::function<rt_status(int)>& job) {
  std::vector<rt_status> st((size_t)n, RT_OK);
  std::vector<std::string> msg((size_t)n);
  std::vector<std::thread> th;
  for (int k = 0; k < n; ++k)
    th.emplace_back([&, k]() {
      st[k] = job(k);
      if (st[k] != RT_OK) msg[k] = g_err;
    });
  for (auto& t : th) t.join();
  for (int k = 0; k < n; ++k)
    if (st[k] != RT_OK) return fail(st[k], msg[k]);
  return RT_OK;
}

// The host-merge path's stats: device_ms is the slowest device's (they run concurrently).
static rt_stats merge_host_stats(const std::vector<rt_stats>& ps) {
  rt_stats out = unpack_stats(kStatsInit);
  for (const rt_stats& s : ps) {
    merge_stats(&out, s);
    out.device_ms = std::max(out.device_ms, s.device_ms);
  }
  return out;
}
// The merged counters the peer-write path copied to m->h_stats (device_ms and kernel_launches are the caller's).
static rt_stats merge_raw_stats(const rt_multi* m) {
  rt_stats out = unpack_stats(kStatsInit);
  for (size_t k = 0; k < m->cams.size(); ++k) merge_stats(&out, unpack_stats(m->h_stats + k * kStatCount));
  return out;
}

static void free_multi(rt_multi* m) {
  if (!m) return;
  for (rt_camera* c : m->cams) free_camera(c);
  if (!m->devices.empty()) {
    DeviceGuard g(m->devices[0]);
    dev_free(m->d_rgb8);
    dev_free(m->d_linear);
    dev_free(m->d_color);
    dev_free(m->d_moments);
  }
  for (size_t k = 0; k < m->done.size(); ++k)
    if (m->done[k]) { DeviceGuard g(m->devices[k]); cudaEventDestroy(m->done[k]); }
  for (size_t k = 0; k < m->rendered.size(); ++k)
    if (m->rendered[k]) { DeviceGuard g(m->devices[k]); cudaEventDestroy(m->rendered[k]); }
  if (m->h_stats) cudaFreeHost(m->h_stats);
  delete m;
}

extern "C" {

rt_status rt_multi_create(const rt_scene_desc* scene, const rt_render_opts* opts, int32_t n_devices, const int32_t* devices, rt_multi** out) {
  if (!scene || !opts || !out) return fail(RT_ERR_INVALID_ARGUMENT, "null argument");
  *out = nullptr;
  rt_multi* m = nullptr;
  try {
    std::shared_ptr<HostScene> hs;
    double ms = 0;
    rt_status st = compile_shared(scene, opts, hs, ms); // scene errors first, like the reference, GPU or not
    if (st != RT_OK) return st;
    const int ndev = rt_device_count();
    if (ndev <= 0) return fail(RT_ERR_NO_DEVICE, "no CUDA device visible; this library has no CPU fallback");
    if (n_devices <= 0) n_devices = ndev;
    m = new rt_multi();
    for (int k = 0; k < n_devices; ++k) {
      const int d = devices ? devices[k] : k;
      if (d < 0 || d >= ndev) { free_multi(m); return fail(RT_ERR_INVALID_ARGUMENT, "device ordinal out of range"); }
      for (int prev : m->devices)
        if (prev == d) { free_multi(m); return fail(RT_ERR_INVALID_ARGUMENT, "device listed twice"); }
      m->devices.push_back(d);
    }
    // RT_B200_MULTI_PARTS=n (development switch): n parts dealt to the devices in turn, each with its own camera, stream
    // and events, so that the partitioned passes, the cross-stream waits and both paths run with several parts on one GPU
    if (const char* e = getenv("RT_B200_MULTI_PARTS")) {
      const int parts = atoi(e);
      if (parts >= 1) {
        const std::vector<int> given = m->devices;
        m->devices.clear();
        for (int k = 0; k < parts; ++k) m->devices.push_back(given[(size_t)k % given.size()]);
        n_devices = parts;
      }
    }
    // every device must be able to write device[0]'s memory, else the host-merge path is used
    m->p2p = true;
    for (int k = 1; k < n_devices && m->p2p; ++k) {
      if (m->devices[k] == m->devices[0]) continue; // a part on device[0] itself needs no peer mapping
      int can = 0;
      if (cudaDeviceCanAccessPeer(&can, m->devices[k], m->devices[0]) != cudaSuccess || !can) { cudaGetLastError(); m->p2p = false; break; }
      DeviceGuard g(m->devices[k]);
      const cudaError_t e = cudaDeviceEnablePeerAccess(m->devices[0], 0);
      if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) m->p2p = false;
      cudaGetLastError();
    }
    if (getenv("RT_B200_MULTI_NO_P2P")) m->p2p = false; // development switch: exercise the host-merge path
    for (int k = 0; k < n_devices; ++k) {
      rt_render_opts o = *opts;
      o.device = m->devices[k];
      o.part_index = k;
      o.part_count = n_devices;
      rt_camera* c = nullptr;
      st = camera_from_host(hs, &o, &c, k == 0 ? ms : 0.0);
      if (st != RT_OK) { free_multi(m); return st; }
      m->cams.push_back(c);
      DeviceGuard g(m->devices[k]);
      cudaEvent_t ev = nullptr, ev_r = nullptr;
      // each device renders on its own non-blocking stream: the legacy default stream would serialise them
      if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess || cudaEventCreateWithFlags(&ev, cudaEventDisableTiming) != cudaSuccess ||
          cudaEventCreateWithFlags(&ev_r, cudaEventDisableTiming) != cudaSuccess) {
        if (ev) cudaEventDestroy(ev);
        const std::string msg = cudaGetErrorString(cudaGetLastError());
        free_multi(m);
        return fail(RT_ERR_CUDA, "rt_multi_create: stream/event: " + msg);
      }
      c->owns_stream = true;
      m->done.push_back(ev);
      m->rendered.push_back(ev_r);
    }
    if (cudaMallocHost(&m->h_stats, sizeof(unsigned long long) * kStatCount * (size_t)n_devices) != cudaSuccess) {
      cudaGetLastError();
      free_multi(m);
      return fail(RT_ERR_CUDA, "rt_multi_create: pinned stats buffer");
    }
    *out = m;
    return RT_OK;
  } catch (const std::exception& e) {
    if (m) free_multi(m);
    return fail(RT_ERR_INVALID_ARGUMENT, std::string("rt_multi_create: ") + e.what());
  }
}

rt_status rt_multi_destroy(rt_multi* m) {
  free_multi(m);
  return RT_OK;
}

rt_status rt_multi_get_info(const rt_multi* m, rt_camera_info* info, int32_t* n_devices, int32_t* peer_writes) {
  if (!m || m->cams.empty()) return fail(RT_ERR_INVALID_ARGUMENT, "null argument");
  if (n_devices) *n_devices = (int32_t)m->cams.size();
  if (peer_writes) *peer_writes = m->p2p ? 1 : 0;
  return info ? rt_camera_get_info(m->cams[0], info) : RT_OK;
}

rt_status rt_multi_render_region(rt_multi* m, const rt_region* region, uint8_t* rgb8, size_t rgb8_len, float* linear, rt_stats* stats) {
  RT_GUARD_BEGIN
  if (!m || m->cams.empty()) return fail(RT_ERR_INVALID_ARGUMENT, "null argument");
  const int n = (int)m->cams.size();
  rt_camera* c0 = m->cams[0];
  const int W = c0->hs->image_width, H = c0->hs->image_height;
  const size_t npx = (size_t)W * H;
  if (rgb8 && rgb8_len < npx * 3) return fail(RT_ERR_BUFFER_TOO_SMALL, "rgb8 buffer smaller than width*height*3");
  if (stats) std::memset(stats, 0, sizeof(*stats));
  if (!m->p2p && n > 1) {
    // host merge: one thread per device, each copies the blocks it owns into the caller's buffer
    std::vector<rt_stats> ps((size_t)n);
    rt_status st = on_every_device(n, [&](int k) { return render_host(m->cams[k], region, rgb8, rgb8_len, linear, nullptr, &ps[k]); });
    if (st != RT_OK) return st;
    if (stats) *stats = merge_host_stats(ps);
    return RT_OK;
  }
  // ---- peer-write path ----
  {
    DeviceGuard g0(m->devices[0]);
    if (rgb8 && !m->d_rgb8) CU(dev_alloc(&m->d_rgb8, npx * 3));
    if (linear && !m->d_linear) CU(dev_alloc(&m->d_linear, npx * 3 * sizeof(float)));
  }
  RenderParams P0{};
  int launches_total = 0;
  for (int k = 0; k < n; ++k) {
    rt_camera* c = m->cams[k];
    DeviceGuard g(c->device);
    RenderParams P;
    rt_status st = clip_region(c, region, P);
    if (st != RT_OK) return st;
    P.rgb8 = rgb8 ? m->d_rgb8 : nullptr;       // device 0's framebuffer, peer-mapped on device k
    P.linear = linear ? m->d_linear : nullptr;
    int launches = 0;
    if ((st = timed_render(c, P, c->ev1, m->h_stats + (size_t)k * kStatCount, &launches)) != RT_OK) return st;
    CU(cudaEventRecord(m->done[k], c->stream));
    launches_total += launches;
    if (k == 0) P0 = P;
  }
  {
    DeviceGuard g0(m->devices[0]);
    for (int k = 1; k < n; ++k) CU(cudaStreamWaitEvent(c0->stream, m->done[k], 0)); // peers' pixels have landed in device 0's memory
    if (rgb8) CU(copy_region(rgb8, m->d_rgb8, 3, P0, W, cudaMemcpyDeviceToHost, c0->stream));
    if (linear) CU(copy_region(linear, m->d_linear, 12, P0, W, cudaMemcpyDeviceToHost, c0->stream));
    CU(cudaStreamSynchronize(c0->stream));
  }
  if (stats) {
    double ms_max = 0;
    for (int k = 0; k < n; ++k) {
      DeviceGuard g(m->cams[k]->device);
      float ms = 0;
      CU(cudaEventElapsedTime(&ms, m->cams[k]->ev0, m->cams[k]->ev1));
      ms_max = std::max(ms_max, (double)ms);
    }
    *stats = merge_raw_stats(m);
    stats->device_ms = ms_max; // the slowest device (they run concurrently)
    stats->kernel_launches = launches_total;
  }
  return RT_OK;
  RT_GUARD_END
}

// The row bands of the denoiser on several parts: one per part, or RT_B200_DENOISE_BANDS=n (development switch) bands dealt
// to the parts in turn, with `poison` set: their buffers are filled with NaN first (denoise_features).
static int dn_band_count(int n_parts, bool* poison) {
  const char* e = getenv("RT_B200_DENOISE_BANDS");
  *poison = e && atoi(e) >= 1;
  return *poison ? atoi(e) : n_parts;
}
// Band b of n_bands: contiguous rows [b0, b1) of the region of P; some bands are empty when the region has fewer rows.
static void band_rows(const RenderParams& P, int b, int n_bands, int& b0, int& b1) {
  const int rh = P.y1 - P.y0;
  b0 = P.y0 + (int)((long long)b * rh / n_bands);
  b1 = P.y0 + (int)((long long)(b + 1) * rh / n_bands);
}

// Denoised render on every device (include/rt_b200.h).  Peer-write path: every device renders its blocks' colour and
// moments straight into device 0's d_color / d_moments, then, after every device's render, filters its band of the
// region's rows (dn_halo's ghost zones, recomputed instead of exchanged) with prepare reading the colour and moments over
// the peer mapping, and writes the band's rows of d_linear / d_rgb8 on device 0.  The output never aliases d_color: other
// bands still read it.  Host-merge path: the colour and moments are merged on the host, and device 0 filters the region.
// RT_B200_DENOISE_BANDS=n (development switch): n bands dealt to the devices in turn, each band's buffers filled with
// NaN first, so that the band and halo logic runs, and a read outside a band's computed rows shows, on one GPU.
rt_status rt_multi_render_denoised(rt_multi* m, const rt_region* region, uint8_t* rgb8, size_t rgb8_len, float* linear,
                                   const rt_denoise_opts* opts, rt_stats* stats) {
  RT_GUARD_BEGIN
  if (!m || m->cams.empty()) return fail(RT_ERR_INVALID_ARGUMENT, "null argument");
  DenoiseParams D{};
  rt_status st = dn_options(opts, D);
  if (st != RT_OK) return st;
  const int n = (int)m->cams.size();
  rt_camera* c0 = m->cams[0];
  const int W = c0->hs->image_width, H = c0->hs->image_height;
  const size_t npx = (size_t)W * H;
  if (rgb8 && rgb8_len < npx * 3) return fail(RT_ERR_BUFFER_TOO_SMALL, "rgb8 buffer smaller than width*height*3");
  if (c0->hs->cam.mode != RT_MODE_DEFAULT) return fail(RT_ERR_UNSUPPORTED, "denoised renders need the default render mode");
  RenderParams P0;
  st = clip_region(c0, region, P0);
  if (st != RT_OK) return st;
  const int rw = P0.x1 - P0.x0, rh = P0.y1 - P0.y0;
  bool poison = false;
  const int n_bands = dn_band_count(n, &poison);
  auto band = [&](int b, int& b0, int& b1) { band_rows(P0, b, n_bands, b0, b1); };
  {
    DeviceGuard g0(m->devices[0]);
    if (!m->d_color) CU(dev_alloc(&m->d_color, npx * 3 * sizeof(float)));
    if (!m->d_moments) CU(dev_alloc(&m->d_moments, npx * 8 * sizeof(float)));
    if (!m->d_linear) CU(dev_alloc(&m->d_linear, npx * 3 * sizeof(float)));
    if (rgb8 && !m->d_rgb8) CU(dev_alloc(&m->d_rgb8, npx * 3));
  }
  uint8_t* out8 = rgb8 ? m->d_rgb8 : nullptr;
  int launches_total = 0;
  if (!m->p2p && n > 1) {
    // host merge: one thread per device renders its blocks' colour and moments into host arrays, device 0 filters
    std::vector<float> hc(npx * 3), hm(npx * 8);
    std::vector<rt_stats> ps((size_t)n);
    st = on_every_device(n, [&](int k) { return render_host(m->cams[k], region, nullptr, 0, hc.data(), hm.data(), &ps[k]); });
    if (st != RT_OK) return st;
    DeviceGuard g0(m->devices[0]);
    CU(cudaEventRecord(c0->ev0, c0->stream));
    if (rw > 0 && rh > 0) {
      CU(copy_region(m->d_color, hc.data(), 12, P0, W, cudaMemcpyHostToDevice, c0->stream));
      CU(copy_region(m->d_moments, hm.data(), 32, P0, W, cudaMemcpyHostToDevice, c0->stream));
      for (int b = 0; b < n_bands; ++b) {
        int b0, b1, l = 0;
        band(b, b0, b1);
        st = denoise_band(c0, P0, b0, b1, D, m->d_color, m->d_moments, m->d_linear, out8, poison, &l);
        if (st != RT_OK) return st;
        launches_total += l;
      }
    }
    CU(cudaEventRecord(c0->ev1, c0->stream));
    if (stats) {
      *stats = merge_host_stats(ps);
      float ms = 0;
      CU(cudaEventSynchronize(c0->ev1));
      CU(cudaEventElapsedTime(&ms, c0->ev0, c0->ev1));
      stats->device_ms += ms; // the slowest render, then the upload and the filter
      stats->kernel_launches += launches_total;
    }
  } else {
    // ---- peer-write path ----
    std::vector<RenderParams> Ps((size_t)n);
    for (int k = 0; k < n; ++k) {
      rt_camera* c = m->cams[k];
      DeviceGuard g(c->device);
      RenderParams& P = Ps[k];
      st = clip_region(c, region, P);
      if (st != RT_OK) return st;
      P.rgb8 = nullptr; // RGB8 is written from the filtered image
      P.linear = m->d_color; // device 0's buffers, peer-mapped on device k
      P.moments = m->d_moments;
      int launches = 0;
      if ((st = timed_render(c, P, m->rendered[k], m->h_stats + (size_t)k * kStatCount, &launches)) != RT_OK) return st;
      launches_total += launches;
    }
    if (rw > 0 && rh > 0) {
      for (int k = 0; k < n; ++k) { // a band's passes read rows other devices rendered
        DeviceGuard g(m->cams[k]->device);
        for (int j = 0; j < n; ++j)
          if (j != k) CU(cudaStreamWaitEvent(m->cams[k]->stream, m->rendered[j], 0));
      }
      for (int b = 0; b < n_bands; ++b) {
        rt_camera* c = m->cams[b % n];
        DeviceGuard g(c->device);
        int b0, b1, l = 0;
        band(b, b0, b1);
        st = denoise_band(c, Ps[b % n], b0, b1, D, m->d_color, m->d_moments, m->d_linear, out8, poison, &l);
        if (st != RT_OK) return st;
        launches_total += l;
      }
    }
    for (int k = 1; k < n; ++k) {
      DeviceGuard g(m->cams[k]->device);
      CU(cudaEventRecord(m->done[k], m->cams[k]->stream));
    }
    DeviceGuard g0(m->devices[0]);
    for (int k = 1; k < n; ++k) CU(cudaStreamWaitEvent(c0->stream, m->done[k], 0)); // every band has landed in device 0's memory
    CU(cudaEventRecord(c0->ev1, c0->stream));
    if (stats) {
      CU(cudaEventSynchronize(c0->ev1));
      float ms = 0;
      CU(cudaEventElapsedTime(&ms, c0->ev0, c0->ev1));
      *stats = merge_raw_stats(m);
      stats->device_ms = ms; // device 0, from its render to the last band's last kernel
      stats->kernel_launches = launches_total;
    }
  }
  DeviceGuard g0(m->devices[0]);
  if (rgb8) CU(copy_region(rgb8, m->d_rgb8, 3, P0, W, cudaMemcpyDeviceToHost, c0->stream));
  if (linear) CU(copy_region(linear, m->d_linear, 12, P0, W, cudaMemcpyDeviceToHost, c0->stream));
  CU(cudaStreamSynchronize(c0->stream));
  return RT_OK;
  RT_GUARD_END
}

} // extern "C"

// Progressive render on every device (rt_multi_render_progressive*, include/rt_b200.h): the passes and caps of
// progressive_host, each pass rendered, filtered (`dn`) and delivered the way rt_multi_render_region and
// rt_multi_render_denoised deliver a one-shot call.  Each camera keeps its PixelStats and fixed-point sums in its own
// memory between the passes.  With `dn` the features are computed in the first pass only, and the filter never writes
// the colour it reads (d_color, or the host-merge path's upload of it): a pixel that converged in an earlier pass is not
// rendered again, and its noisy colour must survive for the next pass's filter.
// Ordering between passes: pass k+1's render on any device writes colour rows that other devices' pass-k band filters
// read (the halos), and framebuffer rows that device 0's pass-k copy reads.  This relies on the host synchronisation that
// precedes on_pass: device 0's stream waits on every device's `done` event, recorded after that device's last kernel of
// the pass (the host-merge path synchronises every device's stream), and the host enqueues pass k+1 only after
// cudaStreamSynchronize of that stream has returned.
static rt_status multi_progressive(rt_multi* m, const rt_region* region, uint8_t* rgb8, size_t rgb8_len, float* linear,
                                   float* moments, int32_t n_passes, rt_progress_fn on_pass, void* user, rt_stats* stats,
                                   const DenoiseParams* dn) {
  const int n = (int)m->cams.size();
  rt_camera* c0 = m->cams[0];
  const int W = c0->hs->image_width, H = c0->hs->image_height;
  const size_t npx = (size_t)W * H;
  if (rgb8 && rgb8_len < npx * 3) return fail(RT_ERR_BUFFER_TOO_SMALL, "rgb8 buffer smaller than width*height*3");
  if (dn && c0->hs->cam.mode != RT_MODE_DEFAULT) return fail(RT_ERR_UNSUPPORTED, "denoised renders need the default render mode");
  RenderParams P0;
  rt_status st = clip_region(c0, region, P0);
  if (st != RT_OK) return st;
  const bool filter = dn && P0.x1 > P0.x0 && P0.y1 > P0.y0;
  const bool host_merge = !m->p2p && n > 1;
  bool poison = false;
  const int n_bands = dn_band_count(n, &poison);
  {
    DeviceGuard g0(m->devices[0]);
    if (dn && !m->d_color) CU(dev_alloc(&m->d_color, npx * 3 * sizeof(float)));
    if (dn && !m->d_moments) CU(dev_alloc(&m->d_moments, npx * 8 * sizeof(float)));
    if ((dn || (linear && !host_merge)) && !m->d_linear) CU(dev_alloc(&m->d_linear, npx * 3 * sizeof(float)));
    if (rgb8 && (dn || !host_merge) && !m->d_rgb8) CU(dev_alloc(&m->d_rgb8, npx * 3));
  }
  uint8_t* out8 = rgb8 ? m->d_rgb8 : nullptr;
  // Features (first pass) and filter of every band, band b on cams[b % parts].  With the switch's poison, a part's
  // buffers are filled with NaN before its first band's features only: its later passes filter every band on them.
  auto filter_bands = [&](int parts, bool first, int* launches) -> rt_status {
    for (int b = 0; first && b < n_bands; ++b) {
      rt_camera* c = m->cams[b % parts];
      DeviceGuard g(c->device);
      int b0, b1, l = 0;
      band_rows(P0, b, n_bands, b0, b1);
      rt_status s = denoise_features(c, P0, b0, b1, dn->iterations, poison && b < parts, &l);
      if (s != RT_OK) return s;
      *launches += l;
    }
    for (int b = 0; b < n_bands; ++b) {
      rt_camera* c = m->cams[b % parts];
      DeviceGuard g(c->device);
      int b0, b1, l = 0;
      band_rows(P0, b, n_bands, b0, b1);
      rt_status s = denoise_filter(c, P0, b0, b1, *dn, m->d_color, m->d_moments, m->d_linear, out8, &l);
      if (s != RT_OK) return s;
      *launches += l;
    }
    return RT_OK;
  };
  // host merge, denoised: every device's blocks of the colour and moments, uploaded to device 0 for the filter
  std::vector<float> hc, hm;
  float* h_mom = moments;
  if (dn && host_merge) {
    hc.resize(npx * 3);
    if (!h_mom) { hm.resize(npx * 8); h_mom = hm.data(); }
  }
  const int S = c0->hs->cam.samples;
  const bool stream = c0->hs->cam.adaptive || c0->hs->cam.mode != 0 || dn; // as progressive_host
  const std::vector<int> caps = camera_pass_caps(c0, n_passes);
  rt_stats total = unpack_stats(kStatsInit);
  int prev = 0;
  bool first = true;
  for (int k = 1; k <= n_passes; ++k) {
    const int cap = caps[(size_t)k - 1];
    if (cap < 0) continue;
    const ProgPass pass{prev, cap, first};
    const ProgPass* pp = (S > 0 && n_passes > 1) ? &pass : nullptr;
    rt_stats ps;
    double ms = 0;
    int launches = 0;
    if (host_merge) {
      std::vector<rt_stats> dev((size_t)n);
      st = on_every_device(n, [&](int j) {
        return dn ? render_host(m->cams[j], region, nullptr, 0, hc.data(), h_mom, &dev[j], nullptr, pp)
                  : render_host(m->cams[j], region, rgb8, rgb8_len, linear, nullptr, &dev[j], nullptr, pp);
      });
      if (st != RT_OK) return st;
      ps = merge_host_stats(dev);
      ms = ps.device_ms; // the slowest device
      launches = ps.kernel_launches;
      if (dn) { // device 0 filters the region
        DeviceGuard g0(m->devices[0]);
        CU(cudaEventRecord(c0->ev0, c0->stream));
        if (filter) {
          CU(copy_region(m->d_color, hc.data(), 12, P0, W, cudaMemcpyHostToDevice, c0->stream));
          CU(copy_region(m->d_moments, h_mom, 32, P0, W, cudaMemcpyHostToDevice, c0->stream));
          if ((st = filter_bands(1, first, &launches)) != RT_OK) return st;
        }
        CU(cudaEventRecord(c0->ev1, c0->stream));
        if (rgb8) CU(copy_region(rgb8, m->d_rgb8, 3, P0, W, cudaMemcpyDeviceToHost, c0->stream));
        if (linear) CU(copy_region(linear, m->d_linear, 12, P0, W, cudaMemcpyDeviceToHost, c0->stream));
        CU(cudaStreamSynchronize(c0->stream));
        float f = 0;
        CU(cudaEventElapsedTime(&f, c0->ev0, c0->ev1));
        ms += f; // the slowest render, then the upload and the filter
      }
    } else {
      // ---- peer-write path: every device writes its blocks into device 0's buffers ----
      for (int j = 0; j < n; ++j) {
        rt_camera* c = m->cams[j];
        DeviceGuard g(c->device);
        RenderParams P;
        if ((st = clip_region(c, region, P)) != RT_OK) return st;
        P.rgb8 = rgb8 && !dn ? m->d_rgb8 : nullptr; // the denoised form writes RGB8 from the filtered image
        P.linear = dn ? m->d_color : linear ? m->d_linear : nullptr;
        P.moments = dn ? m->d_moments : nullptr;
        int l = 0;
        if ((st = timed_render(c, P, dn ? m->rendered[j] : c->ev1, m->h_stats + (size_t)j * kStatCount, &l, pp)) != RT_OK) return st;
        launches += l;
        if (!dn) CU(cudaEventRecord(m->done[j], c->stream));
      }
      if (dn) {
        if (filter) {
          for (int j = 0; j < n; ++j) { // a band's passes read rows other devices rendered
            DeviceGuard g(m->cams[j]->device);
            for (int i = 0; i < n; ++i)
              if (i != j) CU(cudaStreamWaitEvent(m->cams[j]->stream, m->rendered[i], 0));
          }
          if ((st = filter_bands(n, first, &launches)) != RT_OK) return st;
        }
        for (int j = 1; j < n; ++j) {
          DeviceGuard g(m->cams[j]->device);
          CU(cudaEventRecord(m->done[j], m->cams[j]->stream));
        }
      }
      DeviceGuard g0(m->devices[0]);
      for (int j = 1; j < n; ++j) CU(cudaStreamWaitEvent(c0->stream, m->done[j], 0)); // every device's part of the pass has landed
      if (dn) CU(cudaEventRecord(c0->ev1, c0->stream));
      if (rgb8) CU(copy_region(rgb8, m->d_rgb8, 3, P0, W, cudaMemcpyDeviceToHost, c0->stream));
      if (linear) CU(copy_region(linear, m->d_linear, 12, P0, W, cudaMemcpyDeviceToHost, c0->stream));
      if (moments) CU(copy_region(moments, m->d_moments, 32, P0, W, cudaMemcpyDeviceToHost, c0->stream));
      CU(cudaStreamSynchronize(c0->stream));
      if (dn) { // device 0, from its render to the last band's last kernel
        float f = 0;
        CU(cudaEventElapsedTime(&f, c0->ev0, c0->ev1));
        ms = f;
      } else { // the slowest device
        for (int j = 0; j < n; ++j) {
          DeviceGuard g(m->cams[j]->device);
          float f = 0;
          CU(cudaEventElapsedTime(&f, m->cams[j]->ev0, m->cams[j]->ev1));
          ms = std::max(ms, (double)f);
        }
      }
      ps = merge_raw_stats(m);
    }
    ps.kernel_launches = launches;
    fold_pass_stats(&total, ps, ms, stream, cap);
    prev = cap;
    first = false;
    if (on_pass && on_pass(user, k, n_passes, (int32_t)cap, &total) != 0) break; // every device stops after this pass
  }
  if (stats) *stats = total;
  return RT_OK;
}

extern "C" {

rt_status rt_multi_render_progressive(rt_multi* m, const rt_region* region, uint8_t* rgb8, size_t rgb8_len, float* linear,
                                      int32_t n_passes, rt_progress_fn on_pass, void* user, rt_stats* stats) {
  RT_GUARD_BEGIN
  if (!m || m->cams.empty()) return fail(RT_ERR_INVALID_ARGUMENT, "null argument");
  if (n_passes < 1) return fail(RT_ERR_INVALID_ARGUMENT, "n_passes must be >= 1");
  return multi_progressive(m, region, rgb8, rgb8_len, linear, nullptr, n_passes, on_pass, user, stats, nullptr);
  RT_GUARD_END
}

rt_status rt_multi_render_progressive_denoised(rt_multi* m, const rt_region* region, uint8_t* rgb8, size_t rgb8_len, float* linear,
                                               float* moments, int32_t n_passes, const rt_denoise_opts* opts, rt_progress_fn on_pass,
                                               void* user, rt_stats* stats) {
  RT_GUARD_BEGIN
  if (!m || m->cams.empty()) return fail(RT_ERR_INVALID_ARGUMENT, "null argument");
  if (n_passes < 1) return fail(RT_ERR_INVALID_ARGUMENT, "n_passes must be >= 1");
  DenoiseParams D{};
  rt_status st = dn_options(opts, D);
  if (st != RT_OK) return st;
  return multi_progressive(m, region, rgb8, rgb8_len, linear, moments, n_passes, on_pass, user, stats, &D);
  RT_GUARD_END
}

int32_t rt_progressive_caps(int32_t samples, int32_t batch, int32_t n_passes, int32_t* caps) {
  if (samples < 0 || batch < 1 || n_passes < 1 || !caps) return -1;
  try {
    const std::vector<int> v = pass_caps(samples, batch, n_passes);
    int32_t run = 0;
    for (int k = 0; k < n_passes; ++k) {
      caps[k] = v[(size_t)k];
      run += v[(size_t)k] >= 0;
    }
    return run;
  } catch (const std::exception&) { return -1; }
}

// ---- framebuffer shared between the one-process-per-GPU ranks of a node (CUDA IPC) ----
rt_status rt_shared_buffer_create(int32_t device, size_t bytes, void** dev_ptr, uint8_t handle[64]) {
  if (!dev_ptr || !handle || bytes == 0) return fail(RT_ERR_INVALID_ARGUMENT, "null argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  if (rt_device_count() <= 0) return fail(RT_ERR_NO_DEVICE, "no CUDA device visible");
  if (device < 0) { if (cudaGetDevice(&device) != cudaSuccess) device = 0; }
  DeviceGuard g(device);
  void* p = nullptr;
  CU(cudaMalloc(&p, bytes)); // a plain allocation of its own: IPC handles name whole allocations
  cudaIpcMemHandle_t h;
  const cudaError_t e = cudaIpcGetMemHandle(&h, p);
  if (e != cudaSuccess) { cudaFree(p); return fail(RT_ERR_CUDA, std::string("cudaIpcGetMemHandle: ") + cudaGetErrorString(e)); }
  std::memcpy(handle, &h, 64);
  *dev_ptr = p;
  return RT_OK;
}
rt_status rt_shared_buffer_open(int32_t device, const uint8_t handle[64], void** dev_ptr) {
  if (!dev_ptr || !handle) return fail(RT_ERR_INVALID_ARGUMENT, "null argument");
  if (rt_device_count() <= 0) return fail(RT_ERR_NO_DEVICE, "no CUDA device visible");
  if (device < 0) { if (cudaGetDevice(&device) != cudaSuccess) device = 0; }
  DeviceGuard g(device);
  cudaIpcMemHandle_t h;
  std::memcpy(&h, handle, 64);
  void* p = nullptr;
  const cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
  if (e != cudaSuccess) { cudaGetLastError(); return fail(RT_ERR_CUDA, std::string("cudaIpcOpenMemHandle: ") + cudaGetErrorString(e)); }
  *dev_ptr = p;
  return RT_OK;
}
rt_status rt_shared_buffer_release(int32_t device, void* dev_ptr, int32_t opened) {
  if (!dev_ptr) return RT_OK;
  if (device < 0) { if (cudaGetDevice(&device) != cudaSuccess) device = 0; }
  DeviceGuard g(device);
  const cudaError_t e = opened ? cudaIpcCloseMemHandle(dev_ptr) : cudaFree(dev_ptr);
  if (e != cudaSuccess) { cudaGetLastError(); return fail(RT_ERR_CUDA, std::string("rt_shared_buffer_release: ") + cudaGetErrorString(e)); }
  return RT_OK;
}

} // extern "C"

// ---------------------------------------------------------------------------------------------
// per-function parity hooks: stage the records (rounded to FP32 where `Vec3.create` would round them,
// src/geometry/vec3.ts:263), run one thread per record, copy the answers back.  Synchronous.
// ---------------------------------------------------------------------------------------------
namespace {
struct DbgBuf { // device scratch of one hook call, returned to the cache on scope exit
  std::vector<void*> ptrs;
  ~DbgBuf() { for (void* p : ptrs) dev_free(p); }
  template <class T>
  cudaError_t up(const std::vector<T>& h, T** d) {
    cudaError_t e = dev_alloc(d, std::max<size_t>(h.size(), 1) * sizeof(T));
    if (e != cudaSuccess) return e;
    ptrs.push_back(*d);
    return h.empty() ? cudaSuccess : cudaMemcpy(*d, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice);
  }
  template <class T>
  cudaError_t out(size_t n, T** d) {
    cudaError_t e = dev_alloc(d, std::max<size_t>(n, 1) * sizeof(T));
    if (e == cudaSuccess) ptrs.push_back(*d);
    return e;
  }
};
std::vector<float> to_f32(const double* p, size_t n) {
  std::vector<float> v(n);
  for (size_t i = 0; i < n; ++i) v[i] = (float)p[i];
  return v;
}
struct DbgHitH { float ro[3], rd[3], p[3], n[3]; int front, pad; }; // = rt::DbgHit (rt_debug.cuh)
static_assert(sizeof(DbgHitH) == 56 && sizeof(rt_debug_scatter_out) == 44, "debug record layouts");
} // namespace


extern "C" {

rt_status rt_debug_scatter(rt_camera* c, int32_t object_index, int32_t n, const rt_debug_hit* hits, const double* uniforms,
                           rt_debug_scatter_out* out) {
  RT_GUARD_BEGIN
  if (!c || n < 0 || (n > 0 && (!hits || !uniforms || !out))) return fail(RT_ERR_INVALID_ARGUMENT, "null argument");
  int root = -1;
  for (const I2& si : c->hs->slot_info)
    if ((si.y & 0x3fffffff) == object_index) { root = si.x; break; }
  if (root < 0) return fail(RT_ERR_INVALID_ARGUMENT, "object_index out of range");
  if (n == 0) return RT_OK;
  DeviceGuard g(c->device);
  std::vector<DbgHitH> hh((size_t)n);
  for (int i = 0; i < n; ++i)
    for (int a = 0; a < 3; ++a) {
      hh[i].ro[a] = (float)hits[i].ray_origin[a]; hh[i].rd[a] = (float)hits[i].ray_dir[a];
      hh[i].p[a] = (float)hits[i].p[a]; hh[i].n[a] = (float)hits[i].normal[a];
      hh[i].front = hits[i].front_face; hh[i].pad = 0;
    }
  DbgBuf B;
  DbgHitH* d_h = nullptr; float* d_u = nullptr; rt_debug_scatter_out* d_o = nullptr;
  CU(B.up(hh, &d_h)); CU(B.up(to_f32(uniforms, (size_t)n * RT_DEBUG_UNIFORMS), &d_u)); CU(B.out((size_t)n, &d_o));
  CU(launch_debug_scatter(c->ds, root, n, d_h, d_u, d_o, c->stream));
  CU(cudaMemcpyAsync(out, d_o, (size_t)n * sizeof(*out), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return RT_OK;
  RT_GUARD_END
}

rt_status rt_debug_get_ray(rt_camera* c, int32_t n, const int32_t* ij, const double* uniforms, float* ray_out, int32_t* used) {
  RT_GUARD_BEGIN
  if (!c || n < 0 || (n > 0 && (!ij || !uniforms || !ray_out))) return fail(RT_ERR_INVALID_ARGUMENT, "null argument");
  if (n == 0) return RT_OK;
  DeviceGuard g(c->device);
  DbgBuf B;
  int* d_ij = nullptr; float* d_u = nullptr; float* d_o = nullptr; int* d_used = nullptr;
  CU(B.up(std::vector<int>(ij, ij + 2 * (size_t)n), &d_ij));
  CU(B.up(to_f32(uniforms, (size_t)n * RT_DEBUG_UNIFORMS), &d_u));
  CU(B.out((size_t)n * 6, &d_o)); CU(B.out((size_t)n, &d_used));
  CU(launch_debug_get_ray(c->ds, n, d_ij, d_u, d_o, d_used, c->stream));
  CU(cudaMemcpyAsync(ray_out, d_o, (size_t)n * 6 * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  if (used) CU(cudaMemcpyAsync(used, d_used, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return RT_OK;
  RT_GUARD_END
}

rt_status rt_debug_light_pdf(rt_camera* c, int32_t light, int32_t n, const double* origin, const double* direction, float* value) {
  RT_GUARD_BEGIN
  if (!c || n < 0 || (n > 0 && (!origin || !direction || !value))) return fail(RT_ERR_INVALID_ARGUMENT, "null argument");
  if (light < 0 || light >= (int)c->hs->lights.size()) return fail(RT_ERR_INVALID_ARGUMENT, "light_index out of range");
  if (n == 0) return RT_OK;
  DeviceGuard g(c->device);
  DbgBuf B;
  float *d_o = nullptr, *d_d = nullptr, *d_v = nullptr;
  CU(B.up(to_f32(origin, 3 * (size_t)n), &d_o)); CU(B.up(to_f32(direction, 3 * (size_t)n), &d_d)); CU(B.out((size_t)n, &d_v));
  CU(launch_debug_light_pdf(c->ds, light, n, d_o, d_d, d_v, c->stream));
  CU(cudaMemcpyAsync(value, d_v, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return RT_OK;
  RT_GUARD_END
}

rt_status rt_debug_light_random_vec(rt_camera* c, int32_t light, int32_t n, const double* origin, const double* uniforms, float* out) {
  RT_GUARD_BEGIN
  if (!c || n < 0 || (n > 0 && (!origin || !uniforms || !out))) return fail(RT_ERR_INVALID_ARGUMENT, "null argument");
  if (light < 0 || light >= (int)c->hs->lights.size()) return fail(RT_ERR_INVALID_ARGUMENT, "light_index out of range");
  if (n == 0) return RT_OK;
  DeviceGuard g(c->device);
  DbgBuf B;
  float *d_o = nullptr, *d_u = nullptr, *d_v = nullptr;
  CU(B.up(to_f32(origin, 3 * (size_t)n), &d_o)); CU(B.up(to_f32(uniforms, (size_t)n * RT_DEBUG_UNIFORMS), &d_u)); CU(B.out(3 * (size_t)n, &d_v));
  CU(launch_debug_light_random(c->ds, light, n, d_o, d_u, d_v, c->stream));
  CU(cudaMemcpyAsync(out, d_v, 3 * (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return RT_OK;
  RT_GUARD_END
}

rt_status rt_debug_diffuse_bounce(rt_camera* c, int32_t n, const double* p, const double* normal, const double* uniforms, float* out) {
  RT_GUARD_BEGIN
  if (!c || n < 0 || (n > 0 && (!p || !normal || !uniforms || !out))) return fail(RT_ERR_INVALID_ARGUMENT, "null argument");
  if (n == 0) return RT_OK;
  DeviceGuard g(c->device);
  DbgBuf B;
  float *d_p = nullptr, *d_n = nullptr, *d_u = nullptr, *d_v = nullptr;
  CU(B.up(to_f32(p, 3 * (size_t)n), &d_p)); CU(B.up(to_f32(normal, 3 * (size_t)n), &d_n));
  CU(B.up(to_f32(uniforms, (size_t)n * RT_DEBUG_UNIFORMS), &d_u)); CU(B.out(6 * (size_t)n, &d_v));
  CU(launch_debug_diffuse(c->ds, n, d_p, d_n, d_u, d_v, c->stream));
  CU(cudaMemcpyAsync(out, d_v, 6 * (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return RT_OK;
  RT_GUARD_END
}

} // extern "C"

// ---- tiny device helper: raw stats -> rt_stats on the device (for the no-sync entry point) ----
namespace rt {
__global__ void k_finalize_stats(const unsigned long long* raw, rt_stats* out, int launches) {
  if (threadIdx.x || blockIdx.x) return;
  rt_stats s;
  s.pixels = raw[kStatPixels];
  s.samples_total = raw[kStatSamples];
  s.bounces_total = raw[kStatBounces];
  s.rays = raw[kStatRays];
  s.samples_min = (int32_t)raw[kStatSamplesMin];
  s.samples_max = (int32_t)raw[kStatSamplesMax];
  s.bounces_min = (int32_t)raw[kStatBouncesMin];
  s.bounces_max = (int32_t)raw[kStatBouncesMax];
  s.device_ms = 0;
  s.kernel_launches = launches;
  s.reserved = 0;
  s.node_visits = raw[kStatNodeVisits];
  s.prim_tests = raw[kStatPrimTests];
  *out = s;
}
cudaError_t launch_finalize_stats(const unsigned long long* raw, rt_stats* out, int launches, cudaStream_t st) {
  k_finalize_stats<<<1, 32, 0, st>>>(raw, out, launches);
  return cudaGetLastError();
}
} // namespace rt
