// rt_megakernel.cu — register-resident path tracer ("megakernel" integrator) and the
// primary-visibility parity kernel, for sm_100a.
//
// Work decomposition (all render kernels): persistent grid (resident CTAs only) pulling work items
// from an atomic queue, so the tail of a render is one item long instead of one wave long, and a GPU
// that owns only 1/8 of the tiles still fills its SMs evenly.
//
// k_render_pool<KIND, POOL> and k_render_trav (fixed spp, default mode — the benchmark path) are
// warp-persistent: a work item is (8x4 pixel block, sample chunk) and belongs to ONE warp; there is no
// CTA-wide barrier after scene staging.  Lanes take (pixel, sample) pairs from a warp-level queue
// (ballot + popc prefix over a warp-uniform cursor) whenever their path ends, so every iteration every
// lane generates one Philox block, traces one ray and shades one hit.  Radiance is accumulated per
// pixel in exact 64-bit fixed point, so the image does not depend on which lane took which sample, on
// the chunking or on the number of GPUs.
//   * k_render_pool<LIST>: tiny scenes, all primitives in shared memory, converged brute-force loop.
//   * k_render_pool<SAH>: small and medium trees, one whole while-while tree walk per iteration.
//   * k_render_trav (big SAH trees): traversal is resumable; a warp alternates traversal bursts (a few
//     node visits for every lane that is mid-ray) with shading/regeneration for the lanes whose ray
//     finished, switching when few lanes still traverse — the warp never waits for its longest
//     traversal with idle lanes.
//   * k_render_sorted (SORTED integrator): CTA-wide counting sort of the hits by material class between
//     the trace and the shade phase.
//
// k_render_stream / k_render_stream_trav (adaptive sampling / render modes / moments): a lane owns one pixel
// at a time and runs the reference's loop (src/camera.ts:400-423) in sample order, as the adaptive exit rule
// requires; lanes pull the next pixel from their warp's stream when theirs stops.
//
// k_render_adaptive (plain adaptive renders — the reference's DEFAULT options — of every scene the whole-query kernels serve):
// the exit rule needs a pixel's batch to be complete, not to have run on one lane.  A warp item is one batch of a group of
// pixels; its (pixel, sample) pairs go through the pair queue of k_render_pool, every finished sample is a 16-byte record, and
// one lane per pixel then adds the records in sample order and decides — bit for bit the sums and decisions of k_render_stream.
//
// All path state lives in registers; HBM sees the scene reads (L1/L2 resident), 24 B of atomics per
// (pixel, chunk) when chunks > 1, and 3 bytes per pixel of output.
#include <algorithm>

#include "rt_device.cuh"

namespace rt {

static constexpr int kTile = 16;
#ifndef RT_MIN_BLOCKS
#define RT_MIN_BLOCKS 2
#endif
// CTA geometry of k_render_pool<LIST> (warp-persistent: the CTA only shares the staged scene, so its size is free):
// threads x resident CTAs decides the register cap (65536 / (threads x CTAs), granularity 8) and the warps per SM.
#ifndef RT_LIST_THREADS
#define RT_LIST_THREADS 256
#endif
#ifndef RT_LIST_BLOCKS
#define RT_LIST_BLOCKS 3
#endif
// ... and of k_render_trav (deep trees: latency-bound on node fetches, so warps per SM matter more than spill-free registers)
#ifndef RT_TRAV_THREADS
#define RT_TRAV_THREADS 256
#endif
#ifndef RT_TRAV_BLOCKS
#define RT_TRAV_BLOCKS RT_MIN_BLOCKS
#endif
#ifndef RT_TRAV_MIN_LANES
#define RT_TRAV_MIN_LANES 20 // leave the traversal phase when this many lanes or fewer still traverse
#endif

RT_DEV unsigned long long warp_sum(unsigned long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
RT_DEV int warp_min(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
RT_DEV int warp_max(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// index 0..255 -> pixel inside the tile: each group of 32 covers an 8x4 block
RT_DEV void tile_pixel(int idx, int& px, int& py) {
  int lane = idx & 31, w = idx >> 5;
  px = (w & 1) * 8 + (lane & 7);
  py = (w >> 1) * 4 + (lane >> 3);
}

template <int KIND>
RT_DEV ListSmem stage_list(const DevScene& S, ListSmemData& sm) {
  if (KIND == BVH_LIST) {
    for (int s = threadIdx.x; s < S.n_slots; s += blockDim.x) {
      sm.p0[s] = ldg4(S.p0 + s);
      sm.p1[s] = ldg4(S.p1 + s);
      const F4 q2 = ldg4(S.p2 + s);
      sm.p2[s] = q2;
      sm.p3[s] = ldg4(S.p3 + s);
      I2 info = ldgi2(S.slot_info + s);
      const int ty = (info.y >> 30) & 3;
      // axis-aligned quads get one warp-uniform code per axis so the converged loop never selects components
      sm.type[s] = ty == OBJ_AAQUAD ? OBJ_AAQUAD + 1 + __float_as_int(q2.y) : ty;
      sm.mat[s] = info.x;
    }
    __syncthreads();
  }
  // the handle is made by a volatile asm placed after the barrier: every ld.shared depends on it, none can move above
  uint32_t base = KIND == BVH_LIST ? (uint32_t)__cvta_generic_to_shared(&sm) : 0u;
  asm volatile("mov.u32 %0, %0;" : "+r"(base));
  return ListSmem{base};
}

template <int KIND, bool LEAF_LOOP = true> // LEAF_LOOP: see leaves_intersect (rt_device.cuh)
RT_DEV bool closest_hit(const DevScene& S, const SmemList& L, const Ray& r, float& t, int& slot, WorkCount& wc) {
  RayPre pre = precompute(r, true); // LIST uses idir too (axis-aligned quads); unused parts are dead code
  t = CUDART_INF_F;
  slot = -1;
  ++wc.rays;
  if (KIND == BVH_LIST) { RT_COUNT_PRIMS(wc, S.n_slots); trace_list(S, L, r, pre, t, slot); }
  else if (KIND == BVH_SAH) trace_sah<LEAF_LOOP>(S, r, pre, t, slot, wc);
  else trace_ref(S, r, pre, t, slot);
  return slot >= 0;
}
template <int KIND, bool LEAF_LOOP = true>
RT_DEV bool closest_hit(const DevScene& S, const SmemList& L, const Ray& r, float& t, int& slot) {
  WorkCount wc;
  return closest_hit<KIND, LEAF_LOOP>(S, L, r, t, slot, wc);
}

struct PathState {
  Ray ray;
  V3 tp, radiance;
  int bounces;
  float listed_w; // shadow-ray estimator only: weight of a LISTED light's emission met by ps.ray (1, or the scattered ray's MIS weight)
};

// rayColor, part 1 (camera.ts:228-245): depth limit and Russian roulette.  True = the path ended.
RT_DEV bool path_pre(const DevCamera& cam, PathState& ps, Rng& g) {
  bool done = ps.bounces >= cam.depth;
  if (!done && cam.roulette && ps.bounces >= cam.rr_depth) {
    float p = fminf(maxc(ps.tp), 0.95f);
    done = g.next() > p;
    ps.tp = ps.tp * rcp_approx(p);
  }
  return done;
}

// rayColor, part 2 (camera.ts:249-319) given the closest hit (slot < 0: miss).  True = the path ended
// (its radiance is complete); otherwise ps.ray / ps.tp / ps.bounces describe the next call.
template <int KIND, bool LV = true> // LV: light records by 128-bit loads (light_ld4, rt_device.cuh)
RT_DEV bool path_post(const DevScene& S, const ListSmem* sm, const MixW& mw, PathState& ps, Rng& g, float t, int slot) {
  const DevCamera& cam = S.cam;
  if (slot < 0) { // camera.ts:252-258
    V3 ud = normalize3(ps.ray.d);
    float a = 0.5f * (ud.y + 1.0f);
    V3 bg = ld3(cam.bg_top) * (1.0f - a) + ld3(cam.bg_bottom) * a;
    ps.radiance = ps.radiance + bg * ps.tp;
    return true;
  }
  int type, root;
  F4 p0;
  if (KIND == BVH_LIST) { type = sm->type(slot); root = sm->mat(slot); p0 = sm->p0(slot); }
  else { I2 info = ldgi2(S.slot_info + slot); type = (info.y >> 30) & 3; root = info.x; p0 = ldg4(S.p0 + slot); }
  const Surf sf = surface_at(type, p0, ps.ray, t);
  const I4 mb = ldgi4(S.matB + root);
  const F4 ma = ldg4(S.matA + root);
  if (mb.w) { // emitted * throughput (camera.ts:261)
    F4 e = ldg4(S.matE + root);
    ps.radiance = ps.radiance + xyz(e) * ps.tp;
  }
  Scatter sc;
  if (mb.x == MAT_LAMBERT) { sc.kind = SCATTER_DIFFUSE; sc.attenuation = xyz(ma); sc.dir = mk3(0, 0, 0); }
  else if (mb.x == MAT_LIGHT) return true; // scatter == null: emitted only, bounce not counted (camera.ts:267-269)
  else sc = scatter_material(S, root, mb, ma, ps.ray.d, sf, g);
  if (sc.kind == SCATTER_NONE) return true;
  ++ps.bounces;
  if (sc.kind == SCATTER_SPECULAR) { // camera.ts:275-282
    ps.tp = ps.tp * sc.attenuation;
    ps.ray = Ray{sf.p, sc.dir};
    return false;
  }
  // camera.ts:285-315 with the mixture pdf of pdf.ts:57-99
  const float u_sel = g.next(), r1 = g.next(), r2 = g.next();
  V3 dir;
  float cosv, pdf_value;
  diffuse_bounce<LV>(S, mw, sf.p, sf.n, u_sel, r1, r2, dir, cosv, pdf_value);
  if (!(pdf_value > 0.0001f)) return true; // camera.ts:298-301 (NaN also ends the path)
  ps.tp = ps.tp * (sc.attenuation * (cosv * rcp_approx(pdf_value)));
  ps.ray = Ray{sf.p, dir};
  return false;
}

// One whole rayColor call on the path's current ray.
template <int KIND, bool LEAF_LOOP = true, bool LV = true>
RT_DEV bool path_step(const DevScene& S, const SmemList& L, const ListSmem& sm, const MixW& mw, PathState& ps, Rng& g,
                      WorkCount& wc) {
  if (path_pre(S.cam, ps, g)) return true;
  float t;
  int slot;
  closest_hit<KIND, LEAF_LOOP>(S, L, ps.ray, t, slot, wc); // world.hit(r, (0.001, inf)) — camera.ts:249
  return path_post<KIND, LV>(S, &sm, mw, ps, g, t, slot);
}

// ---------------------------------------------------------------------------------------------------
// RT_LIGHTS_SHADOW_RAYS — rayColor with next-event estimation instead of the reference's one-sample mixture (rt_b200.h).
// At a diffuse scatter the reference draws ONE direction from 0.5 cosine + 0.5 p_light and follows it.  Here the two
// halves become two rays: a shadow ray along a direction drawn from p_light (the light list's own generators and pdfs,
// pdf.ts:57-99 / quad.ts / sphere.ts) answers "which listed light does this direction meet first" and carries that
// light's emission; the scattered ray is cosine-distributed and carries everything else.  Where the scattered ray itself
// meets a listed light both rays estimate the same emission, and the two estimates are combined with the balance
// heuristic (weights p_light / (p_light + p_cos) and p_cos / (p_light + p_cos)): next-event estimation alone has a
// 1/d^2 singularity next to a light (the ceiling around the Cornell light, 0.01 above it) that the reference's mixture
// does not have.  Each part is unbiased, the weights sum to 1: the pixel's expectation is the reference's
// (tests/test_gpu_shadow_rays.py compares converged images with the oracle's mixture estimator).  Depth limit,
// roulette, bounce counting, specular scatter and the pdf <= 1e-4 cut of camera.ts:298-301 are the reference's.
// ---------------------------------------------------------------------------------------------------
RT_DEV bool is_listed_light(const DevScene& S, int slot) {
  bool listed = false;
  for (int k = 0; k < S.n_lights; ++k) listed |= S.lights[k].slot == slot;
  return listed;
}
RT_DEV float light_list_pdf(const DevScene& S, const MixW& mw, V3 p, V3 dir) { // HittableListPDF.value, pdf.ts:74-86
  float sum = 0.f;
  for (int k = 0; k < mw.nl; ++k) sum += light_pdf_value(S, S.lights[k], p, dir);
  return sum / (float)mw.nl;
}
template <int KIND>
RT_DEV bool path_post_shadow(const DevScene& S, const SmemList& L, const ListSmem* sm, const MixW& mw, PathState& ps, Rng& g, float t,
                             int slot, WorkCount& wc) {
  const DevCamera& cam = S.cam;
  if (slot < 0) { // camera.ts:252-258
    V3 ud = normalize3(ps.ray.d);
    float a = 0.5f * (ud.y + 1.0f);
    V3 bg = ld3(cam.bg_top) * (1.0f - a) + ld3(cam.bg_bottom) * a;
    ps.radiance = ps.radiance + bg * ps.tp;
    return true;
  }
  int type, root;
  F4 p0;
  if (KIND == BVH_LIST) { type = sm->type(slot); root = sm->mat(slot); p0 = sm->p0(slot); }
  else { I2 info = ldgi2(S.slot_info + slot); type = (info.y >> 30) & 3; root = info.x; p0 = ldg4(S.p0 + slot); }
  const Surf sf = surface_at(type, p0, ps.ray, t);
  const I4 mb = ldgi4(S.matB + root);
  const F4 ma = ldg4(S.matA + root);
  if (mb.w) { // emitted * throughput (camera.ts:261); a listed light met by a scattered ray shares it with the shadow ray
    F4 e = ldg4(S.matE + root);
    const float w = ps.listed_w < 1.f && is_listed_light(S, slot) ? ps.listed_w : 1.f;
    ps.radiance = ps.radiance + xyz(e) * ps.tp * w;
  }
  Scatter sc;
  if (mb.x == MAT_LAMBERT) { sc.kind = SCATTER_DIFFUSE; sc.attenuation = xyz(ma); sc.dir = mk3(0, 0, 0); }
  else if (mb.x == MAT_LIGHT) return true;
  else sc = scatter_material(S, root, mb, ma, ps.ray.d, sf, g);
  if (sc.kind == SCATTER_NONE) return true;
  ++ps.bounces;
  ps.listed_w = 1.f;
  if (sc.kind == SCATTER_SPECULAR) {
    ps.tp = ps.tp * sc.attenuation;
    ps.ray = Ray{sf.p, sc.dir};
    return false;
  }
  const Onb onb = make_onb<true>(sf.n);
  const float kInvPi = 0.31830988618f;
  if (mw.nl > 0) {
    // ---- the shadow ray: one listed light chosen uniformly (pdf.ts:88-99 picks its generator the same way) ----
    const float u_sel = g.next(), r1 = g.next(), r2 = g.next();
    const int chosen = min((int)(u_sel * (float)mw.nl), mw.nl - 1);
    const V3 ldir = light_random_vec(S.lights[chosen], sf.p, r1, r2);
    const float p_cos = dot3(ldir, onb.w) * kInvPi;
    const float p_light = light_list_pdf(S, mw, sf.p, ldir);
    if (p_cos > 0.f && p_light > 0.0001f) { // (NaN pdfs — a sphere light seen from inside — fail the comparison)
      float ts;
      int ss;
      closest_hit<KIND, false>(S, L, Ray{sf.p, ldir}, ts, ss, wc);
      if (ss >= 0 && is_listed_light(S, ss)) {
        int root_l;
        if (KIND == BVH_LIST) root_l = sm->mat(ss);
        else root_l = ldgi2(S.slot_info + ss).x;
        if (ldgi4(S.matB + root_l).w) {
          const F4 e = ldg4(S.matE + root_l);
          // f / p_light * w_light = (albedo p_cos) / (p_light + p_cos)
          ps.radiance = ps.radiance + xyz(e) * (ps.tp * sc.attenuation) * (p_cos * rcp_approx(p_light + p_cos));
        }
      }
    }
  }
  // ---- the scattered ray: cosine-distributed, pdf = scatter pdf, so the weight is the albedo ----
  const float r3 = g.next(), r4 = g.next();
  const V3 dir = onb_local(onb, cosine_direction(r3, r4));
  const float p_cos2 = dot3(dir, onb.w) * kInvPi;
  if (!(p_cos2 > 0.0001f)) return true; // camera.ts:298-301
  if (mw.nl > 0) {
    const float p_light2 = light_list_pdf(S, mw, sf.p, dir);
    ps.listed_w = p_light2 > 0.0001f ? p_cos2 * rcp_approx(p_light2 + p_cos2) : 1.f; // the shadow ray never takes a direction of pdf <= 1e-4
  }
  ps.tp = ps.tp * sc.attenuation;
  ps.ray = Ray{sf.p, dir};
  return false;
}
template <int KIND>
RT_DEV bool path_step_shadow(const DevScene& S, const SmemList& L, const ListSmem& sm, const MixW& mw, PathState& ps, Rng& g,
                             WorkCount& wc) {
  if (path_pre(S.cam, ps, g)) return true;
  float t;
  int slot;
  closest_hit<KIND, false>(S, L, ps.ray, t, slot, wc);
  return path_post_shadow<KIND>(S, L, &sm, mw, ps, g, t, slot, wc);
}

// writeColorToBuffer (camera.ts:455-472) of one channel: sqrt gamma, then the Uint8ClampedArray store
// (NaN/negative -> 0, >255 -> 255).  Shared by write_pixel and the denoiser's output (rt_denoise.cuh).
RT_DEV uint8_t gamma_rgb8(float c) {
  const double v = floor(255.999 * sqrt((double)c));
  return !(v > 0.0) ? 0 : (v >= 255.0 ? 255 : (uint8_t)v);
}
// finalColor (camera.ts:326-340, default mode) + writeColorToBuffer (camera.ts:455-472)
RT_DEV void write_pixel(const RenderParams& R, size_t pi, V3 fc) {
  if (R.rgb8) {
    R.rgb8[pi * 3] = gamma_rgb8(fc.x);
    R.rgb8[pi * 3 + 1] = gamma_rgb8(fc.y);
    R.rgb8[pi * 3 + 2] = gamma_rgb8(fc.z);
  }
  if (R.linear) { R.linear[pi * 3] = fc.x; R.linear[pi * 3 + 1] = fc.y; R.linear[pi * 3 + 2] = fc.z; }
}

// RenderStats contribution of a lane (renderStats.ts:21-35): warp-reduce, one atomic each.
// n_pixels pixels were completed, each with pixel_samples samples; n_samples paths were traced.
// (px_smin, px_smax): fewest / most samples of any pixel this lane completed.
RT_DEV void flush_work(const RenderParams& R, const WorkCount& wc) { // instrumented build only: executed traversal work
#ifdef RT_COUNT_EVENTS
  if (!R.stats) return;
  const unsigned long long v = warp_sum((unsigned long long)wc.visits), p = warp_sum((unsigned long long)wc.prims);
  if ((threadIdx.x & 31) == 0 && (v || p)) { atomicAdd(R.stats + kStatNodeVisits, v); atomicAdd(R.stats + kStatPrimTests, p); }
#else
  (void)R; (void)wc;
#endif
}
RT_DEV void flush_stats_range(const RenderParams& R, unsigned n_pixels, int px_smin, int px_smax, unsigned n_samples,
                              unsigned bounces_sum, unsigned rays, int min_b, int max_b) {
  if (!R.stats) return;
  unsigned long long px = warp_sum((unsigned long long)n_pixels);
  unsigned long long ss = warp_sum((unsigned long long)n_samples);
  unsigned long long bs = warp_sum((unsigned long long)bounces_sum);
  unsigned long long rs = warp_sum((unsigned long long)rays);
  int smin = warp_min(n_pixels ? px_smin : 0x7fffffff), smax = warp_max(n_pixels ? px_smax : 0);
  int bmin = warp_min(n_samples ? min_b : 0x7fffffff), bmax = warp_max(n_samples ? max_b : 0);
  if ((threadIdx.x & 31) == 0 && (ss || px || rs)) {
    atomicAdd(R.stats + kStatPixels, px);
    atomicAdd(R.stats + kStatSamples, ss);
    atomicAdd(R.stats + kStatBounces, bs);
    atomicAdd(R.stats + kStatRays, rs);
    atomicMin(R.stats + kStatSamplesMin, (unsigned long long)smin);
    atomicMax(R.stats + kStatSamplesMax, (unsigned long long)smax);
    atomicMin(R.stats + kStatBouncesMin, (unsigned long long)bmin);
    atomicMax(R.stats + kStatBouncesMax, (unsigned long long)bmax);
  }
}
RT_DEV void flush_stats(const RenderParams& R, unsigned n_pixels, int pixel_samples, unsigned n_samples, unsigned bounces_sum,
                        unsigned rays, int min_b, int max_b) {
  flush_stats_range(R, n_pixels, pixel_samples, pixel_samples, n_samples, bounces_sum, rays, min_b, max_b);
}

// radiance -> 2^-32 fixed point.  NaN and negatives count as 0, a single sample saturates at 65536
// (the reference has no clamp; a 15-unit light needs a 4000x throughput spike to get there).
RT_DEV unsigned long long to_fixed(float x) {
  x = fminf(fmaxf(x, 0.f), 65536.f); // fmaxf(NaN, 0) = 0
  return __float2ull_rz(x * 4294967296.f);
}
RT_DEV float from_fixed(unsigned long long s, int samples) { return (float)(((double)s * (1.0 / 4294967296.0)) / (double)samples); }

// ---------------------------------------------------------------------------------------------------
// Warp-level work items: (8x4 pixel block, sample chunk)
// ---------------------------------------------------------------------------------------------------
struct WarpItem {
  int blk, px0, py0, s_begin, s_end;
};
// Pops items until one touches the region.  False = queue exhausted.
// One GPU: items = (block of the region's tile grid, chunk).  Several GPUs: items = (run of part_count consecutive blocks,
// chunk) and the block is the ONE this part owns in that run (owned_block_of_run) — a GPU never pops another GPU's work
// (round 1 popped every block of the image and skipped 7 of 8: at 8 GPUs that was 166 dependent atomics per warp, most of
// the ~0.8 ms each GPU lost against the ideal eighth of the one-GPU time).
RT_DEV bool next_warp_item(const RenderParams& R, int samples, int blocks_per_row, unsigned lane, WarpItem& it) {
  const int chunks = R.chunks;
  const int blocks_x = R.tiles_x * 2, blocks_y = R.tiles_y * 4; // 8x4 blocks covering the tile grid
  const int n_items = (R.part_count > 1 ? R.n_runs : blocks_x * blocks_y) * chunks;
  for (;;) {
    int item = 0;
    if (lane == 0) item = atomicAdd(R.queue, 1);
    item = __shfl_sync(0xffffffffu, item, 0);
    if (item >= n_items) return false;
    const int blk = item / chunks, chunk = item - blk * chunks;
    if (R.part_count > 1) {
      const unsigned i = owned_block_of_run((unsigned)(R.run0 + blk), R.part_index, R.part_count);
      it.px0 = (int)(i % (unsigned)blocks_per_row) * 8;
      it.py0 = (int)(i / (unsigned)blocks_per_row) * 4;
    } else {
      const int bx = blk % blocks_x, by = blk / blocks_x;
      it.px0 = (R.x0 / kTile) * kTile + bx * 8;
      it.py0 = (R.y0 / kTile) * kTile + by * 4;
    }
    if (it.px0 >= R.x1 || it.py0 >= R.y1 || it.px0 + 8 <= R.x0 || it.py0 + 4 <= R.y0) continue; // block outside the region
    it.blk = blk;
    const int cnt = R.s_cnt > 0 ? R.s_cnt : samples; // progressive pass: a window of the pixel's samples
    it.s_begin = R.s0 + (int)(((long long)cnt * chunk) / chunks);
    it.s_end = R.s0 + (int)(((long long)cnt * (chunk + 1)) / chunks);
    return true;
  }
}

// Per-warp pixel accumulators: 32 pixels x (r, g, b) x three 21-bit limbs of the fixed-point sums.  A limb
// accumulator absorbs 2048 additions before it can overflow, so the adds need no carry and no return
// value: they are fire-and-forget shared-memory reductions.
RT_DEV void acc_clear(unsigned int* acc, unsigned lane) {
#pragma unroll
  for (int k = 0; k < 9; ++k) acc[lane * 9 + k] = 0;
  __syncwarp();
}
RT_DEV void acc_add(unsigned int* acc, int lp, V3 radiance) {
  const float c[3] = {radiance.x, radiance.y, radiance.z};
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const unsigned long long v = to_fixed(c[k]); // < 2^49
    const unsigned l0 = (unsigned)v & 0x1fffffu, l1 = (unsigned)(v >> 21) & 0x1fffffu, l2 = (unsigned)(v >> 42);
    atomicAdd(&acc[lp * 9 + 3 * k], l0);
    atomicAdd(&acc[lp * 9 + 3 * k + 1], l1);
    if (l2) atomicAdd(&acc[lp * 9 + 3 * k + 2], l2); // radiance >= 1024: rare
  }
}
RT_DEV void acc_read(const unsigned int* acc, unsigned lane, unsigned long long sum[3]) {
#pragma unroll
  for (int k = 0; k < 3; ++k)
    sum[k] = (unsigned long long)acc[lane * 9 + 3 * k] + ((unsigned long long)acc[lane * 9 + 3 * k + 1] << 21) +
             ((unsigned long long)acc[lane * 9 + 3 * k + 2] << 42);
}

// Item epilogue: lane k owns pixel k of the block.  chunks == 1: write the pixel.  Otherwise add the
// chunk's sums to `accum` and let the warp that completes the block's last chunk write it.
// Returns 1 when this lane wrote its pixel.
RT_DEV unsigned item_epilogue(const RenderParams& R, const DevCamera& cam, const WarpItem& it, unsigned lane, const unsigned long long sum[3]) {
  const int i = it.px0 + (int)(lane & 7u), j = it.py0 + (int)(lane >> 3);
  const bool active = i >= R.x0 && i < R.x1 && j >= R.y0 && j < R.y1;
  const size_t pi = (size_t)j * cam.width + i;
  const int div = R.div_samples > 0 ? R.div_samples : cam.samples; // progressive pass: samples taken so far
  unsigned wrote = 0;
  if (R.chunks == 1 && !R.keep_accum) {
    if (active) {
      wrote = 1;
      write_pixel(R, pi, mk3(from_fixed(sum[0], div), from_fixed(sum[1], div), from_fixed(sum[2], div)));
    }
  } else {
    if (active) {
      atomicAdd(R.accum + pi * 4 + 0, sum[0]);
      atomicAdd(R.accum + pi * 4 + 1, sum[1]);
      atomicAdd(R.accum + pi * 4 + 2, sum[2]);
    }
    __threadfence();
    __syncwarp();
    int last = 0;
    if (lane == 0) last = atomicAdd(R.tile_done + it.blk, 1) == R.chunks - 1;
    last = __shfl_sync(0xffffffffu, last, 0);
    if (last) { // every partial sum of the block is in `accum`
      __threadfence();
      if (active) {
        wrote = 1;
        const unsigned long long* a = R.accum + pi * 4;
        write_pixel(R, pi, mk3(from_fixed(__ldcg(a), div), from_fixed(__ldcg(a + 1), div), from_fixed(__ldcg(a + 2), div)));
      }
    }
  }
  return wrote;
}

// =========================================================================================
// k_render_pool — fixed spp, default mode, whole closest-hit query per iteration.
// POOL = true : the (pixel, sample) pairs of the item are one pool shared by the 32 lanes.
// POOL = false: lane k keeps pixel k and walks its samples in order with register accumulators
//               (neighbouring pixels cost about the same: the shared-memory reductions and the queue
//               arithmetic are not worth their ~1-2 %).
// Both give bit-identical images (exact fixed-point sums).
// =========================================================================================
// Register budget: the LIST kernel runs 3 CTAs/SM (<= 80 registers, a few spilled words): measured +3 %
// over 2 CTAs/SM on Cornell; tree kernels keep 2 (their traversal stacks live in local memory already).
// Code placement.  The hot loops of these kernels sit at the edge of the instruction cache, and their speed depends on where the
// loop starts relative to the 128-byte instruction lines: an unrelated change that moved the tree walk of k_render_pool<SAH> by ONE
// instruction cost weekend-final 5.8 % (36.1 -> 38.2 ms at 64 spp, same loop body; profiles/r02c_c3_regression.log).  CUDA C++ has
// no alignment control for code, so the kernels can be shifted by N one-instruction no-ops executed once at kernel entry
// (RT_PAD_SAH, swept in profiles/r02c_code_pad_sweep.log; k_render_pool<LIST>, k_render_trav, k_render_sorted and k_render_adaptive
// were swept too and do not care: profiles/r02c_code_pad_sweep2.log).
#ifndef RT_PAD_LIST
#define RT_PAD_LIST 0
#endif
#ifndef RT_PAD_SAH
#define RT_PAD_SAH 3 // weekend-final at 64 spp, pads 0..7 (with the vector light loads): 38.1 38.4 38.0 36.9 37.2 37.3 37.8 38.2 ms; with member reads 36.0 (pad 0), 35.9 (pad 3); the LIST kernel does not care (26.44-26.54)
#endif
template <int N>
RT_DEV void code_pad() {
#pragma unroll
  for (int k = 0; k < N; ++k) asm volatile("nanosleep.u32 0;");
}
template <int KIND, bool POOL>
__global__ void __launch_bounds__(KIND == BVH_LIST ? RT_LIST_THREADS : 256, KIND == BVH_LIST ? RT_LIST_BLOCKS : RT_MIN_BLOCKS)
k_render_pool(const DevScene S, const RenderParams R) {
  code_pad<KIND == BVH_SAH ? RT_PAD_SAH : (KIND == BVH_LIST && !POOL ? RT_PAD_LIST : 0)>();
  __shared__ ListSmemData sm_data;
  __shared__ unsigned int s_acc[POOL ? (KIND == BVH_LIST ? RT_LIST_THREADS : 256) / 32 : 1][32 * 9];
  const ListSmem sm = stage_list<KIND>(S, sm_data);
  const ListSmem& L = sm;
  const DevCamera& cam = S.cam;
  const MixW mw = make_mixw(S);
  const unsigned lane = threadIdx.x & 31u;
  const unsigned lt_mask = (1u << lane) - 1u;
  unsigned int* acc = s_acc[POOL ? (threadIdx.x >> 5) : 0];

  // RenderStats partials of this lane over all items of its warp
  unsigned int st_pixels = 0, st_paths = 0, st_bounces = 0;
  WorkCount wc;
  int st_bmin = 0x7fffffff, st_bmax = 0;

  WarpItem it;
  while (next_warp_item(R, cam.samples, (cam.width + 7) >> 3, lane, it)) {
    const int pool = 32 * (it.s_end - it.s_begin); // (pixel, sample) pairs of this item
    if (POOL) acc_clear(acc, lane);

    PathState ps{Ray{mk3(0, 0, 0), mk3(0, 0, 1)}, mk3(1, 1, 1), mk3(0, 0, 0), 0};
    int lp = (int)lane, sample = 0; // current pair
    int pi_x = it.px0 + (int)(lane & 7u), pi_y = it.py0 + (int)(lane >> 3);
    int next = POOL ? 0 : it.s_begin; // POOL: warp-uniform cursor into the pool; else this lane's next sample
    bool have = false, retired = false;
    unsigned long long own[3] = {0, 0, 0}; // !POOL: this lane's pixel sums
    Rng g;
    if (!POOL) retired = !(pi_x >= R.x0 && pi_x < R.x1 && pi_y >= R.y0 && pi_y < R.y1);

    for (;;) {
      const bool want = !have && !retired;
      bool fresh = false;
      if (POOL) {
        // ---- warp-level queue: lanes without a path take the next (pixel, sample) pairs in lane order ----
        const unsigned m = __ballot_sync(0xffffffffu, want);
        if (want) {
          const int idx = next + __popc(m & lt_mask);
          if (idx >= pool) retired = true;
          else {
            lp = idx & 31;
            sample = it.s_begin + (idx >> 5);
            pi_x = it.px0 + (lp & 7);
            pi_y = it.py0 + (lp >> 3);
            // pairs of pixels outside the region are dropped; the lane takes another one next round
            fresh = pi_x >= R.x0 && pi_x < R.x1 && pi_y >= R.y0 && pi_y < R.y1;
            have = fresh;
          }
        }
        next += __popc(m);
      } else if (want) {
        if (next >= it.s_end) retired = true;
        else { sample = next++; fresh = true; have = true; }
      }
      if (__all_sync(0xffffffffu, retired)) break;
      bool ended = false;
      if (have) {
        const uint32_t pixel = (uint32_t)pi_y * (uint32_t)cam.width + (uint32_t)pi_x;
        if (fresh) { ps.tp = mk3(1, 1, 1); ps.radiance = mk3(0, 0, 0); ps.bounces = 0; }
        g.begin(pixel, (uint32_t)sample, (uint32_t)ps.bounces, S.seed_lo, S.seed_hi); // one Philox block per bounce
        if (fresh) ps.ray = camera_ray(cam, pi_x, pi_y, g, true);
        // LV (light_ld4): member reads for the lane-keeps-pixel LIST kernel and for the tree walk — the vector loads cost them
        // 1.9 % (Cornell) and 3 % (weekend-final, which has no light at all: register allocation and code placement of the walk)
        ended = path_step<KIND, true, (KIND == BVH_LIST && POOL) || KIND == BVH_REFERENCE>(S, L, sm, mw, ps, g, wc);
      }
      // every way a path can end (miss, light, absorbed, roulette, depth, pdf 0) meets here: ONE copy of the end-of-path code
      // instead of one per exit of path_step (measured on Cornell 1024^2 @256: 31.45 -> 30.19 ms)
      __syncwarp();
      if (ended) { // pixel.add(rayColor, bounces) — renderStats.ts:76-88
        if (POOL) acc_add(acc, lp, ps.radiance);
        else { own[0] += to_fixed(ps.radiance.x); own[1] += to_fixed(ps.radiance.y); own[2] += to_fixed(ps.radiance.z); }
        ++st_paths;
        st_bounces += (unsigned)ps.bounces;
        st_bmin = min(st_bmin, ps.bounces);
        st_bmax = max(st_bmax, ps.bounces);
        have = false;
      }
    }
    __syncwarp();
    unsigned long long sum[3] = {own[0], own[1], own[2]};
    if (POOL) acc_read(acc, lane, sum);
    st_pixels += item_epilogue(R, cam, it, lane, sum);
    __syncwarp(); // acc is cleared at the top of the next item
  }
  flush_stats(R, st_pixels, cam.samples, st_paths, st_bounces, wc.rays, st_bmin, st_bmax);
  flush_work(R, wc);
}

// =========================================================================================
// k_render_sorted — fixed spp, default mode: CTA-wide path pool, hits sorted by material class
// between the trace and the shade phase.
//
// In k_render_pool about half of the issued instructions are shading code run by 10-50 % of a warp's
// lanes (every lane's hit has its own material: walls, light, glass, miss).  Here the 256 threads of a
// CTA share one pool of (pixel, sample) pairs (the eight warp items the warps popped), and every
// iteration is
//   A  trace      all threads, one ray each (converged: LIST tests every primitive for every ray)
//   B  sort       class = material type of the hit | miss | idle; counting sort over the CTA:
//                 match.any + popc inside a warp, 64 (class, warp) counts in shared memory, one
//                 redundant 64-entry scan per warp (no third barrier)
//   C  exchange   a thread writes its path (six 16-byte records) at the sorted position and takes the
//                 path at position threadIdx.x: warps now hold one class each
//   D  shade      path_post for the hit, exact fixed-point accumulation of finished paths, a new pair
//                 from the pool for their threads (warp-aggregated shared atomic), then the Philox
//                 block + roulette test of the next bounce for everybody
// Two barriers per iteration.  A path killed by the roulette test keeps its thread for one idle trace
// phase (slot = -2) so accumulation has a single call site.  Which thread runs which pair is
// scheduling-dependent; the image is not (counter-based RNG + exact sums), so the output is
// bit-identical to k_render_pool's.
// =========================================================================================
enum : int { CLS_MISS = 6, CLS_IDLE = 7, CLS_COUNT = 8 };

struct SortSmem {
  float4 st[6][256];            // G0 (o, t) G1 (d, slot) G2 (tp, bounces) G3 (radiance, item<<5|pixel) G4 (q0..q3) G5 (q4, avail|block<<3, pixel, sample)
  unsigned int acc[8][32 * 9];  // per warp item: 32 pixels x 9 limbs (acc_add)
  int cnt[CLS_COUNT * 8];       // [class][warp]
  int it_px0[8], it_py0[8], it_sb[8], it_se[8], it_blk[8];
  int cursor;
};

template <int KIND>
__global__ void __launch_bounds__(256, 3) k_render_sorted(const DevScene S, const RenderParams R) {
  __shared__ ListSmemData sm_data;
  __shared__ SortSmem ss;
  const ListSmem sm = stage_list<KIND>(S, sm_data);
  const ListSmem& L = sm;
  const DevCamera& cam = S.cam;
  const MixW mw = make_mixw(S);
  const unsigned tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
  const unsigned lt_mask = (1u << lane) - 1u;
  const unsigned full = 0xffffffffu;

  unsigned int st_pixels = 0, st_paths = 0, st_bounces = 0, st_rays = 0;
  int st_bmin = 0x7fffffff, st_bmax = 0;

  for (;;) {
    // ---- CTA item = the eight warp items popped by the eight warps ----
    {
      WarpItem it{0, 0, 0, 0, 0};
      const bool got = next_warp_item(R, cam.samples, (cam.width + 7) >> 3, lane, it);
      if (lane == 0) {
        ss.it_px0[warp] = it.px0; ss.it_py0[warp] = it.py0; ss.it_blk[warp] = it.blk;
        ss.it_sb[warp] = got ? it.s_begin : 0; ss.it_se[warp] = got ? it.s_end : 0;
      }
      acc_clear(ss.acc[warp], lane);
      if (tid == 0) ss.cursor = 0;
    }
    __syncthreads();
    int maxlen = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) maxlen = max(maxlen, ss.it_se[k] - ss.it_sb[k]);
    if (maxlen == 0) break; // the queue is exhausted for every warp
    const int pool = maxlen * 256; // pair idx -> item idx & 7, pixel (idx >> 3) & 31, sample (idx >> 8); short items drop theirs

    PathState ps{Ray{mk3(0, 0, 0), mk3(0, 0, 1)}, mk3(1, 1, 1), mk3(0, 0, 0), 0};
    Rng g;
    g.seed_lo = S.seed_lo; g.seed_hi = S.seed_hi;
    g.k0 = g.k1 = g.stream = g.block = 0; g.q0 = g.q1 = g.q2 = g.q3 = g.q4 = 0; g.avail = 0;
    uint32_t pixel = 0, sample = 0;
    int wl = 0;
    bool have = false, dead = false;

    for (;;) {
      // ---- A: trace ----
      float t = CUDART_INF_F;
      int slot = -1, key = CLS_IDLE;
      if (have) {
        int type = CLS_MISS;
        if (dead) slot = -2;
        else {
          ++st_rays;
          closest_hit<KIND>(S, L, ps.ray, t, slot); // world.hit(r, (0.001, inf)) — camera.ts:249
          if (slot >= 0) {
            const int root = KIND == BVH_LIST ? sm.mat(slot) : ldgi2(S.slot_info + slot).x;
            type = __ldg(&S.matB[root].x);
          }
        }
        // sort order: lambert, light, miss, metal, glass, mixed, layered — the class that shades longest
        // comes first (its range starts warp-aligned) and shares its one mixed warp with the cheapest classes
        key = (int)((0x2651430u >> (4 * type)) & 7u);
      }
      // ---- B: counting sort by class over the CTA ----
      const unsigned grp = __match_any_sync(full, key);
      if (lane < CLS_COUNT) ss.cnt[lane * 8 + warp] = 0;
      __syncwarp();
      if ((grp & lt_mask) == 0) ss.cnt[key * 8 + warp] = __popc(grp);
      __syncthreads();
      const int c0 = ss.cnt[2 * lane], c1 = ss.cnt[2 * lane + 1];
      int incl = c0 + c1;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(full, incl, o);
        if (lane >= (unsigned)o) incl += v;
      }
      const int excl = incl - (c0 + c1);
      const int e = key * 8 + (int)warp;
      int dst = __shfl_sync(full, excl, e >> 1);
      const int c0e = __shfl_sync(full, c0, e >> 1);
      if (e & 1) dst += c0e;
      dst += __popc(grp & lt_mask);
      const int n_live = __shfl_sync(full, excl, (CLS_IDLE * 8) >> 1); // paths in flight = first idle position
      const bool exhausted = ss.cursor >= pool;
      if (n_live == 0 && exhausted) break;
      // ---- C: exchange ----
      if (have) {
        ss.st[0][dst] = make_float4(ps.ray.o.x, ps.ray.o.y, ps.ray.o.z, t);
        ss.st[1][dst] = make_float4(ps.ray.d.x, ps.ray.d.y, ps.ray.d.z, __int_as_float(slot));
        ss.st[2][dst] = make_float4(ps.tp.x, ps.tp.y, ps.tp.z, __int_as_float(ps.bounces));
        ss.st[3][dst] = make_float4(ps.radiance.x, ps.radiance.y, ps.radiance.z, __int_as_float(wl));
        ss.st[4][dst] = make_float4(__uint_as_float(g.q0), __uint_as_float(g.q1), __uint_as_float(g.q2), __uint_as_float(g.q3));
        ss.st[5][dst] = make_float4(__uint_as_float(g.q4), __int_as_float(g.avail | (int)(g.block << 3)), __uint_as_float(pixel),
                                    __uint_as_float(sample));
      }
      __syncthreads();
      have = (int)tid < n_live;
      if (have) {
        const float4 a0 = ss.st[0][tid], a1 = ss.st[1][tid], a2 = ss.st[2][tid], a3 = ss.st[3][tid], a4 = ss.st[4][tid],
                     a5 = ss.st[5][tid];
        ps.ray.o = mk3(a0.x, a0.y, a0.z); t = a0.w;
        ps.ray.d = mk3(a1.x, a1.y, a1.z); slot = __float_as_int(a1.w);
        ps.tp = mk3(a2.x, a2.y, a2.z); ps.bounces = __float_as_int(a2.w);
        ps.radiance = mk3(a3.x, a3.y, a3.z); wl = __float_as_int(a3.w);
        g.q0 = __float_as_uint(a4.x); g.q1 = __float_as_uint(a4.y); g.q2 = __float_as_uint(a4.z); g.q3 = __float_as_uint(a4.w);
        g.q4 = __float_as_uint(a5.x);
        const int ab = __float_as_int(a5.y);
        g.avail = ab & 7; g.block = (uint32_t)ab >> 3;
        pixel = __float_as_uint(a5.z); sample = __float_as_uint(a5.w);
        g.k0 = pixel; g.k1 = sample; g.stream = (uint32_t)ps.bounces;
      }
      // ---- D: shade, retire, refill, start the next bounce ----
      bool start = false, fresh = false;
      if (have) {
        const bool fin = slot == -2 || path_post<KIND>(S, &sm, mw, ps, g, t, slot);
        if (fin) { // pixel.add(rayColor, bounces) — renderStats.ts:76-88
          acc_add(ss.acc[wl >> 5], wl & 31, ps.radiance);
          ++st_paths;
          st_bounces += (unsigned)ps.bounces;
          st_bmin = min(st_bmin, ps.bounces);
          st_bmax = max(st_bmax, ps.bounces);
          have = false;
        } else start = true;
      }
      int px = 0, py = 0;
      const unsigned need = __ballot_sync(full, !have);
      if (need != 0u && !exhausted) {
        const int leader = __ffs(need) - 1;
        int base = 0;
        if ((int)lane == leader) base = atomicAdd(&ss.cursor, __popc(need));
        base = __shfl_sync(full, base, leader);
        const int idx = base + __popc(need & lt_mask);
        if (!have && idx < pool) {
          const int w = idx & 7, lp = (idx >> 3) & 31;
          const int smp = ss.it_sb[w] + (idx >> 8);
          px = ss.it_px0[w] + (lp & 7);
          py = ss.it_py0[w] + (lp >> 3);
          if (smp < ss.it_se[w] && px >= R.x0 && px < R.x1 && py >= R.y0 && py < R.y1) {
            have = fresh = start = true;
            wl = w * 32 + lp;
            sample = (uint32_t)smp;
            pixel = (uint32_t)py * (uint32_t)cam.width + (uint32_t)px;
            ps.tp = mk3(1, 1, 1); ps.radiance = mk3(0, 0, 0); ps.bounces = 0;
          }
        }
      }
      dead = false;
      if (start) {
        g.begin(pixel, sample, (uint32_t)ps.bounces, S.seed_lo, S.seed_hi); // one Philox block per bounce
        if (fresh) ps.ray = camera_ray(cam, px, py, g, true);
        dead = path_pre(cam, ps, g);
      }
    }
    __syncthreads(); // everybody has left the loop; accumulators are final
    {
      unsigned long long sum[3];
      acc_read(ss.acc[warp], lane, sum);
      const WarpItem it{ss.it_blk[warp], ss.it_px0[warp], ss.it_py0[warp], ss.it_sb[warp], ss.it_se[warp]};
      if (it.s_end > it.s_begin) st_pixels += item_epilogue(R, cam, it, lane, sum);
    }
    __syncthreads(); // descriptors and accumulators are rewritten at the top
  }
  flush_stats(R, st_pixels, cam.samples, st_paths, st_bounces, st_rays, st_bmin, st_bmax);
}

// =========================================================================================
// k_render_trav — fixed spp, default mode, SAH trees: traversal interleaved with shading.
// Lane states: NONE (needs a pair) -> BEGIN (bounce not started) -> TRACE (mid-traversal, advanced in
// bursts) -> HIT (closest hit known, not shaded) -> BEGIN | NONE.
// =========================================================================================
enum : int { ST_NONE = 0, ST_BEGIN = 1, ST_TRACE = 2, ST_HIT = 3 };

__global__ void __launch_bounds__(RT_TRAV_THREADS, RT_TRAV_BLOCKS) k_render_trav(const DevScene S, const RenderParams R) {
  __shared__ unsigned int s_acc[RT_TRAV_THREADS / 32][32 * 9];
  const DevCamera& cam = S.cam;
  const MixW mw = make_mixw(S);
  const unsigned lane = threadIdx.x & 31u;
  const unsigned lt_mask = (1u << lane) - 1u;
  unsigned int* acc = s_acc[threadIdx.x >> 5];
  TravStack stack;

  unsigned int st_pixels = 0, st_paths = 0, st_bounces = 0;
  WorkCount wc;
  int st_bmin = 0x7fffffff, st_bmax = 0;

  WarpItem it;
  while (next_warp_item(R, cam.samples, (cam.width + 7) >> 3, lane, it)) {
    const int pool = 32 * (it.s_end - it.s_begin);
    acc_clear(acc, lane);

    PathState ps{Ray{mk3(0, 0, 0), mk3(0, 0, 1)}, mk3(1, 1, 1), mk3(0, 0, 0), 0};
    int lp = 0, sample = 0, pi_x = 0, pi_y = 0;
    int next = 0;
    int st = ST_NONE;
    bool retired = false, fresh = false;
    Trav tv{-1, 0, CUDART_INF_F, -1};
    BoxPre bp{mk3(0, 0, 0), mk3(0, 0, 0)};
    Rng g;

    for (;;) {
      // ---- shading phase, part 1: finish the bounce of lanes whose ray is done ----
      if (st == ST_HIT) {
        const bool done = path_post<BVH_SAH>(S, nullptr, mw, ps, g, tv.tbest, tv.sbest);
        st = done ? ST_NONE : ST_BEGIN;
        if (done) {
          acc_add(acc, lp, ps.radiance);
          ++st_paths;
          st_bounces += (unsigned)ps.bounces;
          st_bmin = min(st_bmin, ps.bounces);
          st_bmax = max(st_bmax, ps.bounces);
        }
      }
      // ---- warp-level queue: lanes without a path take the next (pixel, sample) pairs in lane order.  AFTER the shading above:
      //      a lane whose path just ended (a third of the shaded lanes on the 100 k-sphere scene) starts its next path in this
      //      very round; with the queue at the top of the loop it sat out the whole traversal phase that follows ----
      const bool want = st == ST_NONE && !retired;
      const unsigned m = __ballot_sync(0xffffffffu, want);
      if (want) {
        const int idx = next + __popc(m & lt_mask);
        if (idx >= pool) retired = true;
        else {
          lp = idx & 31;
          sample = it.s_begin + (idx >> 5);
          pi_x = it.px0 + (lp & 7);
          pi_y = it.py0 + (lp >> 3);
          if (pi_x >= R.x0 && pi_x < R.x1 && pi_y >= R.y0 && pi_y < R.y1) { st = ST_BEGIN; fresh = true; }
        }
      }
      next += __popc(m);
      if (__all_sync(0xffffffffu, st == ST_NONE && retired)) break;

      // ---- shading phase, part 2: start the next bounce / the new path ----
      if (st == ST_BEGIN) {
        const uint32_t pixel = (uint32_t)pi_y * (uint32_t)cam.width + (uint32_t)pi_x;
        if (fresh) { ps.tp = mk3(1, 1, 1); ps.radiance = mk3(0, 0, 0); ps.bounces = 0; }
        g.begin(pixel, (uint32_t)sample, (uint32_t)ps.bounces, S.seed_lo, S.seed_hi); // one Philox block per bounce
        if (fresh) { ps.ray = camera_ray(cam, pi_x, pi_y, g, true); fresh = false; }
        if (path_pre(cam, ps, g)) { // ended by the depth limit or the roulette: nothing to trace
          acc_add(acc, lp, ps.radiance);
          ++st_paths;
          st_bounces += (unsigned)ps.bounces;
          st_bmin = min(st_bmin, ps.bounces);
          st_bmax = max(st_bmax, ps.bounces);
          st = ST_NONE;
        } else {
          ++wc.rays;
          RT_COUNT_PRIMS(wc, S.n_unbounded);
          trav_begin(S, ps.ray, tv);
          bp = box_precompute(ps.ray);
          st = tv.cur >= 0 ? ST_TRACE : ST_HIT;
        }
      }

      // ---- traversal phase, in bursts: a lane walks up to R.trav_burst inner nodes until it holds a leaf
      //      (while-while), the warp reconverges at the end of that loop and intersects the leaves together.
      //      One vote per burst; the phase ends when few lanes still traverse and others have work waiting.
      //      (Two votes per node visit with separate inner / leaf rounds measured 171 ms on the 100 k-sphere
      //      scene at 8 spp; bursts of 2 / 4 / 8 / 16: 138 / 128 / 127 / 140 ms.) ----
      //      Keeping the leaves of a burst parked until they outnumber the traversing lanes (bursts + the old
      //      ST_LEAF rounds) was measured too: 136-139 ms against 126-129 ms.
      for (;;) {
        const unsigned tt = __ballot_sync(0xffffffffu, st == ST_TRACE);
        if (tt == 0) break;
        if (__popc(tt) <= R.trav_min_lanes) {
          // lanes that could do something else: shade a finished ray, start a bounce, take a new pair
          if (__any_sync(0xffffffffu, st == ST_HIT || st == ST_BEGIN || (st == ST_NONE && !retired))) break;
        }
        if (st == ST_TRACE) {
          int steps = 0;
          TravLeaves lv{0, 0, 0, 0};
#pragma unroll 1 // unrolled copies of the node visit cost more instruction cache than they save
          while (tv.cur >= 0 && lv.a == 0 && steps < R.trav_burst) { trav_inner(S, bp, tv, stack, lv); ++steps; RT_COUNT_VISIT(wc); }
          RT_COUNT_LEAVES(wc, lv);
          if (lv.a != 0) trav_leaves(S, ps.ray, bp, tv, lv);
          st = tv.cur >= 0 ? ST_TRACE : ST_HIT;
        }
      }
    }
    __syncwarp();
    unsigned long long sum[3];
    acc_read(acc, lane, sum);
    st_pixels += item_epilogue(R, cam, it, lane, sum);
    __syncwarp();
  }
  flush_stats(R, st_pixels, cam.samples, st_paths, st_bounces, wc.rays, st_bmin, st_bmax);
  flush_work(R, wc);
}

// =========================================================================================
// k_render_stream — adaptive sampling, render modes, moments.  One lane = one pixel at a time, its samples in
// order (the adaptive exit of camera.ts:348-368 is sequential: src/camera.ts:400-423 is this loop), FP64
// sum(ill), sum(ill^2) and an FP32 colour sum like the reference.  A lane whose pixel stopped takes the next
// pixel of its warp's stream instead of waiting for a tile: with adaptive sampling neighbouring pixels
// differ 10x in sample count.  The stream = 8x4 pixel blocks popped from the global queue whenever the
// current block runs out, so a warp never drains before the render does.  Measured against the
// tile-synchronous kernel it replaced (one thread per pixel, CTA = 16x16 tile; identical output): 100 k
// spheres 3037 -> 1925 ms, 480 spheres 497 -> 416 ms, layered/mixed 500 -> 483 ms, Cornell 157 -> 170 ms
// (its cheap all-black pixels now share warps with the expensive ones).
// =========================================================================================
// Per-pixel second moment for the parity tests: sum of squared deviations from the running mean (Welford), so a
// pixel whose samples differ in the 4th digit only (sky gradient under pixel jitter) still gets its variance —
// sum(c^2) - n mean^2 in FP32 cancels to noise there.  `color` already holds the new sample; n = samples so far.
RT_DEV void moments_add(V3 color, V3 x, int n, float& m2x, float& m2y, float& m2z) {
  if (n < 2) return;
  const float ip = 1.0f / (float)(n - 1), in = 1.0f / (float)n;
  const V3 mean_old = (color - x) * ip, mean_new = color * in;
  m2x = fmaf(x.x - mean_old.x, x.x - mean_new.x, m2x);
  m2y = fmaf(x.y - mean_old.y, x.y - mean_new.y, m2y);
  m2z = fmaf(x.z - mean_old.z, x.z - mean_new.z, m2z);
}

// pixelConverged (camera.ts:348-368) on the FP64 sums, WITHOUT its two divisions and two square roots:
//   variance = (s2 - s1^2 / n) / (n - 1),  mean = s1 / n,  converged  <=>  variance <= 0 | NaN  |  1.96 sqrt(variance / n) <= tol mean
// and for s1 > 0 the last condition is  1.96^2 (n s2 - s1^2) <= tol^2 (n - 1) s1^2  (both sides of the reference's inequality are
// non-negative, multiply through by n^2 (n - 1) and square); for s1 <= 0 the right-hand side of the reference is <= 0 and only the
// variance <= 0 branch can hold.  Six FP64 operations instead of ~100 instructions of DDIV / DSQRT sequences: lanes reach their checks
// at different iterations, so that block used to run in nearly every iteration of the warp's sample loop for one or two lanes.
RT_DEV bool pixel_converged(double s1, double s2, int samples, float tol) {
  const double n = (double)samples;
  const double D = fma(n, s2, -(s1 * s1)); // n (n - 1) variance
  if (!(D > 0.0)) return true;             // variance <= 0 or NaN (camera.ts:360)
  const double t2 = (double)tol * (double)tol * (n - 1.0);
  return s1 > 0.0 && 3.8416 * D <= t2 * (s1 * s1);
}

// Out of line on purpose: these run once per pixel / per 64 pixels, and the sample loop of k_render_stream is
// instruction-cache bound like every kernel here (measured: with them inlined the Cornell loop is 13 % slower).
__device__ __noinline__ void stream_write_pixel(uint8_t* rgb8, float* linear, float* moments, int width, int mode, int depth, int max_samples,
                                                int i, int j, int samples, unsigned bounces_sum, float cx, float cy, float cz, float m2x,
                                                float m2y, float m2z) {
  V3 fc; // finalColor (camera.ts:326-340)
  if (mode == 1) {
    float avg = samples > 0 ? (float)((double)bounces_sum / (double)samples) : 0.f;
    fc = mk3(0, 0, fminf(avg / (float)depth, 1.0f));
  } else if (mode == 2) {
    fc = mk3(fminf((float)samples / (float)max_samples, 1.0f), 0, 0);
  } else {
    fc = mk3(cx, cy, cz) * (float)(1.0 / (double)samples);
  }
  const size_t pi = (size_t)j * width + i;
  RenderParams out{};
  out.rgb8 = rgb8;
  out.linear = linear;
  write_pixel(out, pi, fc);
  if (moments) {
    float* m = moments + pi * 8;
    m[0] = cx; m[1] = cy; m[2] = cz; m[3] = m2x; m[4] = m2y; m[5] = m2z;
    m[6] = (float)samples; m[7] = (float)bounces_sum;
  }
}
// PixelStats of a pixel between two passes of a progressive render.  Out of line: once per pixel per pass.
__device__ __noinline__ int pixstate_load(const PixState* ps, size_t pi, float& cx, float& cy, float& cz, double& s1, double& s2, int& samples,
                                          unsigned& bounces) {
  const PixState p = ps[pi];
  cx = p.color[0]; cy = p.color[1]; cz = p.color[2];
  s1 = p.sum_ill; s2 = p.sum_ill2; samples = p.samples; bounces = p.bounces;
  return p.done;
}
__device__ __noinline__ void pixstate_store(PixState* ps, size_t pi, float cx, float cy, float cz, double s1, double s2, int samples,
                                            unsigned bounces, int done) {
  PixState p;
  p.color[0] = cx; p.color[1] = cy; p.color[2] = cz;
  p.sum_ill = s1; p.sum_ill2 = s2; p.samples = samples; p.bounces = bounces; p.done = done;
  ps[pi] = p;
}
// Welford second moment of a pixel a later progressive pass picks up: stream_write_pixel left it in the moments buffer at
// the end of the previous pass (FP32 in, FP32 out, so the sequence continues as in the one-shot render).  Not in PixState,
// whose layout k_render_adaptive's 64-bit accessors rely on.  Out of line like pixstate_load.
__device__ __noinline__ V3 moments_m2_load(const float* moments, size_t pi) {
  const float* m = moments + pi * 8;
  return mk3(m[3], m[4], m[5]);
}

// The warp's pixel stream: lanes named in `want` take the next pixels, in lane order, from the current 8x4 block;
// when it runs out the next block that belongs to this GPU and touches the region is popped from the queue.
// Called by the whole warp, only when some lane needs a pixel (rare next to the sample loop).
struct StreamTake {
  int i, j, got;                 // this lane's new pixel
  int cursor, blk_x0, blk_y0;    // the stream after the call (warp-uniform)
  int queue_empty;
};
__device__ __noinline__ StreamTake stream_take(unsigned want, int cursor, int blk_x0, int blk_y0, bool queue_empty, int* queue,
                                               int n_items, int tiles_x, int rx0, int ry0, int rx1, int ry1, int part_index, int part_count,
                                               int run0, int blocks_per_row, unsigned lane) {
  StreamTake tk{0, 0, 0, cursor, blk_x0, blk_y0, queue_empty ? 1 : 0};
  const unsigned lt_mask = (1u << lane) - 1u, full = 0xffffffffu;
  bool mine = (want >> lane) & 1u;
  while (want != 0u) {
    if (tk.cursor >= 32) {
      if (tk.queue_empty) break;
      bool found = false;
      for (;;) {
        int item = 0;
        if (lane == 0) item = atomicAdd(queue, 1);
        item = __shfl_sync(full, item, 0);
        if (item >= n_items) { tk.queue_empty = 1; break; }
        int bx, by;
        if (part_count > 1) { // item = a run of part_count blocks: the one block this part owns in it
          const unsigned i = owned_block_of_run((unsigned)(run0 + item), part_index, part_count);
          bx = (int)(i % (unsigned)blocks_per_row) * 8;
          by = (int)(i / (unsigned)blocks_per_row) * 4;
        } else {
          const int tile = item >> 3, sub = item & 7;
          const int tx = (rx0 / kTile) + tile % tiles_x, ty = (ry0 / kTile) + tile / tiles_x;
          bx = tx * kTile + (sub & 1) * 8;
          by = ty * kTile + (sub >> 1) * 4;
        }
        if (bx >= rx1 || by >= ry1 || bx + 8 <= rx0 || by + 4 <= ry0) continue;
        tk.blk_x0 = bx; tk.blk_y0 = by; tk.cursor = 0;
        found = true;
        break;
      }
      if (!found) break;
    }
    const int p = tk.cursor + __popc(want & lt_mask);
    if (mine && p < 32) {
      const int pi = tk.blk_x0 + (p & 7), pj = tk.blk_y0 + (p >> 3);
      if (pi >= rx0 && pi < rx1 && pj >= ry0 && pj < ry1) { tk.i = pi; tk.j = pj; tk.got = 1; mine = false; } // else: skipped, ask again
    }
    tk.cursor = min(32, tk.cursor + __popc(want));
    want = __ballot_sync(full, mine);
  }
  return tk;
}

#ifndef RT_STREAM_LIST_BLOCKS
#define RT_STREAM_LIST_BLOCKS RT_MIN_BLOCKS
#endif
// SHADOW: the shadow-ray estimator (path_post_shadow).  RESUME: a later progressive pass (k_render_stream_resume), which
// picks pixels up from R.pixstate.  Its warps may take only pixels that stopped in earlier passes, so a warp left without a
// pixel goes on taking until the stream is exhausted; with moments it also reloads each pixel's Welford M2
// (moments_m2_load).  One-shot renders never take such a pixel, so a warp with no pixel after a take has exhausted the
// stream.  Separate instantiations keep their kernels as they were: the reload in a shared kernel cost the one-shot
// moments render 0.3 % and changed the spills of another (profiles/README.md section 9.2).
template <int KIND, bool SHADOW, bool RESUME>
__device__ __forceinline__ void render_stream(const DevScene& S, const RenderParams& R) {
  __shared__ ListSmemData sm_data;
  const ListSmem sm = stage_list<KIND>(S, sm_data);
  const ListSmem& L = sm;
  const DevCamera& cam = S.cam;
  const MixW mw = make_mixw(S);
  const unsigned lane = threadIdx.x & 31u, full = 0xffffffffu;
  const int n_items = R.part_count > 1 ? R.n_runs : R.tiles_x * R.tiles_y * 8; // 8x4 blocks, eight per 16x16 tile | one owned block per run

  // the warp's stream (warp-uniform)
  int blk_x0 = 0, blk_y0 = 0, cursor = 32;
  bool queue_empty = false;
  // this lane's pixel: PixelStats (renderStats.ts:67-88)
  bool have_px = false, need_path = true;
  int i = 0, j = 0, samples = 0;
  V3 color = mk3(0, 0, 0);
  unsigned int bounces_sum = 0;
  double sum_ill = 0, sum_ill2 = 0; // PixelStats.sumIll / sumIll2 up to the last check
  float b_ill = 0, b_ill2 = 0;      // ... plus the current batch (<= aBatch samples) in FP32
  int countdown = 1;                // samples until the next convergence check
  float m2x = 0, m2y = 0, m2z = 0;
  PathState ps{Ray{mk3(0, 0, 0), mk3(0, 0, 1)}, mk3(1, 1, 1), mk3(0, 0, 0), 0};
  Rng g;
  // RenderStats tallies of this lane over all its pixels
  unsigned int t_pixels = 0, t_samples = 0, t_bounces = 0;
  WorkCount wc;
  int t_smin = 0x7fffffff, t_smax = 0, t_bmin = 0x7fffffff, t_bmax = 0;

  // progressive pass: the pixel stops at `cap` samples (a multiple of aBatch) and its PixelStats wait in R.pixstate
  const int cap = R.pass_cap > 0 ? min(R.pass_cap, cam.samples) : cam.samples;
  int samples0 = 0;
  unsigned int bounces0 = 0;
  auto finish_pixel = [&](bool final_) {
    stream_write_pixel(R.rgb8, R.linear, R.moments, cam.width, cam.mode, cam.depth, cam.samples, i, j, samples, bounces_sum, color.x,
                       color.y, color.z, m2x, m2y, m2z);
    if (R.pixstate) pixstate_store(R.pixstate, (size_t)j * cam.width + i, color.x, color.y, color.z, sum_ill, sum_ill2, samples, bounces_sum, final_ ? 1 : 0);
    if (final_) { // RenderStats.addPixel (renderStats.ts:21-35) once per pixel, when it is complete
      ++t_pixels;
      t_smin = min(t_smin, samples);
      t_smax = max(t_smax, samples);
    }
    t_samples += (unsigned)(samples - samples0); // the work of this pass
    t_bounces += bounces_sum - bounces0;
    have_px = false;
  };

  for (;;) {
    // ---- lanes without a pixel take the next pixels of the stream, in lane order ----
    const unsigned want = __ballot_sync(full, !have_px);
    if (want != 0u) {
      const StreamTake tk = stream_take(want, cursor, blk_x0, blk_y0, queue_empty, R.queue, n_items, R.tiles_x, R.x0, R.y0, R.x1,
                                        R.y1, R.part_index, R.part_count, R.run0, (cam.width + 7) >> 3, lane);
      cursor = tk.cursor; blk_x0 = tk.blk_x0; blk_y0 = tk.blk_y0; queue_empty = tk.queue_empty != 0;
      if (tk.got) {
        i = tk.i; j = tk.j;
        have_px = true;
        need_path = true;
        samples = 0; bounces_sum = 0;
        color = mk3(0, 0, 0);
        sum_ill = 0; sum_ill2 = 0;
        b_ill = b_ill2 = 0.f;
        countdown = cam.a_batch;
        m2x = m2y = m2z = 0;
        samples0 = 0; bounces0 = 0;
        if (R.pixstate && R.s0 > 0) { // a later pass (s0 = the previous cap): pick the pixel up where the last pass left it
          if (pixstate_load(R.pixstate, (size_t)j * cam.width + i, color.x, color.y, color.z, sum_ill, sum_ill2, samples, bounces_sum)) have_px = false;
          else if constexpr (RESUME) {
            if (R.moments) { const V3 m2 = moments_m2_load(R.moments, (size_t)j * cam.width + i); m2x = m2.x; m2y = m2.y; m2z = m2.z; }
          }
          samples0 = samples; bounces0 = bounces_sum;
        }
      }
    }
    if (__all_sync(full, !have_px)) {
      if constexpr (RESUME) {
        if (!(queue_empty && cursor >= 32)) continue; // every pixel taken had stopped in an earlier pass: take more
      }
      break; // stream exhausted and every pixel written
    }

    bool stop = have_px && cam.samples <= 0; // while (0 < 0): the pixel gets no sample at all
    bool final_ = stop;
    bool ended = false;
    if (have_px && !stop) {
      const uint32_t pixel = (uint32_t)j * (uint32_t)cam.width + (uint32_t)i;
      if (need_path) { ps.tp = mk3(1, 1, 1); ps.radiance = mk3(0, 0, 0); ps.bounces = 0; ps.listed_w = 1.f; }
      g.begin(pixel, (uint32_t)samples, (uint32_t)ps.bounces, S.seed_lo, S.seed_hi);
      if (need_path) {
        ps.ray = camera_ray(cam, i, j, g, true);
        need_path = false;
      }
      ended = SHADOW ? path_step_shadow<KIND>(S, L, sm, mw, ps, g, wc) : path_step<KIND, false>(S, L, sm, mw, ps, g, wc);
    }
    __syncwarp(); // every way a path can end meets here: ONE copy of the end-of-sample code (see k_render_pool)
    {
      if (ended) { // pixel.add(rayColor, bounces, useAdaptiveSampling)
        color = color + ps.radiance;
        ++samples;
        bounces_sum += (unsigned)ps.bounces;
        t_bmin = min(t_bmin, ps.bounces);
        t_bmax = max(t_bmax, ps.bounces);
        if (cam.adaptive) { // illuminance (vec3.ts:239-242); FP32 partial sums of one batch, folded into FP64 at the check
          const float il = fmaf(0.299f, ps.radiance.x, fmaf(0.587f, ps.radiance.y, 0.114f * ps.radiance.z));
          b_ill += il;
          b_ill2 = fmaf(il, il, b_ill2);
        }
        if (R.moments) moments_add(color, ps.radiance, samples, m2x, m2y, m2z);
        need_path = true;
        // while (pixel.samples < samples && !pixelConverged(pixel)) — camera.ts:406, evaluated for the next sample
        final_ = samples >= cam.samples;
        // the check runs when samples % aBatch == 0 (camera.ts:348-368): a countdown instead of a division per sample
        bool check = false;
        if (cam.adaptive && --countdown == 0) {
          countdown = cam.a_batch;
          sum_ill += (double)b_ill;
          sum_ill2 += (double)b_ill2;
          b_ill = b_ill2 = 0.f;
          check = samples >= 2;
        }
        if (!final_ && check) final_ = pixel_converged(sum_ill, sum_ill2, samples, cam.a_tol);
        stop = final_ || samples >= cap;
      }
    }
    if (stop) finish_pixel(final_);
  }
  flush_stats_range(R, t_pixels, t_smin, t_smax, t_samples, t_bounces, wc.rays, t_bmin, t_bmax);
  flush_work(R, wc);
}
template <int KIND, bool SHADOW = false>
__global__ void __launch_bounds__(256, KIND == BVH_LIST ? RT_STREAM_LIST_BLOCKS : RT_MIN_BLOCKS) k_render_stream(const DevScene S, const RenderParams R) {
  render_stream<KIND, SHADOW, false>(S, R);
}
template <int KIND, bool SHADOW = false>
__global__ void __launch_bounds__(256, KIND == BVH_LIST ? RT_STREAM_LIST_BLOCKS : RT_MIN_BLOCKS) k_render_stream_resume(const DevScene S, const RenderParams R) {
  render_stream<KIND, SHADOW, true>(S, R);
}

// =========================================================================================
// k_render_stream_trav — k_render_stream for deep SAH trees: the pixel stream of k_render_stream with the
// resumable traversal of k_render_trav (bursts interleaved with shading), so a lane whose ray finished
// early shades, takes its next sample or its next pixel while the others still walk the tree.  Per-pixel
// arithmetic and its order are those of k_render_stream: identical output.  RESUME as in render_stream.
// =========================================================================================
template <bool RESUME>
__device__ __forceinline__ void render_stream_trav(const DevScene& S, const RenderParams& R) {
  const DevCamera& cam = S.cam;
  const MixW mw = make_mixw(S);
  const unsigned lane = threadIdx.x & 31u, full = 0xffffffffu;
  const int n_items = R.part_count > 1 ? R.n_runs : R.tiles_x * R.tiles_y * 8; // 8x4 blocks, eight per 16x16 tile | one owned block per run
  TravStack stack;

  int blk_x0 = 0, blk_y0 = 0, cursor = 32; // the warp's pixel stream (warp-uniform)
  bool queue_empty = false;
  bool have_px = false; // this lane's pixel: PixelStats (renderStats.ts:67-88)
  int i = 0, j = 0, samples = 0;
  V3 color = mk3(0, 0, 0);
  unsigned int bounces_sum = 0;
  double sum_ill = 0, sum_ill2 = 0;
  float b_ill = 0, b_ill2 = 0;
  int countdown = 1;
  float m2x = 0, m2y = 0, m2z = 0;
  PathState ps{Ray{mk3(0, 0, 0), mk3(0, 0, 1)}, mk3(1, 1, 1), mk3(0, 0, 0), 0}; // this lane's path
  Rng g;
  int st = ST_NONE;
  bool fresh = false;
  Trav tv{-1, 0, CUDART_INF_F, -1};
  BoxPre bp{mk3(0, 0, 0), mk3(0, 0, 0)};
  unsigned int t_pixels = 0, t_samples = 0, t_bounces = 0;
  WorkCount wc;
  int t_smin = 0x7fffffff, t_smax = 0, t_bmin = 0x7fffffff, t_bmax = 0;

  const int cap = R.pass_cap > 0 ? min(R.pass_cap, cam.samples) : cam.samples; // progressive pass (see k_render_stream)
  int samples0 = 0;
  unsigned int bounces0 = 0;
  auto finish_pixel = [&](bool final_) {
    stream_write_pixel(R.rgb8, R.linear, R.moments, cam.width, cam.mode, cam.depth, cam.samples, i, j, samples, bounces_sum, color.x,
                       color.y, color.z, m2x, m2y, m2z);
    if (R.pixstate) pixstate_store(R.pixstate, (size_t)j * cam.width + i, color.x, color.y, color.z, sum_ill, sum_ill2, samples, bounces_sum, final_ ? 1 : 0);
    if (final_) {
      ++t_pixels;
      t_smin = min(t_smin, samples);
      t_smax = max(t_smax, samples);
    }
    t_samples += (unsigned)(samples - samples0);
    t_bounces += bounces_sum - bounces0;
    have_px = false;
  };
  // pixel.add(rayColor, bounces, useAdaptiveSampling) + the loop condition of camera.ts:406 for the next sample
  auto end_sample = [&]() {
    color = color + ps.radiance;
    ++samples;
    bounces_sum += (unsigned)ps.bounces;
    t_bmin = min(t_bmin, ps.bounces);
    t_bmax = max(t_bmax, ps.bounces);
    if (cam.adaptive) {
      const float il = fmaf(0.299f, ps.radiance.x, fmaf(0.587f, ps.radiance.y, 0.114f * ps.radiance.z));
      b_ill += il;
      b_ill2 = fmaf(il, il, b_ill2);
    }
    if (R.moments) moments_add(color, ps.radiance, samples, m2x, m2y, m2z);
    bool final_ = samples >= cam.samples;
    bool check = false;
    if (cam.adaptive && --countdown == 0) {
      countdown = cam.a_batch;
      sum_ill += (double)b_ill;
      sum_ill2 += (double)b_ill2;
      b_ill = b_ill2 = 0.f;
      check = samples >= 2;
    }
    if (!final_ && check) final_ = pixel_converged(sum_ill, sum_ill2, samples, cam.a_tol); // camera.ts:348-368
    if (final_ || samples >= cap) { finish_pixel(final_); st = ST_NONE; }
    else { st = ST_BEGIN; fresh = true; }
  };

  for (;;) {
    // ---- lanes without a pixel take the next pixels of the stream ----
    const unsigned want = __ballot_sync(full, st == ST_NONE && !have_px);
    if (want != 0u) {
      const StreamTake tk = stream_take(want, cursor, blk_x0, blk_y0, queue_empty, R.queue, n_items, R.tiles_x, R.x0, R.y0, R.x1,
                                        R.y1, R.part_index, R.part_count, R.run0, (cam.width + 7) >> 3, lane);
      cursor = tk.cursor; blk_x0 = tk.blk_x0; blk_y0 = tk.blk_y0; queue_empty = tk.queue_empty != 0;
      if (tk.got) {
        i = tk.i; j = tk.j;
        have_px = true;
        samples = 0; bounces_sum = 0;
        color = mk3(0, 0, 0);
        sum_ill = 0; sum_ill2 = 0;
        b_ill = b_ill2 = 0.f;
        countdown = cam.a_batch;
        m2x = m2y = m2z = 0;
        samples0 = 0; bounces0 = 0;
        bool skip = false;
        if (R.pixstate && R.s0 > 0) {
          skip = pixstate_load(R.pixstate, (size_t)j * cam.width + i, color.x, color.y, color.z, sum_ill, sum_ill2, samples, bounces_sum) != 0;
          samples0 = samples; bounces0 = bounces_sum;
        }
        if constexpr (RESUME) {
          if (!skip && R.moments) { const V3 m2 = moments_m2_load(R.moments, (size_t)j * cam.width + i); m2x = m2.x; m2y = m2.y; m2z = m2.z; }
        }
        if (skip) have_px = false;
        else if (cam.samples <= 0) finish_pixel(true); // while (0 < 0): the pixel gets no sample at all
        else { st = ST_BEGIN; fresh = true; }
      }
    }
    if (__all_sync(full, st == ST_NONE && !have_px)) {
      if constexpr (RESUME) {
        if (!(queue_empty && cursor >= 32)) continue; // every pixel taken had stopped in an earlier pass: take more
      }
      break; // stream exhausted and every pixel written
    }

    // ---- shading phase: finish the bounce of lanes whose ray is done, start the next bounce / sample ----
    if (st == ST_HIT) {
      if (path_post<BVH_SAH>(S, nullptr, mw, ps, g, tv.tbest, tv.sbest)) end_sample();
      else st = ST_BEGIN;
    }
    if (st == ST_BEGIN) {
      const uint32_t pixel = (uint32_t)j * (uint32_t)cam.width + (uint32_t)i;
      if (fresh) { ps.tp = mk3(1, 1, 1); ps.radiance = mk3(0, 0, 0); ps.bounces = 0; }
      g.begin(pixel, (uint32_t)samples, (uint32_t)ps.bounces, S.seed_lo, S.seed_hi);
      if (fresh) { ps.ray = camera_ray(cam, i, j, g, true); fresh = false; }
      if (path_pre(cam, ps, g)) end_sample(); // ended by the depth limit or the roulette: nothing to trace
      else {
        ++wc.rays;
        RT_COUNT_PRIMS(wc, S.n_unbounded);
        trav_begin(S, ps.ray, tv);
        bp = box_precompute(ps.ray);
        st = tv.cur >= 0 ? ST_TRACE : ST_HIT;
      }
    }

    // ---- traversal bursts (see k_render_trav) ----
    for (;;) {
      const unsigned tt = __ballot_sync(full, st == ST_TRACE);
      if (tt == 0) break;
      if (__popc(tt) <= R.trav_min_lanes) {
        if (__any_sync(full, st == ST_HIT || st == ST_BEGIN || (st == ST_NONE && !(queue_empty && cursor >= 32)))) break;
      }
      if (st == ST_TRACE) {
        int steps = 0;
          TravLeaves lv{0, 0, 0, 0};
#pragma unroll 1
        while (tv.cur >= 0 && lv.a == 0 && steps < R.trav_burst) { trav_inner(S, bp, tv, stack, lv); ++steps; RT_COUNT_VISIT(wc); }
        RT_COUNT_LEAVES(wc, lv);
        if (lv.a != 0) trav_leaves(S, ps.ray, bp, tv, lv);
        st = tv.cur >= 0 ? ST_TRACE : ST_HIT;
      }
    }
  }
  flush_stats_range(R, t_pixels, t_smin, t_smax, t_samples, t_bounces, wc.rays, t_bmin, t_bmax);
  flush_work(R, wc);
}
__global__ void __launch_bounds__(256, RT_MIN_BLOCKS) k_render_stream_trav(const DevScene S, const RenderParams R) {
  render_stream_trav<false>(S, R);
}
__global__ void __launch_bounds__(256, RT_MIN_BLOCKS) k_render_stream_trav_resume(const DevScene S, const RenderParams R) {
  render_stream_trav<true>(S, R);
}

// =========================================================================================
// k_render_adaptive — adaptive sampling (the reference's default) at the lane occupancy of the fixed-spp kernels.
//
// k_render_stream gives a pixel to ONE lane until it converges: camera.ts:348-368 decides after every aBatch samples whether
// the pixel goes on, so its samples cannot be dealt out freely.  But the decision only needs the batch to be COMPLETE, not to
// have run on one lane.  Here the unit of work is one batch of a GROUP of pixels (1-4 8x4 blocks): the (pixel, sample)
// pairs of the group's still active pixels x aBatch samples form a pool that the 32 lanes drain with the pair queue of
// k_render_pool<.., true> (a lane whose path ends takes the next pair: no lane waits for a neighbour's long pixel); every
// finished sample is written as a 16-byte record (radiance, bounces) into the warp's slice of a scratch array; when the pool
// is dry each pixel's records are added to its PixelStats IN SAMPLE ORDER by one lane — the very sequence of FP32 / FP64
// additions k_render_stream performs — followed by the convergence test.  Same streams, same sums, same decisions: the image
// and the statistics are those of k_render_stream bit for bit (tests/test_gpu_parity.py compares the two kernels).
// A group's batches must run one after the other; the groups are independent.  The queue deals out (batch r, group g)
// batch-major, a warp that pops (r, g) waits for tile_done[g] == r (by then (r - 1, g) was popped a whole round of groups
// earlier: the wait is almost never taken; every CTA of the persistent grid is resident, so the owner of (r - 1, g) runs),
// and groups whose pixels are all final are skipped with one load.  No kernel-wide barrier between batches, and the tail of
// the render is one batch of one group instead of one whole pixel (17 ms at 1024 spp).
// =========================================================================================
// CTA shape per scene kind (Cornell 1024 spp / weekend-final 512 spp with the reference's defaults, ms): the list walk runs best
// at 20 warps of 96 registers (128 x 5: 114.6; 256 x 2: 120.3; 128 x 6 at 80 registers: 124.0; 192 x 3: 116.8), the tree walks
// at 16 warps of 128 (256 x 2: 209; 128 x 5: 256; 128 x 6: 303) — r02c_adaptive_variants2.log
#ifndef RT_ADAPT_LIST_THREADS
#define RT_ADAPT_LIST_THREADS 128
#endif
#ifndef RT_ADAPT_LIST_BLOCKS
#define RT_ADAPT_LIST_BLOCKS 5
#endif
#ifndef RT_ADAPT_BLOCKS
#define RT_ADAPT_BLOCKS 2
#endif
#ifndef RT_ADAPT_THREADS
#define RT_ADAPT_THREADS 256
#endif
__host__ __device__ constexpr int ad_threads(int kind) { return kind == BVH_LIST ? RT_ADAPT_LIST_THREADS : RT_ADAPT_THREADS; }
__host__ __device__ constexpr int ad_blocks(int kind) { return kind == BVH_LIST ? RT_ADAPT_LIST_BLOCKS : RT_ADAPT_BLOCKS; }
// PixelStats between two batches.  Written by one SM, read by another a batch later: L2 accesses (ld.cg / st.cg), the L1 of the
// reading SM may still hold the line from an earlier batch.
RT_DEV void adstate_load(const PixState* ps, size_t pi, float& cx, float& cy, float& cz, double& s1, double& s2, int& samples, unsigned& bounces) {
  const long long* p = reinterpret_cast<const long long*>(ps + pi); // 40 bytes, 8-byte aligned
  const long long w0 = __ldcg(p), w1 = __ldcg(p + 1), w2 = __ldcg(p + 2), w3 = __ldcg(p + 3), w4 = __ldcg(p + 4);
  cx = __int_as_float((int)(w0 & 0xffffffffLL)); cy = __int_as_float((int)(w0 >> 32));
  cz = __int_as_float((int)(w1 & 0xffffffffLL)); samples = (int)(w1 >> 32);
  s1 = __longlong_as_double(w2); s2 = __longlong_as_double(w3);
  bounces = (unsigned)(w4 & 0xffffffffLL);
}
RT_DEV void adstate_store(PixState* ps, size_t pi, float cx, float cy, float cz, double s1, double s2, int samples, unsigned bounces, int done) {
  long long* p = reinterpret_cast<long long*>(ps + pi);
  auto pack = [](unsigned lo, unsigned hi) { return (long long)(((unsigned long long)hi << 32) | lo); };
  __stcg(p, pack((unsigned)__float_as_int(cx), (unsigned)__float_as_int(cy)));
  __stcg(p + 1, pack((unsigned)__float_as_int(cz), (unsigned)samples));
  __stcg(p + 2, __double_as_longlong(s1));
  __stcg(p + 3, __double_as_longlong(s2));
  __stcg(p + 4, pack(bounces, (unsigned)done));
}
#ifndef RT_ADAPT_MAXBLOCKS
#define RT_ADAPT_MAXBLOCKS 4
#endif
constexpr int kAdMaxBlocks = RT_ADAPT_MAXBLOCKS;        // 8x4 blocks per group (the slot index k * 32 + lane is a byte: <= 8)
constexpr int kAdMaxRecords = 320 * kAdMaxBlocks;       // records per warp slice: ad_blocks * 32 * aBatch <= this

template <int KIND>
__global__ void __launch_bounds__(ad_threads(KIND), ad_blocks(KIND)) k_render_adaptive(const DevScene S, const RenderParams R) {
  constexpr int kAdWarps = ad_threads(KIND) / 32;
  __shared__ ListSmemData sm_data;
  __shared__ unsigned char s_slot[kAdWarps][kAdMaxBlocks * 32]; // per warp: the group's active pixels (index inside the group), packed
  __shared__ int s_blk[kAdWarps][2 * kAdMaxBlocks];             // per warp: pixel origin of each block of the group
  const ListSmem sm = stage_list<KIND>(S, sm_data);
  const ListSmem& L = sm;
  const DevCamera& cam = S.cam;
  const MixW mw = make_mixw(S);
  const unsigned lane = threadIdx.x & 31u, full = 0xffffffffu, lt_mask = (1u << lane) - 1u;
  const int warp = (int)(threadIdx.x >> 5);
  unsigned char* slot_px = s_slot[warp];
  int* blk = s_blk[warp];
  const int B = cam.a_batch, GB = R.ad_blocks;
  AdRecord* rec = R.adrec + (size_t)(blockIdx.x * kAdWarps + warp) * (size_t)(GB * 32 * B);
  const int blocks_x = R.tiles_x * 2, blocks_per_row = (cam.width + 7) >> 3;
  const int n_blocks = R.part_count > 1 ? R.n_runs : blocks_x * R.tiles_y * 4;
  const int n_groups = (n_blocks + GB - 1) / GB;
  const int n_rounds = (cam.samples + B - 1) / B;
  const int n_items = n_groups * n_rounds;

  unsigned int t_pixels = 0, t_samples = 0, t_bounces = 0;
  WorkCount wc;
  int t_smin = 0x7fffffff, t_smax = 0, t_bmin = 0x7fffffff, t_bmax = 0;

  for (;;) {
    int item = 0;
    if (lane == 0) item = atomicAdd(R.queue, 1);
    item = __shfl_sync(full, item, 0);
    if (item >= n_items) break;
    const int round = item / n_groups, g = item - round * n_groups;
    // ---- the group's earlier batches must be complete ----
    volatile int* done_rounds = R.tile_done + g;
    int have = 0;
    if (lane == 0) {
      while ((have = *done_rounds) < round) __nanosleep(200);
    }
    have = __shfl_sync(full, have, 0);
    if (have > round) continue; // INT_MAX: every pixel of the group is final
    __threadfence();            // the PixelStats written by the warp that ran the previous batch
    // ---- the group's blocks and its active pixels ----
    if ((int)lane < GB) {
      const int b = g * GB + (int)lane;
      int bx = -(1 << 20), by = -(1 << 20);
      if (b < n_blocks) {
        if (R.part_count > 1) {
          const unsigned i = owned_block_of_run((unsigned)(R.run0 + b), R.part_index, R.part_count);
          bx = (int)(i % (unsigned)blocks_per_row) * 8;
          by = (int)(i / (unsigned)blocks_per_row) * 4;
        } else {
          bx = (R.x0 / kTile) * kTile + (b % blocks_x) * 8;
          by = (R.y0 / kTile) * kTile + (b / blocks_x) * 4;
        }
      }
      blk[2 * lane] = bx;
      blk[2 * lane + 1] = by;
    }
    __syncwarp();
    const int s_done = round * B, Bc = min(B, cam.samples - s_done); // every active pixel of the group has s_done samples
    int n_active = 0;
    for (int k = 0; k < GB; ++k) {
      const int x = blk[2 * k] + (int)(lane & 7u), y = blk[2 * k + 1] + (int)(lane >> 3);
      bool act = x >= R.x0 && x < R.x1 && y >= R.y0 && y < R.y1;
      if (act && round > 0) act = __ldcg(&R.adstate[(size_t)y * cam.width + x].done) == 0;
      const unsigned m = __ballot_sync(full, act);
      if (act) slot_px[n_active + __popc(m & lt_mask)] = (unsigned char)(k * 32 + (int)lane);
      n_active += __popc(m);
    }
    __syncwarp();
    if (n_active == 0) { // nothing of this group lies in the region
      if (lane == 0) *done_rounds = 0x7fffffff;
      continue;
    }
    // ---- the pool: n_active pixels x Bc samples, sample-major (neighbouring lanes run the same sample of different pixels) ----
    const int pool = n_active * Bc;
    {
      PathState ps{Ray{mk3(0, 0, 0), mk3(0, 0, 1)}, mk3(1, 1, 1), mk3(0, 0, 0), 0};
      Rng gen;
      int slot = 0, s_in = 0, pi_x = 0, pi_y = 0, next = 0;
      bool have_path = false, retired = false;
      for (;;) {
        const bool want = !have_path && !retired;
        bool fresh = false;
        const unsigned m = __ballot_sync(full, want);
        if (want) {
          const int idx = next + __popc(m & lt_mask);
          if (idx >= pool) retired = true;
          else {
            s_in = idx / n_active;
            slot = idx - s_in * n_active;
            const int q = slot_px[slot];
            pi_x = blk[2 * (q >> 5)] + (q & 7);
            pi_y = blk[2 * (q >> 5) + 1] + ((q >> 3) & 3);
            fresh = true;
            have_path = true;
          }
        }
        next += __popc(m);
        if (__all_sync(full, retired)) break;
        bool ended = false;
        if (have_path) {
          const uint32_t pixel = (uint32_t)pi_y * (uint32_t)cam.width + (uint32_t)pi_x;
          if (fresh) { ps.tp = mk3(1, 1, 1); ps.radiance = mk3(0, 0, 0); ps.bounces = 0; }
          gen.begin(pixel, (uint32_t)(s_done + s_in), (uint32_t)ps.bounces, S.seed_lo, S.seed_hi);
          if (fresh) ps.ray = camera_ray(cam, pi_x, pi_y, gen, true);
          ended = path_step<KIND, false, KIND != BVH_LIST>(S, L, sm, mw, ps, gen, wc); // (LV: Cornell defaults 60.2 -> 58.2 ms at 512 spp without the vector loads)
        }
        __syncwarp(); // one copy of the end-of-sample code (see k_render_pool)
        if (ended) {
          AdRecord r{ps.radiance.x, ps.radiance.y, ps.radiance.z, ps.bounces};
          __stcg(reinterpret_cast<float4*>(rec + slot * B + s_in), *reinterpret_cast<const float4*>(&r));
          t_bmin = min(t_bmin, ps.bounces);
          t_bmax = max(t_bmax, ps.bounces);
          have_path = false;
        }
      }
    }
    __syncwarp(); // the records of every lane are visible to the lane that folds the pixel
    // ---- pixel.add(...) of the batch in sample order + the loop condition of camera.ts:406, one lane per pixel ----
    int remaining = 0;
    for (int slot = (int)lane; slot < n_active; slot += 32) {
      const int q = slot_px[slot];
      const int x = blk[2 * (q >> 5)] + (q & 7), y = blk[2 * (q >> 5) + 1] + ((q >> 3) & 3);
      const size_t pi = (size_t)y * cam.width + x;
      float cx = 0.f, cy = 0.f, cz = 0.f;
      double s1 = 0.0, s2 = 0.0;
      int samples = 0;
      unsigned bounces = 0;
      if (round > 0) adstate_load(R.adstate, pi, cx, cy, cz, s1, s2, samples, bounces);
      float b_ill = 0.f, b_ill2 = 0.f;
      for (int k = 0; k < Bc; ++k) {
        const float4 v = __ldcg(reinterpret_cast<const float4*>(rec + slot * B + k));
        cx += v.x; cy += v.y; cz += v.z;
        bounces += (unsigned)__float_as_int(v.w);
        const float il = fmaf(0.299f, v.x, fmaf(0.587f, v.y, 0.114f * v.z)); // illuminance (vec3.ts:239-242)
        b_ill += il;
        b_ill2 = fmaf(il, il, b_ill2);
        t_bounces += (unsigned)__float_as_int(v.w);
      }
      samples += Bc;
      t_samples += (unsigned)Bc;
      s1 += (double)b_ill;
      s2 += (double)b_ill2;
      bool final_ = samples >= cam.samples;
      if (!final_ && Bc == B && samples >= 2) final_ = pixel_converged(s1, s2, samples, cam.a_tol); // camera.ts:348-368
      if (final_) {
        stream_write_pixel(R.rgb8, R.linear, nullptr, cam.width, 0, cam.depth, cam.samples, x, y, samples, bounces, cx, cy, cz, 0.f, 0.f, 0.f);
        ++t_pixels;
        t_smin = min(t_smin, samples);
        t_smax = max(t_smax, samples);
      } else ++remaining;
      adstate_store(R.adstate, pi, cx, cy, cz, s1, s2, samples, bounces, final_ ? 1 : 0);
    }
    const unsigned any_left = __ballot_sync(full, remaining > 0);
    __threadfence();
    __syncwarp();
    if (lane == 0) *done_rounds = any_left ? round + 1 : 0x7fffffff;
  }
  flush_stats_range(R, t_pixels, t_smin, t_smax, t_samples, t_bounces, wc.rays, t_bmin, t_bmax);
  flush_work(R, wc);
}

// =========================================================================================
// primary visibility (parity hook): pixel-centre rays, no jitter, no defocus
// =========================================================================================
template <int KIND>
__global__ void __launch_bounds__(256) k_trace_primary(const DevScene S, const RenderParams R, int* obj_id, float* t_out,
                                                       float* normal, uint8_t* front) {
  __shared__ ListSmemData sm_data;
  const ListSmem sm = stage_list<KIND>(S, sm_data);
  const ListSmem& L = sm;
  const int tx = (R.x0 / kTile) + blockIdx.x, ty = (R.y0 / kTile) + blockIdx.y;
  int lx, ly;
  tile_pixel(threadIdx.x, lx, ly);
  const int i = tx * kTile + lx, j = ty * kTile + ly;
  if (!(i >= R.x0 && i < R.x1 && j >= R.y0 && j < R.y1)) return;
  Rng g{};
  Ray ray = camera_ray(S.cam, i, j, g, false);
  float t;
  int slot;
  bool hit = closest_hit<KIND>(S, L, ray, t, slot);
  const size_t pi = (size_t)j * S.cam.width + i;
  Surf sf{mk3(0, 0, 0), mk3(0, 0, 0), false};
  int obj = -1;
  if (hit) {
    I2 info = ldgi2(S.slot_info + slot);
    obj = info.y & 0x3fffffff;
    sf = surface_at((info.y >> 30) & 3, ldg4(S.p0 + slot), ray, t);
  }
  if (obj_id) obj_id[pi] = obj;
  if (t_out) t_out[pi] = hit ? t : CUDART_INF_F;
  if (normal) { normal[pi * 3] = sf.n.x; normal[pi * 3 + 1] = sf.n.y; normal[pi * 3 + 2] = sf.n.z; }
  if (front) front[pi] = hit && sf.front ? 1 : 0;
}

// =========================================================================================
// FP32 peak microbenchmark: 8 independent FFMA chains per thread
// =========================================================================================
__global__ void __launch_bounds__(256) k_fp32_peak(float* out, int iters, float a, float b) {
  float x0 = threadIdx.x * 1e-3f, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int u = 0; u < 16; ++u) {
      x0 = fmaf(x0, a, b); x1 = fmaf(x1, a, b); x2 = fmaf(x2, a, b); x3 = fmaf(x3, a, b);
      x4 = fmaf(x4, a, b); x5 = fmaf(x5, a, b); x6 = fmaf(x6, a, b); x7 = fmaf(x7, a, b);
    }
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
}

// =========================================================================================
// launchers (called from rt_api.cu)
// =========================================================================================
void render_tile_grid(const RenderParams& R, int* tiles_x, int* tiles_y) {
  int tx0 = R.x0 / kTile, ty0 = R.y0 / kTile;
  int tx1 = (R.x1 - 1) / kTile, ty1 = (R.y1 - 1) / kTile;
  *tiles_x = tx1 - tx0 + 1;
  *tiles_y = ty1 - ty0 + 1;
}

// k_render_adaptive: plain adaptive renders (default mode, no moments, one shot) of every scene the whole-query kernels serve.
// Returns the group size in 8x4 blocks (0 = the pixel-stream kernels render this), and the number of warps whose record
// slices `adrec` must hold.
constexpr int kTravNodesAdaptive = 16384; // deep trees keep k_render_stream_trav (resumable traversal)
int render_adaptive_blocks(const DevScene& S, const RenderParams& R, int sms, int* warps) {
  static const bool off = getenv("RT_B200_NO_ADAPTIVE_POOL") != nullptr; // development switch
  if (off || !S.cam.adaptive || S.cam.mode != 0 || R.moments || S.cam.shadow_rays || R.pixstate || R.pass_cap > 0) return 0;
  if (S.cam.samples < 1 || S.cam.a_batch < 1 || S.cam.a_batch * 32 > kAdMaxRecords) return 0;
  if (S.bvh_kind == BVH_SAH && S.n_nodes >= kTravNodesAdaptive) return 0;
  int per_sm = 0;
  cudaError_t e;
  switch (S.bvh_kind) {
    case BVH_LIST: e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_render_adaptive<BVH_LIST>, ad_threads(BVH_LIST), 0); break;
    case BVH_SAH: e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_render_adaptive<BVH_SAH>, ad_threads(BVH_SAH), 0); break;
    default: e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_render_adaptive<BVH_REFERENCE>, ad_threads(BVH_REFERENCE), 0); break;
  }
  if (e != cudaSuccess || per_sm < 1) return 0;
  const long long n_warps = (long long)sms * per_sm * (ad_threads(S.bvh_kind) / 32);
  const long long n_blocks = R.part_count > 1 ? R.n_runs : (long long)R.tiles_x * R.tiles_y * 8;
  // groups as large as the record slice allows (longer pools, shorter tails) while every warp still finds two groups
  long long gb = std::min<long long>(kAdMaxBlocks, kAdMaxRecords / (32 * S.cam.a_batch));
  while (gb > 1 && n_blocks / gb < 2 * n_warps) --gb;
  const long long n_groups = (n_blocks + gb - 1) / gb, n_rounds = (S.cam.samples + S.cam.a_batch - 1) / S.cam.a_batch;
  if (n_groups * n_rounds >= (1LL << 30)) return 0;
  if (warps) *warps = (int)n_warps;
  return (int)gb;
}

bool render_needs_full(const DevScene& S, const RenderParams& R) {
  static const bool force = getenv("RT_B200_FORCE_PIXELS") != nullptr; // development switch
  return force || S.cam.adaptive || S.cam.mode != 0 || R.moments != nullptr || S.cam.shadow_rays;
}

// ctas_of_work counts 256-thread CTAs (eight warp items each); kernels with another CTA size scale it.
template <class K>
static cudaError_t launch_persistent(K kernel, const DevScene& S, const RenderParams& R, long long ctas_of_work, int sms, cudaStream_t st,
                                     int threads = 256) {
  int per_sm = 0;
  cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, 0);
  if (e != cudaSuccess) return e;
  if (per_sm < 1) per_sm = 1;
  ctas_of_work = ctas_of_work * 256 / threads;
  long long resident = (long long)sms * per_sm;
  int grid = (int)(ctas_of_work < resident ? ctas_of_work : resident);
  if (grid < 1) grid = 1;
  kernel<<<grid, threads, 0, st>>>(S, R);
  return cudaGetLastError();
}

// A later progressive pass picks pixels up from R.pixstate: the _resume kernels (see render_stream).
static bool stream_resumes(const RenderParams& R) { return R.pixstate && R.s0 > 0; }
template <int KIND, bool SHADOW = false>
static cudaError_t launch_stream(const DevScene& S, const RenderParams& R, long long tiles, int sms, cudaStream_t st) {
  if (stream_resumes(R)) return launch_persistent(k_render_stream_resume<KIND, SHADOW>, S, R, tiles, sms, st);
  return launch_persistent(k_render_stream<KIND, SHADOW>, S, R, tiles, sms, st);
}

cudaError_t launch_render_mega(const DevScene& S, const RenderParams& R, int sms, cudaStream_t st) {
  if (R.x1 <= R.x0 || R.y1 <= R.y0) return cudaSuccess;
  const long long tiles = (long long)R.tiles_x * R.tiles_y;
  constexpr int kTravNodes = 16384; // tree size from which resumable traversal beats the whole-query walk (see case BVH_SAH below)
  constexpr int kTravNodesFixed = 6144; // ... for fixed-spp renders (k_render_pool<SAH> vs k_render_trav)
  if (render_needs_full(S, R)) {
    static const bool no_stream_trav = getenv("RT_B200_NO_STREAM_TRAV") != nullptr; // development switch
    if (S.cam.shadow_rays) { // whole-query walks for every tree size: the shadow ray is traced inside the shading step
      switch (S.bvh_kind) {
        case BVH_LIST: return launch_stream<BVH_LIST, true>(S, R, tiles, sms, st);
        case BVH_SAH: return launch_stream<BVH_SAH, true>(S, R, tiles, sms, st);
        default: return launch_stream<BVH_REFERENCE, true>(S, R, tiles, sms, st);
      }
    }
    if (R.ad_blocks > 0) { // chosen by render_adaptive_blocks (rt_api.cu sizes adstate / adrec from it)
      switch (S.bvh_kind) {
        case BVH_LIST: return launch_persistent(k_render_adaptive<BVH_LIST>, S, R, 1LL << 40, sms, st, ad_threads(BVH_LIST));
        case BVH_SAH: return launch_persistent(k_render_adaptive<BVH_SAH>, S, R, 1LL << 40, sms, st, ad_threads(BVH_SAH));
        default: return launch_persistent(k_render_adaptive<BVH_REFERENCE>, S, R, 1LL << 40, sms, st, ad_threads(BVH_REFERENCE));
      }
    }
    switch (S.bvh_kind) {
      case BVH_LIST: return launch_stream<BVH_LIST>(S, R, tiles, sms, st);
      case BVH_SAH:
        if (S.n_nodes >= kTravNodes && !no_stream_trav)
          return launch_persistent(stream_resumes(R) ? k_render_stream_trav_resume : k_render_stream_trav, S, R, tiles, sms, st);
        return launch_stream<BVH_SAH>(S, R, tiles, sms, st);
      default: return launch_stream<BVH_REFERENCE>(S, R, tiles, sms, st);
    }
  }
  // a tile = 8 warp blocks and a CTA runs 8 warps: `tiles * chunks` CTAs' worth of warp items
  const long long work = tiles * R.chunks;
  static const bool pool_list = getenv("RT_B200_POOL_LIST") != nullptr;   // development switches
  static const bool no_trav = getenv("RT_B200_NO_TRAV") != nullptr;
  static const bool env_sorted = getenv("RT_B200_SORTED") != nullptr;
  // k_render_sorted ends its CTA loop when no warp holds samples, so it cannot write the pixels of an image with
  // zero samples per pixel (black image, camera.ts:406); k_render_pool's epilogue runs for every item.
  const bool sorted_list = (env_sorted || R.sorted) && S.cam.samples > 0;
  switch (S.bvh_kind) {
    case BVH_LIST:
      // Lane-keeps-pixel (POOL = false) has no queue arithmetic but its lanes finish an item at different times; with short
      // items (a GPU that owns 1/8 of the blocks cuts its pixels' samples into ~18 chunks to keep 20 rounds of warps busy)
      // that intra-warp tail costs more than the pair queue.  Cornell 1024 spp, bit-identical images: whole image, 341
      // samples per item: 107.1 vs 107.8 ms; one part of eight, 57 samples per item: 14.35 vs 13.87 ms (ideal 13.39).
      if (pool_list || (R.s_cnt > 0 ? R.s_cnt : S.cam.samples) / (R.chunks > 0 ? R.chunks : 1) < 128)
        return launch_persistent(k_render_pool<BVH_LIST, true>, S, R, work, sms, st, RT_LIST_THREADS);
      if (sorted_list) {
        // 3 CTAs x 43.4 KB fit the 132 KB split; the rest stays L1.  Function attributes are per device, and one
        // process may drive several GPUs, so this is set at every launch (microseconds, once per render).
        const cudaError_t carve = cudaFuncSetAttribute(k_render_sorted<BVH_LIST>, cudaFuncAttributePreferredSharedMemoryCarveout, 57);
        if (carve != cudaSuccess) return carve;
        return launch_persistent(k_render_sorted<BVH_LIST>, S, R, work, sms, st);
      }
      return launch_persistent(k_render_pool<BVH_LIST, false>, S, R, work, sms, st, RT_LIST_THREADS);
    case BVH_SAH:
      // Whole-query while-while walk (k_render_pool) vs traversal bursts interleaved with shading (k_render_trav),
      // rain scene at 1 k ... 100 k spheres with the 4-wide tree (scripts/gpu_trav_threshold.py; n_nodes counts
      // 64-byte slots; final tree layout): 11.7 / 15.2 ms at 8 k slots (8 000 spheres), 19.2 / 18.1 at 20 k,
      // 27.5 / 22.9 at 48.5 k: regenerating paths mid-traversal pays once lanes diverge by many node visits.
      if (sorted_list && (S.n_nodes < kTravNodes || no_trav)) {
        const cudaError_t carve = cudaFuncSetAttribute(k_render_sorted<BVH_SAH>, cudaFuncAttributePreferredSharedMemoryCarveout, 57);
        if (carve != cudaSuccess) return carve;
        return launch_persistent(k_render_sorted<BVH_SAH>, S, R, work, sms, st);
      }
      static const bool trav_always = getenv("RT_B200_TRAV_ALWAYS") != nullptr;
      // fixed spp: crossover re-measured after the pair queue moved behind the shading (scripts/gpu_trav_threshold.py, rain scenes
      // at 8 spp, pool / trav ms): 2730 node slots 7.08 / 7.85, 7956: 10.61 / 10.06, 15944: 16.08 / 12.32 (profiles/r02c_trav_threshold.log)
      if (!trav_always && (no_trav || S.n_nodes < kTravNodesFixed)) return launch_persistent(k_render_pool<BVH_SAH, true>, S, R, work, sms, st);
      // (Measured and removed, round 2: TWO paths per lane — the active one in registers, the other parked in shared memory,
      //  swapped in when the active ray finishes so the lane keeps traversing; bit-identical image, 100 k spheres at 32 spp
      //  390 -> 417-436 ms over every min-lanes / burst setting: the swaps, the second service pass and the second traversal
      //  stack cost more than the idle lanes they fill.)
      return launch_persistent(k_render_trav, S, R, work, sms, st, RT_TRAV_THREADS);
    default: return launch_persistent(k_render_pool<BVH_REFERENCE, true>, S, R, work, sms, st);
  }
}

cudaError_t launch_trace_primary(const DevScene& S, const RenderParams& R, int* obj_id, float* t, float* normal,
                                 uint8_t* front, cudaStream_t st) {
  if (R.x1 <= R.x0 || R.y1 <= R.y0) return cudaSuccess;
  int gx, gy;
  render_tile_grid(R, &gx, &gy);
  dim3 grid((unsigned)gx, (unsigned)gy, 1), block(256);
  switch (S.bvh_kind) {
    case BVH_LIST: k_trace_primary<BVH_LIST><<<grid, block, 0, st>>>(S, R, obj_id, t, normal, front); break;
    case BVH_SAH: k_trace_primary<BVH_SAH><<<grid, block, 0, st>>>(S, R, obj_id, t, normal, front); break;
    default: k_trace_primary<BVH_REFERENCE><<<grid, block, 0, st>>>(S, R, obj_id, t, normal, front); break;
  }
  return cudaGetLastError();
}

cudaError_t launch_fp32_peak(float* out, int blocks, int iters, cudaStream_t st) {
  k_fp32_peak<<<blocks, 256, 0, st>>>(out, iters, 0.999f, 0.001f);
  return cudaGetLastError();
}

} // namespace rt

#include "rt_wavefront.cuh" // the wavefront integrator shares every helper above
#include "rt_debug.cuh"     // per-function parity hooks: the same device functions on explicit inputs
#include "rt_denoise.cuh"   // first-hit feature buffers and the a-trous denoiser
