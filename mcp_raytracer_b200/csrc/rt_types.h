// rt_types.h — POD layouts shared by the host scene compiler and the sm_100a kernels.
//
// Data layout in HBM (all arrays 16-byte aligned, read-only during a render):
//   nodes   [n_nodes]  4 x float4 = 64 B   REFERENCE trees: two child boxes + two child refs (pair layout, Node);
//                                          SAH trees: 4-wide nodes of two slots each (WideNode, 128 B)
//   p0      [n_slots]  float4              sphere: (cx,cy,cz,r) | planar: (nx,ny,nz,D)
//   p1,p2   [n_slots]  float4              planar only: (A.xyz, q.A) and (B.xyz, q.B) with
//                                          A = v x w, B = w x u  =>  alpha = p.A - q.A,
//                                          beta = p.B - q.B  (plane.ts:71-74 rewritten by the
//                                          scalar-triple-product identity)
//   p3      [n_slots]  float4              planar only: (|A|_1, |B|_1, 4eps|q.A|, 4eps|q.B|), the
//                                          per-primitive constants of the FP32 error bound
//   slot_info [n_slots] int2               (material root, original object index | type<<30)
//   exact   [n_slots]  ExactPrim 96 B      FP32 vectors + FP64 scalars exactly as the reference
//                                          holds them; touched only by the guarded FP64 re-test
//   matA    [n_mats]   float4              (r,g,b,param)
//   matB    [n_mats]   int4                (type, child0, child1, has_emission)
//   matE    [n_mats]   float4              precomputed emitted() of the subtree rooted here
//   matF    [n_mats]   float4              feature albedo of the subtree rooted here (the denoiser demodulates by it)
//   lights  [n_lights] DevLight
// Slots are primitives in BVH-leaf order, so a leaf is a contiguous slot range.
#pragma once
#include <stddef.h>
#include <stdint.h>

#ifdef __CUDACC__
#define RT_HD __host__ __device__
#else
#define RT_HD
#endif

namespace rt {

// OBJ_AAQUAD is a device-side specialisation of OBJ_QUAD chosen by the scene compiler (u, v axis-aligned);
// slot records p1/p2 then hold (c, lo_I, lo_J, hi_I), (hi_J, axis bits, -, -) instead of the general ones.
enum : int { OBJ_SPHERE = 0, OBJ_PLANE = 1, OBJ_QUAD = 2, OBJ_AAQUAD = 3 };
enum : int { MAT_LAMBERT = 0, MAT_METAL = 1, MAT_GLASS = 2, MAT_LIGHT = 3, MAT_MIXED = 4, MAT_LAYERED = 5 };
enum : int { BVH_REFERENCE = 1, BVH_SAH = 2, BVH_LIST = 3 };

struct F4 { float x, y, z, w; };
struct I4 { int x, y, z, w; };
struct I2 { int x, y; };

// Child reference encoding: >= 0 internal node index; < 0 leaf with v = ~ref:
//   first slot = v >> 6, count = ((v >> 4) & 3) + 1, planar mask = v & 15.
// kEmptyRef marks a child that is never entered (its box is inverted as well).
static const int kEmptyRef = 0x7fffffff;
RT_HD inline int make_leaf_ref(int first, int count, int planar_mask) {
  return ~((first << 6) | ((count - 1) << 4) | (planar_mask & 15));
}

struct alignas(16) Node { // 64 B
  float lmin[3], lmax[3];
  float rmin[3], rmax[3];
  int left, right;
  int flags; // bit0/bit1: left/right subtree holds an inverted box => test it with the reference's per-axis rule
  int pad1;
};

// SAH trees: four children per node (the binary tree collapsed, rt_scene.cpp), 128 B = two Node slots.
// box[k] = (centre.xyz, half-extent.xyz) of child k — the slab test is then three FFMA per axis and no per-axis min / max
// (trav_inner, rt_device.cuh); the half-extents are rounded up so that the stored box contains the builder's box; an
// unbounded axis is (0, +inf); ref[k] as above; unused children: half-extent -inf + kEmptyRef.
struct alignas(16) WideNode {
  float box[4][6];
  int ref[4];
  int pad[4];
};

struct alignas(16) ExactPrim { // 96 B
  float q[3];  // sphere centre | planar corner
  float u[3], v[3], n[3], w[3];
  int type;
  int rank;    // position in the reference's visiting order (tie-break on exactly equal t)
  double D;    // plane.ts:39
  double r;    // sphere radius (JS double)
  double area; // quad.ts:37
};

struct alignas(16) DevLight { // light = object with light:true that is a Sphere or a Quad (scenes.ts:74-79)
  F4 p0, p1, p2, p3;  // same records as the slot arrays
  float q[3], u[3], v[3];
  float area;     // quad
  float radius;   // sphere
  int type;
  int slot;
  int pad;
};
static_assert(sizeof(DevLight) == 128 && offsetof(DevLight, q) == 64, "light_f4 (rt_device.cuh) reads DevLight as eight float4");

struct DevCamera {
  float center[3], p00[3], du[3], dv[3], ddu[3], ddv[3];
  float bg_top[3], bg_bottom[3];
  int width, height;
  int samples, depth, rr_depth, a_batch, mode;
  float a_tol;
  int roulette, adaptive, jitter, defocus;
  int shadow_rays; // rt_render_opts.light_sampling == RT_LIGHTS_SHADOW_RAYS (next-event estimation)
};

struct DevScene {
  DevCamera cam;
  const F4* nodes; // 4 per node
  const F4* p0;
  const F4* p1;
  const F4* p2;
  const F4* p3;
  const I2* slot_info;
  const ExactPrim* exact;
  const F4* matA;
  const I4* matB;
  const F4* matE;
  const DevLight* lights;
  const F4* matF;
  int n_nodes, n_slots, n_unbounded, n_mats, n_lights;
  int bvh_kind;
  int planar_any; // scene has planes/quads
  int list_n[6];  // LIST: slots per kind, in slot order: spheres, axis-aligned quads x/y/z, general quads, planes
  float sph_cmax, sph_r2max; // LIST: max |centre component| and max r^2 over the spheres
  uint32_t seed_lo, seed_hi;
};

// Image partition across GPUs (one process per GPU, or rt_multi_* inside one process).  The unit is the 8x4 pixel
// block — one warp work item.  Blocks are numbered row-major over the WHOLE image (bx = x / 8, by = y / 4,
// blocks_per_row = ceil(width / 8)); every run of `n` consecutive blocks gives each part exactly one block, in an
// order rotated by a hash of the run's index.  Parts are therefore balanced to one block per run (64x4 pixels at
// n = 8) whatever the image content — no diagonal, row or column structure that could alias with the scene, as the
// round-1 rule owner = (tile_x + tile_y) % n had — and ownership does not depend on the render region.
RT_HD inline int block_owner(int bx, int by, int blocks_per_row, int n) {
  const unsigned i = (unsigned)by * (unsigned)blocks_per_row + (unsigned)bx;
  const unsigned g = i / (unsigned)n, r = i - g * (unsigned)n;
  unsigned h = g * 0x9E3779B1u;
  h ^= h >> 15; h *= 0x85EBCA77u; h ^= h >> 13;
  return (int)((r + h) % (unsigned)n);
}

// The block part `part` owns in run g (inverse of block_owner): linear index over the whole image.
RT_HD inline unsigned owned_block_of_run(unsigned g, int part, int n) {
  unsigned h = g * 0x9E3779B1u;
  h ^= h >> 15; h *= 0x85EBCA77u; h ^= h >> 13;
  const unsigned r = ((unsigned)part + (unsigned)n - h % (unsigned)n) % (unsigned)n;
  return g * (unsigned)n + r;
}

// Per-render launch parameters.
struct RenderParams {
  int x0, y0, x1, y1;          // region, clipped to the image
  int part_index, part_count;  // this GPU renders the 8x4 blocks with block_owner(...) == part_index
  int run0, n_runs;            // part_count > 1: the runs of part_count consecutive blocks that overlap the region's block rows
  uint8_t* rgb8;               // [H][W][3] or null
  float* linear;               // [H][W][3] or null
  float* moments;              // [H][W][8] or null
  unsigned long long* stats;   // device RenderStats accumulator (see kStat*)
  // Work decomposition of the render kernels: work item = (tile, sample chunk).  A pixel's samples
  // are cut into `chunks` contiguous ranges that different CTAs may run.  Radiance sums are kept in
  // 64-bit fixed point (2^-32 units), so adding them is exact and order-independent: the image is
  // bit-identical whatever the chunking, the scheduling or the number of GPUs.  Partial sums of a
  // chunk go to `accum` [H][W][4] with atomics; the CTA that finishes a tile last writes its pixels.
  int tiles_x, tiles_y;        // tile grid covering the region
  int chunks;
  unsigned long long* accum;   // [H][W][4] (r, g, b, unused), zero before the launch; chunks > 1 only
  int* queue;                  // [0] = next work item
  int* tile_done;              // [8x4 blocks] finished chunks per block
  int trav_min_lanes;          // k_render_trav: leave the traversal phase when <= this many lanes still traverse
  int trav_burst;              // k_render_trav: inner-node visits a lane may do between two votes
  int sorted;                  // use k_render_sorted (CTA-wide sort of hits by material class) where it exists
  // ---- progressive rendering (rt_camera_render_progressive): one launch = one pass ----
  // fixed spp: this launch renders samples [s0, s0 + s_cnt) of every pixel on top of `accum` (kept from the earlier passes) and
  // writes the pixel as sum / div_samples; s_cnt == 0: the whole range [0, samples), divisor = samples
  int s0, s_cnt, div_samples;
  int keep_accum;              // sums go through `accum` even when chunks == 1
  // pixel stream (adaptive sampling / modes): a pixel runs until it converges, reaches `samples` or reaches pass_cap samples;
  // its PixelStats live in pixstate between passes (null: one-shot render)
  struct PixState* pixstate;
  int pass_cap;
  // ---- batch-parallel adaptive sampling (k_render_adaptive) ----
  // PixelStats of every pixel between two batches live in `adstate` [H][W]; a warp item = one batch (aBatch samples) of the still
  // active pixels of a group of ad_blocks 8x4 blocks, its per-sample records in this warp's slice of `adrec`; tile_done[group] =
  // batches the group has completed (INT_MAX: every pixel final)
  struct PixState* adstate;
  struct AdRecord* adrec; // [resident warps][ad_blocks * 32 * aBatch]
  int ad_blocks;
};
struct alignas(16) AdRecord { // one finished sample: pixel.add(rayColor, bounces) waiting for its turn in the pixel's sum
  float r, g, b;
  int bounces;
};
// PixelStats of one pixel between two passes of a progressive render (renderStats.ts:67-88)
struct alignas(8) PixState {
  float color[3];
  int samples;
  double sum_ill, sum_ill2;
  unsigned int bounces;
  int done; // converged or all samples taken: later passes skip the pixel
};
static_assert(sizeof(PixState) == 40 && offsetof(PixState, samples) == 12 && offsetof(PixState, sum_ill) == 16 && offsetof(PixState, bounces) == 32,
              "adstate_load / adstate_store (rt_megakernel.cu) move a PixState as five 64-bit words");
// ---- denoiser (rt_denoise.cuh): one filter launch sequence over the pixels of a region ----
// Every buffer is indexed by whole-image pixel (y * width + x); only pixels inside [x0, x1) x [y0, y1) are read or written.
// A launch computes the rows [wy0, wy1) of the region (its window); taps and gradients test the region, not the window.
struct DenoiseParams {
  int width;
  int x0, y0, x1, y1;
  int wy0, wy1;
  const float* color;   // [H][W][3] linear colour (the pixel mean)
  const float* albedo;  // [H][W][3] feature albedo
  const float* normal;  // [H][W][3] feature normal (zero on a miss)
  const float* depth;   // [H][W] feature depth (-1 on a miss)
  const float* moments; // [H][W][8] as rt_camera_render_moments writes them
  F4* buf[2];           // (demodulated colour, luminance variance); x = NaN marks a pixel the filter passes through
  F4* feat;             // (normal, depth)
  float* grad;          // [H][W][2] depth gradient
  int iterations;
  float sigma_l, sigma_n, sigma_z;
  float* out;           // [H][W][3] linear result; may be `color` when one band covers the region (read and written pixel by pixel)
  uint8_t* rgb8;        // [H][W][3] or null
};
// Filtering a band of rows [b0, b1) on its own (ghost zones, no exchange between passes): pass k (step 2^k) reads up to
// 2^(k+1) rows away (taps at +-2 * 2^k, the variance blur at +-1), so of K passes, pass k computes h = 2^(K+1) - 2^(k+2)
// rows beyond each side of the band and the last pass exactly the band.  stage -1 = prepare: 2^(K+1) - 2 rows; the
// features are needed one row further (the depth gradient reads +-1).  Every window is clipped to the region.
inline int dn_halo(int iterations, int stage) { return (1 << (iterations + 1)) - (1 << (stage + 2)); }
// ---- wavefront integrator (rt_wavefront.cuh): path pool + queues in HBM ----
struct U2 { uint32_t x, y; };
enum : int { WF_TAGS = 3 };
enum : int { // indices into WfBuffers::counters (device ints)
  WFC_NEXT_PAIR = 0,   // next (pixel, sample) pair index (64-bit: two ints)
  WFC_NEXT_PAIR_HI,
  WFC_N_EXTEND,        // rays queued for the next extend
  WFC_EXTEND_CURSOR,   // extend's dynamic-fetch cursor
  WFC_N_SHADE0, WFC_N_SHADE1, WFC_N_SHADE2,
  WFC_N_FREE,          // free slots queued for the next generate
  WFC_COUNT
};
struct WfBuffers {
  F4* ray_o;   // o.xyz, hit t
  F4* ray_d;   // d.xyz, hit slot (int bits)
  F4* tp;      // throughput.xyz, bounces (int bits)
  F4* rad;     // radiance.xyz, draws already taken from the current bounce's stream (int bits)
  U2* pix;     // pixel index, sample index
  int* q_extend;
  int* q_shade[WF_TAGS];
  int* q_free;
  int* counters;
  int n_slots;
  unsigned long long total_pairs; // owned 8x4 blocks * 32 * samples
};
struct WfHost { // device allocations owned by the camera (rt_api.cu)
  WfBuffers W;
  int* q_extend[2];
  int* q_free[2];
  int* owned_blocks;
  int* h_counters; // pinned host
  int n_owned, blocks_x;
  int owned_capacity;
};

enum : int {
  kStatPixels = 0, kStatSamples, kStatBounces, kStatRays,
  kStatSamplesMin, kStatSamplesMax, kStatBouncesMin, kStatBouncesMax,
  kStatNodeVisits, kStatPrimTests, // instrumented build (-DRT_COUNT_EVENTS) only; 0 otherwise
  kStatCount
};

} // namespace rt
