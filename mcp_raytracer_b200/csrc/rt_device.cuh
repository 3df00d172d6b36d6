// rt_device.cuh — device-side building blocks of the sm_100a path tracer.
//
// Everything the reference evaluates per ray (src/camera.ts:221-319 and callees) as FP32
// device functions written for SIMT convergence: the primitive tests are branch-free
// (every lane computes t, alpha, beta / both roots and decides with predicates), and each
// carries a cheap conservative bound on its own FP32 error.  A test whose outcome lies within
// that bound of a decision threshold (hit/miss, interval end, quad edge, equal-distance tie) or
// whose t is not good to ~2e-5 relative returns "ambiguous" and is re-evaluated with the
// reference's exact formula in FP64 from the reference's FP32-stored operands (ExactPrim).
// That keeps primary-hit object ids identical to the reference's FP64-scalar arithmetic
// without paying FP64 on the common path.
#pragma once
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stddef.h>
#include <stdint.h>

#include "rt_types.h"

namespace rt {

#define RT_DEV __device__ __forceinline__

static constexpr float kEps32 = 5.9604645e-08f; // 2^-24
static constexpr float kRayTMin = 0.001f;       // camera.ts:249

// ---------------------------------------------------------------------------------------
// small vector helpers
// ---------------------------------------------------------------------------------------
struct V3 {
  float x, y, z;
};
RT_DEV V3 mk3(float x, float y, float z) { return V3{x, y, z}; }
RT_DEV V3 ld3(const float* p) { return V3{p[0], p[1], p[2]}; }
RT_DEV V3 xyz(F4 v) { return V3{v.x, v.y, v.z}; }
RT_DEV V3 operator+(V3 a, V3 b) { return V3{a.x + b.x, a.y + b.y, a.z + b.z}; }
RT_DEV V3 operator-(V3 a, V3 b) { return V3{a.x - b.x, a.y - b.y, a.z - b.z}; }
RT_DEV V3 operator*(V3 a, V3 b) { return V3{a.x * b.x, a.y * b.y, a.z * b.z}; }
RT_DEV V3 operator*(V3 a, float s) { return V3{a.x * s, a.y * s, a.z * s}; }
RT_DEV V3 operator-(V3 a) { return V3{-a.x, -a.y, -a.z}; }
RT_DEV float dot3(V3 a, V3 b) { return fmaf(a.x, b.x, fmaf(a.y, b.y, a.z * b.z)); }
RT_DEV V3 cross3(V3 a, V3 b) { return V3{a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }
RT_DEV V3 fma3(float s, V3 a, V3 b) { return V3{fmaf(s, a.x, b.x), fmaf(s, a.y, b.y), fmaf(s, a.z, b.z)}; } // s*a+b
RT_DEV float l1norm(V3 a) { return fabsf(a.x) + fabsf(a.y) + fabsf(a.z); }
RT_DEV float maxabs(V3 a) { return fmaxf(fabsf(a.x), fmaxf(fabsf(a.y), fabsf(a.z))); }
RT_DEV float maxc(V3 a) { return fmaxf(a.x, fmaxf(a.y, a.z)); }
RT_DEV V3 sel3(bool c, V3 a, V3 b) { return V3{c ? a.x : b.x, c ? a.y : b.y, c ? a.z : b.z}; }
RT_DEV float rcp_approx(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
RT_DEV float rsqrt_approx(float x) {
  float r;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
RT_DEV V3 normalize3(V3 a) { // gl-matrix normalize: zero stays zero
  float l = dot3(a, a);
  float s = l > 0.f ? rsqrt_approx(l) : 0.f;
  // rsqrt.approx is good to 2 ulp: unit vectors are unit to 2.4e-7, the level of the FP32 roundings around every use
  // (directions are never required to be unit by the tests that consume them: a = |d|^2 is carried, camera.ts:176-210)
  return a * s;
}

RT_DEV F4 ldg4(const F4* p) {
  float4 v = __ldg(reinterpret_cast<const float4*>(p));
  return F4{v.x, v.y, v.z, v.w};
}
// 256-bit read-only load (sm_100: LDG.E.256).  Every lane of a deep-tree walk reads its own node; the 96 bytes of boxes as
// 3 x 256 bits + the refs as 128 bits are four load requests where 7 x 128 bits were seven (ncu, k_wf_extend on the 100 k-sphere
// scene: global-load requests 35.2 M -> 21.2 M, L1 data-pipe wavefronts 79 % -> 72 % of peak, 1.82 -> 1.69 ms).  p must be
// 32-byte aligned.
struct F8 {
  float v[8];
};
RT_DEV F8 ldg8(const void* p) {
  F8 r;
  asm("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
      : "=f"(r.v[0]), "=f"(r.v[1]), "=f"(r.v[2]), "=f"(r.v[3]), "=f"(r.v[4]), "=f"(r.v[5]), "=f"(r.v[6]), "=f"(r.v[7])
      : "l"(p));
  return r;
}
RT_DEV I4 ldgi4(const I4* p) {
  int4 v = __ldg(reinterpret_cast<const int4*>(p));
  return I4{v.x, v.y, v.z, v.w};
}
RT_DEV I2 ldgi2(const I2* p) {
  int2 v = __ldg(reinterpret_cast<const int2*>(p));
  return I2{v.x, v.y};
}

// ---------------------------------------------------------------------------------------
// Philox4x32-7, keyed (pixel, sample), counter (block, stream, seed_lo, seed_hi).  Seven rounds: the fewest that are
// crush-resistant (Salmon et al., SC'11, table 2; Random123 ships known-answer vectors for them, pinned on the oracle's
// copy by tests/test_oracle_reference_vectors.py); ten is Random123's default margin.  The block is generated once per
// bounce by every lane, 11 % of the Cornell kernel's instructions at ten rounds: 10 -> 7 measured 106.9 -> 104.7 ms
// (Cornell), 38.0 -> 36.9 (480 spheres), 198 -> 191 (100 k spheres).  The oracle uses the same count (ORC_PHILOX_ROUNDS).
// Stream b serves the rayColor call entered with `bounces == b`; the camera-ray draws of a
// path are the first draws of its stream 0.  One Philox block yields FIVE 24-bit uniforms:
// the high 24 bits of each word plus one assembled from the low bytes of words 0..2, so the
// common bounce (roulette + mixture select + two sampling numbers, or pixel jitter + select +
// two) costs exactly one block, generated by all lanes together at the top of the bounce.
// ---------------------------------------------------------------------------------------
#ifndef RT_PHILOX_ROUNDS
#define RT_PHILOX_ROUNDS 7
#endif
RT_DEV uint4 philox4x32(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t a, uint32_t b) {
#pragma unroll
  for (int r = 0; r < RT_PHILOX_ROUNDS; ++r) {
    uint32_t h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
    uint32_t h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
    c0 = h1 ^ c1 ^ a; c1 = l1; c2 = h0 ^ c3 ^ b; c3 = l0;
    a += 0x9E3779B9u; b += 0xBB67AE85u;
  }
  return make_uint4(c0, c1, c2, c3);
}
// out-of-line copy for the rare draws beyond the first block of a bounce (keeps the hot loop small)
__device__ __noinline__ uint4 philox4x32_slow(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t a, uint32_t b) {
  return philox4x32(c0, c1, c2, c3, a, b);
}

struct Rng {
  uint32_t k0, k1, seed_lo, seed_hi, stream, block;
  uint32_t q0, q1, q2, q3, q4; // pending 24-bit integers, q0 next
  int avail;
  RT_DEV void load(uint4 w) {
    q0 = w.x >> 8; q1 = w.y >> 8; q2 = w.z >> 8; q3 = w.w >> 8;
    q4 = ((w.x & 0xffu) << 16) | ((w.y & 0xffu) << 8) | (w.z & 0xffu);
    avail = 5;
  }
  // start stream s of path (pixel, sample) and generate its first block (convergent call site)
  RT_DEV void begin(uint32_t pixel, uint32_t sample, uint32_t s, uint32_t slo, uint32_t shi) {
    k0 = pixel; k1 = sample; seed_lo = slo; seed_hi = shi; stream = s; block = 1;
    load(philox4x32(0u, s, slo, shi, pixel, sample));
  }
  RT_DEV float next() {
    if (avail == 0) {
      load(philox4x32_slow(block, stream, seed_lo, seed_hi, k0, k1));
      ++block;
    }
    uint32_t w = q0;
    q0 = q1; q1 = q2; q2 = q3; q3 = q4;
    --avail;
    return (float)w * 5.9604645e-08f;
  }
};

// Explicit uniforms instead of a Philox stream: the per-function parity hooks (rt_debug_*, rt_debug.cuh) drive
// the very same device functions with the sequence the CPU oracle is given.  Past the end of the list: 0.5.
struct ListRng {
  const float* u;
  int n, used;
  RT_DEV float next() {
    const float v = used < n ? u[used] : 0.5f;
    ++used;
    return v;
  }
};

// ---------------------------------------------------------------------------------------
// Ray with the per-ray invariants the tests share
// ---------------------------------------------------------------------------------------
struct Ray {
  V3 o, d;
};
struct RayPre {
  float a, inva, l1d; // |d|^2, 1/|d|^2, L1 norm of d
  float omax175, dmax; // 1.75*max|o_i| (bounds sum|n_i o_i| for unit n), max|d_i|
  V3 idir;            // 1/d
  V3 oid;             // o * idir
};
RT_DEV RayPre precompute(const Ray& r, bool need_box) {
  RayPre p;
  p.a = dot3(r.d, r.d);
  // MUFU reciprocals (1-2 ulp; measured +7 % on Cornell against IEEE division): the primitive tests' error bounds have
  // that much slack built in (8 eps on t), and box tests pad tmax by 4 ulp
  p.inva = rcp_approx(p.a);
  p.l1d = l1norm(r.d);
  p.omax175 = 1.75f * maxabs(r.o);
  p.dmax = maxabs(r.d);
  if (need_box) {
    p.idir = V3{rcp_approx(r.d.x), rcp_approx(r.d.y), rcp_approx(r.d.z)};
    p.oid = r.o * p.idir;
  } else {
    p.idir = V3{0, 0, 0};
    p.oid = V3{0, 0, 0};
  }
  return p;
}

// ---------------------------------------------------------------------------------------
// Exact (FP64) re-tests: the reference's formulas on the reference's operands, no FMA
// contraction (__d*_rn), so results agree with V8 double arithmetic.
// ---------------------------------------------------------------------------------------
RT_DEV double ddot(const float* a, V3 b) {
  return __dadd_rn(__dadd_rn(__dmul_rn((double)a[0], (double)b.x), __dmul_rn((double)a[1], (double)b.y)),
                   __dmul_rn((double)a[2], (double)b.z));
}
RT_DEV double ddot(V3 a, V3 b) {
  return __dadd_rn(__dadd_rn(__dmul_rn((double)a.x, (double)b.x), __dmul_rn((double)a.y, (double)b.y)),
                   __dmul_rn((double)a.z, (double)b.z));
}
// One primitive, the reference's formula in FP64 over the open interval (tmin, tmax):
// sphere.ts:45-66, plane.ts:55-77 + quad.ts:60 (quad: inclusive inside test; plane: none).
__device__ __noinline__ bool prim_exact(const ExactPrim* e, Ray r, double tmin, double tmax, double& t_out) {
  if (e->type == OBJ_SPHERE) {
    V3 c = ld3(e->q);
    V3 oc = V3{__fsub_rn(r.o.x, c.x), __fsub_rn(r.o.y, c.y), __fsub_rn(r.o.z, c.z)};
    double a = ddot(r.d, r.d);
    double hb = ddot(oc, r.d);
    double rr = e->r;
    double cc = __dsub_rn(ddot(oc, oc), __dmul_rn(rr, rr));
    double disc = __dsub_rn(__dmul_rn(hb, hb), __dmul_rn(a, cc));
    if (disc < 0) return false;
    double sq = sqrt(disc);
    double root = (-hb - sq) / a;
    if (!(tmin < root && root < tmax)) {
      root = (-hb + sq) / a;
      if (!(tmin < root && root < tmax)) return false;
    }
    t_out = root;
    return true;
  }
  double denom = ddot(e->n, r.d);
  if (fabs(denom) < 1e-8) return false;
  double t = (e->D - ddot(e->n, r.o)) / denom;
  if (!(tmin < t && t < tmax)) return false;
  if (e->type == OBJ_QUAD) {
    // r.at(t): scale then add, each rounded to FP32 (ray.ts:25-28)
    V3 sd = V3{(float)__dmul_rn((double)r.d.x, t), (float)__dmul_rn((double)r.d.y, t), (float)__dmul_rn((double)r.d.z, t)};
    V3 ip = V3{__fadd_rn(r.o.x, sd.x), __fadd_rn(r.o.y, sd.y), __fadd_rn(r.o.z, sd.z)};
    V3 hp = V3{__fsub_rn(ip.x, e->q[0]), __fsub_rn(ip.y, e->q[1]), __fsub_rn(ip.z, e->q[2])};
    auto crossf = [](V3 a, V3 b) {
      double ax = a.x, ay = a.y, az = a.z, bx = b.x, by = b.y, bz = b.z;
      return V3{(float)__dsub_rn(__dmul_rn(ay, bz), __dmul_rn(az, by)), (float)__dsub_rn(__dmul_rn(az, bx), __dmul_rn(ax, bz)),
                (float)__dsub_rn(__dmul_rn(ax, by), __dmul_rn(ay, bx))};
    };
    double alpha = ddot(e->w, crossf(hp, ld3(e->v)));
    double beta = ddot(e->w, crossf(ld3(e->u), hp));
    if (alpha < 0 || alpha > 1 || beta < 0 || beta > 1) return false;
  }
  t_out = t;
  return true;
}

// Decide in FP64 whether slot `slot` beats the current best (tbest from slot sbest).  When
// the two distances agree to FP32 resolution the incumbent is re-evaluated in FP64 too and
// the comparison is the reference's strict `<` (interval.ts:51-53): on an exact tie the
// primitive the reference visits first keeps the hit (hittableList.ts:76-84 / bvh.ts:139-145).
__device__ __noinline__ bool exact_closer(const ExactPrim* ex, int slot, int sbest, float tbest, Ray r, float& t_out) {
  double tn;
  if (!prim_exact(ex + slot, r, 0.001, (double)CUDART_INF_F, tn)) return false;
  if (sbest >= 0) {
    double tb = (double)tbest;
    if (tn > tb * (1.0 + 4.0 * (double)kEps32)) return false;
    if (tn >= tb * (1.0 - 4.0 * (double)kEps32)) {
      double te;
      if (prim_exact(ex + sbest, r, 0.001, (double)CUDART_INF_F, te)) tb = te;
      if (!(tn < tb || (tn == tb && ex[slot].rank < ex[sbest].rank))) return false;
    }
  }
  t_out = (float)tn;
  return true;
}

// ---------------------------------------------------------------------------------------
// FP32 primitive tests, branch-free.  Return 1 = hit (t_out valid), 0 = miss, 2 = ambiguous.
// The interval is the open (0.001, tbest) of camera.ts:249 / hittableList.ts:76-84.
// ---------------------------------------------------------------------------------------
// sphere.ts:45-66 rewritten for FP32: disc/a = r^2 - |oc - (oc.d/a) d|^2 (cancellation-free
// form), roots -s -/+ sqrt(disc)/a, near root first then far root (sphere.ts:59-65).
// EARLY_MISS: leave as soon as the line is known to pass the sphere.  For the LIST loops over many small
// spheres, where nearly always every lane of the warp takes that exit (the rest of the test is then skipped
// by the whole warp); the plain form stays branch-free.
// e_quick: a per-ray upper bound of E for every sphere of the list (sphere_quick_bound), so that most misses
// leave before E itself is computed.
template <bool EARLY_MISS = false>
RT_DEV int sphere_test(F4 s, const Ray& r, const RayPre& pre, float tbest, float& t_out, float e_quick = 3.0e38f) {
  V3 oc = r.o - xyz(s);
  float hb = dot3(oc, r.d);
  float sp = hb * pre.inva;
  V3 l = fma3(-sp, r.d, oc);
  float l2 = dot3(l, l);
  float r2 = s.w * s.w;
  float da = r2 - l2;
  if (EARLY_MISS && da < -e_quick) { t_out = 0.f; return 0; }
  float el = 4.f * kEps32 * fmaf(fabsf(sp), pre.l1d, l1norm(oc)); // bound on each component of the error of l
  float E = fmaf(2.f * l1norm(l), el, 8.f * kEps32 * (r2 + l2));  // bound on the error of da
  if (EARLY_MISS && da < -E) { t_out = 0.f; return 0; }
  float q = fmaxf(da, 0.f) * pre.inva;
  float rs = rsqrt_approx(q);
  float sqd = q * rs; // NaN when q == 0: then da <= E and the answer below does not depend on it
  float terr = fmaf(0.5f * E * pre.inva, rs, 8.f * kEps32 * (fabsf(sp) + sqd));
  float t0 = -sp - sqd, t1 = -sp + sqd;
  float m0 = fminf(t0 - kRayTMin, tbest - t0);
  float m1 = fminf(t1 - kRayTMin, tbest - t1);
  bool in0 = m0 > terr, out0 = m0 < -terr;
  bool in1 = m1 > terr, out1 = m1 < -terr;
  float t = in0 ? t0 : t1;
  bool root_ok = in0 | (out0 & in1);
  bool root_none = out0 & out1;
  bool real = da > E;
  bool sure_hit = real & root_ok & (terr <= 2e-5f * t);
  bool sure_miss = (da < -E) | (real & root_none);
  t_out = t;
  return sure_hit ? 1 : (sure_miss ? 0 : 2);
}

// plane.ts:55-77 / quad.ts:50-63.  p0 = (n, D), p1 = (A, q.A), p2 = (B, q.B),
// p3 = (|A|_1, |B|_1, 4eps|q.A|, 4eps|q.B|)  — see rt_types.h.
RT_DEV int planar_test(F4 p0, F4 p1, F4 p2, F4 p3, bool is_quad, const Ray& r, const RayPre& pre, float tbest, float& t_out) {
  V3 n = xyz(p0);
  float denom = dot3(n, r.d);
  float num = p0.w - dot3(n, r.o);
  float inv = rcp_approx(denom);
  float t = num * inv;
  // |error of t| <= (4eps(|D| + sum|n_i o_i|))/|denom| + (rcp, mul roundings) * |t|
  float terr = fmaf(4.f * kEps32 * (fabsf(p0.w) + pre.omax175), fabsf(inv), 8.f * kEps32 * fabsf(t));
  float mt = fminf(t - kRayTMin, tbest - t);
  bool ok_d = fabsf(denom) >= 1e-8f; // plane.ts:58
  bool in_t = mt > terr, out_t = mt < -terr;
  bool in_ab = true, out_ab = false;
  if (is_quad) {
    V3 p = fma3(t, r.d, r.o);
    float alpha = dot3(p, xyz(p1)) - p1.w;
    float beta = dot3(p, xyz(p2)) - p2.w;
    // |error of alpha| <= |A|_1 (4eps max|p_i| + terr max|d_i|) + 4eps|q.A|
    float k = fmaf(terr, pre.dmax, 4.f * kEps32 * fmaf(fabsf(t), pre.dmax, pre.omax175));
    float ea = fmaf(p3.x, k, p3.z), eb = fmaf(p3.y, k, p3.w);
    float ma = fminf(alpha, 1.f - alpha), mb = fminf(beta, 1.f - beta); // >= 0 inside [0,1] (inclusive, quad.ts:60)
    in_ab = fminf(ma - ea, mb - eb) >= 0.f;
    out_ab = fminf(ma + ea, mb + eb) < 0.f;
  }
  bool sure_hit = ok_d & in_t & in_ab;
  bool sure_miss = !ok_d | out_t | out_ab;
  t_out = t;
  return sure_hit ? 1 : (sure_miss ? 0 : 2);
}

// Axis-aligned quad (u and v each along one coordinate axis; the scene compiler detects them):
// the plane is x_K = c and the inside test is an interval test on the two other coordinates —
// the same set as plane.ts:55-77 + quad.ts:60 describe, at a third of the arithmetic.
//   p1 = (c, lo_I, lo_J, hi_I), p2 = (hi_J, axis bits, -, -), I = (K+1)%3, J = (K+2)%3.
template <int K>
RT_DEV int aaquad_test(F4 p1, F4 p2, const Ray& r, const RayPre& pre, float tbest, float& t_out) {
  constexpr int I = (K + 1) % 3, J = (K + 2) % 3;
  const float o[3] = {r.o.x, r.o.y, r.o.z}, d[3] = {r.d.x, r.d.y, r.d.z};
  const float id[3] = {pre.idir.x, pre.idir.y, pre.idir.z};
  const float t = (p1.x - o[K]) * id[K];
  const float terr = fmaf(4.f * kEps32 * (fabsf(p1.x) + fabsf(o[K])), fabsf(id[K]), 8.f * kEps32 * fabsf(t));
  const float mt = fminf(t - kRayTMin, tbest - t);
  const float pi = fmaf(t, d[I], o[I]), pj = fmaf(t, d[J], o[J]);
  const float ei = fmaf(terr, fabsf(d[I]), 4.f * kEps32 * (fabsf(o[I]) + fabsf(t * d[I])));
  const float ej = fmaf(terr, fabsf(d[J]), 4.f * kEps32 * (fabsf(o[J]) + fabsf(t * d[J])));
  const float mi = fminf(pi - p1.y, p1.w - pi), mj = fminf(pj - p1.z, p2.x - pj); // >= 0 inside (inclusive, quad.ts:60)
  const bool ok_d = fabsf(d[K]) >= 1e-8f; // plane.ts:58 with n = +-e_K
  const bool sure_hit = ok_d & (mt > terr) & (fminf(mi - ei, mj - ej) >= 0.f);
  const bool sure_miss = !ok_d | (mt < -terr) | (fminf(mi + ei, mj + ej) < 0.f);
  t_out = t;
  return sure_hit ? 1 : (sure_miss ? 0 : 2);
}

// One primitive slot against the ray; updates (tbest, sbest) on a closer hit.
// type: OBJ_SPHERE / OBJ_PLANE / OBJ_QUAD / OBJ_AAQUAD (axis in p2.y) / OBJ_AAQUAD + 1 + axis (LIST staging).
template <class Scene>
RT_DEV void test_slot(const Scene& S, int slot, int type, F4 p0, F4 p1, F4 p2, F4 p3, const Ray& r, const RayPre& pre,
                      float& tbest, int& sbest) {
  float t;
  int res;
  if (type == OBJ_SPHERE) res = sphere_test(p0, r, pre, tbest, t); // (an early return on sure misses: no gain in tree leaves, measured)
  else if (type >= OBJ_AAQUAD) {
    const int axis = type > OBJ_AAQUAD ? type - OBJ_AAQUAD - 1 : __float_as_int(p2.y);
    if (axis == 0) res = aaquad_test<0>(p1, p2, r, pre, tbest, t);
    else if (axis == 1) res = aaquad_test<1>(p1, p2, r, pre, tbest, t);
    else res = aaquad_test<2>(p1, p2, r, pre, tbest, t);
  }
  else res = planar_test(p0, p1, p2, p3, type == OBJ_QUAD, r, pre, tbest, t);
  if (res == 2) res = exact_closer(S.exact, slot, sbest, tbest, r, t) ? 1 : 0;
  if (res == 1) { tbest = t; sbest = slot; }
}

// ---------------------------------------------------------------------------------------
// Box tests
// ---------------------------------------------------------------------------------------
// True slab test, conservative (tmax padded by 4 ulp); NaNs from 0*inf are dropped by
// fminf/fmaxf.  Returns the entry distance through tnear.
RT_DEV bool slab_hit(const float* mn, const float* mx, const RayPre& pre, float tmin, float tmax, float& tnear) {
  float x0 = fmaf(mn[0], pre.idir.x, -pre.oid.x), x1 = fmaf(mx[0], pre.idir.x, -pre.oid.x);
  float y0 = fmaf(mn[1], pre.idir.y, -pre.oid.y), y1 = fmaf(mx[1], pre.idir.y, -pre.oid.y);
  float z0 = fmaf(mn[2], pre.idir.z, -pre.oid.z), z1 = fmaf(mx[2], pre.idir.z, -pre.oid.z);
  float tn = fmaxf(fmaxf(fminf(x0, x1), fminf(y0, y1)), fmaxf(fminf(z0, z1), tmin));
  float tf = fminf(fminf(fmaxf(x0, x1), fmaxf(y0, y1)), fminf(fmaxf(z0, z1), tmax));
  tnear = tn;
  return tn <= tf * 1.0000005f + 1e-30f;
}
// The reference's own rule (aabb.ts:30-59): each axis independently against the original
// interval, NaN comparisons fall through as "overlap" — padded so FP32 never rejects what
// FP64 accepts.  Used only on the ancestors of inverted boxes (negative-radius spheres), where
// this rule — not geometry — decides what the reference can reach.
RT_DEV bool ref_box_hit(const float* mn, const float* mx, const Ray& r, const RayPre& pre, float tmin, float tmax) {
  const float o[3] = {r.o.x, r.o.y, r.o.z};
  const float id[3] = {pre.idir.x, pre.idir.y, pre.idir.z};
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    float t0 = (mn[a] - o[a]) * id[a];
    float t1 = (mx[a] - o[a]) * id[a];
    if (id[a] < 0.f) { float tt = t0; t0 = t1; t1 = tt; }
    float lo = t0 > tmin ? t0 : tmin;
    float hi = t1 < tmax ? t1 : tmax;
    float pad = 8.f * kEps32 * (fabsf(lo) + fabsf(hi));
    if (hi + pad <= lo) return false;
  }
  return true;
}

// ---------------------------------------------------------------------------------------
// Closest hit over (0.001, inf): the device form of world.hit (camera.ts:249).
// ---------------------------------------------------------------------------------------
struct Node4 {
  F4 a, b, c, d;
};
RT_DEV Node4 load_node(const F4* nodes, int idx) {
  const F4* p = nodes + 4 * (size_t)idx;
  return Node4{ldg4(p), ldg4(p + 1), ldg4(p + 2), ldg4(p + 3)};
}

template <class Scene>
RT_DEV void intersect_leaf(const Scene& S, int ref, const Ray& r, const RayPre& pre, float& tbest, int& sbest) {
  int v = ~ref;
  int first = v >> 6, count = ((v >> 4) & 3) + 1, mask = v & 15;
#pragma unroll 1
  for (int k = 0; k < count; ++k) {
    int slot = first + k;
    F4 p0 = ldg4(S.p0 + slot);
    if ((mask >> k) & 1) {
      int type = (ldgi2(S.slot_info + slot).y >> 30) & 3;
      test_slot(S, slot, type, p0, ldg4(S.p1 + slot), ldg4(S.p2 + slot), ldg4(S.p3 + slot), r, pre, tbest, sbest);
    } else {
      F4 z{0, 0, 0, 0};
      test_slot(S, slot, OBJ_SPHERE, p0, z, z, z, r, pre, tbest, sbest);
    }
  }
}

// LIST: every slot in the reference's visiting order; records come from shared memory and
// the primitive type is warp-uniform, so the loop runs fully converged.
// The kernels hold ONE `__shared__ ListSmemData`; everything else sees it through `ListSmem`, a handle that is the
// 32-bit shared-space address of that object: each access is `ld.shared` at base + compile-time offset + 16 s.
// (Through C++ pointers or references the compiler rebuilt the shared-window base in every loop iteration —
// S2UR SR_CgaCtaId, UMOV, ULEA: three of the ~50 instructions of a quad test — and round 1's struct of four
// pointers cost four registers on top.)
static constexpr int kListMax = 128;
struct ListSmemData {
  F4 p0[kListMax], p1[kListMax], p2[kListMax], p3[kListMax];
  int type[kListMax];
  int mat[kListMax];
};
RT_DEV F4 lds_f4(uint32_t a) {
  F4 v;
  asm("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
  return v;
}
RT_DEV float lds_f(uint32_t a) {
  float v;
  asm("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
  return v;
}
RT_DEV int lds_i(uint32_t a) {
  int v;
  asm("ld.shared.s32 %0, [%1];" : "=r"(v) : "r"(a));
  return v;
}
struct ListSmem {
  uint32_t base; // shared-space address of the ListSmemData, taken AFTER the staging barrier (stage_list)
  RT_DEV F4 p0(int s) const { return lds_f4(base + (uint32_t)offsetof(ListSmemData, p0) + 16u * (uint32_t)s); }
  RT_DEV F4 p1(int s) const { return lds_f4(base + (uint32_t)offsetof(ListSmemData, p1) + 16u * (uint32_t)s); }
  RT_DEV F4 p2(int s) const { return lds_f4(base + (uint32_t)offsetof(ListSmemData, p2) + 16u * (uint32_t)s); }
  RT_DEV F4 p3(int s) const { return lds_f4(base + (uint32_t)offsetof(ListSmemData, p3) + 16u * (uint32_t)s); }
  RT_DEV float p2x(int s) const { return lds_f(base + (uint32_t)offsetof(ListSmemData, p2) + 16u * (uint32_t)s); }
  RT_DEV int type(int s) const { return lds_i(base + (uint32_t)offsetof(ListSmemData, type) + 4u * (uint32_t)s); }
  RT_DEV int mat(int s) const { return lds_i(base + (uint32_t)offsetof(ListSmemData, mat) + 4u * (uint32_t)s); }
};
using SmemList = ListSmem;
RT_DEV void take_hit(const ExactPrim* ex, int res, float t, int slot, const Ray& r, float& tbest, int& sbest) {
  if (res == 2) { // the FP64 re-test writes through a pointer: a variable of its own, so `t` itself never lives in local memory
    float te;
    res = exact_closer(ex, slot, sbest, tbest, r, te) ? 1 : 0;
    if (res) t = te;
  }
  if (res == 1) { tbest = t; sbest = slot; }
}
// All axis-aligned quads with normal along K, slots [s, e): aaquad_test<K> with the per-ray parts of its
// error bounds hoisted out of the loop, the two in-plane bounds merged into one, and |t| <= (|c| + |o_K|)|1/d_K|
// used so that each bound needs ONE per-ray constant (the loop runs under an 80-register cap: constants the
// compiler cannot keep are recomputed every iteration):
//   |error of t|      <= 4eps(|c| + |o_K|)|1/d_K| + 8eps|t|  <=  12eps |1/d_K| (|c| + |o_K|)          = aK (|c| + |o_K|)
//   |error of p_I,J|  <= terr max|d| + 4eps(max|o| + |t| max|d|)  =  max|d| (terr + 4eps|t|) + c0   (>= aaquad_test's ei, ej)
// so the "sure" sets only shrink and everything in between still goes to the FP64 re-test.
template <int K>
RT_DEV void aaquad_run(const ExactPrim* ex, const SmemList& L, int& s, const int e, const Ray& r, const RayPre& pre, float& tbest,
                       int& sbest) {
  constexpr int I = (K + 1) % 3, J = (K + 2) % 3;
  const float o[3] = {r.o.x, r.o.y, r.o.z}, d[3] = {r.d.x, r.d.y, r.d.z};
  const float id[3] = {pre.idir.x, pre.idir.y, pre.idir.z};
  if (!(fabsf(d[K]) >= 1e-8f)) { s = e; return; } // plane.ts:58 with n = +-e_K: a ray parallel to the planes misses them all
  const float aK = 12.f * kEps32 * fabsf(id[K]);
  const float c0 = 4.f * kEps32 * pre.omax175;
#pragma unroll 1 // the kernel is instruction-cache bound: an unrolled copy of take_hit's FP64 branch costs more than it saves
  for (; s < e; ++s) {
    const F4 p1 = L.p1(s);
    const float hiJ = L.p2x(s);
    const float t = (p1.x - o[K]) * id[K];
    const float terr = aK * (fabsf(p1.x) + fabsf(o[K]));
    const float mt = fminf(t - kRayTMin, tbest - t);
    const float pi = fmaf(t, d[I], o[I]), pj = fmaf(t, d[J], o[J]);
    const float err = fmaf(pre.dmax, fmaf(4.f * kEps32, fabsf(t), terr), c0);
    const float m = fminf(fminf(pi - p1.y, p1.w - pi), fminf(pj - p1.z, hiJ - pj)); // >= 0 inside (inclusive, quad.ts:60)
    const bool sure_hit = (mt > terr) & (m >= err);
    const bool sure_miss = (mt < -terr) | (m < -err);
    take_hit(ex, sure_hit ? 1 : (sure_miss ? 0 : 2), t, s, r, tbest, sbest);
  }
}

// Slots are grouped by kind (S.list_n): one tight loop per kind, each loading only its own records.
template <class Scene>
RT_DEV void trace_list(const Scene& S, const SmemList& L, const Ray& r, const RayPre& pre, float& tbest, int& sbest) {
  int s = 0;
  float t;
  // early exit on a sure miss: with many small spheres the whole warp nearly always takes it (49-sphere box:
  // 109.5 -> 93.9 ms; Cornell with its two big spheres: +1 %)
  // A bound of E that holds for every sphere of the list, from per-ray and per-scene constants only:
  // with M >= |oc|_1 (M = 3 (max|o| + max|c|)):  |l|_1 <= sqrt3 |l|_2 <= sqrt3 M (l is the part of oc
  // perpendicular to d),  |sp| |d|_1 <= sqrt3 |oc|_2 <= sqrt3 M,  l2 <= M^2, hence
  // el <= 4eps (1 + sqrt3) M and E <= eps (38.1 M^2 + 8 (r2 + M^2)) <= eps (47 M^2 + 8 r2max); 64 / 16 below.
  const float M = 3.f * (pre.omax175 + S.sph_cmax);
  const float e_quick = kEps32 * fmaf(64.f * M, M, 16.f * S.sph_r2max);
#pragma unroll 1
  for (const int e = s + S.list_n[0]; s < e; ++s)
    take_hit(S.exact, sphere_test<true>(L.p0(s), r, pre, tbest, t, e_quick), t, s, r, tbest, sbest);
  aaquad_run<0>(S.exact, L, s, s + S.list_n[1], r, pre, tbest, sbest);
  aaquad_run<1>(S.exact, L, s, s + S.list_n[2], r, pre, tbest, sbest);
  aaquad_run<2>(S.exact, L, s, s + S.list_n[3], r, pre, tbest, sbest);
  for (const int e = s + S.list_n[4]; s < e; ++s)
    take_hit(S.exact, planar_test(L.p0(s), L.p1(s), L.p2(s), L.p3(s), true, r, pre, tbest, t), t, s, r, tbest, sbest);
  for (const int e = s + S.list_n[5]; s < e; ++s)
    take_hit(S.exact, planar_test(L.p0(s), L.p1(s), L.p2(s), L.p3(s), false, r, pre, tbest, t), t, s, r, tbest, sbest);
}

// SAH traversal in resumable steps: trav_begin() tests the unbounded prefix and parks the ray at the root,
// trav_inner() visits one node (both child boxes) and hands back leaf children, trav_leaves() intersects
// them.  trace_sah() strings them into a whole query; k_render_trav and the wavefront extend kernel run them
// in bursts interleaved with shading so that lanes whose ray finished early do not idle until the longest
// traversal of the warp is over.
// Work actually executed by a lane: closest-hit queries, and — only in the instrumented build (-DRT_COUNT_EVENTS,
// libmcprt_b200_count.so: the roofline's "executed" figure for tree scenes) — wide-node visits and primitive tests.
struct WorkCount {
  unsigned rays = 0;
#ifdef RT_COUNT_EVENTS
  unsigned visits = 0, prims = 0;
#endif
};
#ifdef RT_COUNT_EVENTS
#define RT_COUNT_VISIT(wc) (++(wc).visits)
#define RT_COUNT_LEAVES(wc, lv) ((wc).prims += leaf_prims((lv).a) + leaf_prims((lv).b) + leaf_prims((lv).c) + leaf_prims((lv).d))
#define RT_COUNT_PRIMS(wc, n) ((wc).prims += (unsigned)(n))
RT_DEV unsigned leaf_prims(int ref) { return ref == 0 ? 0u : (unsigned)(((~ref) >> 4) & 3) + 1u; }
#else
#define RT_COUNT_VISIT(wc) ((void)0)
#define RT_COUNT_LEAVES(wc, lv) ((void)0)
#define RT_COUNT_PRIMS(wc, n) ((void)0)
#endif

struct Trav {
  int cur; // node to visit next, -1 = traversal finished
  int sp;
  float tbest;
  int sbest;
};
struct BoxPre {
  V3 idir, oid; // 1/d, o/d
};
RT_DEV BoxPre box_precompute(const Ray& r) {
  BoxPre b;
  // like precompute(): MUFU reciprocals, the slab tests pad the exit distance by 4 ulp
  b.idir = V3{rcp_approx(r.d.x), rcp_approx(r.d.y), rcp_approx(r.d.z)};
  b.oid = r.o * b.idir;
  return b;
}
RT_DEV bool slab_hit(const float* mn, const float* mx, const BoxPre& pre, float tmin, float tmax, float& tnear) {
  float x0 = fmaf(mn[0], pre.idir.x, -pre.oid.x), x1 = fmaf(mx[0], pre.idir.x, -pre.oid.x);
  float y0 = fmaf(mn[1], pre.idir.y, -pre.oid.y), y1 = fmaf(mx[1], pre.idir.y, -pre.oid.y);
  float z0 = fmaf(mn[2], pre.idir.z, -pre.oid.z), z1 = fmaf(mx[2], pre.idir.z, -pre.oid.z);
  float tn = fmaxf(fmaxf(fminf(x0, x1), fminf(y0, y1)), fmaxf(fminf(z0, z1), tmin));
  float tf = fminf(fminf(fmaxf(x0, x1), fmaxf(y0, y1)), fminf(fmaxf(z0, z1), tmax));
  tnear = tn;
  return tn <= tf * 1.0000005f + 1e-30f;
}
// The wide nodes hold (centre, half-extent) boxes: per axis the slab is entered at tc - h|1/d| and left at tc + h|1/d| with
// tc = c/d - o/d — three FFMA (the |.| is an operand modifier) and no min / max to order the two planes.  The deep-tree
// kernels are bound by the ALU pipe (FMNMX, SEL, compares: 54-66 % busy at 47-65 % issue in ncu) while the FMA pipe idles
// at 12-20 %: 5 ALU instructions per box instead of 11.  NaNs (0 * inf on an axis the ray is parallel to) are dropped by
// fminf / fmaxf as before, which keeps the test conservative.
RT_DEV bool slab_hit_ch(const float* c, const float* h, const BoxPre& pre, float tmin, float tmax, float& tnear) {
  const float tx = fmaf(c[0], pre.idir.x, -pre.oid.x), ty = fmaf(c[1], pre.idir.y, -pre.oid.y), tz = fmaf(c[2], pre.idir.z, -pre.oid.z);
  const float ax = fabsf(pre.idir.x), ay = fabsf(pre.idir.y), az = fabsf(pre.idir.z);
  const float tn = fmaxf(fmaxf(fmaf(-h[0], ax, tx), fmaf(-h[1], ay, ty)), fmaxf(fmaf(-h[2], az, tz), tmin));
  const float tf = fminf(fminf(fmaf(h[0], ax, tx), fmaf(h[1], ay, ty)), fminf(fmaf(h[2], az, tz), tmax));
  tnear = tn;
  return tn <= tf * 1.0000005f + 1e-30f;
}
template <class Scene>
RT_DEV void trav_begin(const Scene& S, const Ray& r, Trav& tv) {
  tv.tbest = CUDART_INF_F;
  tv.sbest = -1;
  tv.sp = 0;
  if (S.n_unbounded > 0) {
    const RayPre pre = precompute(r, true); // the prefix may hold axis-aligned quads (they use 1/d)
    for (int s = 0; s < S.n_unbounded; ++s) {
      int type = (ldgi2(S.slot_info + s).y >> 30) & 3;
      test_slot(S, s, type, ldg4(S.p0 + s), ldg4(S.p1 + s), ldg4(S.p2 + s), ldg4(S.p3 + s), r, pre, tv.tbest, tv.sbest);
    }
  }
  tv.cur = S.n_nodes > 0 ? 0 : -1;
}

// One node visit: trav_inner() tests the two child boxes, descends / pushes / pops, and parks leaf children in
// leaf_a / leaf_b (0 = none, nearer one first); trav_leaves() intersects them (while-while with postponed leaves).
// (Storing the entry distance with each pending child and skipping unreachable entries on pop was measured:
// 4-9 % slower on all three tree scenes — the second local-memory array costs more than the skipped visits.)
struct TravStack {
  int ref[128]; // a visit pushes up to three pending children: depth <= 42 wide levels (checked by the scene compiler)
};
struct TravLeaves { // leaf children of the last visit whose boxes were hit, packed to the front; 0 = none
  int a, b, c, d;
};
// One visit of a 4-wide node (WideNode, rt_types.h): four slab tests; hit leaves are parked in `lv`, hit inner
// children are sorted by entry distance (5 compare-exchanges), the nearest becomes the next node and the
// others go on the stack, farthest first.  (Prefetching pending nodes / leaf records was measured: 5 % slower.)
// SORT = false (whole-query walks of small trees, trace_sah): only the NEAREST hit inner child is singled out, the others are
// pushed in child order — one integer min instead of the sorting network.  Measured: 480 spheres 36.55 -> 35.85 ms, 100 spheres
// 7.75 -> 7.57 ms; on the 100 k-sphere tree the unsorted stack costs more visits than it saves (388 -> 422 ms), so the
// deep-tree kernels keep the sort.
template <bool SORT = true, class Scene>
RT_DEV void trav_inner(const Scene& S, const BoxPre& bp, Trav& tv, TravStack& stack, TravLeaves& lv) {
  const float tmin = kRayTMin;
  const F4* p = S.nodes + 8 * (size_t)tv.cur;
  const F8 w0 = ldg8(p), w1 = ldg8(p + 2), w2 = ldg8(p + 4); // 3 x 256 bits: the four boxes
  const F4 q6 = ldg4(p + 6);                                 // the four refs
  const float b0[6] = {w0.v[0], w0.v[1], w0.v[2], w0.v[3], w0.v[4], w0.v[5]}, b1[6] = {w0.v[6], w0.v[7], w1.v[0], w1.v[1], w1.v[2], w1.v[3]};
  const float b2[6] = {w1.v[4], w1.v[5], w1.v[6], w1.v[7], w2.v[0], w2.v[1]}, b3[6] = {w2.v[2], w2.v[3], w2.v[4], w2.v[5], w2.v[6], w2.v[7]};
  int r0 = __float_as_int(q6.x), r1 = __float_as_int(q6.y), r2 = __float_as_int(q6.z), r3 = __float_as_int(q6.w);
  float t0, t1, t2, t3;
  const bool h0 = slab_hit_ch(b0, b0 + 3, bp, tmin, tv.tbest, t0) && r0 != kEmptyRef;
  const bool h1 = slab_hit_ch(b1, b1 + 3, bp, tmin, tv.tbest, t1) && r1 != kEmptyRef;
  const bool h2 = slab_hit_ch(b2, b2 + 3, bp, tmin, tv.tbest, t2) && r2 != kEmptyRef;
  const bool h3 = slab_hit_ch(b3, b3 + 3, bp, tmin, tv.tbest, t3) && r3 != kEmptyRef;
  // leaves, in child order
  lv.a = lv.b = lv.c = lv.d = 0;
  if (h3 && r3 < 0) { lv.a = r3; }
  if (h2 && r2 < 0) { lv.d = lv.c; lv.c = lv.b; lv.b = lv.a; lv.a = r2; }
  if (h1 && r1 < 0) { lv.d = lv.c; lv.c = lv.b; lv.b = lv.a; lv.a = r1; }
  if (h0 && r0 < 0) { lv.d = lv.c; lv.c = lv.b; lv.b = lv.a; lv.a = r0; }
  if (!SORT) {
    // Entry distances are >= tmin > 0, so their bit patterns order like the floats: the two low mantissa bits carry the
    // child index and one integer min finds distance and index together.
    const int kNone = 0x7f800000;
    const int k0 = h0 && r0 >= 0 ? (__float_as_int(t0) & ~3) : kNone, k1 = h1 && r1 >= 0 ? (__float_as_int(t1) & ~3) | 1 : kNone;
    const int k2 = h2 && r2 >= 0 ? (__float_as_int(t2) & ~3) | 2 : kNone, k3 = h3 && r3 >= 0 ? (__float_as_int(t3) & ~3) | 3 : kNone;
    const int kmin = min(min(k0, k1), min(k2, k3));
    if (kmin != kNone) {
      const int near = kmin & 3;
      if (k3 != kNone && near != 3) stack.ref[tv.sp++] = r3;
      if (k2 != kNone && near != 2) stack.ref[tv.sp++] = r2;
      if (k1 != kNone && near != 1) stack.ref[tv.sp++] = r1;
      if (k0 != kNone && near != 0) stack.ref[tv.sp++] = r0;
      tv.cur = near == 0 ? r0 : (near == 1 ? r1 : (near == 2 ? r2 : r3));
    } else tv.cur = tv.sp > 0 ? stack.ref[--tv.sp] : -1;
    return;
  }
  // inner children: key = entry distance, +inf when not a hit inner child
  float k0 = h0 && r0 >= 0 ? t0 : CUDART_INF_F, k1 = h1 && r1 >= 0 ? t1 : CUDART_INF_F;
  float k2 = h2 && r2 >= 0 ? t2 : CUDART_INF_F, k3 = h3 && r3 >= 0 ? t3 : CUDART_INF_F;
#define RT_CSWAP(ka, ra, kb, rb)                    \
  {                                                 \
    const bool sw = kb < ka;                        \
    const float kt = sw ? kb : ka; const int rt_ = sw ? rb : ra; \
    kb = sw ? ka : kb; rb = sw ? ra : rb;           \
    ka = kt; ra = rt_;                              \
  }
  RT_CSWAP(k0, r0, k1, r1)
  RT_CSWAP(k2, r2, k3, r3)
  RT_CSWAP(k0, r0, k2, r2)
  RT_CSWAP(k1, r1, k3, r3)
  RT_CSWAP(k1, r1, k2, r2)
#undef RT_CSWAP
  if (k3 < CUDART_INF_F) stack.ref[tv.sp++] = r3;
  if (k2 < CUDART_INF_F) stack.ref[tv.sp++] = r2;
  if (k1 < CUDART_INF_F) stack.ref[tv.sp++] = r1;
  if (k0 < CUDART_INF_F) tv.cur = r0;
  else tv.cur = tv.sp > 0 ? stack.ref[--tv.sp] : -1;
  // (measured and dropped, 100 k spheres at 32 spp: prefetch.global.L1 of the next node 389 -> 403 ms, of the parked leaf's record
  //  398 ms, both 415 ms; speculative while-while — lanes that hold leaves walk on while others still search — 394 ms)
}
// The (up to four) parked leaves of one visit, one after the other through ONE copy of the primitive tests: the
// tree kernels are instruction-cache bound (with four inlined copies `no_instruction` was the top stall of
// k_render_trav, 1.6 per issued instruction): 100 k spheres 108.0 -> 102.4 ms, 480 spheres 39.6 -> 37.7 ms.
// LOOP = false keeps the four copies for k_render_stream<SAH>, the one kernel that measured slower with the
// loop (adaptive 480 spheres: 307 vs 332 ms).
template <bool LOOP = true, class Scene>
RT_DEV void leaves_intersect(const Scene& S, TravLeaves lv, const Ray& r, const RayPre& pre, float& tbest, int& sbest) {
  if (!LOOP) {
    intersect_leaf(S, lv.a, r, pre, tbest, sbest);
    if (lv.b != 0) intersect_leaf(S, lv.b, r, pre, tbest, sbest);
    if (lv.c != 0) intersect_leaf(S, lv.c, r, pre, tbest, sbest);
    if (lv.d != 0) intersect_leaf(S, lv.d, r, pre, tbest, sbest);
  } else {
#pragma unroll 1
    while (lv.a != 0) {
      intersect_leaf(S, lv.a, r, pre, tbest, sbest);
      lv.a = lv.b; lv.b = lv.c; lv.c = lv.d; lv.d = 0;
    }
  }
}
template <class Scene>
RT_DEV void trav_leaves(const Scene& S, const Ray& r, const BoxPre& bp, Trav& tv, const TravLeaves& lv) {
  RayPre pre = precompute(r, false);
  pre.idir = bp.idir; // axis-aligned quads reuse the traversal's reciprocal direction
  leaves_intersect(S, lv, r, pre, tv.tbest, tv.sbest);
}
// SAH, whole query, while-while: descend through inner nodes until this lane holds a leaf (or is done); the
// lanes of the warp reconverge at the end of the inner loop and intersect their leaves together.  With leaves
// tested on the spot (trace_sah_ifif) the sphere tests ran with 19 % of the lanes (ncu, 480-sphere scene).
template <bool LEAF_LOOP = true, class Scene>
RT_DEV void trace_sah(const Scene& S, const Ray& r, const RayPre& pre, float& tbest, int& sbest, WorkCount& wc) {
  RT_COUNT_PRIMS(wc, S.n_unbounded);
  for (int s = 0; s < S.n_unbounded; ++s) {
    int type = (ldgi2(S.slot_info + s).y >> 30) & 3;
    test_slot(S, s, type, ldg4(S.p0 + s), ldg4(S.p1 + s), ldg4(S.p2 + s), ldg4(S.p3 + s), r, pre, tbest, sbest);
  }
  if (S.n_nodes == 0) return;
  TravStack stack;
  Trav tv{0, 0, tbest, sbest};
  const BoxPre bp{pre.idir, pre.oid};
  for (;;) {
    TravLeaves lv{0, 0, 0, 0};
    while (tv.cur >= 0 && lv.a == 0) { trav_inner<false>(S, bp, tv, stack, lv); RT_COUNT_VISIT(wc); }
    if (lv.a == 0) break;
    RT_COUNT_LEAVES(wc, lv);
    leaves_intersect<LEAF_LOOP>(S, lv, r, pre, tv.tbest, tv.sbest);
  }
  tbest = tv.tbest;
  sbest = tv.sbest;
}

// REFERENCE: depth-first, left subtree completely before the right box is (re)tested with
// the shrunken interval — bvh.ts:128-146.
template <class Scene>
RT_DEV void trace_ref(const Scene& S, const Ray& r, const RayPre& pre, float& tbest, int& sbest) {
  const float tmin = kRayTMin;
  int stack[64]; // node indices whose RIGHT child is pending
  int sp = 0;
  int cur = 0;
  bool enter_right = false; // cur's left side is done; evaluate its right child
  for (;;) {
    Node4 nd = load_node(S.nodes, cur);
    const int flags = __float_as_int(nd.d.z);
    int next = -1;
    float tn;
    if (!enter_right) {
      const float lmn[3] = {nd.a.x, nd.a.y, nd.a.z}, lmx[3] = {nd.a.w, nd.b.x, nd.b.y};
      int lref = __float_as_int(nd.d.x), rref = __float_as_int(nd.d.y);
      if (rref != kEmptyRef) stack[sp++] = cur;
      if (lref != kEmptyRef && ((flags & 1) ? ref_box_hit(lmn, lmx, r, pre, tmin, tbest) : slab_hit(lmn, lmx, pre, tmin, tbest, tn))) {
        if (lref < 0) intersect_leaf(S, lref, r, pre, tbest, sbest);
        else next = lref;
      }
    } else {
      const float rmn[3] = {nd.b.z, nd.b.w, nd.c.x}, rmx[3] = {nd.c.y, nd.c.z, nd.c.w};
      int rref = __float_as_int(nd.d.y);
      if ((flags & 2) ? ref_box_hit(rmn, rmx, r, pre, tmin, tbest) : slab_hit(rmn, rmx, pre, tmin, tbest, tn)) {
        if (rref < 0) intersect_leaf(S, rref, r, pre, tbest, sbest);
        else next = rref;
      }
    }
    if (next >= 0) { cur = next; enter_right = false; continue; }
    if (sp == 0) return;
    cur = stack[--sp];
    enter_right = true;
  }
}

// ---------------------------------------------------------------------------------------
// Surface at a hit: rec.p, rec.normal (face-forwarded), rec.frontFace
// (sphere.ts:68-84, plane.ts:93-97, quad.ts:64-67).
// ---------------------------------------------------------------------------------------
struct Surf {
  V3 p, n;
  bool front;
};
RT_DEV Surf surface_at(int type, F4 p0, const Ray& r, float t) {
  Surf s;
  s.p = fma3(t, r.d, r.o);
  V3 ns = (s.p - xyz(p0)) * rcp_approx(p0.w);
  V3 n = sel3(type == OBJ_SPHERE, ns, xyz(p0));
  s.front = dot3(r.d, n) <= 0.f;
  s.n = sel3(s.front, n, mk3(0.f - n.x, 0.f - n.y, 0.f - n.z)); // 0-x: negate() canonicalises -0 (vec3.ts:60-70)
  return s;
}

// ---------------------------------------------------------------------------------------
// Sampling — vec3.ts:272-364, onbasis.ts:18-51, pdf.ts:32-51
// ---------------------------------------------------------------------------------------
struct Onb {
  V3 u, v, w;
};
template <bool UNIT = false> // UNIT: n is already a unit vector (surface normals), skip the renormalisation
RT_DEV Onb make_onb(V3 n) { // onbasis.ts:18-25
  Onb b;
  b.w = UNIT ? n : normalize3(n);
  bool xmajor = fabsf(b.w.x) > 0.9f;
  // v = unit(w x a) with a = (0,1,0) or (1,0,0), written out
  V3 c = xmajor ? mk3(-b.w.z, 0.f, b.w.x) : mk3(0.f, b.w.z, -b.w.y);
  b.v = normalize3(c);
  b.u = cross3(b.w, b.v);
  return b;
}
RT_DEV V3 onb_local(const Onb& b, V3 a) { return fma3(a.x, b.u, fma3(a.y, b.v, b.w * a.z)); }
RT_DEV V3 cosine_direction(float r1, float r2) { // vec3.ts:325-337
  // phi = 2 pi r1 folded to [-pi, pi) so the MUFU sin / cos stay in their accurate range (absolute error ~5e-7, the
  // level of the FP32 roundings around it); sincospif costs ~25 instructions more per diffuse bounce.
  // Measured (1024^2 @256 / 2048^2 @64 / 1920x1080 @64): Cornell 30.23 -> 29.77 ms, layered 88.96 -> 88.40, weekend 37.86 -> 37.09.
  const float rr = r1 - (r1 >= 0.5f ? 1.f : 0.f);
  const float sn = __sinf(6.28318530718f * rr);
  const float cs = __cosf(6.28318530718f * rr);
  const float s = sqrtf(r2);
  return mk3(cs * s, sn * s, sqrtf(1.f - r2));
}
template <class G>
RT_DEV V3 random_in_unit_sphere(G& g) {
  for (;;) {
    float x = fmaf(2.f, g.next(), -1.f), y = fmaf(2.f, g.next(), -1.f), z = fmaf(2.f, g.next(), -1.f);
    V3 p = mk3(x, y, z);
    if (dot3(p, p) < 1.f) return p;
  }
}
// The Philox stream: a trial needs three uniforms and a block yields five, so the second trial of the rejection loop (48 % of
// the fuzzy-metal hits, 23 % need a third ...) ran into Rng::next()'s out-of-line refill in the middle of a trial — one lane at a
// time (ncu, 100 k metal spheres: that call at 2 of 32 lanes).  Here the block is generated at the TOP of a trial that cannot be
// served from what is pending: the lanes in the same trial number do it together.  Same draws in the same order (leftovers first).
RT_DEV V3 random_in_unit_sphere(Rng& g) {
  for (;;) {
    uint32_t a, b, c;
    if (g.avail >= 3) {
      a = g.q0; b = g.q1; c = g.q2;
      g.q0 = g.q3; g.q1 = g.q4;
      g.avail -= 3;
    } else {
      const int left = g.avail; // 0, 1 or 2 pending values go first
      const uint32_t l0 = g.q0, l1 = g.q1;
      g.load(philox4x32(g.block, g.stream, g.seed_lo, g.seed_hi, g.k0, g.k1));
      ++g.block;
      const int take = 3 - left; // from the new block
      a = left >= 1 ? l0 : g.q0;
      b = left == 2 ? l1 : (left == 1 ? g.q0 : g.q1);
      c = left == 2 ? g.q0 : (left == 1 ? g.q1 : g.q2);
      const uint32_t n1 = g.q1, n2 = g.q2, n3 = g.q3, n4 = g.q4;
      g.q0 = take == 1 ? n1 : (take == 2 ? n2 : n3);
      g.q1 = take == 1 ? n2 : (take == 2 ? n3 : n4);
      g.q2 = take == 1 ? n3 : n4;
      g.q3 = n4;
      g.avail = 5 - take;
    }
    const float x = fmaf(2.f, (float)a * 5.9604645e-08f, -1.f), y = fmaf(2.f, (float)b * 5.9604645e-08f, -1.f),
                z = fmaf(2.f, (float)c * 5.9604645e-08f, -1.f);
    const V3 p = mk3(x, y, z);
    if (dot3(p, p) < 1.f) return p;
  }
}
RT_DEV float cosine_pdf_value(V3 w_unit, V3 dir) { // pdf.ts:43-46
  float c = dot3(normalize3(dir), w_unit);
  return c <= 0.f ? 0.f : c * 0.31830988618f;
}

// Light pdfs — quad.ts:123-158, sphere.ts:106-147.  A pdf evaluation is one single-primitive
// hit test, never a traced ray.
// The light records are read with 128-bit loads (DevLight is 16-byte aligned, p0..p3 at offset 0, q/u/v at 64): through a
// `const DevLight&` the compiler read p0..p3 and q, u, v as 25 scalar LDG per diffuse bounce.
RT_DEV const F4* light_f4(const DevLight& L) { return reinterpret_cast<const F4*>(&L); }
// LV = false keeps the plain member reads: k_render_pool<LIST, false> — the bench kernel, at its 80-register cap — loses 1.9 %
// to the four consecutive registers a vector load needs (Cornell 512 spp: 53.22 vs 54.24 ms, profiles/r02c_list_kernel_layout.log),
// every other kernel gains (pair-queue LIST kernel 26.82 -> 26.48 ms at 256 spp, layered/mixed 72.4 -> 70.3 ms).
template <bool LV>
RT_DEV F4 light_ld4(const F4* p) { return LV ? ldg4(p) : *p; }
#define RT_LIGHT_LD4(p) light_ld4<LV>(p)
template <bool LV = true, class Scene>
RT_DEV float light_pdf_value(const Scene& S, const DevLight& L, V3 origin, V3 dir) {
  Ray r{origin, dir};
  float t;
  RayPre pre = precompute(r, false);
  if (L.type == OBJ_QUAD) {
    // (the axis-aligned specialisation of the LIST loops was measured here too: 16% slower on Cornell,
    //  it needs 1/d per axis for a single test)
    const F4* lp = light_f4(L);
    const F4 p0 = RT_LIGHT_LD4(lp);
    int res = planar_test(p0, RT_LIGHT_LD4(lp + 1), RT_LIGHT_LD4(lp + 2), RT_LIGHT_LD4(lp + 3), true, r, pre, CUDART_INF_F, t);
    if (res == 2) res = exact_closer(S.exact, L.slot, -1, CUDART_INF_F, r, t) ? 1 : 0;
    float d2 = t * t * pre.a; // |rec.p - origin|^2
    float cosine = fabsf(dot3(dir, xyz(p0)));
    return res == 1 ? d2 / (L.area * cosine) : 0.f;
  }
  const F4 s0 = RT_LIGHT_LD4(light_f4(L));
  int res = sphere_test(s0, r, pre, CUDART_INF_F, t);
  if (res == 2) res = exact_closer(S.exact, L.slot, -1, CUDART_INF_F, r, t) ? 1 : 0;
  if (res != 1) return 0.f;
  V3 oc = xyz(s0) - origin;
  float d2 = dot3(oc, oc), r2 = L.radius * L.radius;
  if (d2 <= r2) return 0.07957747155f; // 1/(4 pi)
  float cos_theta = sqrtf(1.f - r2 / d2);
  return 1.f / (6.28318530718f * (1.f - cos_theta));
}
template <bool LV = true>
RT_DEV V3 light_random_vec(const DevLight& L, V3 origin, float r1, float r2) {
  if (L.type == OBJ_QUAD) { // quad.ts:148-158 (alpha = r1, beta = r2)
    const F4 a = RT_LIGHT_LD4(light_f4(L) + 4), b = RT_LIGHT_LD4(light_f4(L) + 5); // q.xyz u.x | u.yz v.xy
    const float vz = L.v[2];
    V3 rp = fma3(r2, mk3(b.z, b.w, vz), fma3(r1, mk3(a.w, b.x, b.y), mk3(a.x, a.y, a.z)));
    return normalize3(rp - origin);
  }
  V3 oc = xyz(ldg4(light_f4(L))) - origin; // sphere.ts:140-147, vec3.ts:345-351
  float d2 = dot3(oc, oc);
  Onb b = make_onb(oc);
  float z = 1.f + r2 * (sqrtf(1.f - L.radius * L.radius / d2) - 1.f);
  float sn, cs;
  sincospif(2.f * r1, &sn, &cs);
  float s = sqrtf(1.f - z * z);
  return onb_local(b, mk3(cs * s, sn * s, z));
}

// MixturePDF([cosine, lights...], [0.5, 0.5/n ...]) constants — camera.ts:287-288, pdf.ts:66-72
struct MixW {
  int nl;
  float wl, total_w, inv_total_w;
};
template <class Scene>
RT_DEV MixW make_mixw(const Scene& S) {
  MixW m;
  m.nl = S.n_lights;
  m.wl = m.nl > 0 ? 0.5f / (float)m.nl : 0.f;
  m.total_w = 0.5f;
  for (int k = 0; k < m.nl; ++k) m.total_w += m.wl; // summed like weights.reduce (pdf.ts:71)
  m.inv_total_w = 1.0f / m.total_w;
  return m;
}
// The diffuse branch of rayColor, camera.ts:285-308 with the mixture pdf of pdf.ts:57-99, at hit point p with unit
// normal n: `u_sel` picks the component (cosine | light k), (r1, r2) feed whichever generator was picked.
// Out: the direction, cosv = the scatter pdf's value for it (pdf.ts:43-46), pdf_value = the mixture's.
template <bool LV = true, class Scene>
RT_DEV void diffuse_bounce(const Scene& S, const MixW& mw, V3 p, V3 n, float u_sel, float r1, float r2, V3& dir, float& cosv,
                           float& pdf_value) {
  const Onb onb = make_onb<true>(n);
  const float rnd = u_sel * mw.total_w;
  dir = onb_local(onb, cosine_direction(r1, r2));
  if (mw.nl > 0) {
    float partial = 0.5f;
    int chosen = mw.nl - 1;
    for (int k = 0; k < mw.nl; ++k) {
      partial += mw.wl;
      if (rnd < partial) { chosen = k; break; }
    }
    V3 ldir = light_random_vec<LV>(S.lights[chosen], p, r1, r2);
    dir = sel3(rnd < 0.5f, dir, ldir);
  }
  const float cz = dot3(dir, onb.w); // all three generators return unit vectors
  cosv = cz <= 0.f ? 0.f : cz * 0.31830988618f;
  float sum = 0.5f * cosv;
  for (int k = 0; k < mw.nl; ++k) sum = fmaf(mw.wl, light_pdf_value<LV>(S, S.lights[k], p, dir), sum);
  pdf_value = sum * mw.inv_total_w;
}

// ---------------------------------------------------------------------------------------
// Materials — one stackless walk over the material node table.  Mixed and Layered each
// tail-call exactly one child (mixedMaterial.ts:38-45, layeredMaterial.ts:36-53), so the
// recursion of the reference is a loop here.
// ---------------------------------------------------------------------------------------
enum : int { SCATTER_NONE = 0, SCATTER_SPECULAR = 1, SCATTER_DIFFUSE = 2 };
struct Scatter {
  int kind;
  V3 attenuation;
  V3 dir; // specular: scattered direction
};
RT_DEV V3 reflect3(V3 v, V3 n) { return fma3(-2.f * dot3(v, n), n, v); }

// dielectric.ts:44-84.  Returns true when the ray was reflected.
template <class G>
RT_DEV bool dielectric_dir(V3 din, V3 n, bool front, float ior, G& g, V3& out) {
  float ratio = front ? 1.0f / ior : ior;
  V3 ud = normalize3(din);
  float cos_t = fminf(-dot3(ud, n), 1.0f);
  float sin_t = sqrtf(fmaxf(0.f, 1.0f - cos_t * cos_t));
  bool cannot = ratio * sin_t > 1.0f;
  bool refl = cannot;
  if (!cannot) {
    float r0 = (1.f - ratio) / (1.f + ratio);
    r0 *= r0;
    float m = 1.f - cos_t, m2 = m * m;
    float reflectance = fmaf(1.f - r0, m2 * m2 * m, r0);
    refl = reflectance > g.next();
  }
  V3 rd = reflect3(ud, n);
  V3 perp = fma3(cos_t, n, ud) * ratio; // vec3.ts:193-209
  float k = -sqrtf(fabsf(1.0f - dot3(perp, perp)));
  V3 td = fma3(k, n, perp);
  out = sel3(refl, rd, td);
  return refl;
}

// Everything except a plain Lambertian root (handled inline by the caller).
template <class Scene, class G>
RT_DEV Scatter scatter_material(const Scene& S, int root, I4 b, F4 a, V3 din, const Surf& sf, G& g) {
  Scatter out;
  out.kind = SCATTER_NONE;
  out.attenuation = mk3(0, 0, 0);
  out.dir = mk3(0, 0, 0);
  int node = root;
  for (;;) {
    switch (b.x) {
      case MAT_MIXED:
        node = g.next() < a.w ? b.y : b.z;
        break;
      case MAT_LAYERED: {
        V3 d;
        if (dielectric_dir(din, sf.n, sf.front, a.w, g, d)) {
          out.kind = SCATTER_SPECULAR;
          out.attenuation = mk3(1, 1, 1);
          out.dir = d;
          return out;
        }
        din = d; // inner.scatter(refracted ray, same rec)
        node = b.y;
        break;
      }
      case MAT_LAMBERT:
        out.kind = SCATTER_DIFFUSE;
        out.attenuation = xyz(a);
        return out;
      case MAT_METAL: { // metal.ts:29-50
        V3 refl = reflect3(normalize3(din), sf.n);
        if (a.w > 0.f) refl = fma3(a.w, random_in_unit_sphere(g), refl);
        if (dot3(refl, sf.n) <= 0.f) return out; // absorbed
        out.kind = SCATTER_SPECULAR;
        out.attenuation = xyz(a);
        out.dir = refl;
        return out;
      }
      case MAT_GLASS: {
        V3 d;
        dielectric_dir(din, sf.n, sf.front, a.w, g, d);
        out.kind = SCATTER_SPECULAR;
        out.attenuation = mk3(1, 1, 1);
        out.dir = d;
        return out;
      }
      default: // MAT_LIGHT: DefaultMaterial.scatter -> null (material.ts:50-52)
        return out;
    }
    b = ldgi4(S.matB + node);
    a = ldg4(S.matA + node);
  }
}

// ---------------------------------------------------------------------------------------
// Camera rays — camera.ts:176-210 with the reference's FP32 rounding sequence
// (scale then add, each rounded: __fmul_rn/__fadd_rn block FMA contraction), so the ray is
// bit-identical to the oracle's for the same random numbers.
// ---------------------------------------------------------------------------------------
RT_DEV V3 mul_rn(V3 a, float s) { return V3{__fmul_rn(a.x, s), __fmul_rn(a.y, s), __fmul_rn(a.z, s)}; }
RT_DEV V3 add_rn(V3 a, V3 b) { return V3{__fadd_rn(a.x, b.x), __fadd_rn(a.y, b.y), __fadd_rn(a.z, b.z)}; }
RT_DEV V3 sub_rn(V3 a, V3 b) { return V3{__fsub_rn(a.x, b.x), __fsub_rn(a.y, b.y), __fsub_rn(a.z, b.z)}; }

template <class G>
RT_DEV Ray camera_ray(const DevCamera& c, int i, int j, G& g, bool jitter_and_defocus) {
  V3 p00 = ld3(c.p00), du = ld3(c.du), dv = ld3(c.dv), center = ld3(c.center);
  V3 pc = add_rn(add_rn(p00, mul_rn(du, (float)i)), mul_rn(dv, (float)j));
  V3 ps = pc;
  if (jitter_and_defocus && c.jitter) {
    float px = -0.5f + g.next();
    float py = -0.5f + g.next();
    ps = add_rn(add_rn(pc, mul_rn(du, px)), mul_rn(dv, py));
  }
  Ray r;
  r.o = center;
  r.d = sub_rn(ps, center);
  if (jitter_and_defocus && c.defocus) {
    float x, y;
    do { // vec3.ts:357-364
      x = fmaf(2.f, g.next(), -1.f);
      y = fmaf(2.f, g.next(), -1.f);
    } while (!(fmaf(x, x, y * y) < 1.f));
    V3 off = add_rn(mul_rn(ld3(c.ddu), x), mul_rn(ld3(c.ddv), y));
    r.o = add_rn(center, off);
    r.d = sub_rn(ps, r.o);
  }
  return r;
}

} // namespace rt
