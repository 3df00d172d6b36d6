// rt_denoise.cuh — opt-in denoiser: first-hit feature buffers and the spatial filter of SVGF (Schied et al., HPG 2017,
// without its temporal part).  Included at the end of rt_megakernel.cu: the feature kernel regenerates a render's camera
// rays with the same device functions the render kernels inline.  The filter is specified by tests/denoise_reference.py
// (float64 numpy); DESIGN.md section 4.2d gives the algorithm and what it does not do.
#pragma once

namespace rt {

// =========================================================================================
// features: camera rays of samples 0..n_samples-1 of every pixel, exactly as the render kernels draw them (random
// streams are keyed by (pixel, sample), and the camera ray takes the first draws of bounce 0), traced to their first hit
// =========================================================================================
template <int KIND>
__global__ void __launch_bounds__(256) k_render_features(const DevScene S, const RenderParams R, int n_samples, float* albedo,
                                                         float* normal, float* depth) {
  __shared__ ListSmemData sm_data;
  const ListSmem sm = stage_list<KIND>(S, sm_data);
  const ListSmem& L = sm;
  const int tx = (R.x0 / kTile) + blockIdx.x, ty = (R.y0 / kTile) + blockIdx.y;
  int lx, ly;
  tile_pixel(threadIdx.x, lx, ly);
  const int i = tx * kTile + lx, j = ty * kTile + ly;
  if (!(i >= R.x0 && i < R.x1 && j >= R.y0 && j < R.y1)) return;
  const uint32_t pixel = (uint32_t)j * (uint32_t)S.cam.width + (uint32_t)i;
  V3 a = mk3(0, 0, 0), n = mk3(0, 0, 0);
  float z = 0.f;
  int hits = 0;
  for (int s = 0; s < n_samples; ++s) {
    Rng g;
    g.begin(pixel, (uint32_t)s, 0u, S.seed_lo, S.seed_hi);
    const Ray ray = camera_ray(S.cam, i, j, g, true); // jitter only when samples > 1, defocus when the aperture is open
    float t;
    int slot;
    if (closest_hit<KIND>(S, L, ray, t, slot)) {
      const I2 info = ldgi2(S.slot_info + slot);
      const Surf sf = surface_at((info.y >> 30) & 3, ldg4(S.p0 + slot), ray, t);
      a = a + xyz(ldg4(S.matF + info.x));
      n = n + sf.n;
      z += t * sqrtf(dot3(ray.d, ray.d)); // camera directions are not unit vectors (camera.ts:176-210)
      ++hits;
    } else {
      a = a + mk3(1, 1, 1);
    }
  }
  const size_t pi = (size_t)j * S.cam.width + i;
  a = a * (1.0f / (float)n_samples);
  if (hits > 1) { // the mean of one normal is that normal, bit for bit
    const float l2 = dot3(n, n);
    if (l2 > 0.f) n = n * (1.0f / sqrtf(l2));
  }
  if (albedo) { albedo[pi * 3] = a.x; albedo[pi * 3 + 1] = a.y; albedo[pi * 3 + 2] = a.z; }
  if (normal) { normal[pi * 3] = n.x; normal[pi * 3 + 1] = n.y; normal[pi * 3 + 2] = n.z; }
  if (depth) depth[pi] = hits ? z / (float)hits : -1.f;
}

// =========================================================================================
// filter: prepare (demodulate, variance, depth gradient) -> K a-trous passes -> finish (remodulate, RGB8)
// =========================================================================================
constexpr float kDnAlbedoMin = 1e-3f; // demodulation floor
RT_DEV float dn_lum(float r, float g, float b) { return 0.299f * r + 0.587f * g + 0.114f * b; } // the project's illuminance weights
RT_DEV bool dn_finite3(const float* p) { return isfinite(p[0]) && isfinite(p[1]) && isfinite(p[2]); }
// the filter kernels run 16x16 blocks over the launch's window of rows and each thread strides over rows by the grid's
// height: CUDA caps gridDim.y at 65535, so on a window taller than 65535 * 16 rows a thread filters more than one pixel of
// its column
constexpr int kDnBlock = 16;
constexpr unsigned kDnMaxGridY = 65535;
RT_DEV int dn_x(const DenoiseParams& D) { return D.x0 + (int)(blockIdx.x * blockDim.x + threadIdx.x); }
RT_DEV int dn_y0(const DenoiseParams& D) { return D.wy0 + (int)(blockIdx.y * blockDim.y + threadIdx.y); }
RT_DEV int dn_ystride() { return (int)(gridDim.y * blockDim.y); }
RT_DEV bool dn_inside(const DenoiseParams& D, int x, int y) { return x >= D.x0 && x < D.x1 && y >= D.y0 && y < D.y1; }

// depth usable for a gradient: inside the region and a hit
RT_DEV bool dn_depth_at(const DenoiseParams& D, int x, int y, float& z) {
  if (!dn_inside(D, x, y)) return false;
  z = D.depth[(size_t)y * D.width + x];
  return isfinite(z) && z >= 0.f;
}
// central difference, one-sided at region borders and next to misses, 0 with neither neighbour
RT_DEV float dn_gradient(const DenoiseParams& D, int x, int y, int ax, int ay, float zc) {
  float zl, zh;
  const bool l = dn_depth_at(D, x - ax, y - ay, zl), h = dn_depth_at(D, x + ax, y + ay, zh);
  if (l && h) return 0.5f * (zh - zl);
  if (h) return zh - zc;
  if (l) return zc - zl;
  return 0.f;
}

RT_DEV void dn_prepare_pixel(const DenoiseParams& D, int x, int y) {
  const size_t p = (size_t)y * D.width + x;
  const float* c = D.color + p * 3;
  const float* a = D.albedo + p * 3;
  const float* n = D.normal + p * 3;
  const float* m = D.moments + p * 8;
  const float z = D.depth[p];
  const float ar = fmaxf(a[0], kDnAlbedoMin), ag = fmaxf(a[1], kDnAlbedoMin), ab = fmaxf(a[2], kDnAlbedoMin);
  const float ir = c[0] / ar, ig = c[1] / ag, ib = c[2] / ab;
  // variance of the luminance of the pixel mean: (sum_c w_c sd_c)^2 / n (exact for perfectly correlated channels),
  // demodulated by the albedo's luminance; unknown (+inf: luminance weights 1) below two samples
  float var = CUDART_INF_F;
  const float ns = m[6];
  if (ns >= 2.f) {
    const float k = 1.0f / (ns - 1.f);
    const float sd = 0.299f * sqrtf((m[3] > 0.f ? m[3] : 0.f) * k) + 0.587f * sqrtf((m[4] > 0.f ? m[4] : 0.f) * k) +
                     0.114f * sqrtf((m[5] > 0.f ? m[5] : 0.f) * k);
    const float la = fmaxf(dn_lum(a[0], a[1], a[2]), kDnAlbedoMin);
    var = sd * sd / ns / (la * la);
  }
  const bool valid = dn_finite3(c) && dn_finite3(a) && dn_finite3(n) && isfinite(z) && isfinite(ir) && isfinite(ig) && isfinite(ib);
  D.buf[0][p] = valid ? F4{ir, ig, ib, var} : F4{CUDART_NAN_F, CUDART_NAN_F, CUDART_NAN_F, CUDART_NAN_F};
  D.feat[p] = F4{n[0], n[1], n[2], z};
  const bool hit = valid && z >= 0.f;
  D.grad[p * 2] = hit ? dn_gradient(D, x, y, 1, 0, z) : 0.f;
  D.grad[p * 2 + 1] = hit ? dn_gradient(D, x, y, 0, 1, z) : 0.f;
}
__global__ void __launch_bounds__(256) k_denoise_prepare(const DenoiseParams D) {
  const int x = dn_x(D);
  if (x >= D.x1) return;
  for (int y = dn_y0(D); y < D.wy1; y += dn_ystride()) dn_prepare_pixel(D, x, y);
}

// one a-trous pass with step 2^k: 5x5 B3-spline taps weighted by normal, depth and luminance edge stops
RT_DEV void dn_pass_pixel(const DenoiseParams& D, const F4* __restrict__ in, F4* __restrict__ out, int step, int x, int y) {
  const size_t p = (size_t)y * D.width + x;
  const F4 c = in[p];
  if (isnan(c.x)) { out[p] = c; return; }
  // 3x3 (1/4, 1/2, 1/4) blur of the variance over the pixels the filter reads
  const float k3[3] = {0.25f, 0.5f, 0.25f};
  float gv = 0.f, gw = 0.f;
#pragma unroll
  for (int dy = -1; dy <= 1; ++dy)
#pragma unroll
    for (int dx = -1; dx <= 1; ++dx) {
      if (!dn_inside(D, x + dx, y + dy)) continue;
      const F4 q = in[(size_t)(y + dy) * D.width + (x + dx)];
      if (isnan(q.x)) continue;
      const float w = k3[dx + 1] * k3[dy + 1];
      gv += w * q.w;
      gw += w;
    }
  gv /= gw;
  const F4 f = D.feat[p];
  const float gx = D.grad[p * 2], gy = D.grad[p * 2 + 1];
  const bool miss_p = f.w < 0.f;
  const float lp = dn_lum(c.x, c.y, c.z);
  const float z_eps = 1e-3f * f.w + 1e-10f;
  const float h[5] = {1.f / 16, 4.f / 16, 6.f / 16, 4.f / 16, 1.f / 16};
  float sw = 0.f, sr = 0.f, sg = 0.f, sb = 0.f, sv = 0.f;
#pragma unroll
  for (int dy = -2; dy <= 2; ++dy)
#pragma unroll
    for (int dx = -2; dx <= 2; ++dx) {
      const int qx = x + dx * step, qy = y + dy * step;
      if (!dn_inside(D, qx, qy)) continue;
      const size_t q = (size_t)qy * D.width + qx;
      const F4 cq = in[q];
      if (isnan(cq.x)) continue;
      const F4 fq = D.feat[q];
      if (miss_p != (fq.w < 0.f)) continue; // a hit and a miss: w_n = 0
      float w = h[dx + 2] * h[dy + 2];
      if (!miss_p) {
        const float nd = fmaf(f.x, fq.x, fmaf(f.y, fq.y, f.z * fq.z));
        w *= powf(fmaxf(nd, 0.f), D.sigma_n);
        const float dz = D.sigma_z * fabsf(gx * (float)(dx * step) + gy * (float)(dy * step));
        w *= expf(-fabsf(f.w - fq.w) / (dz + z_eps));
      }
      // luminance stop scaled by the larger of the two variances: Monte-Carlo pixels that are bright are also the noisy
      // ones, so a stop scaled by the centre's variance alone lets bright pixels take in dark neighbours but not the
      // reverse, and the image loses energy.  +inf (unknown variance): the weight is 1.
      w *= expf(-fabsf(lp - dn_lum(cq.x, cq.y, cq.z)) / (D.sigma_l * sqrtf(fmaxf(gv, cq.w)) + 1e-10f));
      if (!(w > 0.f)) continue;
      sw += w;
      sr += w * cq.x; sg += w * cq.y; sb += w * cq.z;
      sv += w * w * cq.w;
    }
  out[p] = F4{sr / sw, sg / sw, sb / sw, sv / (sw * sw)};
}
__global__ void __launch_bounds__(256) k_denoise_pass(const DenoiseParams D, const F4* __restrict__ in, F4* __restrict__ out, int step) {
  const int x = dn_x(D);
  if (x >= D.x1) return;
  for (int y = dn_y0(D); y < D.wy1; y += dn_ystride()) dn_pass_pixel(D, in, out, step, x, y);
}

RT_DEV void dn_finish_pixel(const DenoiseParams& D, const F4* __restrict__ in, int x, int y) {
  const size_t p = (size_t)y * D.width + x;
  const F4 c = in[p];
  float o[3];
  if (isnan(c.x)) { // passed through unchanged (a NaN of the pixel stream stays black in RGB8)
    o[0] = D.color[p * 3]; o[1] = D.color[p * 3 + 1]; o[2] = D.color[p * 3 + 2];
  } else {
    const float* a = D.albedo + p * 3;
    o[0] = c.x * fmaxf(a[0], kDnAlbedoMin); o[1] = c.y * fmaxf(a[1], kDnAlbedoMin); o[2] = c.z * fmaxf(a[2], kDnAlbedoMin);
  }
  D.out[p * 3] = o[0]; D.out[p * 3 + 1] = o[1]; D.out[p * 3 + 2] = o[2];
  if (D.rgb8) { D.rgb8[p * 3] = gamma_rgb8(o[0]); D.rgb8[p * 3 + 1] = gamma_rgb8(o[1]); D.rgb8[p * 3 + 2] = gamma_rgb8(o[2]); }
}
__global__ void __launch_bounds__(256) k_denoise_finish(const DenoiseParams D, const F4* __restrict__ in) {
  const int x = dn_x(D);
  if (x >= D.x1) return;
  for (int y = dn_y0(D); y < D.wy1; y += dn_ystride()) dn_finish_pixel(D, in, x, y);
}

// launchers (called from rt_api.cu)
cudaError_t launch_render_features(const DevScene& S, const RenderParams& R, int n_samples, float* albedo, float* normal, float* depth,
                                   cudaStream_t st) {
  if (R.x1 <= R.x0 || R.y1 <= R.y0) return cudaSuccess;
  int gx, gy;
  render_tile_grid(R, &gx, &gy);
  dim3 grid((unsigned)gx, (unsigned)gy, 1), block(256);
  switch (S.bvh_kind) {
    case BVH_LIST: k_render_features<BVH_LIST><<<grid, block, 0, st>>>(S, R, n_samples, albedo, normal, depth); break;
    case BVH_SAH: k_render_features<BVH_SAH><<<grid, block, 0, st>>>(S, R, n_samples, albedo, normal, depth); break;
    default: k_render_features<BVH_REFERENCE><<<grid, block, 0, st>>>(S, R, n_samples, albedo, normal, depth); break;
  }
  return cudaGetLastError();
}

// prepare + `iterations` passes + finish of the rows [b0, b1) of the region: each stage computes the rows the next one
// reads (dn_halo, rt_types.h); b0 = y0, b1 = y1 filters the whole region.  *launches = kernels enqueued
cudaError_t launch_denoise(const DenoiseParams& D0, int b0, int b1, cudaStream_t st, int* launches) {
  *launches = 0;
  if (D0.x1 <= D0.x0 || b1 <= b0) return cudaSuccess;
  DenoiseParams D = D0;
  const dim3 block(kDnBlock, kDnBlock, 1);
  const unsigned cols = (unsigned)((D.x1 - D.x0 + kDnBlock - 1) / kDnBlock);
  auto window = [&](int h) { // rows [b0 - h, b1 + h) clipped to the region -> D.wy0 / D.wy1 and the launch grid
    D.wy0 = std::max(D.y0, b0 - h);
    D.wy1 = std::min(D.y1, b1 + h);
    const unsigned rows = (unsigned)((D.wy1 - D.wy0 + kDnBlock - 1) / kDnBlock);
    return dim3(cols, rows < kDnMaxGridY ? rows : kDnMaxGridY, 1);
  };
  dim3 grid = window(dn_halo(D.iterations, -1));
  k_denoise_prepare<<<grid, block, 0, st>>>(D);
  int cur = 0;
  for (int k = 0; k < D.iterations; ++k, cur ^= 1) {
    grid = window(dn_halo(D.iterations, k));
    k_denoise_pass<<<grid, block, 0, st>>>(D, D.buf[cur], D.buf[cur ^ 1], 1 << k);
  }
  grid = window(0);
  k_denoise_finish<<<grid, block, 0, st>>>(D, D.buf[cur]);
  *launches = D.iterations + 2;
  return cudaGetLastError();
}

} // namespace rt
