// composite.cu — raw2outputs alpha compositing, forward and hand-written backward.
//   replaces DS_NeRF/run_nerf_helpers.py:350-404; backward formula: SURVEY.md §8a'-3.
//
// One warp per ray.  Lane l owns C consecutive samples [l*C, l*C+C): raw is read as float4 per
// sample (16 B, coalesced across the warp), the exclusive cumprod of (1-alpha+1e-10) is a local
// product plus a 5-step multiplicative warp scan, and the five ray sums are warp-shuffle reductions.
// HBM-bound: algorithmic bytes per ray = S*(16 raw + 4 z [+4 noise]) + 12 rays_d read,
// S*4 weights [+S*4 alpha] + 24 written.
#include "common.cuh"

namespace {

constexpr int kWarps = 8;

template <int C>
struct Fwd {
  float a[C], q[C], T[C], w[C], zz[C], e[C], delta[C], sig[C];
  float cr[C], cg[C], cb[C];
  float D, A, R, G, Bc;  // ray sums: depth, acc, rgb
};

// loads one ray's samples and evaluates alpha / transmittance / weights / ray sums
template <int C>
__device__ __forceinline__ void eval_ray(Fwd<C>& f, const float4* __restrict__ raw, const float* __restrict__ z,
                                         const float* __restrict__ noise, float norm, int S, int lane) {
  const int base = lane * C;
  float4 rw[C];
#pragma unroll
  for (int k = 0; k < C; ++k) {
    int i = base + k;
    bool v = i < S;
    rw[k] = v ? __ldg(raw + i) : make_float4(0.f, 0.f, 0.f, 0.f);
    f.zz[k] = v ? __ldg(z + i) : 0.f;
    float nz = (v && noise) ? __ldg(noise + i) : 0.f;
    f.sig[k] = rw[k].w + nz;
  }
  float z_next_lane = __shfl_down_sync(FULL_MASK, f.zz[0], 1);
  float prod = 1.f;
#pragma unroll
  for (int k = 0; k < C; ++k) {
    int i = base + k;
    float zn = (k + 1 < C) ? f.zz[(k + 1 < C) ? k + 1 : k] : z_next_lane;
    float dist = (i + 1 < S) ? (zn - f.zz[k]) : 1e10f;
    f.delta[k] = dist * norm;
    float x = fmaxf(f.sig[k], 0.f) * f.delta[k];
    f.e[k] = expf(-x);
    f.a[k] = (i < S) ? (1.f - f.e[k]) : 0.f;
    f.q[k] = (i < S) ? ((1.f - f.a[k]) + 1e-10f) : 1.f;
    f.T[k] = prod;  // local exclusive product
    prod *= f.q[k];
    f.cr[k] = 1.f / (1.f + expf(-rw[k].x));
    f.cg[k] = 1.f / (1.f + expf(-rw[k].y));
    f.cb[k] = 1.f / (1.f + expf(-rw[k].z));
  }
  // exclusive multiplicative scan of the lane products
  float incl = prod;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    float v = __shfl_up_sync(FULL_MASK, incl, o);
    if (lane >= o) incl *= v;
  }
  float excl = __shfl_up_sync(FULL_MASK, incl, 1);
  if (lane == 0) excl = 1.f;
  float sD = 0.f, sA = 0.f, sR = 0.f, sG = 0.f, sB = 0.f;
#pragma unroll
  for (int k = 0; k < C; ++k) {
    f.T[k] *= excl;
    f.w[k] = f.a[k] * f.T[k];
    sD += f.w[k] * f.zz[k];
    sA += f.w[k];
    sR += f.w[k] * f.cr[k];
    sG += f.w[k] * f.cg[k];
    sB += f.w[k] * f.cb[k];
  }
  f.D = warp_sum(sD);
  f.A = warp_sum(sA);
  f.R = warp_sum(sR);
  f.G = warp_sum(sG);
  f.Bc = warp_sum(sB);
}

// lane-owned run of C floats -> global row (vectorised when the row layout keeps 16/8-byte alignment)
template <int C>
__device__ __forceinline__ void store_row(float* __restrict__ row, const float (&v)[C], int base, int S) {
  if constexpr (C % 4 == 0) {
    if ((S & 3) == 0 && base + C <= S) {
#pragma unroll
      for (int k = 0; k < C; k += 4) *reinterpret_cast<float4*>(row + base + k) = make_float4(v[k], v[k + 1], v[k + 2], v[k + 3]);
      return;
    }
  } else if constexpr (C == 2) {
    if ((S & 1) == 0 && base + 2 <= S) {
      *reinterpret_cast<float2*>(row + base) = make_float2(v[0], v[1]);
      return;
    }
  }
#pragma unroll
  for (int k = 0; k < C; ++k)
    if (base + k < S) row[base + k] = v[k];
}

__device__ __forceinline__ float ray_norm(const float* __restrict__ d) {
  float x = __ldg(d), y = __ldg(d + 1), z = __ldg(d + 2);
  return sqrtf(x * x + y * y + z * z);
}

template <int C>
__global__ void __launch_bounds__(kWarps * 32)
composite_fwd_kernel(const float4* __restrict__ raw, const float* __restrict__ z, const float* __restrict__ rays_d,
                     int d_stride, const float* __restrict__ noise, int64_t n_rays, int S, int white,
                     float* __restrict__ rgb, float* __restrict__ disp, float* __restrict__ acc,
                     float* __restrict__ weights, float* __restrict__ depth, float* __restrict__ alpha) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int64_t ray = (int64_t)blockIdx.x * kWarps + warp; ray < n_rays; ray += (int64_t)gridDim.x * kWarps) {
    Fwd<C> f;
    float norm = ray_norm(rays_d + ray * d_stride);
    eval_ray<C>(f, raw + ray * S, z + ray * S, noise ? noise + ray * S : nullptr, norm, S, lane);
    const int base = lane * C;
    store_row<C>(weights + ray * S, f.w, base, S);
    if (alpha) store_row<C>(alpha + ray * S, f.a, base, S);
    if (lane == 0) {
      float r = f.D / f.A;
      float m = (r != r) ? r : fmaxf(1e-10f, r);  // torch.max propagates NaN (0/0 when every sigma <= 0)
      float bg = white ? (1.f - f.A) : 0.f;
      rgb[ray * 3 + 0] = f.R + bg;
      rgb[ray * 3 + 1] = f.G + bg;
      rgb[ray * 3 + 2] = f.Bc + bg;
      disp[ray] = 1.f / m;
      acc[ray] = f.A;
      depth[ray] = f.D;
    }
  }
}

// kNorm: also d |rays_d| = sum_s dalpha_s relu(sigma_s) dist_s exp(-relu(sigma_s) dist_s |d|), chained to d rays_d [n,3] (d_dir);
// the last dist is 1e10 as in the reference.  The sum is formed with delta_s = dist_s |d| (already in registers) and divided by
// |d| once: d rays_d = (sum_s dalpha_s relu(sigma_s) delta_s e_s) d / |d|^2 (0 when |d| = 0).  relu(sigma) multiplies rather
// than selects, so a NaN dalpha (a ray whose every sigma <= 0: disp = 1/max(1e-10, 0/0)) gives NaN, as the reference's autograd
// does through dists.  d_raw does not depend on the flag.
template <int C, bool kNorm>
__global__ void __launch_bounds__(kWarps * 32)
composite_bwd_kernel(const float4* __restrict__ raw, const float* __restrict__ z, const float* __restrict__ rays_d,
                     int d_stride, const float* __restrict__ noise, int64_t n_rays, int S, int white, int detach_w,
                     const float* __restrict__ g_rgb, const float* __restrict__ g_disp, const float* __restrict__ g_acc,
                     const float* __restrict__ g_depth, const float* __restrict__ g_weights,
                     const float* __restrict__ g_alpha, float4* __restrict__ d_raw, float* __restrict__ d_dir) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int64_t ray = (int64_t)blockIdx.x * kWarps + warp; ray < n_rays; ray += (int64_t)gridDim.x * kWarps) {
    Fwd<C> f;
    float norm = ray_norm(rays_d + ray * d_stride);
    eval_ray<C>(f, raw + ray * S, z + ray * S, noise ? noise + ray * S : nullptr, norm, S, lane);
    float gR = 0.f, gG = 0.f, gB = 0.f;
    if (g_rgb) { gR = __ldg(g_rgb + ray * 3); gG = __ldg(g_rgb + ray * 3 + 1); gB = __ldg(g_rgb + ray * 3 + 2); }
    float gdisp = g_disp ? __ldg(g_disp + ray) : 0.f;
    float gD = g_depth ? __ldg(g_depth + ray) : 0.f;
    float gA = g_acc ? __ldg(g_acc + ray) : 0.f;
    float r = f.D / f.A;
    bool live = !(r <= 1e-10f);  // NaN keeps the path, as torch.max's backward does
    if (live && g_disp) {
      gD += -gdisp * f.A / (f.D * f.D);
      gA += gdisp / f.D;
    }
    if (white) gA -= (gR + gG + gB);
    const int base = lane * C;
    float G[C], Gw[C];
    float local = 0.f;
#pragma unroll
    for (int k = C - 1; k >= 0; --k) {
      int i = base + k;
      float g = f.zz[k] * gD + gA;
      if (!detach_w) g += gR * f.cr[k] + gG * f.cg[k] + gB * f.cb[k];
      if (g_weights && i < S) g += __ldg(g_weights + ray * S + i);
      G[k] = g;
      float gw = (i < S) ? g * f.w[k] : 0.f;
      Gw[k] = local;  // local exclusive suffix
      local += gw;
    }
    // exclusive suffix scan over lanes (sum of totals of higher lanes)
    float incl = local;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      float v = __shfl_down_sync(FULL_MASK, incl, o);
      if (lane + o < 32) incl += v;
    }
    float excl = __shfl_down_sync(FULL_MASK, incl, 1);
    if (lane == 31) excl = 0.f;
    float dnorm = 0.f;
#pragma unroll
    for (int k = 0; k < C; ++k) {
      int i = base + k;
      if (i < S) {
        float suffix = Gw[k] + excl;
        float dalpha = G[k] * f.T[k] - suffix / f.q[k];
        if (g_alpha) dalpha += __ldg(g_alpha + ray * S + i);
        float dsig = (f.sig[k] > 0.f) ? dalpha * f.delta[k] * f.e[k] : 0.f;
        if constexpr (kNorm) dnorm += (f.sig[k] > 0.f) ? dsig * f.sig[k] : dalpha * 0.f;   // 0 * NaN = NaN, as autograd
        float wk = f.w[k];
        float4 o;
        o.x = wk * gR * f.cr[k] * (1.f - f.cr[k]);
        o.y = wk * gG * f.cg[k] * (1.f - f.cg[k]);
        o.z = wk * gB * f.cb[k] * (1.f - f.cb[k]);
        o.w = dsig;
        d_raw[ray * S + i] = o;
      }
    }
    if constexpr (kNorm) {
      dnorm = warp_sum(dnorm);
      if (lane == 0) {
        const float* d = rays_d + ray * d_stride;
        const float inv2 = norm > 0.f ? 1.f / (norm * norm) : 0.f;
        for (int c = 0; c < 3; ++c) d_dir[ray * 3 + c] = dnorm * (__ldg(d + c) * inv2);
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Fast path for the shapes render_rays produces (S = 64 coarse, S = 128 fine): G lanes per ray, 4 consecutive
// samples per lane (S == 4 G), so a warp carries 32 / G rays and nothing is predicated on the sample index.
// Everything a lane needs arrives as 128-bit loads (4 x raw, 1 x z, 1 x noise); weights / alpha / d_raw leave
// as 128-bit stores.  The generic kernels above spend ~165 instructions per sample (IEEE division and expf
// slow paths, index predicates); this path spends ~45, which is what lets HBM become the limit.
// exp / reciprocal are the 2-ulp MUFU forms: the 1e-5 relative tolerance of the path is two orders above them.
// ---------------------------------------------------------------------------------------------
// single-MUFU forms (the non-ftz intrinsics wrap each MUFU in a denormal-range test and two scalings)
__device__ __forceinline__ float ex2_ftz(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rcp_ftz(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rsqrt_ftz(float x) { float y; asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float fast_exp_neg(float x) { return ex2_ftz(x * -1.4426950408889634f); }   // exp(-x)
__device__ __forceinline__ float fast_sigmoid(float x) { return rcp_ftz(1.f + fast_exp_neg(x)); }

// every operand of these kernels is touched once: streaming (evict-first) loads and stores (forward +1 - 2.5 % at 262,144 rays)
#define CLD4(p) __ldcs(p)
#define CST4(p, v) __stcs(p, v)
template <int G>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(FULL_MASK, v, o);
  return v;
}

struct Fast4 {
  float a[4], q[4], T[4], w[4], zz[4], e[4], delta[4], sig[4], cr[4], cg[4], cb[4];
  float D, A, R, G, Bc;
};

template <int G>
__device__ __forceinline__ void eval_ray4(Fast4& f, const float4* __restrict__ raw, const float* __restrict__ z,
                                          const float* __restrict__ noise, const float* __restrict__ d, int sub) {
  float4 rw[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) rw[k] = CLD4(raw + k);
  const float4 z4 = CLD4(reinterpret_cast<const float4*>(z));
  float4 n4 = make_float4(0.f, 0.f, 0.f, 0.f);
  if (noise) n4 = CLD4(reinterpret_cast<const float4*>(noise));
  const float dx = __ldg(d), dy = __ldg(d + 1), dz = __ldg(d + 2);
  const float n2 = dx * dx + dy * dy + dz * dz;
  const float norm = n2 > 0.f ? n2 * rsqrt_ftz(n2) : 0.f;
  f.zz[0] = z4.x; f.zz[1] = z4.y; f.zz[2] = z4.z; f.zz[3] = z4.w;
  f.sig[0] = rw[0].w + n4.x; f.sig[1] = rw[1].w + n4.y; f.sig[2] = rw[2].w + n4.z; f.sig[3] = rw[3].w + n4.w;
  const float z_next = __shfl_down_sync(FULL_MASK, z4.x, 1, G);
  float prod = 1.f;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    float dist = (k < 3) ? (f.zz[(k < 3) ? k + 1 : k] - f.zz[k]) : ((sub == G - 1) ? 1e10f : (z_next - f.zz[3]));
    f.delta[k] = dist * norm;
    f.e[k] = fast_exp_neg(fmaxf(f.sig[k], 0.f) * f.delta[k]);
    f.a[k] = 1.f - f.e[k];
    f.q[k] = (1.f - f.a[k]) + 1e-10f;
    f.T[k] = prod;
    prod *= f.q[k];
    f.cr[k] = fast_sigmoid(rw[k].x);
    f.cg[k] = fast_sigmoid(rw[k].y);
    f.cb[k] = fast_sigmoid(rw[k].z);
  }
  float incl = prod;
#pragma unroll
  for (int o = 1; o < G; o <<= 1) {
    float v = __shfl_up_sync(FULL_MASK, incl, o, G);
    incl *= (sub >= o) ? v : 1.f;
  }
  float excl = __shfl_up_sync(FULL_MASK, incl, 1, G);
  if (sub == 0) excl = 1.f;
  float sD = 0.f, sA = 0.f, sR = 0.f, sG = 0.f, sB = 0.f;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    f.T[k] *= excl;
    f.w[k] = f.a[k] * f.T[k];
    sD = fmaf(f.w[k], f.zz[k], sD);
    sA += f.w[k];
    sR = fmaf(f.w[k], f.cr[k], sR);
    sG = fmaf(f.w[k], f.cg[k], sG);
    sB = fmaf(f.w[k], f.cb[k], sB);
  }
  f.D = group_sum<G>(sD);
  f.A = group_sum<G>(sA);
  f.R = group_sum<G>(sR);
  f.G = group_sum<G>(sG);
  f.Bc = group_sum<G>(sB);
}

// Photometric losses fused into the compositing kernels (img2mse of DS_NeRF/run_nerf_helpers.py:15 as train() applies it to
// rgb / rgb0 / disp, run.py:1000-1027): the forward also returns  sq[0] = sum_rays sum_c (rgb_c - target_rgb_c)^2  and
// sq[1] = sum_rays (disp - target_disp)^2  (deterministic: per-block partials summed in block order by the last block), the
// backward takes d loss / d sq[0..1] from DEVICE memory and adds 2 g (x - target) to the upstream gradients in-kernel.
struct MseArgs {
  const float* target_rgb;    // [N,3] or null
  const float* target_disp;   // [N]   or null
  float* partials;            // forward: [grid][2] scratch
  unsigned int* counter;      // forward: zero-initialised ticket counter (reset by the kernel)
  float* sq_out;              // forward: [2]
  const float* g_sq;          // backward: [2] (device)
};

// four resident blocks per SM (61 registers): 83 % / 87 % of the copy peak at S = 64 / 128 (five blocks, 48 registers: 81 % / 82 %;
// three: 83 % / 77 %; six, with spills: 72 % / 75 %)
template <int G>
__global__ void __launch_bounds__(kWarps * 32, 4)
composite_fwd4_kernel(const float4* __restrict__ raw, const float* __restrict__ z, const float* __restrict__ rays_d,
                      int d_stride, const float* __restrict__ noise, int64_t n_rays, int white,
                      float* __restrict__ rgb, float* __restrict__ disp, float* __restrict__ acc,
                      float* __restrict__ weights, float* __restrict__ depth, float* __restrict__ alpha, const MseArgs mse) {
  float sq_rgb = 0.f, sq_disp = 0.f;
  constexpr int S = 4 * G, RPW = 32 / G;   // samples per ray, rays per warp
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, sub = lane % G;
  const int64_t stride = (int64_t)gridDim.x * kWarps * RPW;
  for (int64_t ray0 = ((int64_t)blockIdx.x * kWarps + warp) * RPW; ray0 < n_rays; ray0 += stride) {
    int64_t ray = ray0 + lane / G;
    const bool live = ray < n_rays;
    if (!live) ray = n_rays - 1;           // keep the shuffles convergent; the duplicate is not stored
    const int64_t off = ray * S + sub * 4;
    Fast4 f;
    eval_ray4<G>(f, raw + off, z + off, noise ? noise + off : nullptr, rays_d + ray * d_stride, sub);
    if (live) {
      CST4(reinterpret_cast<float4*>(weights + off), make_float4(f.w[0], f.w[1], f.w[2], f.w[3]));
      if (alpha) CST4(reinterpret_cast<float4*>(alpha + off), make_float4(f.a[0], f.a[1], f.a[2], f.a[3]));
      if (sub == 0) {
        float r = f.D / f.A;
        float m = (r != r) ? r : fmaxf(1e-10f, r);  // torch.max propagates NaN (0/0 when every sigma <= 0)
        float bg = white ? (1.f - f.A) : 0.f;
        rgb[ray * 3 + 0] = f.R + bg;
        rgb[ray * 3 + 1] = f.G + bg;
        rgb[ray * 3 + 2] = f.Bc + bg;
        disp[ray] = 1.f / m;
        acc[ray] = f.A;
        depth[ray] = f.D;
        if (mse.target_rgb) {
          const float e0 = (f.R + bg) - __ldg(mse.target_rgb + ray * 3), e1 = (f.G + bg) - __ldg(mse.target_rgb + ray * 3 + 1),
                      e2 = (f.Bc + bg) - __ldg(mse.target_rgb + ray * 3 + 2);
          sq_rgb += e0 * e0 + e1 * e1 + e2 * e2;
        }
        if (mse.target_disp) { const float e = 1.f / m - __ldg(mse.target_disp + ray); sq_disp += e * e; }
      }
    }
  }
  if (mse.sq_out) {   // warp -> block -> grid, every level in a fixed order
    __shared__ float part_s[kWarps][2];
    __shared__ bool last_s;
    sq_rgb = warp_sum(sq_rgb);
    sq_disp = warp_sum(sq_disp);
    if (lane == 0) { part_s[warp][0] = sq_rgb; part_s[warp][1] = sq_disp; }
    __syncthreads();
    if (threadIdx.x == 0) {
      float a = 0.f, b = 0.f;
      for (int w = 0; w < kWarps; ++w) { a += part_s[w][0]; b += part_s[w][1]; }
      mse.partials[2 * blockIdx.x] = a;
      mse.partials[2 * blockIdx.x + 1] = b;
      __threadfence();
      last_s = atomicAdd(mse.counter, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (last_s && warp == 0) {
      __threadfence();
      float a = 0.f, b = 0.f;
      for (int i = lane; i < (int)gridDim.x; i += 32) { a += __ldcg(mse.partials + 2 * i); b += __ldcg(mse.partials + 2 * i + 1); }
      a = warp_sum(a);
      b = warp_sum(b);
      if (lane == 0) { mse.sq_out[0] = a; mse.sq_out[1] = b; *mse.counter = 0u; }
    }
  }
}

// resident blocks per SM: S = 64 is fastest at 4 (64 registers, ~100 B of spills: 78.9 % of the copy peak; 2 blocks / 124
// registers: 71.5 %), S = 128 at 2 (no spills: 73.4 % against 69.1 % at 4; 3 blocks are worse for both)
// (the kNorm variant keeps two blocks per SM at S = 64 as well: with 64 registers it would spill the d |rays_d| sum)
template <int G, bool kNorm>
__global__ void __launch_bounds__(kWarps * 32, (G == 32 || kNorm) ? 2 : 4)
composite_bwd4_kernel(const float4* __restrict__ raw, const float* __restrict__ z, const float* __restrict__ rays_d,
                      int d_stride, const float* __restrict__ noise, int64_t n_rays, int white, int detach_w,
                      const float* __restrict__ g_rgb, const float* __restrict__ g_disp, const float* __restrict__ g_acc,
                      const float* __restrict__ g_depth, const float* __restrict__ g_weights,
                      const float* __restrict__ g_alpha, float4* __restrict__ d_raw, const MseArgs mse,
                      float* __restrict__ d_dir) {
  constexpr int S = 4 * G, RPW = 32 / G;
  const float gs_rgb = (mse.g_sq && mse.target_rgb) ? 2.f * __ldg(mse.g_sq) : 0.f;
  const float gs_disp = (mse.g_sq && mse.target_disp) ? 2.f * __ldg(mse.g_sq + 1) : 0.f;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, sub = lane % G;
  const int64_t stride = (int64_t)gridDim.x * kWarps * RPW;
  for (int64_t ray0 = ((int64_t)blockIdx.x * kWarps + warp) * RPW; ray0 < n_rays; ray0 += stride) {
    int64_t ray = ray0 + lane / G;
    const bool live_ray = ray < n_rays;
    if (!live_ray) ray = n_rays - 1;
    const int64_t off = ray * S + sub * 4;
    // upstream gradients first: their latency overlaps the forward recomputation
    float gR = 0.f, gG = 0.f, gB = 0.f;
    if (g_rgb) { gR = __ldg(g_rgb + ray * 3); gG = __ldg(g_rgb + ray * 3 + 1); gB = __ldg(g_rgb + ray * 3 + 2); }
    float gdisp = g_disp ? __ldg(g_disp + ray) : 0.f;
    float tR = 0.f, tG = 0.f, tB = 0.f, tdisp = 0.f;
    if (mse.target_rgb) { tR = __ldg(mse.target_rgb + ray * 3); tG = __ldg(mse.target_rgb + ray * 3 + 1); tB = __ldg(mse.target_rgb + ray * 3 + 2); }
    if (mse.target_disp) tdisp = __ldg(mse.target_disp + ray);
    float gD = g_depth ? __ldg(g_depth + ray) : 0.f;
    float gA = g_acc ? __ldg(g_acc + ray) : 0.f;
    float4 gw4 = make_float4(0.f, 0.f, 0.f, 0.f), ga4 = gw4;
    if (g_weights) gw4 = CLD4(reinterpret_cast<const float4*>(g_weights + off));
    if (g_alpha) ga4 = CLD4(reinterpret_cast<const float4*>(g_alpha + off));
    Fast4 f;
    eval_ray4<G>(f, raw + off, z + off, noise ? noise + off : nullptr, rays_d + ray * d_stride, sub);
    const float r = f.D / f.A;
    if (mse.target_rgb) {             // d (sum of squares) / d rgb_map, from the recomputed forward
      const float bg = white ? (1.f - f.A) : 0.f;
      gR = fmaf(gs_rgb, (f.R + bg) - tR, gR);
      gG = fmaf(gs_rgb, (f.G + bg) - tG, gG);
      gB = fmaf(gs_rgb, (f.Bc + bg) - tB, gB);
    }
    if (mse.target_disp) {
      const float m = (r != r) ? r : fmaxf(1e-10f, r);
      gdisp = fmaf(gs_disp, 1.f / m - tdisp, gdisp);
    }
    if (!(r <= 1e-10f) && (g_disp || mse.target_disp)) {   // NaN keeps the path, as torch.max's backward does
      gD += -gdisp * f.A / (f.D * f.D);
      gA += gdisp / f.D;
    }
    if (white) gA -= (gR + gG + gB);
    const float gwv[4] = {gw4.x, gw4.y, gw4.z, gw4.w}, gav[4] = {ga4.x, ga4.y, ga4.z, ga4.w};
    float Gk[4], Gw[4];
    float local = 0.f;
#pragma unroll
    for (int k = 3; k >= 0; --k) {
      float g = fmaf(f.zz[k], gD, gA) + gwv[k];
      if (!detach_w) g += gR * f.cr[k] + gG * f.cg[k] + gB * f.cb[k];
      Gk[k] = g;
      Gw[k] = local;  // local exclusive suffix
      local = fmaf(g, f.w[k], local);
    }
    float incl = local;   // exclusive suffix scan over the group's lanes
#pragma unroll
    for (int o = 1; o < G; o <<= 1) {
      float v = __shfl_down_sync(FULL_MASK, incl, o, G);
      incl += (sub + o < G) ? v : 0.f;
    }
    float excl = __shfl_down_sync(FULL_MASK, incl, 1, G);
    if (sub == G - 1) excl = 0.f;
    // d_raw of this lane's 4 consecutive samples ...
    float4 o[4];
    float dn = 0.f;   // kNorm: sum of dalpha relu(sigma) delta e over this lane's samples
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float dalpha = Gk[k] * f.T[k] - (Gw[k] + excl) * rcp_ftz(f.q[k]) + gav[k];
      o[k].x = f.w[k] * gR * f.cr[k] * (1.f - f.cr[k]);
      o[k].y = f.w[k] * gG * f.cg[k] * (1.f - f.cg[k]);
      o[k].z = f.w[k] * gB * f.cb[k] * (1.f - f.cb[k]);
      o[k].w = (f.sig[k] > 0.f) ? dalpha * f.delta[k] * f.e[k] : 0.f;
      if constexpr (kNorm) dn += dalpha * fmaxf(f.sig[k], 0.f) * f.delta[k] * f.e[k];   // 0 * NaN = NaN, as autograd
    }
    if constexpr (kNorm) {   // d |rays_d| (see composite_bwd_kernel), summed over the ray's group in a fixed order
      dn = group_sum<G>(dn);
      if (live_ray && sub == 0) {
        const float* d = rays_d + ray * d_stride;
        const float dx = __ldg(d), dy = __ldg(d + 1), dz = __ldg(d + 2);
        const float n2 = dx * dx + dy * dy + dz * dz;
        const float inv2 = n2 > 0.f ? 1.f / n2 : 0.f;
        d_dir[ray * 3 + 0] = dn * (dx * inv2);
        d_dir[ray * 3 + 1] = dn * (dy * inv2);
        d_dir[ray * 3 + 2] = dn * (dz * inv2);
      }
    }
    // ... transposed inside each quad of lanes (lane 4m + j ends up with samples 16m + 4k + j, k = 0..3), so that every store
    // instruction writes 64 contiguous bytes per quad = full 32-byte sectors (16 bytes per lane at a 64-byte stride wrote half
    // sectors: twice the L2 write transactions)
    const int j = lane & 3;
#pragma unroll
    for (int d = 1; d <= 2; d <<= 1) {        // exchange with lane ^ d the elements whose index differs from ours in bit d
      const bool up = (j & d) != 0;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if (k & d) continue;                  // pairs (k, k | d)
        const float4 mine = up ? o[k] : o[k | d];
        float4 got;
        got.x = __shfl_xor_sync(FULL_MASK, mine.x, d);
        got.y = __shfl_xor_sync(FULL_MASK, mine.y, d);
        got.z = __shfl_xor_sync(FULL_MASK, mine.z, d);
        got.w = __shfl_xor_sync(FULL_MASK, mine.w, d);
        if (up) o[k] = got; else o[k | d] = got;
      }
    }
    if (live_ray) {
      const int64_t qoff = ray * S + (sub & ~3) * 4 + j;      // first sample of the quad + our column
#pragma unroll
      for (int k = 0; k < 4; ++k) CST4(d_raw + qoff + 4 * k, o[k]);
    }
  }
}

int grid_for_rays4(int64_t n, int rays_per_warp) {
  int64_t blocks = (n + (int64_t)kWarps * rays_per_warp - 1) / ((int64_t)kWarps * rays_per_warp);
  int64_t cap = (int64_t)mvip_num_sms() * 8;
  return (int)(blocks < cap ? blocks : cap);
}

int grid_for_rays(int64_t n) {
  int64_t blocks = (n + kWarps - 1) / kWarps;
  int64_t cap = (int64_t)mvip_num_sms() * 8;
  return (int)(blocks < cap ? blocks : cap);
}

}  // namespace

#define DISPATCH_C(S, ...)                         \
  do {                                             \
    int c__ = ((S) + 31) / 32;                     \
    if (c__ <= 1) { constexpr int C = 1; __VA_ARGS__; }       \
    else if (c__ <= 2) { constexpr int C = 2; __VA_ARGS__; }  \
    else if (c__ <= 4) { constexpr int C = 4; __VA_ARGS__; }  \
    else if (c__ <= 8) { constexpr int C = 8; __VA_ARGS__; }  \
    else { constexpr int C = 16; __VA_ARGS__; }               \
  } while (0)

extern "C" {

static int composite_forward_impl(const float* raw, const float* z_vals, const float* rays_d, int rays_d_stride,
                                  const float* noise, int64_t n_rays, int n_samples, int white_bkgd, float* rgb, float* disp,
                                  float* acc, float* weights, float* depth, float* alpha, const MseArgs& mse, void* stream) {
  MVIP_REQUIRE(n_rays == 0 || (raw && z_vals && rays_d && rgb && disp && acc && weights && depth), MVIP_E_INVALID,
               "mvip_composite_forward: null pointer");
  MVIP_REQUIRE(n_rays >= 0 && n_samples >= 1 && rays_d_stride >= 3, MVIP_E_INVALID, "mvip_composite_forward: bad shape");
  MVIP_REQUIRE(n_samples <= 512, MVIP_E_UNSUPPORTED, "mvip_composite_forward: n_samples %d > 512", n_samples);
  MVIP_REQUIRE(mvip_aligned(raw, 16) && mvip_aligned(weights, 16) && (!alpha || mvip_aligned(alpha, 16)),
               MVIP_E_INVALID, "mvip_composite_forward: raw/weights/alpha must be 16-byte aligned");
  if (n_rays == 0) {
    if (mse.sq_out) MVIP_CUDA_OK(cudaMemsetAsync(mse.sq_out, 0, 2 * sizeof(float), (cudaStream_t)stream));
    return MVIP_OK;
  }
  const bool vec_ok = mvip_aligned(z_vals, 16) && (!noise || mvip_aligned(noise, 16));
  if (vec_ok && (n_samples == 64 || n_samples == 128)) {
    auto* r4 = reinterpret_cast<const float4*>(raw);
    if (n_samples == 128)
      composite_fwd4_kernel<32><<<grid_for_rays4(n_rays, 1), kWarps * 32, 0, (cudaStream_t)stream>>>(
          r4, z_vals, rays_d, rays_d_stride, noise, n_rays, white_bkgd, rgb, disp, acc, weights, depth, alpha, mse);
    else
      composite_fwd4_kernel<16><<<grid_for_rays4(n_rays, 2), kWarps * 32, 0, (cudaStream_t)stream>>>(
          r4, z_vals, rays_d, rays_d_stride, noise, n_rays, white_bkgd, rgb, disp, acc, weights, depth, alpha, mse);
    MVIP_LAUNCH_OK("composite_fwd4_kernel");
    return MVIP_OK;
  }
  MVIP_REQUIRE(!mse.sq_out, MVIP_E_UNSUPPORTED, "mvip_composite_forward_mse: the fused losses need n_samples = 64 or 128 and 16-byte aligned rows");
  DISPATCH_C(n_samples, (composite_fwd_kernel<C><<<grid_for_rays(n_rays), kWarps * 32, 0, (cudaStream_t)stream>>>(
                            reinterpret_cast<const float4*>(raw), z_vals, rays_d, rays_d_stride, noise, n_rays,
                            n_samples, white_bkgd, rgb, disp, acc, weights, depth, alpha)));
  MVIP_LAUNCH_OK("composite_fwd_kernel");
  return MVIP_OK;
}

static int composite_backward_impl(const float* raw, const float* z_vals, const float* rays_d, int rays_d_stride,
                                   const float* noise, int64_t n_rays, int n_samples, int white_bkgd, int detach_weights,
                                   const float* g_rgb, const float* g_disp, const float* g_acc, const float* g_depth,
                                   const float* g_weights, const float* g_alpha, float* d_raw, const MseArgs& mse, float* d_dir,
                                   void* stream) {
  MVIP_REQUIRE(n_rays == 0 || (raw && z_vals && rays_d && d_raw), MVIP_E_INVALID, "mvip_composite_backward: null pointer");
  MVIP_REQUIRE(n_rays >= 0 && n_samples >= 1 && rays_d_stride >= 3, MVIP_E_INVALID, "mvip_composite_backward: bad shape");
  MVIP_REQUIRE(n_samples <= 512, MVIP_E_UNSUPPORTED, "mvip_composite_backward: n_samples %d > 512", n_samples);
  MVIP_REQUIRE(mvip_aligned(raw, 16) && mvip_aligned(d_raw, 16), MVIP_E_INVALID,
               "mvip_composite_backward: raw/d_raw must be 16-byte aligned");
  if (n_rays == 0) return MVIP_OK;
  const bool vec_ok = mvip_aligned(z_vals, 16) && (!noise || mvip_aligned(noise, 16)) &&
                      (!g_weights || mvip_aligned(g_weights, 16)) && (!g_alpha || mvip_aligned(g_alpha, 16));
  if (vec_ok && (n_samples == 64 || n_samples == 128)) {
    auto* r4 = reinterpret_cast<const float4*>(raw);
    auto* o4 = reinterpret_cast<float4*>(d_raw);
#define MVIP_BWD4(G, NORM)                                                                                                    \
  composite_bwd4_kernel<G, NORM><<<grid_for_rays4(n_rays, 32 / G), kWarps * 32, 0, (cudaStream_t)stream>>>(                  \
      r4, z_vals, rays_d, rays_d_stride, noise, n_rays, white_bkgd, detach_weights, g_rgb, g_disp, g_acc, g_depth, g_weights, \
      g_alpha, o4, mse, d_dir)
    if (n_samples == 128) {
      if (d_dir) MVIP_BWD4(32, true); else MVIP_BWD4(32, false);
    } else {
      if (d_dir) MVIP_BWD4(16, true); else MVIP_BWD4(16, false);
    }
#undef MVIP_BWD4
    MVIP_LAUNCH_OK("composite_bwd4_kernel");
    return MVIP_OK;
  }
  MVIP_REQUIRE(!mse.g_sq, MVIP_E_UNSUPPORTED, "mvip_composite_backward_mse: the fused losses need n_samples = 64 or 128 and 16-byte aligned rows");
  if (d_dir)
    DISPATCH_C(n_samples, (composite_bwd_kernel<C, true><<<grid_for_rays(n_rays), kWarps * 32, 0, (cudaStream_t)stream>>>(
                              reinterpret_cast<const float4*>(raw), z_vals, rays_d, rays_d_stride, noise, n_rays,
                              n_samples, white_bkgd, detach_weights, g_rgb, g_disp, g_acc, g_depth, g_weights, g_alpha,
                              reinterpret_cast<float4*>(d_raw), d_dir)));
  else
    DISPATCH_C(n_samples, (composite_bwd_kernel<C, false><<<grid_for_rays(n_rays), kWarps * 32, 0, (cudaStream_t)stream>>>(
                              reinterpret_cast<const float4*>(raw), z_vals, rays_d, rays_d_stride, noise, n_rays,
                              n_samples, white_bkgd, detach_weights, g_rgb, g_disp, g_acc, g_depth, g_weights, g_alpha,
                              reinterpret_cast<float4*>(d_raw), nullptr)));
  MVIP_LAUNCH_OK("composite_bwd_kernel");
  return MVIP_OK;
}

int mvip_composite_forward(const float* raw, const float* z_vals, const float* rays_d, int rays_d_stride,
                           const float* noise, int64_t n_rays, int n_samples, int white_bkgd, float* rgb, float* disp,
                           float* acc, float* weights, float* depth, float* alpha, void* stream) {
  const MseArgs none = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  return composite_forward_impl(raw, z_vals, rays_d, rays_d_stride, noise, n_rays, n_samples, white_bkgd, rgb, disp, acc, weights,
                                depth, alpha, none, stream);
}

int mvip_composite_backward(const float* raw, const float* z_vals, const float* rays_d, int rays_d_stride,
                            const float* noise, int64_t n_rays, int n_samples, int white_bkgd, int detach_weights,
                            const float* g_rgb, const float* g_disp, const float* g_acc, const float* g_depth,
                            const float* g_weights, const float* g_alpha, float* d_raw, void* stream) {
  const MseArgs none = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  return composite_backward_impl(raw, z_vals, rays_d, rays_d_stride, noise, n_rays, n_samples, white_bkgd, detach_weights, g_rgb,
                                 g_disp, g_acc, g_depth, g_weights, g_alpha, d_raw, none, nullptr, stream);
}

size_t mvip_composite_mse_workspace_bytes(void) { return (size_t)(2 * 1184 + 4) * sizeof(float); }

int mvip_composite_forward_mse(const float* raw, const float* z_vals, const float* rays_d, int rays_d_stride,
                               const float* noise, int64_t n_rays, int n_samples, int white_bkgd, const float* target_rgb,
                               const float* target_disp, float* rgb, float* disp, float* acc, float* weights, float* depth,
                               float* alpha, float* sq_out, void* workspace, void* stream) {
  MVIP_REQUIRE(sq_out && workspace && (target_rgb || target_disp), MVIP_E_INVALID, "mvip_composite_forward_mse: null pointer");
  MVIP_REQUIRE(mvip_num_sms() * 8 <= 1184, MVIP_E_UNSUPPORTED, "mvip_composite_forward_mse: more than 148 SMs");
  float* ws = static_cast<float*>(workspace);
  // workspace: [0] ticket counter (must be zero on the first call: the kernel resets it), [4 ...] per-block partials
  const MseArgs mse = {target_rgb, target_disp, ws + 4, reinterpret_cast<unsigned int*>(ws), sq_out, nullptr};
  return composite_forward_impl(raw, z_vals, rays_d, rays_d_stride, noise, n_rays, n_samples, white_bkgd, rgb, disp, acc, weights,
                                depth, alpha, mse, stream);
}

int mvip_composite_backward_mse(const float* raw, const float* z_vals, const float* rays_d, int rays_d_stride,
                                const float* noise, int64_t n_rays, int n_samples, int white_bkgd, int detach_weights,
                                const float* target_rgb, const float* target_disp, const float* g_sq, const float* g_rgb,
                                const float* g_disp, const float* g_acc, const float* g_depth, const float* g_weights,
                                const float* g_alpha, float* d_raw, void* stream) {
  MVIP_REQUIRE(g_sq && (target_rgb || target_disp), MVIP_E_INVALID, "mvip_composite_backward_mse: null pointer");
  const MseArgs mse = {target_rgb, target_disp, nullptr, nullptr, nullptr, g_sq};
  return composite_backward_impl(raw, z_vals, rays_d, rays_d_stride, noise, n_rays, n_samples, white_bkgd, detach_weights, g_rgb,
                                 g_disp, g_acc, g_depth, g_weights, g_alpha, d_raw, mse, nullptr, stream);
}

int mvip_composite_backward_rays(const float* raw, const float* z_vals, const float* rays_d, int rays_d_stride,
                                 const float* noise, int64_t n_rays, int n_samples, int white_bkgd, int detach_weights,
                                 const float* target_rgb, const float* target_disp, const float* g_sq, const float* g_rgb,
                                 const float* g_disp, const float* g_acc, const float* g_depth, const float* g_weights,
                                 const float* g_alpha, float* d_raw, float* d_rays_d, void* stream) {
  MVIP_REQUIRE(n_rays == 0 || d_rays_d, MVIP_E_INVALID, "mvip_composite_backward_rays: null d_rays_d");
  MVIP_REQUIRE(!g_sq == !(target_rgb || target_disp), MVIP_E_INVALID,
               "mvip_composite_backward_rays: g_sq and a fused-loss target go together");
  const MseArgs mse = {target_rgb, target_disp, nullptr, nullptr, nullptr, g_sq};
  return composite_backward_impl(raw, z_vals, rays_d, rays_d_stride, noise, n_rays, n_samples, white_bkgd, detach_weights, g_rgb,
                                 g_disp, g_acc, g_depth, g_weights, g_alpha, d_raw, mse, d_rays_d, stream);
}

}  // extern "C"
