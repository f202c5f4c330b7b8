// mlp_input_grad.cu — gradient of the fused NeRF MLP with respect to its inputs (the sample points and view directions).
//
// Runs after mvip_mlp_backward on the same stream and reads the bf16 dZ images that call left in its workspace (kDz* in
// mlp_common.cuh).  Per 128-point tile, two tcgen05 GEMMs (cta_group::1, fp32 accumulators in tensor memory):
//   dPE(pts)  [128 x 64] = [dZ_0 | dZ_5] . [W_0 ; W_5,PE]     K = 512  (the skip feeds PE into layer 5 as well)
//   dPE(view) [128 x 64] = dZ_hidden . W_views,PE             K = 128  (27 of the 64 columns are real)
// The A operands are the dZ chunk images as stored (K-major, 128 points x 64 features).  The B operands are the packed
// FORWARD weight chunks 0, 17 and 38: out-rows x 64 inputs, read with an MN-major descriptor (MN = input feature,
// K = output feature), so the blob needs no second copy.  The three chunks (80 KB) stay resident; the dZ images stream
// through a bulk-copy ring.  The epilogue chains dPE through the positional encoding in fp32:
//   dx_j = dPE[j] + sum_k 2^k (cos(2^k x_j) dPE_sin[k][j] - sin(2^k x_j) dPE_cos[k][j])
// with sin / cos recomputed by the forward's own pe_axis from the inputs the forward read.
//
// Output: [P, 6] fp32 per point (d pts | d viewdir).  In rays mode a second kernel sums them per ray in a fixed order
// (one warp per ray, no atomics): d o = sum_s d pts, d d = sum_s z_s d pts, d viewdir = sum_s d view.
#include "mlp_common.cuh"

namespace {
using namespace mlp;

constexpr int kStages = 8;                       // dZ ring: 8 chunk images of 16 KB
constexpr int kChunksPerTile = 10;               // dZ_0 (4), dZ_5 (4), d hidden_pre (2)
constexpr uint32_t kSmW0 = 0, kSmW5 = kW256, kSmWv = 2 * kW256, kSmRing = 2 * kW256 + kW128;
constexpr uint32_t kSmemBytes = kSmRing + kStages * kActChunk + 1024;
constexpr int kThreads = 192;                    // warps 0-3 epilogue, 4 producer, 5 MMA issuer
constexpr uint32_t kTmemCols = 256;              // two accumulator slots of 128 columns (64 pts + 64 view)

__device__ __forceinline__ int dz_chunk(int j) { return j < 4 ? kDzTrunk + 28 + j : (j < 8 ? kDzTrunk + 8 + (j - 4) : kDzHidden + (j - 8)); }

struct Args {
  const uint8_t* packed;
  const uint8_t* dz;
  mvip_points pts;
  float* out6;
  int64_t n_tiles;
};

__global__ void __launch_bounds__(kThreads, 1) mlp_input_grad_kernel(const Args p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ uint64_t bar_w, bar_full[kStages], bar_empty[kStages], bar_acc_full[2], bar_acc_empty[2];
  __shared__ uint32_t tmem_base_s;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    mbar_init(&bar_w, 1);
    for (int s = 0; s < kStages; ++s) { mbar_init(&bar_full[s], 1); mbar_init(&bar_empty[s], 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(&bar_acc_full[s], 1); mbar_init(&bar_acc_empty[s], 4); }
    mbar_fence_init();
  }
  if (warp == 5) tmem_alloc(&tmem_base_s, kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;

  if (warp == 4) {
    // ===================== producer: weights once, then the dZ chunks of every tile of this CTA =====================
    if (elect_one_sync()) {
      mbar_arrive_expect_tx(&bar_w, 2 * kW256 + kW128);
      tma_load_1d(smem + kSmW0, p.packed + fwd_chunk_off(0), kW256, &bar_w);
      tma_load_1d(smem + kSmW5, p.packed + fwd_chunk_off(17), kW256, &bar_w);
      tma_load_1d(smem + kSmWv, p.packed + fwd_chunk_off(38), kW128, &bar_w);
      const uint64_t pol = l2_policy_evict_first();
      int stage = 0;
      uint32_t phase = 0;
      for (int64_t t = blockIdx.x; t < p.n_tiles; t += gridDim.x) {
        const uint8_t* tile = p.dz + (size_t)t * kDzTileBytes;
        for (int j = 0; j < kChunksPerTile; ++j) {
          mbar_wait(&bar_empty[stage], phase ^ 1);
          mbar_arrive_expect_tx(&bar_full[stage], kActChunk);
          tma_load_1d_hint(smem + kSmRing + stage * kActChunk, tile + (size_t)dz_chunk(j) * kActChunk, kActChunk, &bar_full[stage], pol);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 5) {
    // ===================== MMA issuer =====================
    mbar_wait(&bar_w, 0);
    const uint32_t idesc = umma_idesc_bf16(128, 64, 0, 1);   // A K-major (dZ images), B MN-major (forward weight chunks)
    const uint32_t s_base = smem_u32(smem);
    int stage = 0;
    uint32_t phase = 0;
    int it = 0;
    for (int64_t t = blockIdx.x; t < p.n_tiles; t += gridDim.x, ++it) {
      const int slot = it & 1;
      mbar_wait(&bar_acc_empty[slot], ((it >> 1) & 1) ^ 1);
      tc_fence_after();
      for (int j = 0; j < kChunksPerTile; ++j) {
        mbar_wait(&bar_full[stage], phase);
        tc_fence_after();
        // chunk j covers output features 64 (j % 4) .. +63 of its layer = K rows of the weight chunk at 64 rows x 128 B each
        const uint32_t w = j < 4 ? kSmW0 : (j < 8 ? kSmW5 : kSmWv);
        const uint32_t w_rows = (uint32_t)(j & 3) * 64u * 128u;
        const uint32_t d = tmem_base + (uint32_t)slot * 128u + (j < 8 ? 0u : 64u);
        if (elect_one_sync()) {
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) {
            const uint64_t da = umma_desc_sw128(s_base + kSmRing + stage * kActChunk + kk * 32, 16, 1024);
            const uint64_t db = umma_desc_sw128(s_base + w + w_rows + kk * 2048, kW256, 1024);
            umma_bf16(d, da, db, idesc, (kk > 0 || (j != 0 && j != 8)) ? 1u : 0u);
          }
          umma_commit(&bar_empty[stage]);
          if (j == kChunksPerTile - 1) umma_commit(&bar_acc_full[slot]);
        }
        __syncwarp();
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
    }
  } else {
    // ===================== epilogue: TMEM lane = point of the tile =====================
    const int row = warp * 32 + lane;
    const uint32_t lane_base = (uint32_t)(warp * 32) << 16;
    int it = 0;
    for (int64_t t = blockIdx.x; t < p.n_tiles; t += gridDim.x, ++it) {
      const int slot = it & 1;
      const int64_t g = t * kTile + row;
      const bool live = g < p.pts.n_points;
      const int64_t gl = live ? g : 0;
      float x[3], v[3];
      if (p.pts.rays) {   // the forward's own arithmetic: pts = o + d*z
        const int64_t ray = gl / p.pts.n_samples;
        const float* rp = p.pts.rays + ray * p.pts.ray_stride;
        const float zv = __ldg(p.pts.z_vals + gl);
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          x[k] = __fadd_rn(__ldg(rp + k), __fmul_rn(__ldg(rp + 3 + k), zv));
          v[k] = __ldg(rp + p.pts.viewdir_offset + k);
        }
      } else {
        const float* pp = p.pts.pts + gl * p.pts.pts_stride;
        const float* dp = p.pts.dirs + gl * p.pts.dirs_stride;
#pragma unroll
        for (int k = 0; k < 3; ++k) { x[k] = __ldg(pp + k); v[k] = __ldg(dp + k); }
      }
      mbar_wait(&bar_acc_full[slot], (it >> 1) & 1);
      tc_fence_after();
      uint32_t a0[32], a1[32], a2[32];
      const uint32_t col = tmem_base + lane_base + (uint32_t)slot * 128u;
      tmem_ld32(col, a0);
      tmem_ld32(col + 32, a1);
      tmem_ld32(col + 64, a2);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_acc_empty[slot]);
      auto pe_col = [&](int i) { return __uint_as_float(i < 32 ? a0[i] : a1[i - 32]); };
      float out[6];
#pragma unroll
      for (int dd = 0; dd < 3; ++dd) {
        float s[10], c[10];
        pe_axis(x[dd], 10, s, c);
        float acc = pe_col(dd), scale = 1.f;
#pragma unroll
        for (int k = 0; k < 10; ++k) {
          acc = fmaf(scale, fmaf(c[k], pe_col(3 + 6 * k + dd), -s[k] * pe_col(6 + 6 * k + dd)), acc);
          scale *= 2.f;
        }
        out[dd] = acc;
        pe_axis(v[dd], 4, s, c);
        acc = __uint_as_float(a2[dd]);
        scale = 1.f;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          acc = fmaf(scale, fmaf(c[k], __uint_as_float(a2[3 + 6 * k + dd]), -s[k] * __uint_as_float(a2[6 + 6 * k + dd])), acc);
          scale *= 2.f;
        }
        out[3 + dd] = acc;
      }
      if (live) {
        float2* o = reinterpret_cast<float2*>(p.out6 + g * 6);
        o[0] = make_float2(out[0], out[1]);
        o[1] = make_float2(out[2], out[3]);
        o[2] = make_float2(out[4], out[5]);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 5) tmem_dealloc(tmem_base, kTmemCols);
}

// rays mode: one warp per ray; lane-strided partial sums then a fixed xor tree.  Writes every column of the ray's gradient row.
__global__ void __launch_bounds__(256) mlp_input_grad_rays_kernel(const float* __restrict__ d6, const float* __restrict__ z_vals,
                                                                  int64_t n_rays, int S, int stride, int voff,
                                                                  float* __restrict__ d_rays) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t ray = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); ray < n_rays; ray += warps) {
    float a[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int s = lane; s < S; s += 32) {
      const float* q = d6 + (ray * S + s) * 6;
      const float z = __ldg(z_vals + ray * S + s);
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const float dp = __ldg(q + k);
        a[k] += dp;
        a[3 + k] = fmaf(z, dp, a[3 + k]);
        a[6 + k] += __ldg(q + 3 + k);
      }
    }
#pragma unroll
    for (int k = 0; k < 9; ++k) a[k] = warp_sum(a[k]);
    float* row = d_rays + ray * stride;
    for (int c = lane; c < stride; c += 32) {
      float val = 0.f;
      if (c < 6) val += a[c];
      if (c >= voff && c < voff + 3) val += a[6 + c - voff];
      row[c] = val;
    }
  }
}

}  // namespace

extern "C" int mvip_mlp_input_grad(const void* packed, const mvip_points* pts, const void* bwd_workspace, float* d_points,
                                   float* d_rays, void* stream) {
  MVIP_REQUIRE(packed && pts && bwd_workspace && d_points, MVIP_E_INVALID, "mvip_mlp_input_grad: null pointer");
  MVIP_REQUIRE(mvip_aligned(packed, 1024) && mvip_aligned(bwd_workspace, 1024) && mvip_aligned(d_points, 8), MVIP_E_INVALID,
               "mvip_mlp_input_grad: packed / workspace need 1024-byte and d_points 8-byte alignment");
  MVIP_REQUIRE(pts->n_points >= 0, MVIP_E_INVALID, "mvip_mlp_input_grad: negative n_points");
  if (pts->rays) {
    MVIP_REQUIRE(pts->z_vals && pts->n_rays >= 0 && pts->n_samples >= 1 && pts->n_points == pts->n_rays * pts->n_samples,
                 MVIP_E_INVALID, "mvip_mlp_input_grad: rays mode needs z_vals and n_points = n_rays * n_samples");
    MVIP_REQUIRE(pts->ray_stride >= 6 && pts->viewdir_offset >= 0 && pts->viewdir_offset + 3 <= pts->ray_stride, MVIP_E_INVALID,
                 "mvip_mlp_input_grad: bad ray_stride / viewdir_offset (%d, %d)", pts->ray_stride, pts->viewdir_offset);
    MVIP_REQUIRE(d_rays, MVIP_E_INVALID, "mvip_mlp_input_grad: rays mode needs d_rays");
  } else {
    MVIP_REQUIRE(pts->pts && pts->dirs && pts->pts_stride >= 3 && pts->dirs_stride >= 0, MVIP_E_INVALID,
                 "mvip_mlp_input_grad: points mode needs pts and dirs");
  }
  if (pts->n_points == 0) return MVIP_OK;
  Args a;
  a.packed = static_cast<const uint8_t*>(packed);
  a.dz = static_cast<const uint8_t*>(bwd_workspace);   // the dZ images sit at offset 0 of the backward's workspace
  a.pts = *pts;
  a.out6 = d_points;
  a.n_tiles = num_tiles(pts->n_points);
  MVIP_SMEM_OPT_IN(mlp_input_grad_kernel, kSmemBytes);
  const int64_t grid = a.n_tiles < mvip_num_sms() ? a.n_tiles : mvip_num_sms();
  mlp_input_grad_kernel<<<(unsigned)grid, kThreads, kSmemBytes, (cudaStream_t)stream>>>(a);
  MVIP_LAUNCH_OK("mlp_input_grad_kernel");
  if (pts->rays) {
    const int64_t blocks = (pts->n_rays + 7) / 8, cap = (int64_t)mvip_num_sms() * 8;
    mlp_input_grad_rays_kernel<<<(unsigned)(blocks < cap ? blocks : cap), 256, 0, (cudaStream_t)stream>>>(
        d_points, pts->z_vals, pts->n_rays, pts->n_samples, pts->ray_stride, pts->viewdir_offset, d_rays);
    MVIP_LAUNCH_OK("mlp_input_grad_rays_kernel");
  }
  return MVIP_OK;
}
