// rays.cu — camera rays of a pinhole view, written directly as the [N, 8 | 11] ray batch of the hot path (SURVEY.md §8 f1).
//   replaces DS_NeRF/run_nerf_helpers.py:249-260 (get_rays) and the ray-batch assembly of render(), run.py:1171-1207
//   (patch crop, viewdir normalisation, near / far columns, torch.cat).
// Bit-exact against the reference on CPU (verified in the build container against the unmodified get_rays / torch.norm):
//   dirs   = ((j - W/2) / focal, -((i - H/2) / focal), -1)             IEEE division, j / i exact integers
//   rays_d = (dirs.x * R[k][0] + dirs.y * R[k][1]) + dirs.z * R[k][2]    no FMA contraction (torch.sum over 3 products)
//   |v|    = sqrt(fma(v.z, v.z, fma(v.y, v.y, v.x * v.x)))              torch.norm's accumulation order
//   ndc_rays (run_nerf_helpers.py:283-300) fused behind a flag; mvip_rays_pack does the same assembly for given rays.
#include "common.cuh"

namespace {
// NDC warp of one ray (run_nerf_helpers.py:283-300), every op rounded to fp32 in the reference's order:
//   t = -(near + o.z) / d.z;  o' = o + t*d (mul, then add);  sx = (float)(-1/(W/(2 focal))) computed in double by the host;
//   o_ndc = ((sx*o'.x)/o'.z, (sy*o'.y)/o'.z, 1 + (1/o'.z)*2near);  d_ndc = (sx*(d.x/d.z - o'.x/o'.z), sy*(...), (1/o'.z)*(-2near))
//   (`c / tensor` is reciprocal(tensor) * c in torch, Tensor.__rtruediv__).
struct Ndc { int on; float near, sx, sy, two_near, neg_two_near; };

__device__ __forceinline__ void emit_ray(float* __restrict__ o, const float ro[3], const float rd[3], const float v[3],
                                         float near, float far, int use_viewdirs, const Ndc& ndc) {
  if (ndc.on) {
    const float t = __fdiv_rn(-__fadd_rn(ndc.near, ro[2]), rd[2]);
    const float ox = __fadd_rn(ro[0], __fmul_rn(t, rd[0]));
    const float oy = __fadd_rn(ro[1], __fmul_rn(t, rd[1]));
    const float oz = __fadd_rn(ro[2], __fmul_rn(t, rd[2]));
    const float rz = __fdiv_rn(1.f, oz);
    const float qx = __fdiv_rn(ox, oz), qy = __fdiv_rn(oy, oz);
    o[0] = __fdiv_rn(__fmul_rn(ndc.sx, ox), oz);
    o[1] = __fdiv_rn(__fmul_rn(ndc.sy, oy), oz);
    o[2] = __fadd_rn(1.f, __fmul_rn(rz, ndc.two_near));
    o[3] = __fmul_rn(ndc.sx, __fsub_rn(__fdiv_rn(rd[0], rd[2]), qx));
    o[4] = __fmul_rn(ndc.sy, __fsub_rn(__fdiv_rn(rd[1], rd[2]), qy));
    o[5] = __fmul_rn(rz, ndc.neg_two_near);
  } else {
#pragma unroll
    for (int k = 0; k < 3; ++k) { o[k] = ro[k]; o[3 + k] = rd[k]; }
  }
  o[6] = near;
  o[7] = far;
  if (use_viewdirs) {
    const float nrm = __fsqrt_rn(__fmaf_rn(v[2], v[2], __fmaf_rn(v[1], v[1], __fmul_rn(v[0], v[0]))));
    o[8] = __fdiv_rn(v[0], nrm);
    o[9] = __fdiv_rn(v[1], nrm);
    o[10] = __fdiv_rn(v[2], nrm);
  }
}

// camera-frame direction of pixel (row i, column j): ((j - W/2) / focal, -((i - H/2) / focal), -1)
__device__ __forceinline__ void pixel_dir(int i, int j, int H, int W, float focal, float dir[3]) {
  dir[0] = __fdiv_rn(__fsub_rn((float)j, __fmul_rn((float)W, .5f)), focal);
  dir[1] = -__fdiv_rn(__fsub_rn((float)i, __fmul_rn((float)H, .5f)), focal);
  dir[2] = -1.f;
}

// rays_o / rays_d of a direction under pose R, and the view vector under pose Rv ([3,4] row-major each; Rv == R without a
// static camera)
__device__ __forceinline__ void pose_ray(const float* R, const float* Rv, const float dir[3], float ro[3], float rd[3], float v[3]) {
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const float* r = R + 4 * k;
    ro[k] = r[3];
    rd[k] = __fadd_rn(__fadd_rn(__fmul_rn(dir[0], r[0]), __fmul_rn(dir[1], r[1])), __fmul_rn(dir[2], r[2]));
    const float* rv = Rv + 4 * k;
    v[k] = __fadd_rn(__fadd_rn(__fmul_rn(dir[0], rv[0]), __fmul_rn(dir[1], rv[1])), __fmul_rn(dir[2], rv[2]));
  }
}

// block-wide: rows of rays [blk, blk + 256) staged in shared memory -> global, consecutive floats per consecutive thread
__device__ __forceinline__ void flush_rows(const float* rows, float* __restrict__ out, int64_t blk, int64_t n, int stride) {
  __syncthreads();
  const int64_t left = n - blk;
  const int total = (int)(left < 256 ? left : 256) * stride;
  float* dst = out + blk * stride;
  for (int e = threadIdx.x; e < total; e += 256) dst[e] = rows[e];
  __syncthreads();
}

__global__ void __launch_bounds__(256) rays_kernel(const float* __restrict__ c2w, const float* __restrict__ c2w_static, int H, int W,
                                                   float focal, float near, float far, int i0, int j0, int h, int w,
                                                   int use_viewdirs, Ndc ndc, float* __restrict__ out) {
  __shared__ float pose[24];
  if (threadIdx.x < 12) {
    pose[threadIdx.x] = c2w[threadIdx.x];
    pose[12 + threadIdx.x] = c2w_static ? c2w_static[threadIdx.x] : c2w[threadIdx.x];
  }
  __syncthreads();
  __shared__ float rows[256 * 11];   // rows are staged here and leave as consecutive 4-byte stores (a lane per float, not per ray)
  const int stride = use_viewdirs ? 11 : 8;
  const int64_t n = (int64_t)h * w;
  for (int64_t blk = (int64_t)blockIdx.x * blockDim.x; blk < n; blk += (int64_t)gridDim.x * blockDim.x) {
    const int64_t idx = blk + threadIdx.x;
    if (idx < n) {
    const int i = i0 + (int)(idx / w), j = j0 + (int)(idx % w);
    float dir[3], ro[3], rd[3], v[3];
    pixel_dir(i, j, H, W, focal, dir);
    pose_ray(pose + 12, pose, dir, ro, rd, v);   // rays_o / rays_d from the (possibly static) camera
    emit_ray(rows + threadIdx.x * stride, ro, rd, v, near, far, use_viewdirs, ndc);
    }
    flush_rows(rows, out, blk, n, stride);
  }
}

// the `rays=` entry of render() (run.py:1176-1207): given origins / directions -> the same packed batch
__global__ void __launch_bounds__(256) rays_pack_kernel(const float* __restrict__ rays_o, const float* __restrict__ rays_d,
                                                        const float* __restrict__ view_d, int64_t n, float near, float far,
                                                        int use_viewdirs, Ndc ndc, float* __restrict__ out) {
  __shared__ float rows[256 * 11];
  const int stride = use_viewdirs ? 11 : 8;
  for (int64_t blk = (int64_t)blockIdx.x * blockDim.x; blk < n; blk += (int64_t)gridDim.x * blockDim.x) {
    const int64_t idx = blk + threadIdx.x;
    if (idx < n) {
      float ro[3], rd[3], v[3];
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        ro[k] = rays_o[idx * 3 + k];
        rd[k] = rays_d[idx * 3 + k];
        v[k] = view_d ? view_d[idx * 3 + k] : rd[k];
      }
      emit_ray(rows + threadIdx.x * stride, ro, rd, v, near, far, use_viewdirs, ndc);
    }
    flush_rows(rows, out, blk, n, stride);
  }
}

// ---- backward (autograd of the reference's fp32 formulas, in fp32) -------------------------------------------------------------
// d of one packed row (g[stride]) -> d ro, d rd (through ndc_rays when on) and d v (through v / |v|)
__device__ __forceinline__ void ray_row_backward(const float* __restrict__ g, const float ro[3], const float rd[3], const float v[3],
                                                 int use_viewdirs, int voff, const Ndc& ndc, float gro[3], float grd[3], float gv[3]) {
  if (ndc.on) {
    const float go0 = g[0], go1 = g[1], go2 = g[2], gd0 = g[3], gd1 = g[4], gd2 = g[5];
    const float t = -(ndc.near + ro[2]) / rd[2];
    const float ox = ro[0] + t * rd[0], oy = ro[1] + t * rd[1], oz = ro[2] + t * rd[2];
    const float rz = 1.f / oz, rz2 = rz * rz;
    // o_ndc = (sx ox/oz, sy oy/oz, 1 + 2n/oz);  d_ndc = (sx (dx/dz - ox/oz), sy (dy/dz - oy/oz), -2n/oz)
    const float gox = ndc.sx * (go0 - gd0) * rz;
    const float goy = ndc.sy * (go1 - gd1) * rz;
    const float goz = (ndc.sx * ox * (gd0 - go0) + ndc.sy * oy * (gd1 - go1) + ndc.two_near * (gd2 - go2)) * rz2;
    const float rdz = 1.f / rd[2];
    grd[0] = ndc.sx * gd0 * rdz;
    grd[1] = ndc.sy * gd1 * rdz;
    grd[2] = -(ndc.sx * gd0 * rd[0] + ndc.sy * gd1 * rd[1]) * rdz * rdz;
    // o' = o + t d;  t = -(n + o.z) / d.z
    const float gt = gox * rd[0] + goy * rd[1] + goz * rd[2];
    gro[0] = gox; gro[1] = goy; gro[2] = goz - gt * rdz;
    grd[0] += t * gox; grd[1] += t * goy; grd[2] += t * goz + gt * (ndc.near + ro[2]) * rdz * rdz;
  } else {
#pragma unroll
    for (int k = 0; k < 3; ++k) { gro[k] = g[k]; grd[k] = g[3 + k]; }
  }
  gv[0] = gv[1] = gv[2] = 0.f;
  if (use_viewdirs) {   // v_hat = v / |v|:  d v = (g - v_hat (v_hat . g)) / |v|
    const float nrm = sqrtf(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]);
    const float inv = 1.f / nrm;
    const float h0 = v[0] * inv, h1 = v[1] * inv, h2 = v[2] * inv;
    const float gh0 = g[voff], gh1 = g[voff + 1], gh2 = g[voff + 2];
    const float dot = h0 * gh0 + h1 * gh1 + h2 * gh2;
    gv[0] = (gh0 - h0 * dot) * inv;
    gv[1] = (gh1 - h1 * dot) * inv;
    gv[2] = (gh2 - h2 * dot) * inv;
  }
}

__global__ void __launch_bounds__(256) rays_pack_backward_kernel(const float* __restrict__ rays_o, const float* __restrict__ rays_d,
                                                                 const float* __restrict__ view_d, int64_t n, int use_viewdirs, Ndc ndc,
                                                                 const float* __restrict__ g_out, float* __restrict__ g_ro,
                                                                 float* __restrict__ g_rd, float* __restrict__ g_vd) {
  const int stride = use_viewdirs ? 11 : 8;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < n; idx += (int64_t)gridDim.x * blockDim.x) {
    float ro[3], rd[3], v[3], gro[3], grd[3], gv[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      ro[k] = rays_o[idx * 3 + k];
      rd[k] = rays_d[idx * 3 + k];
      v[k] = view_d ? view_d[idx * 3 + k] : rd[k];
    }
    ray_row_backward(g_out + idx * stride, ro, rd, v, use_viewdirs, 8, ndc, gro, grd, gv);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      g_ro[idx * 3 + k] = gro[k];
      if (view_d) { g_rd[idx * 3 + k] = grd[k]; g_vd[idx * 3 + k] = gv[k]; }
      else g_rd[idx * 3 + k] = grd[k] + gv[k];
    }
  }
}

// d c2w [3,4] (and d c2w_static) of a pinhole view: per-pixel terms d R[k][m] = d rays_d[k] dir[m], d t = d rays_o, summed per
// block in a fixed order (thread-strided, then a fixed tree) into partials[block][24]; rays_pose_reduce_kernel adds the blocks
// in block order.  Entries 0..11: the pose rays_o / rays_d come from, 12..23: the pose of the view directions.
constexpr int kPoseCap = 148 * 4;
__global__ void __launch_bounds__(256) rays_pose_backward_kernel(const float* __restrict__ c2w, const float* __restrict__ c2w_static,
                                                                 int H, int W, float focal, int i0, int j0, int h, int w,
                                                                 int use_viewdirs, Ndc ndc, const float* __restrict__ g_out,
                                                                 float* __restrict__ partials) {
  __shared__ float pose[24];
  __shared__ float red[8][24];
  if (threadIdx.x < 12) {
    pose[threadIdx.x] = c2w[threadIdx.x];
    pose[12 + threadIdx.x] = c2w_static ? c2w_static[threadIdx.x] : c2w[threadIdx.x];
  }
  __syncthreads();
  const int stride = use_viewdirs ? 11 : 8;
  const int64_t n = (int64_t)h * w;
  float acc[24];
#pragma unroll
  for (int e = 0; e < 24; ++e) acc[e] = 0.f;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < n; idx += (int64_t)gridDim.x * blockDim.x) {
    const int i = i0 + (int)(idx / w), j = j0 + (int)(idx % w);
    const float dir[3] = {__fdiv_rn(__fsub_rn((float)j, __fmul_rn((float)W, .5f)), focal),
                          -__fdiv_rn(__fsub_rn((float)i, __fmul_rn((float)H, .5f)), focal), -1.f};
    float ro[3], rd[3], v[3], gro[3], grd[3], gv[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const float* R = pose + 12 + 4 * k;
      ro[k] = R[3];
      rd[k] = __fadd_rn(__fadd_rn(__fmul_rn(dir[0], R[0]), __fmul_rn(dir[1], R[1])), __fmul_rn(dir[2], R[2]));
      const float* Rv = pose + 4 * k;
      v[k] = __fadd_rn(__fadd_rn(__fmul_rn(dir[0], Rv[0]), __fmul_rn(dir[1], Rv[1])), __fmul_rn(dir[2], Rv[2]));
    }
    ray_row_backward(g_out + idx * stride, ro, rd, v, use_viewdirs, 8, ndc, gro, grd, gv);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
#pragma unroll
      for (int m = 0; m < 3; ++m) {
        acc[4 * k + m] = fmaf(grd[k], dir[m], acc[4 * k + m]);
        acc[12 + 4 * k + m] = fmaf(gv[k], dir[m], acc[12 + 4 * k + m]);
      }
      acc[4 * k + 3] += gro[k];
    }
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int e = 0; e < 24; ++e) {
    const float s = warp_sum(acc[e]);
    if (lane == 0) red[warp][e] = s;
  }
  __syncthreads();
  if (threadIdx.x < 24) {
    float s = 0.f;
    for (int q = 0; q < 8; ++q) s += red[q][threadIdx.x];
    partials[(size_t)blockIdx.x * 24 + threadIdx.x] = s;
  }
}

// fixed-order sum of the block partials; without a static camera both halves belong to c2w
__global__ void rays_pose_reduce_kernel(const float* __restrict__ partials, int blocks, float* __restrict__ g_c2w,
                                        float* __restrict__ g_c2w_static) {
  const int e = threadIdx.x;
  __shared__ float tot[24];
  if (e < 24) {
    float s = 0.f;
    for (int b = 0; b < blocks; ++b) s += partials[(size_t)b * 24 + e];
    tot[e] = s;
  }
  __syncthreads();
  if (e < 12) {
    if (g_c2w_static) { g_c2w[e] = tot[12 + e]; g_c2w_static[e] = tot[e]; }
    else g_c2w[e] = tot[e] + tot[12 + e];
  }
}

// rays of a table of poses at given pixels: entry k = (view, row, col) -> row k of the batch, bitwise equal to row row*W + col of
// rays_kernel's batch of poses[view] over the whole image.  An entry outside [0,V) x [0,H) x [0,W) gives a row of NaN and reads
// no pose.
__global__ void __launch_bounds__(256) rays_poses_kernel(const float* __restrict__ poses, int V, const int* __restrict__ pixels,
                                                         int64_t n, int H, int W, float focal, float near, float far,
                                                         int use_viewdirs, Ndc ndc, float* __restrict__ out) {
  __shared__ float rows[256 * 11];
  const int stride = use_viewdirs ? 11 : 8;
  for (int64_t blk = (int64_t)blockIdx.x * blockDim.x; blk < n; blk += (int64_t)gridDim.x * blockDim.x) {
    const int64_t idx = blk + threadIdx.x;
    if (idx < n) {
      const int pv = pixels[idx * 3], i = pixels[idx * 3 + 1], j = pixels[idx * 3 + 2];
      float* o = rows + threadIdx.x * stride;
      if (pv >= 0 && pv < V && i >= 0 && i < H && j >= 0 && j < W) {
        const float* P = poses + (int64_t)pv * 12;
        float dir[3], ro[3], rd[3], v[3];
        pixel_dir(i, j, H, W, focal, dir);
        pose_ray(P, P, dir, ro, rd, v);
        emit_ray(o, ro, rd, v, near, far, use_viewdirs, ndc);
      } else {
        for (int e = 0; e < stride; ++e) o[e] = __int_as_float(0x7fc00000);
      }
    }
    flush_rows(rows, out, blk, n, stride);
  }
}

// d poses of rays_poses_kernel.  Block b handles view b / chunks and entries [c * kPosesChunk, +kPosesChunk) of the batch,
// c = b % chunks: each of its entries of that view adds d R[k][m] = (d rays_d[k] + d v[k]) dir[m], d t[k] = d rays_o[k]
// (thread-strided, then a fixed tree) into partials[b][12]; rays_poses_reduce_kernel adds a view's chunks in chunk order.  So
// every sum is taken in an order fixed by `pixels` alone, with no atomics.
// Cost: every block reads the view ids of its whole chunk, so the launch reads V x N ids (4 B each, from L2) besides the N rows
// it differentiates.  At a training batch (N = 4,096, V = 20: 80 blocks, 0.3 MB of ids) that is noise; it stops being
// negligible around V x N ~ 1e7 (e.g. 1,000 views x 65,536 rays: 64 M ids, 0.26 GB of L2 reads per step), where a stable
// sort of the view ids (O(N)) would take its place.
constexpr int kPosesChunk = 1024;
__global__ void __launch_bounds__(256) rays_poses_backward_kernel(const float* __restrict__ poses, const int* __restrict__ pixels,
                                                                  int64_t n, int chunks, int H, int W, float focal,
                                                                  int use_viewdirs, Ndc ndc, const float* __restrict__ g_out,
                                                                  float* __restrict__ partials) {
  __shared__ float red[8][12];
  const int view = (int)(blockIdx.x / chunks);
  const int64_t lo = (int64_t)(blockIdx.x % chunks) * kPosesChunk;
  const int64_t hi = n - lo < kPosesChunk ? n : lo + kPosesChunk;
  const int stride = use_viewdirs ? 11 : 8;
  const float* P = poses + (int64_t)view * 12;
  float acc[12];
#pragma unroll
  for (int e = 0; e < 12; ++e) acc[e] = 0.f;
  for (int64_t idx = lo + threadIdx.x; idx < hi; idx += blockDim.x) {
    if (pixels[idx * 3] != view) continue;
    const int i = pixels[idx * 3 + 1], j = pixels[idx * 3 + 2];
    if (i < 0 || i >= H || j < 0 || j >= W) continue;
    float dir[3], ro[3], rd[3], v[3], gro[3], grd[3], gv[3];
    pixel_dir(i, j, H, W, focal, dir);
    pose_ray(P, P, dir, ro, rd, v);
    ray_row_backward(g_out + idx * stride, ro, rd, v, use_viewdirs, 8, ndc, gro, grd, gv);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const float gk = grd[k] + gv[k];
#pragma unroll
      for (int m = 0; m < 3; ++m) acc[4 * k + m] = fmaf(gk, dir[m], acc[4 * k + m]);
      acc[4 * k + 3] += gro[k];
    }
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int e = 0; e < 12; ++e) {
    const float s = warp_sum(acc[e]);
    if (lane == 0) red[warp][e] = s;
  }
  __syncthreads();
  if (threadIdx.x < 12) {
    float s = 0.f;
    for (int q = 0; q < 8; ++q) s += red[q][threadIdx.x];
    partials[(size_t)blockIdx.x * 12 + threadIdx.x] = s;
  }
}

// g_poses[v][e] = sum over the view's chunks, in chunk order; views no entry uses get 0
__global__ void __launch_bounds__(256) rays_poses_reduce_kernel(const float* __restrict__ partials, int64_t V, int chunks,
                                                                float* __restrict__ g_poses) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= V * 12) return;
  const int64_t view = t / 12, e = t % 12;
  float s = 0.f;
  for (int c = 0; c < chunks; ++c) s += partials[(view * chunks + c) * 12 + e];
  g_poses[t] = s;
}

Ndc make_ndc(int on, int H, int W, double focal, double ndc_near) {
  Ndc c{};
  c.on = on ? 1 : 0;
  if (on) {   // python-double scalars, cast to fp32 when they meet a tensor
    c.near = (float)ndc_near;
    c.sx = (float)(-1. / ((double)W / (2. * focal)));
    c.sy = (float)(-1. / ((double)H / (2. * focal)));
    c.two_near = (float)(2. * ndc_near);
    c.neg_two_near = (float)(-2. * ndc_near);
  }
  return c;
}

unsigned grid_for(int64_t n) {
  int64_t blocks = (n + 255) / 256;
  const int64_t cap = (int64_t)mvip_num_sms() * 16;
  return (unsigned)(blocks > cap ? cap : blocks);
}
}  // namespace

extern "C" int mvip_rays_from_pose_ndc(const float* c2w, const float* c2w_static, int H, int W, double focal, float near,
                                       float far, int i0, int j0, int h, int w, int use_viewdirs, int ndc, double ndc_near,
                                       float* out, void* stream) {
  MVIP_REQUIRE(H > 0 && W > 0 && h >= 0 && w >= 0 && i0 >= 0 && j0 >= 0 && i0 + h <= H && j0 + w <= W, MVIP_E_INVALID,
               "mvip_rays_from_pose: window [%d,+%d) x [%d,+%d) outside the %d x %d image", i0, h, j0, w, H, W);
  MVIP_REQUIRE(focal != 0., MVIP_E_INVALID, "mvip_rays_from_pose: focal == 0");
  const int64_t n = (int64_t)h * w;
  if (n == 0) return MVIP_OK;
  MVIP_REQUIRE(c2w && out, MVIP_E_INVALID, "mvip_rays_from_pose: null pointer");
  rays_kernel<<<grid_for(n), 256, 0, (cudaStream_t)stream>>>(c2w, c2w_static, H, W, (float)focal, near, far, i0, j0, h, w,
                                                             use_viewdirs ? 1 : 0, make_ndc(ndc, H, W, focal, ndc_near), out);
  MVIP_LAUNCH_OK("rays_kernel");
  return MVIP_OK;
}

extern "C" int mvip_rays_from_pose(const float* c2w, const float* c2w_static, int H, int W, float focal, float near,
                                   float far, int i0, int j0, int h, int w, int use_viewdirs, float* out, void* stream) {
  return mvip_rays_from_pose_ndc(c2w, c2w_static, H, W, (double)focal, near, far, i0, j0, h, w, use_viewdirs, 0, 0., out, stream);
}

extern "C" int mvip_rays_pack(const float* rays_o, const float* rays_d, const float* view_d, int64_t n, float near, float far,
                              int use_viewdirs, int ndc, int H, int W, double focal, double ndc_near, float* out, void* stream) {
  MVIP_REQUIRE(n >= 0, MVIP_E_INVALID, "mvip_rays_pack: n < 0");
  if (n == 0) return MVIP_OK;
  MVIP_REQUIRE(rays_o && rays_d && out, MVIP_E_INVALID, "mvip_rays_pack: null pointer");
  MVIP_REQUIRE(!ndc || (H > 0 && W > 0 && focal != 0.), MVIP_E_INVALID, "mvip_rays_pack: ndc needs H, W, focal");
  rays_pack_kernel<<<grid_for(n), 256, 0, (cudaStream_t)stream>>>(rays_o, rays_d, view_d, n, near, far, use_viewdirs ? 1 : 0,
                                                                  make_ndc(ndc, H, W, focal, ndc_near), out);
  MVIP_LAUNCH_OK("rays_pack_kernel");
  return MVIP_OK;
}

extern "C" size_t mvip_rays_from_pose_backward_workspace_bytes(void) { return (size_t)kPoseCap * 24 * sizeof(float); }

extern "C" int mvip_rays_from_pose_backward(const float* c2w, const float* c2w_static, int H, int W, double focal, int i0, int j0,
                                            int h, int w, int use_viewdirs, int ndc, double ndc_near, const float* g_out,
                                            float* g_c2w, float* g_c2w_static, void* workspace, void* stream) {
  MVIP_REQUIRE(H > 0 && W > 0 && h >= 0 && w >= 0 && i0 >= 0 && j0 >= 0 && i0 + h <= H && j0 + w <= W, MVIP_E_INVALID,
               "mvip_rays_from_pose_backward: window [%d,+%d) x [%d,+%d) outside the %d x %d image", i0, h, j0, w, H, W);
  MVIP_REQUIRE(focal != 0., MVIP_E_INVALID, "mvip_rays_from_pose_backward: focal == 0");
  MVIP_REQUIRE(c2w && g_c2w && workspace && (g_out || (int64_t)h * w == 0), MVIP_E_INVALID,
               "mvip_rays_from_pose_backward: null pointer");
  MVIP_REQUIRE(!g_c2w_static == !c2w_static, MVIP_E_INVALID,
               "mvip_rays_from_pose_backward: c2w_static and g_c2w_static must be given together");
  const int64_t n = (int64_t)h * w;
  int64_t blocks = (n + 255) / 256;
  const int64_t cap = mvip_num_sms() * 4 < kPoseCap ? mvip_num_sms() * 4 : kPoseCap;
  blocks = blocks < 1 ? 1 : (blocks > cap ? cap : blocks);
  float* partials = static_cast<float*>(workspace);
  rays_pose_backward_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
      c2w, c2w_static, H, W, (float)focal, i0, j0, h, w, use_viewdirs ? 1 : 0, make_ndc(ndc, H, W, focal, ndc_near), g_out, partials);
  MVIP_LAUNCH_OK("rays_pose_backward_kernel");
  rays_pose_reduce_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(partials, (int)blocks, g_c2w, g_c2w_static);
  MVIP_LAUNCH_OK("rays_pose_reduce_kernel");
  return MVIP_OK;
}

extern "C" int mvip_rays_pack_backward(const float* rays_o, const float* rays_d, const float* view_d, int64_t n, int use_viewdirs,
                                       int ndc, int H, int W, double focal, double ndc_near, const float* g_out, float* g_rays_o,
                                       float* g_rays_d, float* g_view_d, void* stream) {
  MVIP_REQUIRE(n >= 0, MVIP_E_INVALID, "mvip_rays_pack_backward: n < 0");
  if (n == 0) return MVIP_OK;
  MVIP_REQUIRE(rays_o && rays_d && g_out && g_rays_o && g_rays_d && (!view_d || g_view_d), MVIP_E_INVALID,
               "mvip_rays_pack_backward: null pointer");
  MVIP_REQUIRE(!ndc || (H > 0 && W > 0 && focal != 0.), MVIP_E_INVALID, "mvip_rays_pack_backward: ndc needs H, W, focal");
  rays_pack_backward_kernel<<<grid_for(n), 256, 0, (cudaStream_t)stream>>>(rays_o, rays_d, view_d, n, use_viewdirs ? 1 : 0,
                                                                           make_ndc(ndc, H, W, focal, ndc_near), g_out, g_rays_o,
                                                                           g_rays_d, g_view_d);
  MVIP_LAUNCH_OK("rays_pack_backward_kernel");
  return MVIP_OK;
}

namespace {
int64_t poses_chunks(int64_t n) { return n <= kPosesChunk ? 1 : (n + kPosesChunk - 1) / kPosesChunk; }
}  // namespace

extern "C" int mvip_rays_from_poses(const float* poses, int V, const int* pixels, int64_t n, int H, int W, double focal, float near,
                                    float far, int use_viewdirs, int ndc, double ndc_near, float* out, void* stream) {
  MVIP_REQUIRE(V >= 0 && n >= 0 && H > 0 && W > 0, MVIP_E_INVALID, "mvip_rays_from_poses: V = %d, N = %lld, image %d x %d", V,
               (long long)n, H, W);
  MVIP_REQUIRE(focal != 0., MVIP_E_INVALID, "mvip_rays_from_poses: focal == 0");
  if (n == 0) return MVIP_OK;
  MVIP_REQUIRE((poses || V == 0) && pixels && out, MVIP_E_INVALID, "mvip_rays_from_poses: null pointer");
  rays_poses_kernel<<<grid_for(n), 256, 0, (cudaStream_t)stream>>>(poses, V, pixels, n, H, W, (float)focal, near, far,
                                                                   use_viewdirs ? 1 : 0, make_ndc(ndc, H, W, focal, ndc_near), out);
  MVIP_LAUNCH_OK("rays_poses_kernel");
  return MVIP_OK;
}

extern "C" size_t mvip_rays_from_poses_backward_workspace_bytes(int64_t n, int V) {
  return (size_t)(V > 0 ? V : 0) * (size_t)poses_chunks(n < 0 ? 0 : n) * 12 * sizeof(float);
}

extern "C" int mvip_rays_from_poses_backward(const float* poses, int V, const int* pixels, int64_t n, int H, int W, double focal,
                                             int use_viewdirs, int ndc, double ndc_near, const float* g_out, float* g_poses,
                                             void* workspace, void* stream) {
  MVIP_REQUIRE(V >= 0 && n >= 0 && H > 0 && W > 0, MVIP_E_INVALID, "mvip_rays_from_poses_backward: V = %d, N = %lld, image %d x %d",
               V, (long long)n, H, W);
  MVIP_REQUIRE(focal != 0., MVIP_E_INVALID, "mvip_rays_from_poses_backward: focal == 0");
  if (V == 0) return MVIP_OK;
  MVIP_REQUIRE(poses && g_poses && workspace && (n == 0 || (pixels && g_out)), MVIP_E_INVALID,
               "mvip_rays_from_poses_backward: null pointer");
  const int64_t chunks = poses_chunks(n);
  MVIP_REQUIRE((int64_t)V * chunks < (int64_t)1 << 31, MVIP_E_INVALID, "mvip_rays_from_poses_backward: %d views x %lld chunks", V,
               (long long)chunks);
  float* partials = static_cast<float*>(workspace);
  rays_poses_backward_kernel<<<(unsigned)(V * chunks), 256, 0, (cudaStream_t)stream>>>(
      poses, pixels, n, (int)chunks, H, W, (float)focal, use_viewdirs ? 1 : 0, make_ndc(ndc, H, W, focal, ndc_near), g_out, partials);
  MVIP_LAUNCH_OK("rays_poses_backward_kernel");
  rays_poses_reduce_kernel<<<(unsigned)((V * 12 + 255) / 256), 256, 0, (cudaStream_t)stream>>>(partials, V, (int)chunks, g_poses);
  MVIP_LAUNCH_OK("rays_poses_reduce_kernel");
  return MVIP_OK;
}
