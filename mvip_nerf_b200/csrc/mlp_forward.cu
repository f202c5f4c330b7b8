// mlp_forward.cu — fused positional encoding + NeRF MLP forward on tcgen05 tensor cores.
//   replaces DS_NeRF/run.py:1108-1124 (run_network), run_nerf_helpers.py:22-52 (Embedder.embed) and
//   run_nerf_helpers.py:104-127 (NeRF.forward)
//
// ONE kernel, mlp_forward_pair_kernel<kTrain>: CTA pairs (cta_group::2), activations resident in TENSOR MEMORY: the A
// operand of every layer is read from TMEM ("TS" tcgen05.mma), the epilogue writes the next layer's bf16 activations
// straight back to TMEM.  1,443 TFLOP/s at inference on one B200 (87 % of the cuBLAS bf16 burst peak).  Described in the
// comment block above the kernel.  Activations never leave the SM; the only HBM traffic at inference is 16..28 B/point in
// (rays+z) and 16 B/point out (raw).  With a stash pointer (training) every layer's input tile image is also bulk-stored
// for the backward pass (mlp_common.cuh, kStash*).
#include "mlp_pair.cuh"
#include <stdlib.h>

namespace {
using namespace mlp;

constexpr int kNumSteps = 10;

// cycle counters of CTA 0 (debug aid, read with mvip_debug_profile): [0] mma: act wait, [1] mma: weight wait,
// [2] mma: total, [3] epi slot0: acc wait, [4] epi slot0: work, [5] epi slot0: total, [6] producer: empty wait
__device__ unsigned long long g_prof[16];

// Optional event trace of CTA 0 (build with -DMVIP_TRACE): three logs (issuer, epilogue leader of slot 0 / slot 1) of
// (code, clock) pairs for ONE iteration; read with mvip_debug_trace.
#ifdef MVIP_PROF
#define PROF_DECL long long t_act = 0, t_full = 0, t_begin = clock64(), t0_ = 0
#define PROF_T0 t0_ = clock64()
#define PROF_ADD(x) x += clock64() - t0_
#define PROF_STORE do { if (blockIdx.x == 0 && T == 0 && lane == 0) { g_prof[0] = t_act; g_prof[1] = t_full; g_prof[2] = clock64() - t_begin; } } while (0)
#else
#define PROF_DECL
#define PROF_T0
#define PROF_ADD(x)
#define PROF_STORE
#endif
#ifdef MVIP_TRACE
__device__ long long g_trace[3][1024][2];
__device__ int g_trace_n[3];
#define TRACE_DECL(role) int tr_n_ = 0; const int tr_role_ = (role); bool tr_on_ = false
#define TRACE_ARM(cond) tr_on_ = (cond)
#define TRACE(code) do { if (tr_on_ && tr_n_ < 1024) { g_trace[tr_role_][tr_n_][0] = (code); g_trace[tr_role_][tr_n_][1] = clock64(); ++tr_n_; g_trace_n[tr_role_] = tr_n_; } } while (0)
#else
#define TRACE_DECL(role)
#define TRACE_ARM(cond)
#define TRACE(code)
#endif

struct Params {
  const uint8_t* packed;
  mvip_points pts;
  float4* raw;
  uint8_t* stash;
  int64_t n_tiles;
};

// step s: number of 64-wide K chunks of its weight block
__device__ __forceinline__ int step_nchunks(int s) { return s == 0 ? 1 : ((s == 5 || s == 9) ? 5 : 4); }

// one half (4 of the 8 sixteen-byte groups) of a PE row; `half` is warp-uniform
template <int L>
__device__ __forceinline__ void write_pe_half(uint8_t* img, int row, float x, float y, float z, int half) {
  float s[3][10], c[3][10];
  pe_axis(x, L, s[0], c[0]);
  pe_axis(y, L, s[1], c[1]);
  pe_axis(z, L, s[2], c[2]);
  const float in[3] = {x, y, z};
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    if (h == half) {
#pragma unroll
      for (int gg = 0; gg < 4; ++gg) {
        const int g = 4 * h + gg;
        float v[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const int i = g * 8 + e;
          float val = 0.f;
          if (i < 3) val = in[i];
          else if (i < 3 + 6 * L) {
            const int t = i - 3, k = t / 6, r6 = t % 6, d = r6 % 3;
            val = (r6 >= 3) ? c[d][k] : s[d][k];
          }
          v[e] = val;
        }
        *reinterpret_cast<uint4*>(img + chunk_off16(row, g)) =
            make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
      }
    }
  }
}

// bf16x2 pack with fused ReLU (negative -> +0)
__device__ __forceinline__ uint32_t pack_relu_bf16x2(float lo, float hi) {
  uint32_t d;
  asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
  return d;
}

__device__ __forceinline__ float4 lds_f4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ float lds_f1(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
  return v;
}


// =================================================================================================
// CTA-pair kernel (cta_group::2), activations resident in TENSOR MEMORY ("TS" MMAs: A from TMEM, B from smem).
//
// Measured on B200 (scripts/ubench/umma_bench.cu): a 128xNx16 bf16 MMA with A in shared memory takes 171 cycles at N = 256
// (75 % of the tensor-pipe floor, the cuBLAS level) and 107 at N = 128; with A in TMEM it takes 138 / 74 cycles (93 % / 87 %).
// So the layer outputs never go to shared memory: the epilogue packs them to bf16 and writes them straight back
// to TMEM as the next layer's A operand.
//
//   * a cluster of two CTAs works on four 128-point tiles: each CTA owns two tile slots X, Y and the MMAs are
//     256 (2 x 128 points) x 128 x 16: one N-half of a layer at a time;
//   * TMEM per CTA (512 columns): slot T at column 256 T: [0,128) = A operand (256 bf16 features, two per column),
//     [128,256) = fp32 accumulator of one N-half (128 output features);
//   * issue order per layer: X.h0, Y.h0, X.h1, Y.h1.  While the tensor pipe works on Y, X's eight epilogue warps
//     drain X's accumulator half (tcgen05.ld -> +bias, ReLU, bf16 pack).  The h0 result is HELD IN REGISTERS
//     (32 per thread) because X.h1 still reads the old A operand; after X.h1 completes both halves are written
//     to the A columns (tcgen05.st) and X's next layer can start: no tensor-pipe bubble as long as
//     the drain of one half (~600 cycles) fits into the MMAs of the other slot's half (~1200 cycles);
//   * weights: a ring stage holds this CTA's 64 rows of one (layer, N-half, 64-wide K chunk) = 8 KB; a stage
//     is used by X and then Y before it is released, so every weight byte is fetched once per four tiles
//     (1/4 of the L2 -> smem traffic of the 1-CTA kernel) and the ring is 12 deep;
//   * PE(pts) / PE(viewdir) live in shared memory (one 16 KB image per slot) and enter L0, L5 and the views layer as
//     ordinary smem-A MMAs accumulating into the same TMEM columns;
//   * training: the packed bf16 rows are additionally staged in shared memory (32 KB per slot) and bulk-stored to the
//     activation stash; ReLU masks are derived from the packed words.
//   * only the leader CTA (rank 0) issues MMAs; its barriers collect the peer's "weights landed" (relay warp)
//     and "A operand ready / accumulator drained" (remote mbarrier arrive) signals, and tcgen05.commit
//     multicasts "stage free" / "accumulator full" to both CTAs.
// =================================================================================================
constexpr int kThreads2 = 640;
// weight ring: 8 KB slots, filled and released in GROUPS = all K chunks of one (layer, N-half): 1, 4 or 5 slots.
// One full / one empty barrier per group (a successful mbarrier wait costs the issuer ~200 cycles, so per-chunk
// barriers would eat a third of its time).  The producer runs kLag groups ahead.
template <bool kTrain> struct Ring2 {
  static constexpr int kSlots = kTrain ? 12 : 20;
  static constexpr int kLag = kTrain ? 2 : 4;      // any kLag consecutive groups fit: 5+5 <= 12, 4+5+5+4 <= 20
};
constexpr uint32_t kSmemPE2 = 0;                                         // pe[2]: 2 x 16 KB
constexpr uint32_t kSmemSmall2 = 2 * kActChunk;                          // fp32 tail of the packed blob (12,320 B)
constexpr uint32_t kSmemXch2 = kSmemSmall2 + ((kSmallFloats * 4 + 1023) / 1024) * 1024;   // head partials, 2 x 2 KB
constexpr uint32_t kSmemW2 = kSmemXch2 + 2 * 2048;                       // weight ring
constexpr uint32_t kSmemStg2 = kSmemW2 + Ring2<true>::kSlots * kSlotBytes2;   // stash staging: one 4 KB piece (32 rows of a chunk image) per epilogue warp (train)
constexpr uint32_t kSmemMask2 = kSmemStg2 + 16 * 4096;                   // ReLU-mask staging: 512 B per epilogue warp (train)
constexpr uint32_t kSmemBytes2Train = kSmemMask2 + 16 * 512;             // 222,208
constexpr uint32_t kSmemBytes2Infer = kSmemW2 + Ring2<false>::kSlots * kSlotBytes2;   // 214,016
constexpr int kGroupsPerIter2 = 19;

// One accumulator half (row r, 64 of its 128 columns) -> +bias, (ReLU), bf16 pairs in pk[32].
// ONE code instance for all layers (s is warp-uniform): the steady-state loop of the kernel has to stay inside the
// 32 KB instruction cache, otherwise the single MMA-issuing warp starves on instruction fetches.
// s == 7: + alpha head; s == 8 (feature layer): no ReLU; s == 9 (views layer): + rgb head.
template <bool kTrain>
__device__ __forceinline__ void math_half(const uint32_t (&raw)[4][16], uint32_t small_s, int s, int bias_i, int col0,
                                          uint32_t (&pk)[32], uint32_t (&mw)[2], float& alpha_part, float (&rgb_part)[3]) {
#pragma unroll
  for (int b = 0; b < 4; ++b) {
    const uint32_t (&acc)[16] = raw[b];
    const int c0 = col0 + 16 * b;
    float v[16];
#pragma unroll
    for (int j4 = 0; j4 < 4; ++j4) {
      const float4 bb = lds_f4(small_s + (bias_i + c0 + 4 * j4) * 4);
      v[4 * j4 + 0] = __uint_as_float(acc[4 * j4 + 0]) + bb.x;
      v[4 * j4 + 1] = __uint_as_float(acc[4 * j4 + 1]) + bb.y;
      v[4 * j4 + 2] = __uint_as_float(acc[4 * j4 + 2]) + bb.z;
      v[4 * j4 + 3] = __uint_as_float(acc[4 * j4 + 3]) + bb.w;
    }
    if (s == 7) {  // alpha head on CUDA cores, from the fp32 activations (run_nerf_helpers.py:114)
#pragma unroll
      for (int j4 = 0; j4 < 4; ++j4) {
        const float4 w = lds_f4(small_s + (kSmWAlpha + c0 + 4 * j4) * 4);
        alpha_part += fmaxf(v[4 * j4], 0.f) * w.x + fmaxf(v[4 * j4 + 1], 0.f) * w.y + fmaxf(v[4 * j4 + 2], 0.f) * w.z +
                      fmaxf(v[4 * j4 + 3], 0.f) * w.w;
      }
    }
    if (s == 9) {  // rgb head (run_nerf_helpers.py:122)
#pragma unroll 1
      for (int ch = 0; ch < 3; ++ch) {
        float a = 0.f;
#pragma unroll
        for (int j4 = 0; j4 < 4; ++j4) {
          const float4 w = lds_f4(small_s + (kSmWRgb + ch * 128 + c0 + 4 * j4) * 4);
          a += fmaxf(v[4 * j4], 0.f) * w.x + fmaxf(v[4 * j4 + 1], 0.f) * w.y + fmaxf(v[4 * j4 + 2], 0.f) * w.z +
               fmaxf(v[4 * j4 + 3], 0.f) * w.w;
        }
        if (ch == 0) rgb_part[0] += a; else if (ch == 1) rgb_part[1] += a; else rgb_part[2] += a;
      }
    }
    if (s == 8) {
#pragma unroll
      for (int i = 0; i < 8; ++i) pk[8 * b + i] = pack_bf16x2(v[2 * i], v[2 * i + 1]);
    } else {
#pragma unroll
      for (int i = 0; i < 8; ++i) pk[8 * b + i] = pack_relu_bf16x2(v[2 * i], v[2 * i + 1]);
    }
    if (kTrain) {
      // ReLU mask bits of these 16 columns (non-zero bf16 halves), layout: mask_bit_of_column() in mlp_common.cuh
      uint32_t m = 0;
#pragma unroll
      for (int i = 0; i < 8; ++i) m |= (((pk[8 * b + i] + 0x7FFF7FFFu) >> 15) & 0x00010001u) << i;
      mw[b >> 1] |= m << (8 * (b & 1));
    }
  }
}

template <bool kTrain>
__device__ __forceinline__ void ts_epilogue(const Params& p, uint8_t* smem, uint64_t* bar_acc, uint64_t* bar_act, uint64_t* bar_hi,
                                            uint32_t tmem_base, int warp, int lane, uint32_t cta_rank,
                                            int64_t first_it, int64_t n_iters, int64_t it_stride) {
  // epilogue warps are warps 0..15 (the MMA issuer sits in the highest warp: the scheduler favours high warp ids);
  // warp e: slot T = e/8, TMEM lane quarter q = e%4 (== warp%4), column half ch = (e%8)/4 of every accumulator half
  const int e = warp, T = e >> 3, q = e & 3, ch = (e & 7) >> 2;
  const int r = q * 32 + lane;
  const bool leader = (e & 7) == 0 && lane == 0;
  const uint32_t lane_base = (uint32_t)(q * 32) << 16;
  const uint32_t tA = tmem_base + lane_base + T * 256;    // A operand: 128 columns = 256 bf16 features
  const uint32_t tD = tA + 128 + ch * 64;                  // this thread's 64 accumulator columns
  const uint32_t bar_id = 1 + T;
  uint8_t* pe = smem + kSmemPE2 + T * kActChunk;
  // training: every epilogue warp stages and bulk-stores ITS 32 rows of a chunk image (a contiguous 4 KB piece) by itself
  uint8_t* stg = smem + kSmemStg2 + warp * 4096;
  uint8_t* mstg = smem + kSmemMask2 + warp * 512;
  const uint32_t stg_row = smem_u32(stg) + (uint32_t)(lane >> 3) * 1024u + (uint32_t)(lane & 7) * 128u, stg_x7 = (uint32_t)(lane & 7) << 4;
  const uint32_t mstg_row = smem_u32(mstg) + (uint32_t)lane * 16u;
  // shared-window addresses that the hot loop uses, made opaque to the compiler: it otherwise re-derives them from the (generic)
  // dynamic shared-memory pointer before every group of loads / stores (~20 instructions each time, ~100 per accumulator half)
  // instead of holding one register (render-only forward: 1,447 -> 1,476 TFLOP/s)
  uint32_t small_s = smem_u32(smem + kSmemSmall2);
  if (!kTrain) asm volatile("mov.u32 %0, %0;" : "+r"(small_s));       // (training: the register it pins costs more in spills: 882 vs 907 TFLOP/s)
  float4* xch = reinterpret_cast<float4*>(smem + kSmemXch2 + T * 2048) + r;
  uint32_t acc_phase = 0;
  long long t_accw = 0, t_begin = clock64();
  TRACE_DECL(1 + T);

  // two barriers per slot: a signal must be consumed by the issuer before the next one on the same barrier can fire
  // (parity waits); "A[128,256) ready" follows "A[0,128) ready" without any dependence on the issuer, so it has its own.
  // Every epilogue warp signals the issuer by itself (barrier count = 8 warps x 2 CTAs): no named barrier and no
  // single "leader" arrive on the critical path.  Each lane has fenced its own TMEM / smem accesses before.
  auto act_arrive = [&]() {
    __syncwarp();
    if (lane == 0) {
      if (cta_rank == 0) mbar_arrive(&bar_act[T]);
      else mbar_arrive_cluster(mapa_u32(smem_u32(&bar_act[T]), 0));
    }
  };
  auto hi_arrive = [&]() {
    __syncwarp();
    if (lane == 0) {
      if (cta_rank == 0) mbar_arrive(&bar_hi[T]);
      else mbar_arrive_cluster(mapa_u32(smem_u32(&bar_hi[T]), 0));
    }
  };
  auto wait_acc = [&]() {
    long long t0 = clock64();
    mbar_wait(&bar_acc[T], acc_phase);
    t_accw += clock64() - t0;
    acc_phase ^= 1;
    tc_fence_after();
  };

  for (int64_t it = first_it; it < n_iters; it += it_stride) {
    const int64_t tile = 4 * it + 2 * T + (int64_t)cta_rank;
    TRACE_ARM(blockIdx.x == 0 && leader && it == first_it + 3 * it_stride);
    const bool tile_valid = tile < p.n_tiles;
    const int64_t g = tile * kTile + r;
    const bool valid = tile_valid && g < p.pts.n_points;
    uint8_t* stash_tile = kTrain ? p.stash + (size_t)(tile_valid ? tile : 0) * kStashTileBytes : nullptr;

    // This warp's 32 packed bf16 rows (64 features of chunk `chunk`) -> its 4 KB staging piece -> one bulk store into the
    // stash.  Warp-local: no named barrier and no other warp's store on the path (the CTA-wide version - 32 KB per slot
    // behind two 256-thread barriers and a wait on the previous 36 KB store - cost ~1,700 cycles per accumulator half).
    // mask_layer >= 0: this warp's 512 B of ReLU mask words of that layer ([row][h][2 words]) go out with it.
    auto stage_out = [&](int chunk, const uint32_t (&pk)[32], int h, const uint32_t (&mw)[2], bool with_mask, int mask_layer) {
      if (lane == 0) tma_store_wait_read0();    // this warp's previous bulk stores have finished reading its staging pieces
      __syncwarp();
#pragma unroll
      for (int gq = 0; gq < 8; ++gq)      // chunk_off16(lane, gq) = row offset | ((gq ^ (lane & 7)) << 4)
        sts128(stg_row | (((uint32_t)gq << 4) ^ stg_x7), pk[4 * gq], pk[4 * gq + 1], pk[4 * gq + 2], pk[4 * gq + 3]);
      if (with_mask) sts64(mstg_row + h * 8, mw[0], mw[1]);
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0 && tile_valid) {
        // evict-first: the stash is read back a whole backward pass later, never out of L2 (0.664 -> 0.650 ms at P = 524,288)
        const uint64_t spol = l2_policy_evict_first();
        tma_store_1d_hint(stash_tile + (size_t)chunk * kActChunk + q * 4096, stg, 4096, spol);
        if (mask_layer >= 0) tma_store_1d_hint(stash_tile + kStashMaskOff + (size_t)mask_layer * 4096 + ch * 2048 + q * 512, mstg, 512, spol);
        tma_store_commit();
      }
    };

    float px = 0.f, py = 0.f, pz = 0.f, vx = 0.f, vy = 0.f, vz = 0.f;
    if (valid) {
      if (p.pts.rays) {
        const int64_t ray = g / p.pts.n_samples;
        const float* rp = p.pts.rays + ray * p.pts.ray_stride;
        const float zv = __ldg(p.pts.z_vals + g);
        px = __fadd_rn(__ldg(rp + 0), __fmul_rn(__ldg(rp + 3), zv));   // pts = o + d*z   run.py:1783
        py = __fadd_rn(__ldg(rp + 1), __fmul_rn(__ldg(rp + 4), zv));
        pz = __fadd_rn(__ldg(rp + 2), __fmul_rn(__ldg(rp + 5), zv));
        vx = __ldg(rp + p.pts.viewdir_offset);
        vy = __ldg(rp + p.pts.viewdir_offset + 1);
        vz = __ldg(rp + p.pts.viewdir_offset + 2);
      } else {
        const float* pp = p.pts.pts + g * p.pts.pts_stride;
        const float* dp = p.pts.dirs + g * p.pts.dirs_stride;
        px = __ldg(pp); py = __ldg(pp + 1); pz = __ldg(pp + 2);
        vx = __ldg(dp); vy = __ldg(dp + 1); vz = __ldg(dp + 2);
      }
    }
    if (kTrain) {
      if (leader) tma_store_wait_read0();      // PE(viewdir) of the previous tile has been stored
      named_bar_sync(bar_id, 256);
    }
    write_pe_half<10>(pe, r, px, py, pz, ch);
    fence_proxy_async_smem();
    tc_fence_before();
    act_arrive();                              // L0 may start: PE ready, accumulator free
    if (kTrain) {
      named_bar_sync(bar_id, 256);
      if (leader && tile_valid) {
        tma_store_1d_hint(stash_tile + (size_t)kStashPE * kActChunk, pe, kActChunk, l2_policy_evict_first());
        tma_store_commit();
      }
    }

    float alpha_part = 0.f, rgb_part[3] = {0.f, 0.f, 0.f};

    uint32_t pk[32];
#pragma unroll 1
    for (int s = 0; s < kNumSteps; ++s) {
      const int bias_i = (s < 8 ? kSmBiasTrunk + 256 * s : (s == 8 ? kSmBiasFeat : kSmBiasViews));
      const int stash_chunk = (s < 8 ? kStashH + 4 * s : (s == 8 ? kStashFeat : kStashHidden));
      const int nh = (s == 9) ? 1 : 2;
#pragma unroll 1
      for (int h = 0; h < nh; ++h) {
        uint32_t mw[2] = {0u, 0u};
        {
          uint32_t raw[4][16];
          TRACE(s * 16 + 4 * h + 0);
          wait_acc();
          TRACE(s * 16 + 4 * h + 1);
          // h == 1: all MMAs of this layer are complete -> the A operand may be overwritten; pk still holds half 0,
          // i.e. features [0,128) of the next layer's A operand (it could not be stored earlier: half 1 was reading A)
          if (h == 1) tmem_st32(tA + ch * 32, pk);
          load_half(tD, raw);
          if (h == 1) tmem_st_wait();
          TRACE(s * 16 + 4 * h + 2);
          tc_fence_before();
          // h == 0: accumulator drained -> half 1 may be issued;  h == 1: A[0,128) ready + accumulator drained -> the
          // next layer's first K chunks may start.  The math below is off the issuer's critical path.
          if (s < 9) act_arrive();
          TRACE(s * 16 + 4 * h + 3);
          math_half<kTrain>(raw, small_s, s, bias_i, h * 128 + ch * 64, pk, mw, alpha_part, rgb_part);
        }
        if (s < 9 && h == 1) {
          tmem_st32(tA + 64 + ch * 32, pk);
          if (s == 8) {                          // PE(viewdir) replaces PE(pts): L5 has consumed it
            if (kTrain) {                        // ... and the bulk store of PE(pts) into the stash has read it
              if (leader) tma_store_wait_read0();
              named_bar_sync(bar_id, 256);
            }
            write_pe_half<4>(pe, r, vx, vy, vz, ch);
            fence_proxy_async_smem();
          }
          tmem_st_wait();
          tc_fence_before();
          TRACE(s * 16 + 9);
          hi_arrive();                           // A[128,256) (and PE(viewdir)) ready
          if (kTrain && s == 8) {
            named_bar_sync(bar_id, 256);
            if (leader && tile_valid) {
              tma_store_1d_hint(stash_tile + (size_t)kStashVPE * kActChunk, pe, kActChunk, l2_policy_evict_first());
              tma_store_commit();
            }
          }
        }
        if (s == 9) {  // raw = (rgb, alpha): the two column halves of a row meet in shared memory
          if (ch == 1) *xch = make_float4(rgb_part[0], rgb_part[1], rgb_part[2], alpha_part);
          named_bar_sync(bar_id, 256);
          if (ch == 0 && valid) {
            const float4 o = *xch;
            p.raw[g] = make_float4(rgb_part[0] + o.x + lds_f1(small_s + kSmBRgb * 4), rgb_part[1] + o.y + lds_f1(small_s + (kSmBRgb + 1) * 4),
                                   rgb_part[2] + o.z + lds_f1(small_s + (kSmBRgb + 2) * 4), alpha_part + o.w + lds_f1(small_s + kSmBAlpha * 4));
          }
        }
        if (kTrain) {
          const bool last_half = (h == 1) || (s == 9);
          stage_out(stash_chunk + 2 * h + ch, pk, h, mw, s != 8, (s != 8 && last_half) ? (s == 9 ? 8 : s) : -1);
        }
      }
    }
  }
  if (kTrain && lane == 0) tma_store_wait_all0();
  if (blockIdx.x == 0 && warp == 0 && lane == 0) { g_prof[3] = t_accw; g_prof[5] = clock64() - t_begin; }
}

template <bool kTrain>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads2, 1) mlp_forward_pair_kernel(const Params p) {
  constexpr int kSlots = Ring2<kTrain>::kSlots, kLag = Ring2<kTrain>::kLag, kG = kGroupBars2;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ uint64_t bar_gfull[kG], bar_gempty[kG], bar_acc[2], bar_act[2], bar_hi[2];
  __shared__ uint32_t tmem_base_s;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = cluster_ctarank();
  const int64_t n_quads = (p.n_tiles + 3) / 4;
  const int64_t first_it = blockIdx.x >> 1, it_stride = gridDim.x >> 1;

  if (tid == 0) {
    for (int i = 0; i < kG; ++i) {
      mbar_init(&bar_gfull[i], rank == 0 ? 2 : 1);   // leader: own producer + peer relay
      mbar_init(&bar_gempty[i], 2);                  // multicast tcgen05.commit of the two issuer warps
    }
    for (int i = 0; i < 2; ++i) { mbar_init(&bar_acc[i], 1); mbar_init(&bar_act[i], 16); mbar_init(&bar_hi[i], 16); }   // act/hi: 8 epilogue warps x 2 CTAs
    mbar_fence_init();
  }
  if (warp == 17) tmem_alloc_2cta(&tmem_base_s, 512);
  {  // biases + alpha / rgb heads -> shared memory (read ~10^3 times per tile by the epilogue warps)
    const float4* src = reinterpret_cast<const float4*>(p.packed + kSmallOff);
    float4* dst = reinterpret_cast<float4*>(smem + kSmemSmall2);
    for (int i = tid; i < kSmallFloats / 4; i += kThreads2) dst[i] = __ldg(src + i);
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();          // barriers of both CTAs initialised before any remote arrive / multicast commit
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;

  if (warp < 16) {
    reg_inc<104>();   // 16 x 32 x 104 + 4 x 32 x 40 <= 640 x 96 (the CTA's register pool)
    ts_epilogue<kTrain>(p, smem, bar_acc, bar_act, bar_hi, tmem_base, warp, lane, rank, first_it, n_quads, it_stride);
  } else {
    reg_dec<64>();   // 16 x 32 x 104 + 4 x 32 x 64 = 640 x 96: the issuer loop must not spill (local-memory loads on its critical path)
    if (warp == 16) {
      // ===================== TMA producer: this CTA's 64 rows of every (layer, N-half, K chunk), once per quad =====================
      if (lane == 0) {
        uint32_t j = 0; int slot = 0;
        for (int64_t it = first_it; it < n_quads; it += it_stride) {
          int cbase = 0;
          for (int s = 0; s < kNumSteps; ++s) {
            const int n = step_nchunks(s);
            const int nh = (s == 9) ? 1 : 2;
            for (int h = 0; h < nh; ++h, ++j) {
              if (j >= (uint32_t)kLag) mbar_wait(&bar_gempty[(j - kLag) % kG], ((j - kLag) / kG) & 1u);   // the slots are free again
              uint64_t* full = &bar_gfull[j % kG];
              mbar_arrive_expect_tx(full, (uint32_t)n * kSlotBytes2);
              for (int ci = 0; ci < n; ++ci) {
                const uint8_t* src = p.packed + fwd_chunk_off(cbase + ci) + (size_t)(2 * h + (int)rank) * kSlotBytes2;
                tma_load_1d(smem + kSmemW2 + slot * kSlotBytes2, src, kSlotBytes2, full);
                if (++slot == kSlots) slot = 0;
              }
            }
            cbase += n;
          }
        }
      }
    } else if (warp == 19 && rank == 1) {
      // ===================== relay: tell the leader that this CTA's part of a group has landed =====================
      if (lane == 0) {
        uint32_t j = 0;
        for (int64_t it = first_it; it < n_quads; it += it_stride) {
          for (int c = 0; c < kGroupsPerIter2; ++c, ++j) {
            mbar_wait(&bar_gfull[j % kG], (j / kG) & 1u);
            mbar_arrive_cluster(mapa_u32(smem_u32(&bar_gfull[j % kG]), 0));
          }
        }
      }
    } else if (warp >= 18 && rank == 0) {
      // ===================== MMA issuers (leader CTA): warp 18 -> tile slot X, warp 19 -> tile slot Y =====================
      // Two independent issuers: while one sits in an mbarrier wait (~200 cycles even when it succeeds) the other
      // keeps the tensor pipe fed.  The order X.h0, Y.h0, X.h1, Y.h1 emerges from the dependencies.
      // The issue code is straight-line per (layer, N-half) block and spill-free: every cycle this warp loses delays the MMAs.
      const int T = warp - 18;
      uint32_t act_phase = 0, hi_phase = 0, j = 0;
      PROF_DECL;
      TRACE_DECL(0);
      const uint32_t idesc = umma_idesc_bf16(256, 128, 0, 0);
      const uint32_t sbase = smem_u32(smem);
      const uint32_t tA = tmem_base + T * 256;        // A operand columns of this slot
      const uint32_t tDm = tA + 128;                  // accumulator half
      const uint32_t pe_lo = desc_lo2(sbase + kSmemPE2 + T * kActChunk);
      const uint32_t w_lo = desc_lo2(sbase + kSmemW2);
      const uint32_t w_end = w_lo + kSlots * (kSlotBytes2 >> 4);
      uint32_t bpos = w_lo;                           // ring position (descriptor low word) of the next K chunk
      auto next_slot = [&](uint32_t b) { b += (kSlotBytes2 >> 4); return b == w_end ? w_lo : b; };
      for (int64_t it = first_it; it < n_quads; it += it_stride) {
        TRACE_ARM(blockIdx.x == 0 && T == 0 && lane == 0 && it == first_it + 3 * it_stride);
#pragma unroll 1
        for (int s = 0; s < kNumSteps; ++s) {
          const int nh = (s == 9) ? 1 : 2;
#pragma unroll 1
          for (int h = 0; h < nh; ++h, ++j) {
            // chunk order inside the block: [PE (s = 0, 5)] [A cols 0..63: K chunks 1, 2] [A cols 64..127: K chunks 3, 4] [PE(viewdir) (s = 9)]
            const bool pe_first = (s == 0) || (s == 5);
            const uint32_t b0 = bpos;                               // PE chunk (if pe_first)
            const uint32_t b1 = pe_first ? next_slot(b0) : b0;      // K chunk 1
            const uint32_t b2 = next_slot(b1), b3 = next_slot(b2), b4 = next_slot(b3);
            const uint32_t b5 = next_slot(b4);                      // PE(viewdir) chunk (s == 9) / next block
            bpos = (s == 0) ? b1 : ((s == 9) ? next_slot(b5) : b5);
            uint64_t* gempty = &bar_gempty[j % kG];
            PROF_T0;
            mbar_wait(&bar_gfull[j % kG], (j / kG) & 1u);   // both CTAs' parts of the group have landed (normally long ago)
            PROF_ADD(t_full);
            TRACE(s * 64 + h * 32 + 0);
            PROF_T0;
            mbar_wait(&bar_act[T], act_phase);              // s = 0: PE ready; h = 0: A[0,128) ready; always: accumulator drained
            TRACE(s * 64 + h * 32 + 1);
            PROF_ADD(t_act);
            act_phase ^= 1;
            tc_fence_after();
            if (elect_one_sync()) {
              if (pe_first) {
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) mma2_ss(tDm, pe_lo + kk * 2, b0 + kk * 2, idesc, kk > 0 ? 1u : 0u);
              }
              if (s > 0) {
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) mma2_ts(tDm, tA + kk * 8, b1 + kk * 2, idesc, (pe_first || kk > 0) ? 1u : 0u);
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) mma2_ts(tDm, tA + 32 + kk * 8, b2 + kk * 2, idesc, 1u);
              } else {
                umma_commit_2cta(gempty, 3);
                umma_commit_2cta(&bar_acc[T], 3);
              }
            }
            __syncwarp();
            if (s > 0) {
              if (h == 0) {   // A[128,256) is signalled separately by the previous layer's epilogue
                TRACE(s * 64 + h * 32 + 2);
                PROF_T0;
                mbar_wait(&bar_hi[T], hi_phase);
                TRACE(s * 64 + h * 32 + 3);
                PROF_ADD(t_act);
                hi_phase ^= 1;
                tc_fence_after();
              }
              if (elect_one_sync()) {
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) mma2_ts(tDm, tA + 64 + kk * 8, b3 + kk * 2, idesc, 1u);
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) mma2_ts(tDm, tA + 96 + kk * 8, b4 + kk * 2, idesc, 1u);
                if (s == 9) {   // viewdir PE has 27 (< 32) channels: two K steps
                  mma2_ss(tDm, pe_lo, b5, idesc, 1u);
                  mma2_ss(tDm, pe_lo + 2, b5 + 2, idesc, 1u);
                }
                umma_commit_2cta(gempty, 3);            // this issuer is done with the group (both CTAs)
                umma_commit_2cta(&bar_acc[T], 3);
              }
              __syncwarp();
            }
            TRACE(s * 64 + h * 32 + 4);
          }
        }
      }
      PROF_STORE;
    }
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();          // the peer may still signal our barriers / read our smem until it is done too
  if (warp == 17) tmem_dealloc_2cta(tmem_base, 512);
}

int check_points(const char* who, const mvip_points* pts) {
  MVIP_REQUIRE(pts, MVIP_E_INVALID, "%s: null mvip_points", who);
  if (pts->rays) {
    MVIP_REQUIRE(pts->z_vals && pts->n_rays >= 0 && pts->n_samples >= 1, MVIP_E_INVALID, "%s: rays mode needs z_vals", who);
    MVIP_REQUIRE(pts->ray_stride >= 6 && pts->viewdir_offset >= 0 && pts->viewdir_offset + 3 <= pts->ray_stride,
                 MVIP_E_INVALID, "%s: bad ray_stride/viewdir_offset (%d, %d)", who, pts->ray_stride, pts->viewdir_offset);
    MVIP_REQUIRE(pts->n_points == pts->n_rays * pts->n_samples, MVIP_E_INVALID, "%s: n_points != n_rays*n_samples", who);
  } else {
    MVIP_REQUIRE(pts->pts && pts->dirs && pts->pts_stride >= 3 && pts->dirs_stride >= 0, MVIP_E_INVALID,
                 "%s: points mode needs pts and dirs", who);
  }
  MVIP_REQUIRE(pts->n_points >= 0, MVIP_E_INVALID, "%s: negative n_points", who);
  return MVIP_OK;
}

}  // namespace

extern "C" {

int mvip_debug_profile(unsigned long long* out16) {
  MVIP_CUDA_OK(cudaDeviceSynchronize());
  MVIP_CUDA_OK(cudaMemcpyFromSymbol(out16, g_prof, sizeof(unsigned long long) * 16));
  return MVIP_OK;
}

// copies the event trace of a -DMVIP_TRACE build (3 logs x 1024 x (code, clock)); n_out[3] = entries per log
int mvip_debug_trace(long long* out, int* n_out) {
#ifdef MVIP_TRACE
  MVIP_CUDA_OK(cudaDeviceSynchronize());
  MVIP_CUDA_OK(cudaMemcpyFromSymbol(out, g_trace, sizeof(long long) * 3 * 1024 * 2));
  MVIP_CUDA_OK(cudaMemcpyFromSymbol(n_out, g_trace_n, sizeof(int) * 3));
  return MVIP_OK;
#else
  (void)out; (void)n_out;
  mvip_set_error("mvip_debug_trace: library built without -DMVIP_TRACE");
  return MVIP_E_UNSUPPORTED;
#endif
}

size_t mvip_mlp_stash_bytes(int64_t n_points) { return (size_t)mlp::num_tiles(n_points) * mlp::kStashTileBytes; }

int mvip_mlp_forward(const void* packed, const mvip_points* pts, float* raw, void* stash, void* stream) {
  MVIP_REQUIRE(pts, MVIP_E_INVALID, "mvip_mlp_forward: null mvip_points");
  if (pts->n_points == 0) return MVIP_OK;
  MVIP_REQUIRE(packed && raw, MVIP_E_INVALID, "mvip_mlp_forward: null pointer");
  int rc = check_points("mvip_mlp_forward", pts);
  if (rc) return rc;
  MVIP_REQUIRE(mvip_aligned(packed, 1024) && mvip_aligned(raw, 16) && (!stash || mvip_aligned(stash, 1024)),
               MVIP_E_INVALID, "mvip_mlp_forward: packed/stash need 1024-byte and raw 16-byte alignment");
  if (pts->n_points == 0) return MVIP_OK;
  Params p;
  p.packed = static_cast<const uint8_t*>(packed);
  p.pts = *pts;
  p.raw = reinterpret_cast<float4*>(raw);
  p.stash = static_cast<uint8_t*>(stash);
  p.n_tiles = mlp::num_tiles(pts->n_points);
  const int64_t n_quads = (p.n_tiles + 3) / 4;
  const int max_clusters = mvip_num_sms() / 2;
  const int grid2 = 2 * (int)(n_quads < max_clusters ? n_quads : max_clusters);
  const size_t smem2 = (stash ? kSmemBytes2Train : kSmemBytes2Infer) + 1024;
  if (stash) {
    MVIP_SMEM_OPT_IN(mlp_forward_pair_kernel<true>, smem2);
    mlp_forward_pair_kernel<true><<<grid2, kThreads2, smem2, (cudaStream_t)stream>>>(p);
  } else {
    MVIP_SMEM_OPT_IN(mlp_forward_pair_kernel<false>, smem2);
    mlp_forward_pair_kernel<false><<<grid2, kThreads2, smem2, (cudaStream_t)stream>>>(p);
  }
  MVIP_LAUNCH_OK("mlp_forward_pair_kernel");
  return MVIP_OK;
}

}  // extern "C"
