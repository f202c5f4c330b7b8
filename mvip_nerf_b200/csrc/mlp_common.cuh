// mlp_common.cuh — layouts shared by the fused NeRF-MLP kernels (pack / forward / backward).
//
// Network (DS_NeRF/run_nerf_helpers.py:74-127, create_nerf defaults run.py:1487-1489):
//   pts(3)->PE 63, views(3)->PE 27; L0 63->256, L1..L4 256->256, [cat PE] L5 319->256, L6,L7 256->256,
//   alpha 256->1, feature 256->256, [cat PE_v] views 283->128 (ReLU), rgb 128->3.
//
// Operand format everywhere: "chunk image" = R rows x 64 bf16 (128 B/row), 128-byte swizzle
// (chunk_off16 in common.cuh).  A weight chunk has R = 256 (or 128) output rows and 64 input columns
// (K-major B operand); an activation chunk has R = 128 points and 64 features (K-major A operand
// for forward/dgrad; the same bytes are an MN-major operand for wgrad).
#pragma once
#include "common.cuh"

namespace mlp {

constexpr int kTile = 128;                 // points per tile (= TMEM lanes)
constexpr uint32_t kActChunk = 128 * 128;  // bytes of one activation chunk image
constexpr uint32_t kW256 = 256 * 128;      // bytes of a 256-row weight chunk
constexpr uint32_t kW128 = 128 * 128;

// ---- packed blob ---------------------------------------------------------------------------
constexpr int kFwdChunks = 39;   // 34 x 256-row + 5 x 128-row (views layer)
constexpr int kBwdChunks = 34;   // transposed weights for the dgrad chain, all 256-row
constexpr size_t kFwdBytes = 34 * (size_t)kW256 + 5 * (size_t)kW128;
constexpr size_t kBwdBytes = 34 * (size_t)kW256;
// fp32 tail: biases and the two CUDA-core heads
constexpr int kSmBiasTrunk = 0;       // [8][256]
constexpr int kSmBiasFeat = 2048;     // [256]
constexpr int kSmBiasViews = 2304;    // [128]
constexpr int kSmWAlpha = 2432;       // [256]
constexpr int kSmBAlpha = 2688;       // [1] (+3 pad)
constexpr int kSmWRgb = 2692;         // [3][128]
constexpr int kSmBRgb = 3076;         // [3] (+1 pad)
constexpr int kSmallFloats = 3080;
constexpr size_t kSmallOff = kFwdBytes + kBwdBytes;
constexpr size_t kPackedBytes = kSmallOff + kSmallFloats * sizeof(float);

__host__ __device__ inline size_t fwd_chunk_off(int c) { return c < 34 ? (size_t)c * kW256 : 34 * (size_t)kW256 + (size_t)(c - 34) * kW128; }
__host__ __device__ inline uint32_t fwd_chunk_bytes(int c) { return c < 34 ? kW256 : kW128; }

// ---- parameter order of the C ABI ------------------------------------------------------------
__host__ __device__ constexpr int kPW(int layer) { return 2 * layer; }       // pts_linears.{layer}.weight
constexpr int kPViewsW = 16, kPViewsB = 17, kPFeatW = 18, kPFeatB = 19, kPAlphaW = 20, kPAlphaB = 21, kPRgbW = 22,
              kPRgbB = 23;

struct ParamPtrs {
  const float* p[MVIP_MLP_NUM_PARAMS];
};
struct GradPtrs {
  float* p[MVIP_MLP_NUM_PARAMS];
};

// ---- forward stash (per 128-point tile) ---------------------------------------------------------
// chunk images, 16 KB each: 0 = PE(pts); 1+4(l-1)+j = h_l chunk j (l = 1..8); 33..36 = feature;
// 37 = PE(viewdir); 38,39 = hidden (views layer output).  Then ReLU bit masks, 4 KB per layer (layer 8 = hidden):
// [9 layers][2 column halves ch][128 rows][2 N-halves h][2 x u32]: the two words cover the 64 columns 128 h + 64 ch + [0, 64)
// (layer 8 has h = 0 only).  One epilogue warp owns (ch, 32 rows): a contiguous 512 B piece.
constexpr int kStashChunks = 40;
constexpr int kStashPE = 0, kStashH = 1, kStashFeat = 33, kStashVPE = 37, kStashHidden = 38;
constexpr size_t kStashMaskOff = (size_t)kStashChunks * kActChunk;
constexpr size_t kStashMaskBytes = 9 * 128 * 32;
constexpr size_t kStashTileBytes = kStashMaskOff + kStashMaskBytes;

// ---- dZ stash written by the dgrad chain (per tile) ---------------------------------------------
// 0,1 = d hidden_pre; 2..5 = d feature; 6+4t+j = dZ_{7-t} chunk j (t = 0..7 -> layers 7..0)
constexpr int kDzChunks = 38;
constexpr int kDzHidden = 0, kDzFeat = 2, kDzTrunk = 6;
constexpr size_t kDzTileBytes = (size_t)kDzChunks * kActChunk;

// ReLU mask word layout: bit of column j (0..31) inside its 32-column mask word.  The forward epilogue derives
// the bits from packed bf16 pairs of two 16-column blocks, hence the interleave.
__host__ __device__ inline int mask_bit_of_column(int j) { return 16 * (j & 1) + 8 * (j >> 4) + ((j & 15) >> 1); }

// u32 index of the two mask words of (layer, row r, N-half h, column half ch) inside a tile's mask block
__host__ __device__ inline int mask_word_index(int layer, int r, int h, int ch) { return layer * 1024 + ch * 512 + r * 4 + h * 2; }

inline int64_t num_tiles(int64_t n_points) { return (n_points + kTile - 1) / kTile; }

#ifdef __CUDACC__
// ---- positional encoding (forward encoder and the input-gradient chain) ------------------------
// sin/cos(x * 2^k): the phase is reduced in "turns" with a two-float product x/(2 pi) (power-of-two
// scaling and the fractional part are exact), then sin.approx/cos.approx on [-pi, pi].
__device__ __forceinline__ void pe_axis(float x, int L, float* s, float* c) {
  const float kInv2PiHi = 0.15915494f;
  const float kInv2PiLo = 3.0918538e-09f;  // 1/(2 pi) - (double)kInv2PiHi
  float u_hi = x * kInv2PiHi;
  float u_lo = fmaf(x, kInv2PiHi, -u_hi) + x * kInv2PiLo;
  float scale = 1.f;
#pragma unroll
  for (int k = 0; k < 10; ++k) {
    if (k < L) {
      float a = u_hi * scale;
      float ph = (a - rintf(a)) + u_lo * scale;
      float ang = ph * 6.283185307179586f;
      s[k] = __sinf(ang);
      c[k] = __cosf(ang);
      scale *= 2.f;
    }
  }
}
#endif

}  // namespace mlp
