// Tile helpers of the mma.sync training attention kernels, shared by attention_train.cu (Transformer-XL) and
// attention_bert_train.cu (the remix encoder): (q + bias) A-fragments, the content scores of a 64-key tile, the rel-pos
// term through a warp-private "skewed" shared-memory strip, quad reductions and the attention-dropout bits.
//
// Strip geometry: for a 64 x 64 tile whose rel-pos window is the 128 Rk rows D0-64 .. D0+63 (sR0 | sR1), warp w multiplies
// its 16 query rows with window columns 16w .. 16w+79 and stores the 16 x 80 result; strip[r][64 + r - jl] is then the
// term of (query row 16w + r, key jl of the tile) at distance D0 + 16w + r - jl.
#pragma once
#include <cuda_fp16.h>
#include "mma_sync.cuh"
#include "train_kernels.cuh"

namespace dmg {

constexpr int SKEW_LD = 84;    // elements per row of the warp-private skew strip (80 used)
typedef __half skew_t;         // fp16 strip (11-bit mantissa: rounding 5e-4 of the position term) - 2.7 KB per warp
constexpr float ATT_LOG2E = 1.4426950408889634f;
constexpr float ATT_LN2 = 0.6931471805599453f;

// two floats -> packed fp16 pair, saturating to +-65504 instead of overflowing to infinity (lo = first argument)
__device__ __forceinline__ uint32_t pack_half2_sat(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}

// (q + bias) A-fragments: a[ks] covers k = 16*ks..16*ks+15; registers hold (g,2t..),(g+8,2t..),(g,2t+8..),(g+8,2t+8..)
__device__ __forceinline__ uint32_t add_bias2(uint32_t w, float b0, float b1) { return pack_bf16x2(bf16lo(w) + b0, bf16hi(w) + b1); }
__device__ __forceinline__ void q_frags(uint32_t sQ, int w, int lane, const LaneOff& L, const float* __restrict__ u, const float* __restrict__ v,
                                        uint32_t (&qu)[4][4], uint32_t (&qv)[4][4]) {
  const int t = lane & 3;
#pragma unroll
  for (int ks = 0; ks < 4; ks++) {
    uint32_t a[4];
    frag_a(sQ, 16 * w, ks, L, a);
    const int c0 = 16 * ks + 2 * t;
    const float u0 = u[c0], u1 = u[c0 + 1], u8 = u[c0 + 8], u9 = u[c0 + 9];
    const float v0 = v[c0], v1 = v[c0 + 1], v8 = v[c0 + 8], v9 = v[c0 + 9];
    qu[ks][0] = add_bias2(a[0], u0, u1); qu[ks][1] = add_bias2(a[1], u0, u1);
    qu[ks][2] = add_bias2(a[2], u8, u9); qu[ks][3] = add_bias2(a[3], u8, u9);
    qv[ks][0] = add_bias2(a[0], v0, v1); qv[ks][1] = add_bias2(a[1], v0, v1);
    qv[ks][2] = add_bias2(a[2], v8, v9); qv[ks][3] = add_bias2(a[3], v8, v9);
  }
}

// position term of the warp's 16 query rows x the 80 window columns 16w .. 16w+79 into the strip (ends with __syncwarp)
__device__ __forceinline__ void position_strip(const uint32_t (&qv)[4][4], uint32_t sR0, uint32_t sR1, skew_t* skew, int w, int lane,
                                               const LaneOff& L) {
  const int g = lane >> 2, t = lane & 3;
#pragma unroll
  for (int p = 0; p < 5; p++) {
    const int wc = 16 * w + 16 * p;                 // first window column of this pair of n-tiles
    const uint32_t sR = (wc < 64 ? sR0 : sR1) + (wc & 63) * 128;
    float acc[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
#pragma unroll
    for (int ks = 0; ks < 4; ks++) {
      uint32_t r[4];
      frag_b(sR, 0, ks, L, r);
      mma_bf16(acc[0], qv[ks], r[0], r[1]);
      mma_bf16(acc[1], qv[ks], r[2], r[3]);
    }
#pragma unroll
    for (int h = 0; h < 2; h++) {
      const int col = 16 * p + 8 * h + 2 * t;
      *(uint32_t*)(skew + g * SKEW_LD + col) = pack_half2_sat(acc[h][0], acc[h][1]);
      *(uint32_t*)(skew + (g + 8) * SKEW_LD + col) = pack_half2_sat(acc[h][2], acc[h][3]);
    }
  }
  __syncwarp();
}

// skewed read: the strip's term of accumulator element (nt, e) of this lane (row g + 8*(e>>1), key 8*nt + 2*t + (e&1))
__device__ __forceinline__ float skew_at(const skew_t* skew, int g, int t, int nt, int e) {
  const int r = g + 8 * (e >> 1), jl = 8 * nt + 2 * t + (e & 1);
  return __half2float(skew[r * SKEW_LD + 64 + r - jl]);
}

// s[nt][e] = (q + u) K^T of the warp's 16 query rows x the tile's 64 keys
__device__ __forceinline__ void content_scores(const uint32_t (&qu)[4][4], uint32_t sK, const LaneOff& L, float (&s)[8][4]) {
#pragma unroll
  for (int nt = 0; nt < 8; nt++) { s[nt][0] = 0.f; s[nt][1] = 0.f; s[nt][2] = 0.f; s[nt][3] = 0.f; }
#pragma unroll
  for (int ks = 0; ks < 4; ks++) {
#pragma unroll
    for (int np = 0; np < 4; np++) {
      uint32_t r[4];
      frag_b(sK, 16 * np, ks, L, r);
      mma_bf16(s[2 * np], qu[ks], r[0], r[1]);
      mma_bf16(s[2 * np + 1], qu[ks], r[2], r[3]);
    }
  }
}

// s[nt][e] = AC + BD (unscaled) for the warp's 16 query rows x the tile's 64 keys (Transformer-XL: line 1 only).
// sR0 / sR1: the two Rk tiles of the window (distances D0-64..D0-1 and D0..D0+63).
__device__ __forceinline__ void scores_tile(const uint32_t (&qu)[4][4], const uint32_t (&qv)[4][4], uint32_t sK, uint32_t sR0,
                                            uint32_t sR1, skew_t* skew, int w, int lane, const LaneOff& L, float (&s)[8][4]) {
  const int g = lane >> 2, t = lane & 3;
  position_strip(qv, sR0, sR1, skew, w, lane, L);
  content_scores(qu, sK, L, s);
#pragma unroll
  for (int nt = 0; nt < 8; nt++)
#pragma unroll
    for (int e = 0; e < 4; e++) s[nt][e] += skew_at(skew, g, t, nt, e);
  __syncwarp();
}

__device__ __forceinline__ float quad_max(float v) {
  v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 1));
  return fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 2));
}
__device__ __forceinline__ float quad_sum(float v) {
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  return v + __shfl_xor_sync(0xffffffffu, v, 2);
}

// keep factors (0 or drop_scale) of this lane's 4 elements of n-tile nt; drop_base[r] = pair index of (row r, key 0) + t,
// pair index of (bh, row, key j) = ((bh*T + row)*S + j) / 2 (S even) - the layout dmg_train_dropout_mask exports
__device__ __forceinline__ void attn_keep(uint32_t thresh, uint32_t seed, float scale, const uint32_t (&drop_base)[2], int j0, int nt,
                                          float (&keep)[4]) {
#pragma unroll
  for (int r = 0; r < 2; r++) {
    const uint32_t hb = drop_pair_bits(seed, drop_base[r] + (uint32_t)(j0 >> 1) + 4 * nt);
    keep[2 * r] = ((hb & 0xFFFFu) >= thresh) ? scale : 0.f;
    keep[2 * r + 1] = ((hb >> 16) >= thresh) ? scale : 0.f;
  }
}

}  // namespace dmg
