// Flash attention with the Transformer-XL relative-position term for TRAINING (forward + backward), bf16 tensor cores
// (mma.sync m16n8k16, fp32 accumulate), no score tensor in HBM.
//
// Replaces fastai MultiHeadRelativeAttention._apply_attention under autograd (SURVEY.md App. A.3):
//   AC = (q+u) K^T, BD = _line_shift((q+v) Rk^T), P = dropout(softmax((AC+BD)/sqrt(Dh) + mask)), out = P V
// and its backward.  _line_shift is index arithmetic (App. A.4): BD[i,j] = (q_i+v) . Rk[dist], dist = (M+i) - j, for the
// causal region (everything else is masked), so for a 64-query x 64-key tile the needed Rk rows are the 127 distances
// D0-63 .. D0+63 (D0 = M + i0 - j0): each warp multiplies its 16 query rows with its 80-distance window and reads the
// result back "skewed" through a warp-private shared-memory strip.
//
// Layout: q|k|v of the current segment in one [B*T, 3*H*64] bf16 matrix (the QKV GEMM output), k|v of the memory rows in
// a [B*M, 2*H*64] matrix (the memory K/V GEMM output; mems are hidden states in training, re-projected every step with
// the current weights), Rk [M+T, H*64].  T and M are multiples of 64.
//
// Backward = three kernels, none with floating-point atomics on activations:
//   attn_delta_kernel : delta_i = dO_i . O_i
//   attn_bwd_dq_kernel: query-tile owner; recomputes P, forms dS, accumulates dQ (content + position parts -> du, dv),
//                       writes dS in (row, distance) coordinates for the dRk GEMM (ds_dist) and spills P (dropped) and dS
//   attn_bwd_dkv_lite_kernel: key-tile owner; accumulates dK, dV from the spilled P and dS tiles
#include "kernels.cuh"
#include "launch.cuh"
#include "attention_train_common.cuh"

namespace dmg {

namespace {

constexpr int DSK_LD = 88;     // bf16 per row of the warp-private dS strip (80 used); 176-byte rows keep ldmatrix aligned
constexpr float LOG2E = ATT_LOG2E;
constexpr float LN2 = ATT_LN2;

struct MaskP {
  int M, mem_count, win, k;
};
// key j (context coordinates, 0..M+T) visible from query i (0..T)?
__device__ __forceinline__ bool visible(const MaskP& mp, int i, int j) {
  if (j < mp.M) return j >= mp.M - mp.mem_count;
  const int jx = j - mp.M;
  if (jx == 0) return true;                                  // window_mask: column 0 is always visible
  return mp.k == 1 ? jx <= i : jx < (i / mp.win) * mp.win;   // (1,1) causal; (w,0): strictly earlier windows
}

// pointer to the 64-key tile jt of K (kv=0) or V (kv=1) for stream b, head h
__device__ __forceinline__ const bf16* kv_tile_ptr(const AttnTrainArgs& a, int b, int h, int jt, int kv, long long* ld) {
  const int HD = a.H * 64;
  const int j0 = jt * 64;
  if (j0 < a.M) {
    *ld = a.ldm;
    return a.kv_m + ((long long)b * a.M + j0) * a.ldm + kv * HD + h * 64;
  }
  *ld = a.ldx;
  return a.qkv_x + ((long long)b * a.T + (j0 - a.M)) * a.ldx + (1 + kv) * HD + h * 64;
}

// =============================================================================================
// forward
// =============================================================================================
// Pipeline: K / V tiles in an NST-deep ring (cp.async groups, prefetch distance NST-1), Rk tiles in an (NST+1)-slot ring
// (tile rt lives in slot rt % (NST+1)): iteration jt needs Rk tiles rt_hi = (M+i0)/64 - jt and rt_hi - 1, and each
// iteration's load group brings exactly one new Rk tile (the very first brings two).
constexpr int ATT_NST = 3;                 // backward (dq) kernel
constexpr int ATT_NR = ATT_NST + 1;
constexpr int FWD_NST = 2;                 // forward: 2 stages -> 74.75 KB -> three CTAs (12 warps) per SM
constexpr int FWD_NR = FWD_NST + 1;
constexpr int FWD_SMEM = TILE_BYTES /*Q*/ + 2 * FWD_NST * TILE_BYTES /*K,V ring*/ + FWD_NR * TILE_BYTES /*R ring*/ +
                         4 * 16 * SKEW_LD * (int)sizeof(skew_t);

__global__ void __launch_bounds__(128, 3) attn_train_fwd_kernel(const AttnTrainArgs a) {
  extern __shared__ __align__(128) uint8_t smem[];
  uint8_t* sQ = smem;
  uint8_t* sKV = sQ + TILE_BYTES;                   // stage s: K at sKV + 2*s*TILE, V right behind it
  uint8_t* sR = sKV + 2 * FWD_NST * TILE_BYTES;
  skew_t* skew_all = (skew_t*)(sR + FWD_NR * TILE_BYTES);
  const int tid = threadIdx.x, w = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  skew_t* skew = skew_all + w * 16 * SKEW_LD;
  LaneOff L;
  lane_off_init(L, lane, w);

  const int nT = a.T / 64;
  const int it = nT - 1 - (blockIdx.x % nT);        // heavy (late) query tiles first
  const int bh = blockIdx.x / nT, b = bh / a.H, h = bh % a.H;
  const int i0 = it * 64, HD = a.H * 64, S = a.M + a.T;
  const MaskP mp = {a.M, a.mem_count, a.win, a.k};
  const int jt_lo = (a.M - a.mem_count) / 64, jt_hi = (a.M + i0) / 64;
  const int rt_top = (a.M + i0) / 64;               // rt_hi of iteration jt is rt_top - jt

  auto load_stage = [&](int jt) {                   // one cp.async group: K, V of key tile jt and the new Rk tile(s)
    if (jt <= jt_hi) {
      const int st = (jt - jt_lo) % FWD_NST;
      long long ld;
      const bf16* kp = kv_tile_ptr(a, b, h, jt, 0, &ld);
      tile_load_async(sKV + 2 * st * TILE_BYTES, kp, ld, tid, 128);
      const bf16* vp = kv_tile_ptr(a, b, h, jt, 1, &ld);
      tile_load_async(sKV + (2 * st + 1) * TILE_BYTES, vp, ld, tid, 128);
      const int rt_hi = rt_top - jt;
      if (jt == jt_lo) tile_load_async(sR + (rt_hi % FWD_NR) * TILE_BYTES, a.rk + (long long)rt_hi * 64 * HD + h * 64, HD, tid, 128);
      if (rt_hi > 0) tile_load_async(sR + ((rt_hi - 1) % FWD_NR) * TILE_BYTES, a.rk + (long long)(rt_hi - 1) * 64 * HD + h * 64, HD, tid, 128);
    }
    cp_async_commit();
  };

  tile_load_async(sQ, a.qkv_x + ((long long)b * a.T + i0) * a.ldx + h * 64, a.ldx, tid, 128);
  cp_async_commit();
#pragma unroll
  for (int s = 0; s < FWD_NST - 1; s++) load_stage(jt_lo + s);
  cp_async_wait<FWD_NST - 1>();                     // Q has landed (the stage groups may still be in flight)
  __syncthreads();
  uint32_t qu[4][4], qv[4][4];
  q_frags(smem_u32(sQ), w, lane, L, a.u + h * 64, a.v + h * 64, qu, qv);

  float o[8][4];
#pragma unroll
  for (int nt = 0; nt < 8; nt++) { o[nt][0] = 0.f; o[nt][1] = 0.f; o[nt][2] = 0.f; o[nt][3] = 0.f; }
  float m_run[2] = {-INFINITY, -INFINITY}, l_run[2] = {0.f, 0.f};
  const float c = a.scale * LOG2E;
  const int row_g[2] = {i0 + 16 * w + g, i0 + 16 * w + g + 8};
  // dropout pair index of (row, key j) = ((bh*T + row)*S + j) / 2 = drop_base[row] + j/2   (S is even; this thread's j/2 = j0/2 + 4*nt + t)
  const uint32_t drop_base[2] = {(uint32_t)((((long long)bh * a.T + row_g[0]) * S) >> 1) + t,
                                 (uint32_t)((((long long)bh * a.T + row_g[1]) * S) >> 1) + t};

  for (int jt = jt_lo; jt <= jt_hi; jt++) {
    const int j0 = jt * 64;
    const int rt_hi = rt_top - jt, rt_lo = rt_hi > 0 ? rt_hi - 1 : 0;
    cp_async_wait<FWD_NST - 2>();                    // tile jt has landed
    __syncthreads();                                 // ... for everybody; and everybody is done with tile jt-1
    load_stage(jt + FWD_NST - 1);                    // refill the stage tile jt-1 used
    const int st = (jt - jt_lo) % FWD_NST;
    uint8_t* sK = sKV + 2 * st * TILE_BYTES;
    uint8_t* sV = sK + TILE_BYTES;

    float s[8][4];
    scores_tile(qu, qv, smem_u32(sK), smem_u32(sR + (rt_lo % FWD_NR) * TILE_BYTES), smem_u32(sR + (rt_hi % FWD_NR) * TILE_BYTES),
                skew, w, lane, L, s);
    const bool need_mask = (j0 + 63 >= a.M) || (j0 < a.M - a.mem_count);
    // running max kept on the RAW scores (the scale is positive); exp2((s - m) * c) is one FFMA + one MUFU per element
    float mx[2] = {-INFINITY, -INFINITY};
    if (need_mask) {
#pragma unroll
      for (int nt = 0; nt < 8; nt++)
#pragma unroll
        for (int e = 0; e < 4; e++)
          if (!visible(mp, row_g[e >> 1], j0 + 8 * nt + 2 * t + (e & 1))) s[nt][e] = -INFINITY;
    }
#pragma unroll
    for (int nt = 0; nt < 8; nt++) {
      mx[0] = fmaxf(mx[0], fmaxf(s[nt][0], s[nt][1]));
      mx[1] = fmaxf(mx[1], fmaxf(s[nt][2], s[nt][3]));
    }
    float alpha[2], neg_mc[2];
#pragma unroll
    for (int r = 0; r < 2; r++) {
      const float m_new = fmaxf(m_run[r], quad_max(mx[r]));
      alpha[r] = (m_new == -INFINITY) ? 1.f : ex2_fast((m_run[r] - m_new) * c);
      neg_mc[r] = (m_new == -INFINITY) ? 0.f : -m_new * c;
      m_run[r] = m_new;
    }
    float rs[2] = {0.f, 0.f};
    uint32_t pa[4][4];                               // dropped probabilities as A fragments (keys = k dimension)
#pragma unroll
    for (int nt = 0; nt < 8; nt++) {
      float p[4];
#pragma unroll
      for (int e = 0; e < 4; e++) {
        p[e] = ex2_fast(fmaf(s[nt][e], c, neg_mc[e >> 1]));
        rs[e >> 1] += p[e];
      }
      if (a.drop_thresh) {
#pragma unroll
        for (int r = 0; r < 2; r++) {
          const uint32_t hb = drop_pair_bits(a.drop_seed, drop_base[r] + (uint32_t)(j0 >> 1) + 4 * nt);
          p[2 * r] = ((hb & 0xFFFFu) >= a.drop_thresh) ? p[2 * r] * a.drop_scale : 0.f;
          p[2 * r + 1] = ((hb >> 16) >= a.drop_thresh) ? p[2 * r + 1] * a.drop_scale : 0.f;
        }
      }
      pa[nt >> 1][(nt & 1) * 2] = pack_bf16x2(p[0], p[1]);
      pa[nt >> 1][(nt & 1) * 2 + 1] = pack_bf16x2(p[2], p[3]);
    }
#pragma unroll
    for (int r = 0; r < 2; r++) l_run[r] = l_run[r] * alpha[r] + rs[r];
#pragma unroll
    for (int nt = 0; nt < 8; nt++) {
      o[nt][0] *= alpha[0]; o[nt][1] *= alpha[0]; o[nt][2] *= alpha[1]; o[nt][3] *= alpha[1];
    }
    const uint32_t sVa = smem_u32(sV);
#pragma unroll
    for (int ks = 0; ks < 4; ks++) {
#pragma unroll
      for (int np = 0; np < 4; np++) {
        uint32_t r[4];
        frag_b_t(sVa, np, 16 * ks, L, r);
        mma_bf16(o[2 * np], pa[ks], r[0], r[1]);
        mma_bf16(o[2 * np + 1], pa[ks], r[2], r[3]);
      }
    }
  }
#pragma unroll
  for (int r = 0; r < 2; r++) {
    const float l = quad_sum(l_run[r]);
    const float inv = l > 0.f ? 1.f / l : 0.f;
    bf16* orow = a.out + ((long long)b * a.T + row_g[r]) * HD + h * 64;
#pragma unroll
    for (int nt = 0; nt < 8; nt++)
      *(uint32_t*)(orow + 8 * nt + 2 * t) = pack_bf16x2(o[nt][2 * r] * inv, o[nt][2 * r + 1] * inv);
    if (t == 0) a.lse[(long long)bh * a.T + row_g[r]] = (m_run[r] * c + log2f(l)) * LN2;
  }
}

// =============================================================================================
// backward
// =============================================================================================
__global__ void __launch_bounds__(256) attn_delta_kernel(const bf16* __restrict__ out, const bf16* __restrict__ dout,
                                                         float* __restrict__ delta, int rows, int T, int H) {
  const int warp = (blockIdx.x * 256 + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= rows) return;
  const int b = warp / T, i = warp % T;
  const uint32_t* o = (const uint32_t*)(out + (long long)warp * H * 64);
  const uint32_t* d = (const uint32_t*)(dout + (long long)warp * H * 64);
  for (int h = 0; h < H; h++) {
    const uint32_t x = o[h * 32 + lane], y = d[h * 32 + lane];
    float s = bf16lo(x) * bf16lo(y) + bf16hi(x) * bf16hi(y);
    s = warp_sum(s);
    if (lane == 0) delta[((long long)b * H + h) * T + i] = s;
  }
}

// recompute P (normalised), dP and dS for one tile; returns ds (scaled gradient wrt AC+BD) in s
__device__ __forceinline__ void bwd_tile_math(const AttnTrainArgs& a, const MaskP& mp, float (&s)[8][4], float (&dpd)[8][4],
                                              const int (&row_g)[2], const float (&lse2)[2], const float (&dl)[2], int j0,
                                              const uint32_t (&drop_base)[2], int t, bf16* p_row0, bf16* p_row1, bf16* ds_row0,
                                              bf16* ds_row1) {
  // p_row*/ds_row*: the dropped probabilities and dS of this thread's two rows are also written (bf16 pairs) at column
  // offset 8*nt + 2*t of the given row pointers - the input of the dK/dV kernel (attn_bwd_dkv_lite_kernel)
  const float c = a.scale * LOG2E;
  const bool need_mask = (j0 + 63 >= a.M) || (j0 < a.M - a.mem_count);
#pragma unroll
  for (int nt = 0; nt < 8; nt++) {
    float keep[4] = {1.f, 1.f, 1.f, 1.f};
    if (a.drop_thresh) attn_keep(a.drop_thresh, a.drop_seed, a.drop_scale, drop_base, j0, nt, keep);
#pragma unroll
    for (int e = 0; e < 4; e++) {
      const int r = e >> 1;
      float p = ex2_fast(s[nt][e] * c - lse2[r]);
      if (need_mask && !visible(mp, row_g[r], j0 + 8 * nt + 2 * t + (e & 1))) p = 0.f;
      const float dp = dpd[nt][e] * keep[e];
      s[nt][e] = p * (dp - dl[r]) * a.scale;
      keep[e] *= p;                                 // keep[] now holds the dropped probability
    }
    *(uint32_t*)(p_row0 + 8 * nt + 2 * t) = pack_bf16x2(keep[0], keep[1]);
    *(uint32_t*)(p_row1 + 8 * nt + 2 * t) = pack_bf16x2(keep[2], keep[3]);
    *(uint32_t*)(ds_row0 + 8 * nt + 2 * t) = pack_bf16x2(s[nt][0], s[nt][1]);
    *(uint32_t*)(ds_row1 + 8 * nt + 2 * t) = pack_bf16x2(s[nt][2], s[nt][3]);
  }
}

// Same with the probabilities SAVED by the tcgen05 forward (AttnTrainArgs::p_save / m_save): pw[nt][r] holds the bf16 pair
// (row r of this thread, keys 8*nt + 2*t, +1) relative to the block maximum; fac[r] = exp(m_save*scale - lse) rescales it.
// Masked keys were saved as zeros, so no visibility test is needed.
__device__ __forceinline__ void bwd_tile_math_saved(const AttnTrainArgs& a, const uint32_t (&pw)[8][2], const float (&fac)[2],
                                                    float (&s)[8][4], float (&dpd)[8][4], const float (&dl)[2], int j0,
                                                    const uint32_t (&drop_base)[2], int t, bf16* p_row0, bf16* p_row1, bf16* ds_row0,
                                                    bf16* ds_row1) {
#pragma unroll
  for (int nt = 0; nt < 8; nt++) {
    float keep[4] = {1.f, 1.f, 1.f, 1.f};
    if (a.drop_thresh) attn_keep(a.drop_thresh, a.drop_seed, a.drop_scale, drop_base, j0, nt, keep);
#pragma unroll
    for (int e = 0; e < 4; e++) {
      const int r = e >> 1;
      const float p = ((e & 1) ? bf16hi(pw[nt][r]) : bf16lo(pw[nt][r])) * fac[r];
      const float dp = dpd[nt][e] * keep[e];
      s[nt][e] = p * (dp - dl[r]) * a.scale;
      keep[e] *= p;                                 // keep[] now holds the dropped probability
    }
    // p_row0 is never null: the branch only keeps ptxas from hoisting the caller's loads of the next tile's words above these
    // stores, which needs a second set of pw registers (without it the kernel spills at 255 registers)
    if (p_row0) {
      *(uint32_t*)(p_row0 + 8 * nt + 2 * t) = pack_bf16x2(keep[0], keep[1]);
      *(uint32_t*)(p_row1 + 8 * nt + 2 * t) = pack_bf16x2(keep[2], keep[3]);
      *(uint32_t*)(ds_row0 + 8 * nt + 2 * t) = pack_bf16x2(s[nt][0], s[nt][1]);
      *(uint32_t*)(ds_row1 + 8 * nt + 2 * t) = pack_bf16x2(s[nt][2], s[nt][3]);
    }
  }
}

constexpr int DQ_SMEM = 2 * ATT_NST * TILE_BYTES /*K,V ring (Q and dO are staged in its last stage first)*/ + ATT_NR * TILE_BYTES /*R*/ +
                        4 * 16 * SKEW_LD * (int)sizeof(skew_t) + 4 * 16 * DSK_LD * 2;

// PS = true: the probabilities come from the forward's p_save / m_save (no AC / BD / skew / exp recomputation, no (q+u),
// (q+v) fragments, no skew strip): 2 ring stages, <= 168 registers -> three CTAs per SM instead of two.
constexpr int DQ_PS_NST = 3;
constexpr int DQ_PS_MINB = 2;
constexpr int DQ_PS_SMEM = 2 * DQ_PS_NST * TILE_BYTES + (DQ_PS_NST + 1) * TILE_BYTES + 4 * 16 * DSK_LD * 2;

template <bool PS>
__global__ void __launch_bounds__(128, PS ? DQ_PS_MINB : 1) attn_bwd_dq_kernel(const AttnTrainBwdArgs ba) {
  constexpr int NST = PS ? DQ_PS_NST : ATT_NST, NR = NST + 1;
  const AttnTrainArgs& a = ba.f;
  extern __shared__ __align__(128) uint8_t smem[];
  uint8_t* sKV = smem;
  uint8_t* sR = sKV + 2 * NST * TILE_BYTES;
  skew_t* skew_all = (skew_t*)(sR + NR * TILE_BYTES);
  bf16* dsk_all = PS ? (bf16*)skew_all : (bf16*)(skew_all + 4 * 16 * SKEW_LD);
  const int tid = threadIdx.x, w = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  skew_t* skew = skew_all + w * 16 * SKEW_LD;
  LaneOff L;
  lane_off_init(L, lane, w);
  bf16* dsk = dsk_all + w * 16 * DSK_LD;

  const int nT = a.T / 64;
  const int it = nT - 1 - (blockIdx.x % nT);
  const int bh = blockIdx.x / nT, b = bh / a.H, h = bh % a.H;
  const int i0 = it * 64, HD = a.H * 64, S = a.M + a.T;
  const MaskP mp = {a.M, a.mem_count, a.win, a.k};
  const long long bhT = (long long)bh * a.T;
  const int jt_lo = (a.M - a.mem_count) / 64, jt_hi = (a.M + i0) / 64;
  const int rt_top = (a.M + i0) / 64;

  auto load_stage = [&](int jt) {
    if (jt <= jt_hi) {
      const int st = (jt - jt_lo) % NST;
      long long ld;
      const bf16* kp = kv_tile_ptr(a, b, h, jt, 0, &ld);
      tile_load_async(sKV + 2 * st * TILE_BYTES, kp, ld, tid, 128);
      const bf16* vp = kv_tile_ptr(a, b, h, jt, 1, &ld);
      tile_load_async(sKV + (2 * st + 1) * TILE_BYTES, vp, ld, tid, 128);
      const int rt_hi = rt_top - jt;
      if (jt == jt_lo) tile_load_async(sR + (rt_hi % NR) * TILE_BYTES, a.rk + (long long)rt_hi * 64 * HD + h * 64, HD, tid, 128);
      if (rt_hi > 0) tile_load_async(sR + ((rt_hi - 1) % NR) * TILE_BYTES, a.rk + (long long)(rt_hi - 1) * 64 * HD + h * 64, HD, tid, 128);
    }
    cp_async_commit();
  };

  // stage Q and dO through the LAST ring stage (the prologue fills stages 0 .. NST-2) to build the A fragments
  uint8_t* sQst = sKV + 2 * (NST - 1) * TILE_BYTES;
  uint8_t* sdOst = sQst + TILE_BYTES;
  if (!PS) tile_load_async(sQst, a.qkv_x + ((long long)b * a.T + i0) * a.ldx + h * 64, a.ldx, tid, 128);
  tile_load_async(sdOst, ba.dout + ((long long)b * a.T + i0) * HD + h * 64, HD, tid, 128);
  cp_async_commit();
#pragma unroll
  for (int s2 = 0; s2 < NST - 1; s2++) load_stage(jt_lo + s2);
  for (int i = lane; i < 16 * DSK_LD; i += 32) dsk[i] = __float2bfloat16_rn(0.f);   // off-band entries stay zero
  cp_async_wait<NST - 1>();
  __syncthreads();
  uint32_t qu[4][4], qv[4][4], dof[4][4];
  if (!PS) q_frags(smem_u32(sQst), w, lane, L, a.u + h * 64, a.v + h * 64, qu, qv);
#pragma unroll
  for (int ks = 0; ks < 4; ks++) frag_a(smem_u32(sdOst), 16 * w, ks, L, dof[ks]);

  const int row_g[2] = {i0 + 16 * w + g, i0 + 16 * w + g + 8};
  const uint32_t drop_base[2] = {(uint32_t)(((bhT + row_g[0]) * S) >> 1) + t, (uint32_t)(((bhT + row_g[1]) * S) >> 1) + t};
  float lse2[2], dl[2];
#pragma unroll
  for (int r = 0; r < 2; r++) {
    lse2[r] = a.lse[bhT + row_g[r]] * LOG2E;
    dl[r] = ba.delta[bhT + row_g[r]];
  }
  // saved probabilities: this thread's 16 words of a tile (2 rows x 8 n-tiles).  They are consumed by the tile math in the
  // first half of an iteration, and the next tile's words are requested right behind it, so the loads fly during the second
  // half (strip, dQ contractions, dS_dist copy) without a second set of registers.
  const int nblk = S >> 6;
  const uint32_t* psrc[2] = {nullptr, nullptr};
  const float* msrc[2] = {nullptr, nullptr};
  uint32_t pw[8][2];
  float mblk[2] = {0.f, 0.f};
  if (PS) {
#pragma unroll
    for (int r = 0; r < 2; r++) {
      psrc[r] = (const uint32_t*)(a.p_save + (bhT + row_g[r]) * S) + t;
      msrc[r] = a.m_save + (bhT + row_g[r]) * nblk;
    }
#pragma unroll
    for (int nt = 0; nt < 8; nt++)
#pragma unroll
      for (int r = 0; r < 2; r++) pw[nt][r] = __ldg(psrc[r] + ((jt_lo * 64) >> 1) + 4 * nt);
#pragma unroll
    for (int r = 0; r < 2; r++) mblk[r] = __ldg(msrc[r] + jt_lo);
  }
  float dq_ac[8][4], dq_bd[8][4];
#pragma unroll
  for (int nt = 0; nt < 8; nt++)
#pragma unroll
    for (int e = 0; e < 4; e++) { dq_ac[nt][e] = 0.f; dq_bd[nt][e] = 0.f; }

  // distances that no key tile of this row produces (beyond the oldest visible key) must read as zero in the dRk GEMM
  {
    const long long HS = (long long)a.H * S;
    for (int r = 0; r < 16; r++) {
      const int i = i0 + 16 * w + r;
      const int first = a.M + i - jt_lo * 64 + 1;
      bf16* drow = ba.ds_dist + ((long long)b * a.T + i) * HS + (long long)h * S;
      for (int dd = first + lane; dd < S; dd += 32) drow[dd] = __float2bfloat16_rn(0.f);
    }
  }

  const long long HS = (long long)a.H * S;
  bf16* const ds_row_base = ba.ds_dist + ((long long)b * a.T + i0 + 16 * w) * HS + (long long)h * S;
  for (int jt = jt_lo; jt <= jt_hi; jt++) {
    const int j0 = jt * 64;
    const int D0 = a.M + i0 - j0;
    const int rt_hi = D0 / 64, rt_lo = rt_hi > 0 ? rt_hi - 1 : 0;
    cp_async_wait<NST - 2>();
    __syncthreads();                                 // tile jt visible to all; tile jt-1 (and the Q/dO staging) released
    load_stage(jt + NST - 1);
    const int st = (jt - jt_lo) % NST;
    uint8_t* sK = sKV + 2 * st * TILE_BYTES;
    uint8_t* sV = sK + TILE_BYTES;
    const uint32_t sR0 = smem_u32(sR + (rt_lo % NR) * TILE_BYTES), sR1 = smem_u32(sR + (rt_hi % NR) * TILE_BYTES);

    float s[8][4], dpd[8][4];
    if (!PS) scores_tile(qu, qv, smem_u32(sK), sR0, sR1, skew, w, lane, L, s);
    // dPd = dO V^T
#pragma unroll
    for (int nt = 0; nt < 8; nt++) { dpd[nt][0] = 0.f; dpd[nt][1] = 0.f; dpd[nt][2] = 0.f; dpd[nt][3] = 0.f; }
    const uint32_t sVa = smem_u32(sV), sKa = smem_u32(sK);
#pragma unroll
    for (int ks = 0; ks < 4; ks++) {
#pragma unroll
      for (int np = 0; np < 4; np++) {
        uint32_t r[4];
        frag_b(sVa, 16 * np, ks, L, r);
        mma_bf16(dpd[2 * np], dof[ks], r[0], r[1]);
        mma_bf16(dpd[2 * np + 1], dof[ks], r[2], r[3]);
      }
    }
    if (PS) {
      float fac[2];
#pragma unroll
      for (int r = 0; r < 2; r++) fac[r] = ex2_fast(mblk[r] * (a.scale * LOG2E) - lse2[r]);
      const long long o0 = (bhT + row_g[0]) * S + j0, o1 = (bhT + row_g[1]) * S + j0;
      bwd_tile_math_saved(a, pw, fac, s, dpd, dl, j0, drop_base, t, ba.p_buf + o0, ba.p_buf + o1, ba.ds_buf + o0, ba.ds_buf + o1);
      if (jt < jt_hi) {                              // next tile's words and maxima
#pragma unroll
        for (int nt = 0; nt < 8; nt++)
#pragma unroll
          for (int r = 0; r < 2; r++) pw[nt][r] = __ldg(psrc[r] + ((j0 + 64) >> 1) + 4 * nt);
#pragma unroll
        for (int r = 0; r < 2; r++) mblk[r] = __ldg(msrc[r] + jt + 1);
      }
    } else {                                         // spill P (dropped) and dS for the dK/dV kernel: [b*H+h][T][S] bf16
      const long long o0 = (bhT + row_g[0]) * S + j0, o1 = (bhT + row_g[1]) * S + j0;
      bwd_tile_math(a, mp, s, dpd, row_g, lse2, dl, j0, drop_base, t, ba.p_buf + o0, ba.p_buf + o1, ba.ds_buf + o0, ba.ds_buf + o1);
    }

    // dS into the skewed strip (bf16): strip[row][64 + row - jl]
#pragma unroll
    for (int nt = 0; nt < 8; nt++) {
      const int jl = 8 * nt + 2 * t;
      dsk[g * DSK_LD + 64 + g - jl] = __float2bfloat16_rn(s[nt][0]);
      dsk[g * DSK_LD + 63 + g - jl] = __float2bfloat16_rn(s[nt][1]);
      dsk[(g + 8) * DSK_LD + 72 + g - jl] = __float2bfloat16_rn(s[nt][2]);
      dsk[(g + 8) * DSK_LD + 71 + g - jl] = __float2bfloat16_rn(s[nt][3]);
    }
    // dQ_ac += dS K
    uint32_t dsa[4][4];
#pragma unroll
    for (int ks = 0; ks < 4; ks++) {
      dsa[ks][0] = pack_bf16x2(s[2 * ks][0], s[2 * ks][1]);
      dsa[ks][1] = pack_bf16x2(s[2 * ks][2], s[2 * ks][3]);
      dsa[ks][2] = pack_bf16x2(s[2 * ks + 1][0], s[2 * ks + 1][1]);
      dsa[ks][3] = pack_bf16x2(s[2 * ks + 1][2], s[2 * ks + 1][3]);
    }
#pragma unroll
    for (int ks = 0; ks < 4; ks++) {
#pragma unroll
      for (int np = 0; np < 4; np++) {
        uint32_t r[4];
        frag_b_t(sKa, np, 16 * ks, L, r);
        mma_bf16(dq_ac[2 * np], dsa[ks], r[0], r[1]);
        mma_bf16(dq_ac[2 * np + 1], dsa[ks], r[2], r[3]);
      }
    }
    __syncwarp();
    // dQ_bd += strip (16 x 80) * Rwin (80 x 64)
    const uint32_t dska = smem_u32(dsk);
#pragma unroll
    for (int ks = 0; ks < 5; ks++) {
      uint32_t af[4];
      ldsm_x4(dska + (lane & 15) * (DSK_LD * 2) + (2 * ks + (lane >> 4)) * 16, af);
      const int wc = 16 * w + 16 * ks;
      const uint32_t sRx = wc < 64 ? sR0 : sR1;
#pragma unroll
      for (int np = 0; np < 4; np++) {
        uint32_t r[4];
        frag_b_t(sRx, np, wc & 63, L, r);
        mma_bf16(dq_bd[2 * np], af, r[0], r[1]);
        mma_bf16(dq_bd[2 * np + 1], af, r[2], r[3]);
      }
    }
    // dS in (row, distance) coordinates: strip column col <-> distance D0 - 64 + 16w + col; valid band [1+r, 64+r]
    {
      bf16* drow = ds_row_base + (D0 - 64 + 16 * w) + 1 + lane;      // row 16w of this tile, band start of r = 0
      const bf16* srow = dsk + 1 + lane;
      if (D0 - 64 + 16 * w + 1 >= 0) {                                 // every distance of the band is >= 0 (all but the diagonal tiles)
#pragma unroll
        for (int r = 0; r < 16; r++) {
          drow[r] = srow[r * DSK_LD + r];
          drow[r + 32] = srow[r * DSK_LD + r + 32];
          drow += HS;
        }
      } else {
        for (int r = 0; r < 16; r++) {
#pragma unroll
          for (int half = 0; half < 2; half++) {
            const int col = 1 + r + lane + 32 * half;
            if (D0 - 64 + 16 * w + col >= 0) drow[r + 32 * half] = srow[r * DSK_LD + r + 32 * half];
          }
          drow += HS;
        }
      }
    }
    __syncwarp();
  }

  // dq = content part + position part; du / dv = their column sums over all rows
#pragma unroll
  for (int r = 0; r < 2; r++) {
    bf16* qrow = ba.dqkv_x + ((long long)b * a.T + row_g[r]) * a.ldx + h * 64;
#pragma unroll
    for (int nt = 0; nt < 8; nt++)
      *(uint32_t*)(qrow + 8 * nt + 2 * t) =
          pack_bf16x2(dq_ac[nt][2 * r] + dq_bd[nt][2 * r], dq_ac[nt][2 * r + 1] + dq_bd[nt][2 * r + 1]);
  }
#pragma unroll
  for (int nt = 0; nt < 8; nt++) {
#pragma unroll
    for (int e = 0; e < 2; e++) {
      float su = dq_ac[nt][e] + dq_ac[nt][e + 2], sv = dq_bd[nt][e] + dq_bd[nt][e + 2];
#pragma unroll
      for (int o = 4; o < 32; o <<= 1) {
        su += __shfl_xor_sync(0xffffffffu, su, o);
        sv += __shfl_xor_sync(0xffffffffu, sv, o);
      }
      if (g == 0) {
        atomicAdd(ba.du + h * 64 + 8 * nt + 2 * t + e, su);
        atomicAdd(ba.dv + h * 64 + 8 * nt + 2 * t + e, sv);
      }
    }
  }
}

// dK / dV from the spilled P and dS tiles (no recomputation of the scores): key-tile owner, loops over the query tiles that
// see it; per iteration four 64x64 tiles (P, dS, dO, Q) arrive through a double-buffered cp.async ring.
// ALL_QUERIES: every query tile sees every key (the remix encoder's unmasked attention) instead of the causal range.
constexpr int LITE_SMEM = 2 * 4 * TILE_BYTES;

template <bool ALL_QUERIES>
__global__ void __launch_bounds__(128) attn_bwd_dkv_lite_kernel(const AttnTrainBwdArgs ba) {
  const AttnTrainArgs& a = ba.f;
  extern __shared__ __align__(128) uint8_t smem[];
  const int tid = threadIdx.x, w = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  LaneOff L;
  lane_off_init(L, lane, w);
  const int nS = (a.M + a.T) / 64;
  const int jt = blockIdx.x % nS;
  const int bh = blockIdx.x / nS, b = bh / a.H, h = bh % a.H;
  const int j0 = jt * 64, HD = a.H * 64, S = a.M + a.T;
  const long long bhT = (long long)bh * a.T;
  bf16 *dk_dst, *dv_dst;
  long long ldd;
  if (j0 < a.M) {
    ldd = a.ldm;
    dk_dst = ba.dkv_m + ((long long)b * a.M + j0) * a.ldm + h * 64;
    dv_dst = dk_dst + HD;
  } else {
    ldd = a.ldx;
    dk_dst = ba.dqkv_x + ((long long)b * a.T + (j0 - a.M)) * a.ldx + HD + h * 64;
    dv_dst = dk_dst + HD;
  }
  if (j0 < a.M - a.mem_count) {
    for (int i = tid; i < 64 * 32; i += 128) {
      const int r = i >> 5, cidx = (i & 31) * 2;
      *(uint32_t*)(dk_dst + (long long)r * ldd + cidx) = 0u;
      *(uint32_t*)(dv_dst + (long long)r * ldd + cidx) = 0u;
    }
    return;
  }
  const int nT = a.T / 64;
  const int it_lo = (ALL_QUERIES || j0 < a.M) ? 0 : (j0 - a.M) / 64;
  auto load_stage = [&](int it) {
    if (it < nT) {
      uint8_t* st = smem + ((it - it_lo) & 1) * 4 * TILE_BYTES;
      const int i0 = it * 64;
      tile_load_async(st, ba.p_buf + (bhT + i0) * S + j0, S, tid, 128);
      tile_load_async(st + TILE_BYTES, ba.ds_buf + (bhT + i0) * S + j0, S, tid, 128);
      tile_load_async(st + 2 * TILE_BYTES, ba.dout + ((long long)b * a.T + i0) * HD + h * 64, HD, tid, 128);
      tile_load_async(st + 3 * TILE_BYTES, a.qkv_x + ((long long)b * a.T + i0) * a.ldx + h * 64, a.ldx, tid, 128);
    }
    cp_async_commit();
  };
  load_stage(it_lo);
  float dk[8][4], dv[8][4];
#pragma unroll
  for (int nt = 0; nt < 8; nt++)
#pragma unroll
    for (int e = 0; e < 4; e++) { dk[nt][e] = 0.f; dv[nt][e] = 0.f; }
  const float* ub = a.u + h * 64;
  for (int it = it_lo; it < nT; it++) {
    cp_async_wait<0>();
    __syncthreads();
    load_stage(it + 1);
    uint8_t* st = smem + ((it - it_lo) & 1) * 4 * TILE_BYTES;
    uint8_t* sQ = st + 3 * TILE_BYTES;
    // q -> q + u in place, each warp its own 16 query rows (the B operand of the dK contraction)
#pragma unroll
    for (int ks = 0; ks < 4; ks++) {
      const int c0 = 16 * ks + 2 * t;
#pragma unroll
      for (int hh = 0; hh < 2; hh++) {
#pragma unroll
        for (int rr = 0; rr < 2; rr++) {
          uint32_t* ptr = (uint32_t*)(sQ + tile_off(16 * w + g + 8 * rr, 2 * ks + hh) + 4 * t);
          *ptr = pack_bf16x2(bf16lo(*ptr) + ub[c0 + 8 * hh], bf16hi(*ptr) + ub[c0 + 8 * hh + 1]);
        }
      }
    }
    __syncthreads();
    const uint32_t sPa = smem_u32(st), sdSa = smem_u32(st + TILE_BYTES), sdOa = smem_u32(st + 2 * TILE_BYTES), sQua = smem_u32(sQ);
#pragma unroll
    for (int ks = 0; ks < 4; ks++) {
      uint32_t ap[4], as[4];
      frag_a_t(sPa, 16 * ks, L, ap);
      frag_a_t(sdSa, 16 * ks, L, as);
#pragma unroll
      for (int np = 0; np < 4; np++) {
        uint32_t r[4];
        frag_b_t(sdOa, np, 16 * ks, L, r);
        mma_bf16(dv[2 * np], ap, r[0], r[1]);
        mma_bf16(dv[2 * np + 1], ap, r[2], r[3]);
        frag_b_t(sQua, np, 16 * ks, L, r);
        mma_bf16(dk[2 * np], as, r[0], r[1]);
        mma_bf16(dk[2 * np + 1], as, r[2], r[3]);
      }
    }
  }
#pragma unroll
  for (int r = 0; r < 2; r++) {
    const long long ro = (long long)(16 * w + g + 8 * r) * ldd;
#pragma unroll
    for (int nt = 0; nt < 8; nt++) {
      *(uint32_t*)(dk_dst + ro + 8 * nt + 2 * t) = pack_bf16x2(dk[nt][2 * r], dk[nt][2 * r + 1]);
      *(uint32_t*)(dv_dst + ro + 8 * nt + 2 * t) = pack_bf16x2(dv[nt][2 * r], dv[nt][2 * r + 1]);
    }
  }
}

int check_args(const AttnTrainArgs& a) {
  DMG_CHECK(a.T > 0 && a.T % 64 == 0 && a.M % 64 == 0 && a.mem_count % 64 == 0 && a.mem_count <= a.M,
            "training attention: T=%d, M=%d, mem_count=%d must be multiples of 64", a.T, a.M, a.mem_count);
  DMG_CHECK((a.win == 1 && a.k == 1) || (a.win >= 1 && a.k == 0),
            "training attention: window_mask (%d,%d) unsupported (only (1,1) and (w,0), the pairs rand_window_mask draws)", a.win, a.k);
  DMG_CHECK(a.ldx % 8 == 0 && (a.M == 0 || a.ldm % 8 == 0), "training attention: row strides must be multiples of 8");
  DMG_CHECK((long long)a.B * a.H * a.T * (a.M + a.T) < (1ll << 32), "training attention: dropout index exceeds 32 bits");
  return 0;
}

}  // namespace

int attn_train_delta(const AttnTrainBwdArgs& ba, cudaStream_t st) {
  const AttnTrainArgs& a = ba.f;
  const int rows = a.B * a.T;
  return launch_np(attn_delta_kernel, dim3((rows * 32 + 255) / 256), dim3(256), 0, st, (const bf16*)a.out, ba.dout, ba.delta, rows, a.T,
                   a.H);
}

int attn_bwd_dkv_all_queries(const AttnTrainBwdArgs& ba, cudaStream_t st) {
  const AttnTrainArgs& a = ba.f;
  DMG_CHECK(a.M == 0 && ba.p_buf && ba.ds_buf, "attn_bwd_dkv_all_queries: needs M = 0 and the spilled P / dS tiles");
  static bool configured = false;
  if (!configured) {
    DMG_CUDA_OK(cudaFuncSetAttribute(attn_bwd_dkv_lite_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, LITE_SMEM));
    configured = true;
  }
  return launch_np(attn_bwd_dkv_lite_kernel<true>, dim3(a.B * a.H * (a.T / 64)), dim3(128), (size_t)LITE_SMEM, st, ba);
}

int attn_train_fwd(const AttnTrainArgs& a, cudaStream_t st) {
  if (check_args(a)) return -2;
  if (attn_train_fwd_tc_supported(a)) return attn_train_fwd_tc(a, st);
  static bool configured = false;
  if (!configured) {
    DMG_CUDA_OK(cudaFuncSetAttribute(attn_train_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, FWD_SMEM));
    configured = true;
  }
  return launch_np(attn_train_fwd_kernel, dim3(a.B * a.H * (a.T / 64)), dim3(128), (size_t)FWD_SMEM, st, a);
}

int attn_train_bwd(const AttnTrainBwdArgs& ba, cudaStream_t st) {
  const AttnTrainArgs& a = ba.f;
  if (check_args(a)) return -2;
  DMG_CHECK(ba.p_buf && ba.ds_buf, "training attention backward: the P / dS workspaces p_buf and ds_buf are required");
  static bool configured = false;
  if (!configured) {
    DMG_CUDA_OK(cudaFuncSetAttribute(attn_bwd_dq_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, DQ_SMEM));
    DMG_CUDA_OK(cudaFuncSetAttribute(attn_bwd_dq_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, DQ_PS_SMEM));
    DMG_CUDA_OK(cudaFuncSetAttribute(attn_bwd_dkv_lite_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, LITE_SMEM));
    configured = true;
  }
  if (attn_train_delta(ba, st)) return -1;
  if (attn_bwd_dq_tc_supported(ba)) {   // saved probabilities, 128-aligned shapes: dQ on tcgen05
    if (attn_bwd_dq_tc(ba, st)) return -1;
  } else if (a.p_save && a.m_save) {   // the tcgen05 forward saved the probabilities: no score recomputation
    if (launch_np(attn_bwd_dq_kernel<true>, dim3(a.B * a.H * (a.T / 64)), dim3(128), (size_t)DQ_PS_SMEM, st, ba)) return -1;
  } else if (launch_np(attn_bwd_dq_kernel<false>, dim3(a.B * a.H * (a.T / 64)), dim3(128), (size_t)DQ_SMEM, st, ba)) {
    return -1;
  }
  if (attn_bwd_dkv_tc_supported(ba)) return attn_bwd_dkv_tc(ba, st);   // spilled tiles + (q+u): tcgen05 contraction
  return launch_np(attn_bwd_dkv_lite_kernel<false>, dim3(a.B * a.H * ((a.M + a.T) / 64)), dim3(128), (size_t)LITE_SMEM, st, ba);
}

}  // namespace dmg
