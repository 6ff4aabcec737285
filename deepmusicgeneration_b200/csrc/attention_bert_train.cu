// Flash attention of the remix (masked-BERT) encoder for TRAINING: forward with attention dropout and the saved
// log-sum-exp, and the query-tile half of its backward; bf16 mma.sync (m16n8k16, fp32 accumulate), T a multiple of 64.
//
// Replaces MemMultiHeadRelativeAttentionKV._apply_attention (deep_music_remix.py:2078-2104, mem_len 0, r_mask=False) under
// autograd.  _line_shift without a mask keeps three lines alive (SURVEY.md App. A.4):
//   line 1 (j <= i)   : BD[i,j] = (q_i + v) . Rk[i - j]
//   line 2 (j == i+1) : 0
//   line 3 (j >  i+1) : BD[i,j] = (q_{i+1} + v) . Rk[T + 1 + i - j]
// Each line is a skewed strip over its own 128-row Rk window (attention_train_common.cuh): line 1 at D0 = i0 - j0, line 3
// at D0 = T + 1 + i0 - j0 with the NEXT query rows.  The windows run past both ends of the table, so Rk must read as zero
// for rows -64 .. T+127, and q|k|v needs one readable row past the last stream (q of row i0 + 64 of the last tile); the
// entries computed from those rows are discarded by the line selection.
//
// Backward (attn_bert_train_bwd), no floating-point atomics on activations:
//   attn_delta_kernel (attention_train.cu) : delta_i = dO_i . O_i
//   attn_bert_bwd_dq_kernel                : query-tile owner; recomputes P, forms dS, accumulates the content part of dQ
//                                            (-> du), spills the dropped P and dS for the key-tile kernel and writes dS in
//                                            (q-row, distance) coordinates (ds_dist): line-1 entries of row i go to row i,
//                                            line-3 entries of row i to row i + 1 - disjoint writes, every distance once
//   attn_bwd_dkv_lite_kernel<true> (attention_train.cu): key-tile owner; dK = dS^T (q+u), dV = P^T dO over all query tiles
// The position part of dQ (ds_dist . Rk per head, -> dv) and dRk are GEMMs of the trainer (train.cu).
#include "kernels.cuh"
#include "launch.cuh"
#include "attention_train_common.cuh"

namespace dmg {

namespace {

// shared memory of both kernels: Q, Q of the next rows, dO (backward only), K, V, the line-1 and line-3 windows, skew strips
constexpr int BT_SMEM = 9 * TILE_BYTES + 4 * 16 * SKEW_LD * (int)sizeof(skew_t);

struct BertSmem {
  uint8_t *sQ, *sQn, *sdO, *sK, *sV, *sR;
  skew_t* skew;
  __device__ BertSmem(uint8_t* smem, int w) {
    sQ = smem; sQn = sQ + TILE_BYTES; sdO = sQn + TILE_BYTES; sK = sdO + TILE_BYTES; sV = sK + TILE_BYTES; sR = sV + TILE_BYTES;
    skew = (skew_t*)(sR + 4 * TILE_BYTES) + w * 16 * SKEW_LD;
  }
};

// K, V of key tile j0 and the rel-pos windows the tile needs (line 1 when j0 <= i0, line 3 when j0 >= i0): one cp.async group
__device__ __forceinline__ void load_key_tile(const AttnTrainArgs& a, const BertSmem& sm, int b, int h, int i0, int j0, int tid) {
  const int HD = a.H * 64;
  const bf16* kp = a.qkv_x + ((long long)b * a.T + j0) * a.ldx + HD + h * 64;
  tile_load_async(sm.sK, kp, a.ldx, tid, 128);
  tile_load_async(sm.sV, kp + HD, a.ldx, tid, 128);
  const bf16* rk = a.rk + h * 64;
  if (j0 <= i0) {
    const int D0 = i0 - j0;
    tile_load_async(sm.sR, rk + (long long)(D0 - 64) * HD, HD, tid, 128);
    tile_load_async(sm.sR + TILE_BYTES, rk + (long long)D0 * HD, HD, tid, 128);
  }
  if (j0 >= i0) {
    const int D0 = a.T + 1 + i0 - j0;
    tile_load_async(sm.sR + 2 * TILE_BYTES, rk + (long long)(D0 - 64) * HD, HD, tid, 128);
    tile_load_async(sm.sR + 3 * TILE_BYTES, rk + (long long)D0 * HD, HD, tid, 128);
  }
  cp_async_commit();
}

// raw scores (AC + BD, unscaled) of the warp's 16 query rows x the key tile at j0; qvn = (q + v) of the rows one below
__device__ __forceinline__ void bert_scores(const uint32_t (&qu)[4][4], const uint32_t (&qv)[4][4], const uint32_t (&qvn)[4][4],
                                            const BertSmem& sm, int w, int lane, const LaneOff& L, int i0, int j0, float (&s)[8][4]) {
  const int g = lane >> 2, t = lane & 3;
  const int dd = i0 + 16 * w - j0;                  // i - j of element (r, jl) is dd + r - jl
  content_scores(qu, smem_u32(sm.sK), L, s);
  if (j0 <= i0) {
    position_strip(qv, smem_u32(sm.sR), smem_u32(sm.sR + TILE_BYTES), sm.skew, w, lane, L);
#pragma unroll
    for (int nt = 0; nt < 8; nt++)
#pragma unroll
      for (int e = 0; e < 4; e++)
        if (dd + g + 8 * (e >> 1) - (8 * nt + 2 * t + (e & 1)) >= 0) s[nt][e] += skew_at(sm.skew, g, t, nt, e);
    __syncwarp();
  }
  if (j0 >= i0) {
    position_strip(qvn, smem_u32(sm.sR + 2 * TILE_BYTES), smem_u32(sm.sR + 3 * TILE_BYTES), sm.skew, w, lane, L);
#pragma unroll
    for (int nt = 0; nt < 8; nt++)
#pragma unroll
      for (int e = 0; e < 4; e++)
        if (dd + g + 8 * (e >> 1) - (8 * nt + 2 * t + (e & 1)) < -1) s[nt][e] += skew_at(sm.skew, g, t, nt, e);
    __syncwarp();
  }
}

// Q and next-row Q (and dO) of query tile i0 -> fragments (q+u), (q+v), (q_next+v)
__device__ __forceinline__ void load_query_tile(const AttnTrainArgs& a, const BertSmem& sm, const bf16* dout, int b, int h, int i0, int tid) {
  const bf16* qp = a.qkv_x + ((long long)b * a.T + i0) * a.ldx + h * 64;
  tile_load_async(sm.sQ, qp, a.ldx, tid, 128);
  tile_load_async(sm.sQn, qp + a.ldx, a.ldx, tid, 128);
  if (dout) tile_load_async(sm.sdO, dout + ((long long)b * a.T + i0) * (a.H * 64) + h * 64, a.H * 64, tid, 128);
  cp_async_commit();
  cp_async_wait<0>();
  __syncthreads();
}

__global__ void __launch_bounds__(128) attn_bert_train_fwd_kernel(const AttnTrainArgs a) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int tid = threadIdx.x, w = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  const BertSmem sm(smem, w);
  LaneOff L;
  lane_off_init(L, lane, w);
  const int nT = a.T / 64;
  const int it = blockIdx.x % nT, bh = blockIdx.x / nT, b = bh / a.H, h = bh % a.H;
  const int i0 = it * 64, HD = a.H * 64, S = a.T;

  load_query_tile(a, sm, nullptr, b, h, i0, tid);
  uint32_t qu[4][4], qv[4][4], qvn[4][4], unused[4][4];
  q_frags(smem_u32(sm.sQ), w, lane, L, a.u + h * 64, a.v + h * 64, qu, qv);
  q_frags(smem_u32(sm.sQn), w, lane, L, a.v + h * 64, a.v + h * 64, unused, qvn);

  float o[8][4];
#pragma unroll
  for (int nt = 0; nt < 8; nt++) { o[nt][0] = 0.f; o[nt][1] = 0.f; o[nt][2] = 0.f; o[nt][3] = 0.f; }
  float m_run[2] = {-INFINITY, -INFINITY}, l_run[2] = {0.f, 0.f};
  const float c = a.scale * ATT_LOG2E;
  const int row_g[2] = {i0 + 16 * w + g, i0 + 16 * w + g + 8};
  const uint32_t drop_base[2] = {(uint32_t)((((long long)bh * a.T + row_g[0]) * S) >> 1) + t,
                                 (uint32_t)((((long long)bh * a.T + row_g[1]) * S) >> 1) + t};

  for (int jt = 0; jt < nT; jt++) {
    const int j0 = jt * 64;
    __syncthreads();                                 // everybody is done with the previous key tile
    load_key_tile(a, sm, b, h, i0, j0, tid);
    cp_async_wait<0>();
    __syncthreads();
    float s[8][4];
    bert_scores(qu, qv, qvn, sm, w, lane, L, i0, j0, s);
    // running max on the raw scores (the scale is positive); no key is masked, so every score is finite
    float mx[2] = {-INFINITY, -INFINITY};
#pragma unroll
    for (int nt = 0; nt < 8; nt++) {
      mx[0] = fmaxf(mx[0], fmaxf(s[nt][0], s[nt][1]));
      mx[1] = fmaxf(mx[1], fmaxf(s[nt][2], s[nt][3]));
    }
    float alpha[2], neg_mc[2];
#pragma unroll
    for (int r = 0; r < 2; r++) {
      const float m_new = fmaxf(m_run[r], quad_max(mx[r]));
      alpha[r] = ex2_fast((m_run[r] - m_new) * c);
      neg_mc[r] = -m_new * c;
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
        float keep[4];
        attn_keep(a.drop_thresh, a.drop_seed, a.drop_scale, drop_base, j0, nt, keep);
#pragma unroll
        for (int e = 0; e < 4; e++) p[e] *= keep[e];
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
    const uint32_t sVa = smem_u32(sm.sV);
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
    const float inv = 1.f / l;
    bf16* orow = a.out + ((long long)b * a.T + row_g[r]) * HD + h * 64;
#pragma unroll
    for (int nt = 0; nt < 8; nt++)
      *(uint32_t*)(orow + 8 * nt + 2 * t) = pack_bf16x2(o[nt][2 * r] * inv, o[nt][2 * r + 1] * inv);
    if (t == 0) a.lse[(long long)bh * a.T + row_g[r]] = (m_run[r] * c + log2f(l)) * ATT_LN2;
  }
}

__global__ void __launch_bounds__(128) attn_bert_bwd_dq_kernel(const AttnTrainBwdArgs ba) {
  const AttnTrainArgs& a = ba.f;
  extern __shared__ __align__(128) uint8_t smem[];
  const int tid = threadIdx.x, w = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  const BertSmem sm(smem, w);
  LaneOff L;
  lane_off_init(L, lane, w);
  const int nT = a.T / 64;
  const int it = blockIdx.x % nT, bh = blockIdx.x / nT, b = bh / a.H, h = bh % a.H;
  const int i0 = it * 64, S = a.T;
  const long long bhT = (long long)bh * a.T, HS = (long long)a.H * S;
  bf16* const dsd = ba.ds_dist + (long long)b * a.T * HS + (long long)h * S;   // row r, distance x at dsd[r*HS + x]

  if (it == 0 && w == 0)                             // row 0 has no line-3 predecessor: its distances 1 .. T-1 are zero
    for (int x = 1 + lane; x < S; x += 32) dsd[x] = __float2bfloat16_rn(0.f);

  load_query_tile(a, sm, ba.dout, b, h, i0, tid);
  uint32_t qu[4][4], qv[4][4], qvn[4][4], dof[4][4], unused[4][4];
  q_frags(smem_u32(sm.sQ), w, lane, L, a.u + h * 64, a.v + h * 64, qu, qv);
  q_frags(smem_u32(sm.sQn), w, lane, L, a.v + h * 64, a.v + h * 64, unused, qvn);
#pragma unroll
  for (int ks = 0; ks < 4; ks++) frag_a(smem_u32(sm.sdO), 16 * w, ks, L, dof[ks]);

  const int row_g[2] = {i0 + 16 * w + g, i0 + 16 * w + g + 8};
  const uint32_t drop_base[2] = {(uint32_t)(((bhT + row_g[0]) * S) >> 1) + t, (uint32_t)(((bhT + row_g[1]) * S) >> 1) + t};
  const float c = a.scale * ATT_LOG2E;
  float lse2[2], dl[2];
#pragma unroll
  for (int r = 0; r < 2; r++) {
    lse2[r] = a.lse[bhT + row_g[r]] * ATT_LOG2E;
    dl[r] = ba.delta[bhT + row_g[r]];
  }
  float dq[8][4];
#pragma unroll
  for (int nt = 0; nt < 8; nt++)
#pragma unroll
    for (int e = 0; e < 4; e++) dq[nt][e] = 0.f;

  for (int jt = 0; jt < nT; jt++) {
    const int j0 = jt * 64;
    __syncthreads();
    load_key_tile(a, sm, b, h, i0, j0, tid);
    cp_async_wait<0>();
    __syncthreads();
    float s[8][4], dpd[8][4];
    bert_scores(qu, qv, qvn, sm, w, lane, L, i0, j0, s);
    // dPd = dO V^T
#pragma unroll
    for (int nt = 0; nt < 8; nt++) { dpd[nt][0] = 0.f; dpd[nt][1] = 0.f; dpd[nt][2] = 0.f; dpd[nt][3] = 0.f; }
    const uint32_t sVa = smem_u32(sm.sV), sKa = smem_u32(sm.sK);
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
    // P, dS; spill the dropped P and dS ([b*H+h][T][T] bf16) for the key-tile kernel; dS in distance coordinates
    const long long o0 = (bhT + row_g[0]) * S + j0, o1 = (bhT + row_g[1]) * S + j0;
#pragma unroll
    for (int nt = 0; nt < 8; nt++) {
      float keep[4] = {1.f, 1.f, 1.f, 1.f};
      if (a.drop_thresh) attn_keep(a.drop_thresh, a.drop_seed, a.drop_scale, drop_base, j0, nt, keep);
#pragma unroll
      for (int e = 0; e < 4; e++) {
        const int r = e >> 1;
        const float p = ex2_fast(s[nt][e] * c - lse2[r]);
        s[nt][e] = p * (dpd[nt][e] * keep[e] - dl[r]) * a.scale;
        keep[e] *= p;                                // keep[] now holds the dropped probability
        const int i = row_g[r], j = j0 + 8 * nt + 2 * t + (e & 1);
        const bf16 v = __float2bfloat16_rn(s[nt][e]);
        if (j <= i) dsd[(long long)i * HS + (i - j)] = v;                           // line 1: row i, distance i - j
        else if (j > i + 1) dsd[(long long)(i + 1) * HS + (S + 1 + i - j)] = v;     // line 3: row i + 1, distance T + 1 + i - j
      }
      const int c0 = 8 * nt + 2 * t;
      *(uint32_t*)(ba.p_buf + o0 + c0) = pack_bf16x2(keep[0], keep[1]);
      *(uint32_t*)(ba.p_buf + o1 + c0) = pack_bf16x2(keep[2], keep[3]);
      *(uint32_t*)(ba.ds_buf + o0 + c0) = pack_bf16x2(s[nt][0], s[nt][1]);
      *(uint32_t*)(ba.ds_buf + o1 + c0) = pack_bf16x2(s[nt][2], s[nt][3]);
    }
    // dQ (content part) += dS K
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
        mma_bf16(dq[2 * np], dsa[ks], r[0], r[1]);
        mma_bf16(dq[2 * np + 1], dsa[ks], r[2], r[3]);
      }
    }
  }

  // content part of dq; du = its column sum over all rows (the position part and dv follow in the trainer's GEMMs)
#pragma unroll
  for (int r = 0; r < 2; r++) {
    bf16* qrow = ba.dqkv_x + ((long long)b * a.T + row_g[r]) * a.ldx + h * 64;
#pragma unroll
    for (int nt = 0; nt < 8; nt++) *(uint32_t*)(qrow + 8 * nt + 2 * t) = pack_bf16x2(dq[nt][2 * r], dq[nt][2 * r + 1]);
  }
#pragma unroll
  for (int nt = 0; nt < 8; nt++) {
#pragma unroll
    for (int e = 0; e < 2; e++) {
      float su = dq[nt][e] + dq[nt][e + 2];
#pragma unroll
      for (int o = 4; o < 32; o <<= 1) su += __shfl_xor_sync(0xffffffffu, su, o);
      if (g == 0) atomicAdd(ba.du + h * 64 + 8 * nt + 2 * t + e, su);
    }
  }
}

int check_bert_args(const AttnTrainArgs& a) {
  DMG_CHECK(a.T > 0 && a.T % 64 == 0 && a.M == 0 && a.mem_count == 0, "remix training attention: T=%d must be a multiple of 64, no memory (M=%d)",
            a.T, a.M);
  DMG_CHECK(a.win == 1 && a.k == 1, "remix training attention: window mask (%d,%d) unsupported (the encoder has no mask)", a.win, a.k);
  DMG_CHECK(a.ldx % 8 == 0, "remix training attention: row stride must be a multiple of 8");
  DMG_CHECK((long long)a.B * a.H * a.T * a.T < (1ll << 32), "remix training attention: dropout index exceeds 32 bits");
  return 0;
}

}  // namespace

int attn_bert_train_fwd(const AttnTrainArgs& a, cudaStream_t st) {
  if (check_bert_args(a)) return -2;
  static bool configured = false;
  if (!configured) {
    DMG_CUDA_OK(cudaFuncSetAttribute(attn_bert_train_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, BT_SMEM));
    configured = true;
  }
  return launch_np(attn_bert_train_fwd_kernel, dim3(a.B * a.H * (a.T / 64)), dim3(128), (size_t)BT_SMEM, st, a);
}

int attn_bert_train_bwd(const AttnTrainBwdArgs& ba, cudaStream_t st) {
  const AttnTrainArgs& a = ba.f;
  if (check_bert_args(a)) return -2;
  DMG_CHECK(ba.p_buf && ba.ds_buf && ba.ds_dist, "remix training attention backward: P / dS workspaces missing");
  static bool configured = false;
  if (!configured) {
    DMG_CUDA_OK(cudaFuncSetAttribute(attn_bert_bwd_dq_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, BT_SMEM));
    configured = true;
  }
  if (attn_train_delta(ba, st)) return -1;
  if (launch_np(attn_bert_bwd_dq_kernel, dim3(a.B * a.H * (a.T / 64)), dim3(128), (size_t)BT_SMEM, st, ba)) return -1;
  return attn_bwd_dkv_all_queries(ba, st);
}

}  // namespace dmg
