// Relative-positional attention with segment-recurrence memory (Transformer-XL) - fused kernels.
//
// Reference being replaced (SURVEY.md 2.2 K5-K9, K13): fastai MultiHeadRelativeAttention._apply_attention and its
// in-repo twin MemMultiHeadRelativeAttentionKV._apply_attention (deep_music_remix.py:2078-2104):
//     AC = (q+u) K^T ; BD = _line_shift((q+v) R^T) ; P = softmax((AC+BD)/sqrt(Dh) + mask) ; out = P V
// _line_shift is never materialised: with Rd[dist] = r_attn(PositionalEncoding(dist)) cached per layer,
//     j <= M+i   : BD[i,j] = (q_i+v)     . Rd[M+i-j]
//     j == M+i+1 : BD[i,j] = 0                                   (BERT encoder only; masked in the causal TXL)
//     j >  M+i+1 : BD[i,j] = (q_{i+1}+v) . Rd[S+1+i-j]           (the live wrap-around of the unmasked encoder)
// (SURVEY.md App. A.4).  K/V of past tokens live in a per-(stream, head) ring in HBM, slot = token index mod M.
//
//  * x_len == 1 over the bf16 ring (the HBM-bound kernel of batched generation) lives in attention_decode2.cu.
//  * attn_general_kernel - any x_len (prefill, training-shape forward, BERT encoder), fp32 or bf16 ring,
//    flash-style online softmax over 32x32 tiles on the FFMA pipe.
#include "kernels.cuh"
#include "launch.cuh"

namespace dmg {

constexpr float LOG2E = 1.4426950408889634f;

// =============================================================================================
// general kernel
// =============================================================================================
constexpr int GQ = 32, GK = 32, GLD = 68;   // query tile, key tile, padded row stride (floats)

template <bool BERT>
__host__ __device__ constexpr int gen_smem_floats() {
  return GQ * GLD /*Qu*/ + (GQ + 1) * GLD /*Qv*/ + GK * GLD /*K*/ + GK * GLD /*V*/ + 63 * GLD /*R lower*/ +
         (BERT ? 63 * GLD : 0) /*R upper*/ + GQ * (GK + 1) /*P*/;
}

// VARLEN (BERT only): sequence b has a.lens[b] tokens in rows [b*a.T, b*a.T + a.lens[b]) of the padded layout; query tiles past
// its end do nothing (the caller zeroes those output rows)
template <class T, bool BERT, bool VARLEN>
__global__ void __launch_bounds__(128) attn_general_kernel(AttnGeneralArgs a) {
  extern __shared__ float sm[];
  float* Qu = sm;
  float* Qv = Qu + GQ * GLD;
  float* Ks = Qv + (GQ + 1) * GLD;
  float* Vs = Ks + GK * GLD;
  float* RL = Vs + GK * GLD;
  float* RU = RL + 63 * GLD;
  float* P = RU + (BERT ? 63 * GLD : 0);

  const int tid = threadIdx.x;
  pdl_launch_dependents();
  pdl_wait();
  const int i0 = blockIdx.x * GQ, h = blockIdx.y, b = blockIdx.z;
  const int T_len = VARLEN ? a.lens[b] : a.T, H = a.H, HD = H * 64, M = a.M;
  if (VARLEN && i0 >= T_len) return;
  const int* st = a.state + (size_t)a.state_stride * (a.b0 + b);   // this stream's memory: streams of a batch may hold different counts
  const int pos_total = st[0], m = st[1], S = m + T_len;
  const T* kring = (const T*)a.kring;
  const T* vring = (const T*)a.vring;
  const T* rd = (const T*)a.rd + (size_t)h * a.Dcap * 64;

  // q (+u / +v) rows; Qv holds one extra row (i0+32) for the wrap-around term
  for (int idx = tid; idx < (GQ + 1) * 16; idx += 128) {
    const int r = idx >> 4, c4 = (idx & 15) * 4;
    const int i = i0 + r;
    float4 q = make_float4(0.f, 0.f, 0.f, 0.f);
    if (i < T_len) q = *(const float4*)(a.qkv + ((size_t)b * a.T + i) * 3 * HD + h * 64 + c4);
    const float4 uu = *(const float4*)(a.u + h * 64 + c4), vv = *(const float4*)(a.v + h * 64 + c4);
    if (r < GQ) *(float4*)(Qu + r * GLD + c4) = make_float4(q.x + uu.x, q.y + uu.y, q.z + uu.z, q.w + uu.w);
    *(float4*)(Qv + r * GLD + c4) = make_float4(q.x + vv.x, q.y + vv.y, q.z + vv.z, q.w + vv.w);
  }

  const int qi = tid >> 2, kg = tid & 3;
  const int i = i0 + qi;
  float m_run = -INFINITY, l_run = 0.f;
  float o[16];
#pragma unroll
  for (int e = 0; e < 16; e++) o[e] = 0.f;

  int jend = S;
  if (!BERT) jend = min(S, m + i0 + GQ);   // every mask the reference builds hides keys with jx > i

  for (int j0 = 0; j0 < jend; j0 += GK) {
    __syncthreads();
    // ---- K / V tile: ring slots for memory, the qkv buffer for the segment itself
    {
      const int r = tid >> 2, c16 = (tid & 3) * 16;
      const int j = j0 + r;
      float kv[16], vv[16];
      if (j < S) {
        if (j < m) {
          const int slot = (int)(((long long)pos_total - m + j) % M);
          const size_t off = (((size_t)(a.b0 + b) * H + h) * M + slot) * 64 + c16;
#pragma unroll
          for (int e = 0; e < 16; e++) {
            kv[e] = to_f32(kring[off + e]);
            vv[e] = to_f32(vring[off + e]);
          }
        } else {
          const float* row = a.qkv + ((size_t)b * a.T + (j - m)) * 3 * HD + h * 64 + c16;
#pragma unroll
          for (int e = 0; e < 16; e++) {
            kv[e] = row[HD + e];
            vv[e] = row[2 * HD + e];
          }
        }
      } else {
#pragma unroll
        for (int e = 0; e < 16; e++) kv[e] = vv[e] = 0.f;
      }
#pragma unroll
      for (int e = 0; e < 16; e++) {
        Ks[r * GLD + c16 + e] = kv[e];
        Vs[r * GLD + c16 + e] = vv[e];
      }
    }
    // ---- relative-position key windows: row w <-> (qi - jl + 31)
    {
      const int dLo = m + i0 - j0 - 31;
      const int dUp = S + 1 + i0 - j0 - 31;
      for (int idx = tid; idx < 63 * 16; idx += 128) {
        const int w = idx >> 4, c4 = (idx & 15) * 4;
        int dist = dLo + w;
        float4 val = make_float4(0.f, 0.f, 0.f, 0.f);
        if (dist >= 0 && dist < a.Dcap) {
          const T* p = rd + (size_t)dist * 64 + c4;
          val = make_float4(to_f32(p[0]), to_f32(p[1]), to_f32(p[2]), to_f32(p[3]));
        }
        *(float4*)(RL + w * GLD + c4) = val;
        if (BERT) {
          dist = dUp + w;
          val = make_float4(0.f, 0.f, 0.f, 0.f);
          if (dist >= 0 && dist < a.Dcap) {
            const T* p = rd + (size_t)dist * 64 + c4;
            val = make_float4(to_f32(p[0]), to_f32(p[1]), to_f32(p[2]), to_f32(p[3]));
          }
          *(float4*)(RU + w * GLD + c4) = val;
        }
      }
    }
    __syncthreads();

    // ---- scores
    float sv[8];
    float tmax = -INFINITY;
#pragma unroll
    for (int jj = 0; jj < 8; jj++) {
      const int jl = kg + 4 * jj;
      const int j = j0 + jl;
      bool valid = (i < T_len) && (j < S);
      const float* rrow = RL + (qi - jl + 31) * GLD;
      const float* qvrow = Qv + qi * GLD;
      float bdw = 1.f;
      if (BERT) {
        if (j == m + i + 1) bdw = 0.f;
        else if (j > m + i + 1) {
          rrow = RU + (qi - jl + 31) * GLD;
          qvrow = Qv + (qi + 1) * GLD;
        }
      } else {
        const int jx = j - m;
        if (jx > 0) valid = valid && ((jx / a.win - i / a.win) < a.k);
      }
      const float* qurow = Qu + qi * GLD;
      const float* krow = Ks + jl * GLD;
      float ac = 0.f, bd = 0.f;
#pragma unroll
      for (int d4 = 0; d4 < 64; d4 += 4) {
        const float4 qa = *(const float4*)(qurow + d4), kk = *(const float4*)(krow + d4);
        const float4 qb = *(const float4*)(qvrow + d4), rr = *(const float4*)(rrow + d4);
        ac = fmaf(qa.x, kk.x, ac); ac = fmaf(qa.y, kk.y, ac); ac = fmaf(qa.z, kk.z, ac); ac = fmaf(qa.w, kk.w, ac);
        bd = fmaf(qb.x, rr.x, bd); bd = fmaf(qb.y, rr.y, bd); bd = fmaf(qb.z, rr.z, bd); bd = fmaf(qb.w, rr.w, bd);
      }
      const float s = valid ? (ac + bdw * bd) * a.scale : -INFINITY;
      sv[jj] = s;
      tmax = fmaxf(tmax, s);
    }
    tmax = fmaxf(tmax, __shfl_xor_sync(0xffffffffu, tmax, 1));
    tmax = fmaxf(tmax, __shfl_xor_sync(0xffffffffu, tmax, 2));
    const float m_new = fmaxf(m_run, tmax);
    const float corr = (m_new == -INFINITY) ? 1.f : expf(m_run - m_new);
    float psum = 0.f;
#pragma unroll
    for (int jj = 0; jj < 8; jj++) {
      const float p = (m_new == -INFINITY) ? 0.f : expf(sv[jj] - m_new);
      P[qi * (GK + 1) + kg + 4 * jj] = p;
      psum += p;
    }
    psum += __shfl_xor_sync(0xffffffffu, psum, 1);
    psum += __shfl_xor_sync(0xffffffffu, psum, 2);
    l_run = l_run * corr + psum;
    m_run = m_new;
#pragma unroll
    for (int e = 0; e < 16; e++) o[e] *= corr;
    __syncwarp();

    // ---- P.V : this thread owns output dims [kg*16, kg*16+16) of query qi
#pragma unroll 4
    for (int jl = 0; jl < GK; jl++) {
      const float p = P[qi * (GK + 1) + jl];
      const float* vrow = Vs + jl * GLD + kg * 16;
#pragma unroll
      for (int e4 = 0; e4 < 16; e4 += 4) {
        const float4 vv = *(const float4*)(vrow + e4);
        o[e4] = fmaf(p, vv.x, o[e4]); o[e4 + 1] = fmaf(p, vv.y, o[e4 + 1]);
        o[e4 + 2] = fmaf(p, vv.z, o[e4 + 2]); o[e4 + 3] = fmaf(p, vv.w, o[e4 + 3]);
      }
    }
  }
  if (i < T_len) {
    const float inv = l_run > 0.f ? 1.f / l_run : 0.f;
    T* out = (T*)a.out + ((size_t)b * a.T + i) * HD + h * 64 + kg * 16;
#pragma unroll
    for (int e = 0; e < 16; e++) out[e] = from_f32<T>(o[e] * inv);
  }
}

template <class T, bool BERT, bool VARLEN = false>
static int launch_general(const AttnGeneralArgs& a, cudaStream_t st) {
  const int smem = gen_smem_floats<BERT>() * 4;
  static bool configured = false;
  if (!configured) {
    DMG_CUDA_OK(cudaFuncSetAttribute(attn_general_kernel<T, BERT, VARLEN>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    configured = true;
  }
  dim3 grid((a.T + GQ - 1) / GQ, a.H, a.B);
  return launch_k(attn_general_kernel<T, BERT, VARLEN>, grid, dim3(128), smem, st, 1, a);
}

template <class T>
int attn_general(const AttnGeneralArgs& a, cudaStream_t st) {
  DMG_CHECK(a.win >= 1, "attn_general: window size must be >= 1");
  if (a.B <= 0 || a.T <= 0) return 0;
  if (a.lens) {
    DMG_CHECK(a.bert && a.M == 0, "attn_general: per-sequence lengths need the memory-less BERT encoder");
    return launch_general<T, true, true>(a, st);
  }
  return a.bert ? launch_general<T, true>(a, st) : launch_general<T, false>(a, st);
}
template int attn_general<float>(const AttnGeneralArgs&, cudaStream_t);
template int attn_general<bf16>(const AttnGeneralArgs&, cudaStream_t);

}  // namespace dmg
