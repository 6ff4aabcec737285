// Tensor-core flash attention for INFERENCE segments (x_len > 1) without memory: the Transformer-XL prefill of a seed
// (causal, eval mask) and the masked-BERT remix encoder (no mask, _line_shift wrap-around live), bf16 mma.sync,
// fp32 softmax, no score tensor in HBM.  Same tile machinery as attention_train.cu (64 x 64 tiles, 4 warps, rel-pos term
// by a skewed read of a 16 x 80 strip), forward only, any x_len (ragged last tile: zero-filled loads, masked keys).
//
// Replaces fastai MultiHeadRelativeAttention._apply_attention (SURVEY.md App. A.3) for the first segment after reset()
// and MemMultiHeadRelativeAttentionKV._apply_attention (deep_music_remix.py:2078-2104, r_mask=False):
//   line 1 (j <= i)   : BD[i,j] = (q_i + v) . Rk[i - j]
//   line 2 (j == i+1) : 0
//   line 3 (j >  i+1) : BD[i,j] = (q_{i+1} + v) . Rk[T + 1 + i - j]          (App. A.4; BERT only - the TXL mask hides it)
// Line 3 uses the NEXT query row and a window into Rk shifted by (T + 1) mod 64 rows, so that both windows stay aligned to
// 64-row tiles of their (shifted) table.
#include "kernels.cuh"
#include "launch.cuh"
#include "mma_sync.cuh"

namespace dmg {

namespace {

constexpr int FL_SKEW_LD = 84;
constexpr float FL_LOG2E = 1.4426950408889634f;

__device__ __forceinline__ void cp_async16_zfill(void* smem_dst, const void* gsrc, bool valid) {
  const int n = valid ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(n) : "memory");
}
// 64 x 64 bf16 tile from rows [r0, r0+64) of a matrix with `nrows` valid rows (others read as zero)
__device__ __forceinline__ void tile_load_guard(uint8_t* tile, const bf16* base, long long ld, int r0, int nrows, int tid) {
  const int r = tid >> 3, c = tid & 7;
#pragma unroll
  for (int k = 0; k < 4; k++) {
    const int row = r0 + r + 16 * k;
    const bool ok = row >= 0 && row < nrows;
    cp_async16_zfill(tile + tile_off(r + 16 * k, c), base + (long long)(ok ? row : 0) * ld + c * 8, ok);
  }
}

__device__ __forceinline__ uint32_t fl_add2(uint32_t w, float b0, float b1) { return pack_bf16x2(bf16lo(w) + b0, bf16hi(w) + b1); }
__device__ __forceinline__ void fl_q_frags(uint32_t sQ, int w, int lane, const LaneOff& L, const float* __restrict__ bias,
                                           uint32_t (&out)[4][4]) {
  const int t = lane & 3;
#pragma unroll
  for (int ks = 0; ks < 4; ks++) {
    uint32_t a[4];
    frag_a(sQ, 16 * w, ks, L, a);
    const int c0 = 16 * ks + 2 * t;
    const float b0 = bias[c0], b1 = bias[c0 + 1], b8 = bias[c0 + 8], b9 = bias[c0 + 9];
    out[ks][0] = fl_add2(a[0], b0, b1); out[ks][1] = fl_add2(a[1], b0, b1);
    out[ks][2] = fl_add2(a[2], b8, b9); out[ks][3] = fl_add2(a[3], b8, b9);
  }
}
// acc[nt][e] (+)= A (16 x 64) * K-tile^T
__device__ __forceinline__ void fl_content(const uint32_t (&qa)[4][4], uint32_t sK, const LaneOff& L, float (&s)[8][4]) {
#pragma unroll
  for (int ks = 0; ks < 4; ks++) {
#pragma unroll
    for (int np = 0; np < 4; np++) {
      uint32_t r[4];
      frag_b(sK, 16 * np, ks, L, r);
      mma_bf16(s[2 * np], qa[ks], r[0], r[1]);
      mma_bf16(s[2 * np + 1], qa[ks], r[2], r[3]);
    }
  }
}
// position term through the skewed strip: bd[nt][e] = (q + v)[row] . Rwin[64 + row - jl]   (sR0 | sR1 = the 128-row window)
__device__ __forceinline__ void fl_position(const uint32_t (&qv)[4][4], uint32_t sR0, uint32_t sR1, float* skew, int w, int lane,
                                            const LaneOff& L, float (&bd)[8][4]) {
  const int g = lane >> 2, t = lane & 3;
#pragma unroll
  for (int p = 0; p < 5; p++) {
    const int wc = 16 * w + 16 * p;
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
      *(float2*)(skew + g * FL_SKEW_LD + col) = make_float2(acc[h][0], acc[h][1]);
      *(float2*)(skew + (g + 8) * FL_SKEW_LD + col) = make_float2(acc[h][2], acc[h][3]);
    }
  }
  __syncwarp();
#pragma unroll
  for (int nt = 0; nt < 8; nt++) {
    const int jl = 8 * nt + 2 * t;
    bd[nt][0] = skew[g * FL_SKEW_LD + 64 + g - jl];
    bd[nt][1] = skew[g * FL_SKEW_LD + 63 + g - jl];
    bd[nt][2] = skew[(g + 8) * FL_SKEW_LD + 72 + g - jl];
    bd[nt][3] = skew[(g + 8) * FL_SKEW_LD + 71 + g - jl];
  }
  __syncwarp();
}

struct FlashArgs {
  const bf16* qkv;     // [B*T, 3*HD] bf16: q | k | v
  const bf16* rk;      // rel-pos keys by distance: head h at rk + h*rk_hs, row stride rk_ld, rk_rows rows
  long long rk_hs; int rk_ld, rk_rows;
  const float* u;      // [HD]
  const float* v;
  bf16* out;           // [B*T, HD]
  int B, T, H;
  float scale;
  // per-sequence lengths (BERT): block row bh / H walks sequence seqs[bh / H], whose lens[.] tokens are rows [b*T, b*T + len) of the
  // padded layout (T = the padded length); nTg 64-row query tiles per (sequence, head), tiles past the sequence end do nothing
  const int* lens;
  const int* seqs;
  int nTg;
};

constexpr int FL_SMEM = 4 * TILE_BYTES /*Q, Qnext, K, V*/ + 4 * TILE_BYTES /*two Rk windows*/ + 4 * 16 * FL_SKEW_LD * 4;

template <bool BERT, bool VARLEN>
__global__ void __launch_bounds__(128) attn_flash_kernel(const FlashArgs a) {
  extern __shared__ __align__(128) uint8_t smem[];
  uint8_t* sQ = smem;
  uint8_t* sQn = sQ + TILE_BYTES;
  uint8_t* sK = sQn + TILE_BYTES;
  uint8_t* sV = sK + TILE_BYTES;
  uint8_t* sR = sV + TILE_BYTES;                     // [0],[1]: line-1 window; [2],[3]: line-3 window
  float* skew_all = (float*)(sR + 4 * TILE_BYTES);
  const int tid = threadIdx.x, w = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  float* skew = skew_all + w * 16 * FL_SKEW_LD;
  LaneOff L;
  lane_off_init(L, lane, w);
  pdl_launch_dependents();
  pdl_wait();

  const int nTb = VARLEN ? a.nTg : (a.T + 63) / 64;   // query tiles per block row
  const int it = nTb - 1 - (blockIdx.x % nTb);
  const int bh = blockIdx.x / nTb, b = VARLEN ? a.seqs[bh / a.H] : bh / a.H, h = bh % a.H;
  const int T = VARLEN ? a.lens[b] : a.T;           // this sequence's length
  const int nT = (T + 63) / 64, T64 = nT * 64;
  if (VARLEN && it >= nT) return;
  const int i0 = it * 64, HD = a.H * 64;
  const long long ldx = 3 * HD;
  const bf16* qkv_b = a.qkv + (long long)b * a.T * ldx + h * 64;     // q of (b, h); k at +HD, v at +2*HD
  const bf16* rk_h = a.rk + (long long)h * a.rk_hs;
  const int shift3 = T + 1 - T64;                   // line-3 table: Rk3[x] = Rk[x + shift3], x = T64 + i - j

  tile_load_guard(sQ, qkv_b, ldx, i0, T, tid);
  if (BERT) tile_load_guard(sQn, qkv_b, ldx, i0 + 1, T, tid);
  cp_async_commit();
  cp_async_wait<0>();
  __syncthreads();
  uint32_t qu[4][4], qv[4][4], qvn[4][4];
  fl_q_frags(smem_u32(sQ), w, lane, L, a.u + h * 64, qu);
  fl_q_frags(smem_u32(sQ), w, lane, L, a.v + h * 64, qv);
  if (BERT) fl_q_frags(smem_u32(sQn), w, lane, L, a.v + h * 64, qvn);

  float o[8][4];
#pragma unroll
  for (int nt = 0; nt < 8; nt++) { o[nt][0] = 0.f; o[nt][1] = 0.f; o[nt][2] = 0.f; o[nt][3] = 0.f; }
  float m_run[2] = {-INFINITY, -INFINITY}, l_run[2] = {0.f, 0.f};
  const float c = a.scale * FL_LOG2E;
  const int row_g[2] = {i0 + 16 * w + g, i0 + 16 * w + g + 8};
  const int jt_hi = BERT ? nT - 1 : it;

  for (int jt = 0; jt <= jt_hi; jt++) {
    const int j0 = jt * 64;
    const bool use1 = jt <= it, use3 = BERT && jt >= it;
    __syncthreads();
    tile_load_guard(sK, qkv_b + HD, ldx, j0, T, tid);
    tile_load_guard(sV, qkv_b + 2 * HD, ldx, j0, T, tid);
    if (use1) {                                      // distances D0-64 .. D0+63, D0 = i0 - j0 >= 0
      const int D0 = i0 - j0;
      tile_load_guard(sR, rk_h, a.rk_ld, D0 - 64, a.rk_rows, tid);
      tile_load_guard(sR + TILE_BYTES, rk_h, a.rk_ld, D0, a.rk_rows, tid);
    }
    if (use3) {                                      // Rk3 rows D0-64 .. D0+63, D0 = T64 + i0 - j0 >= 64
      const int D0 = T64 + i0 - j0;
      tile_load_guard(sR + 2 * TILE_BYTES, rk_h, a.rk_ld, D0 - 64 + shift3, a.rk_rows, tid);
      tile_load_guard(sR + 3 * TILE_BYTES, rk_h, a.rk_ld, D0 + shift3, a.rk_rows, tid);
    }
    cp_async_commit();
    cp_async_wait<0>();
    __syncthreads();

    float s[8][4];
#pragma unroll
    for (int nt = 0; nt < 8; nt++) { s[nt][0] = 0.f; s[nt][1] = 0.f; s[nt][2] = 0.f; s[nt][3] = 0.f; }
    fl_content(qu, smem_u32(sK), L, s);
    float bd1[8][4], bd3[8][4];
    if (use1) fl_position(qv, smem_u32(sR), smem_u32(sR + TILE_BYTES), skew, w, lane, L, bd1);
    if (use3) fl_position(qvn, smem_u32(sR + 2 * TILE_BYTES), smem_u32(sR + 3 * TILE_BYTES), skew, w, lane, L, bd3);
    float mx[2] = {-INFINITY, -INFINITY};
#pragma unroll
    for (int nt = 0; nt < 8; nt++) {
#pragma unroll
      for (int e = 0; e < 4; e++) {
        const int i = row_g[e >> 1], j = j0 + 8 * nt + 2 * t + (e & 1);
        float bdv = 0.f;
        if (j <= i) { if (use1) bdv = bd1[nt][e]; }
        else if (BERT && j > i + 1) { if (use3) bdv = bd3[nt][e]; }
        float x = s[nt][e] + bdv;
        const bool vis = BERT ? (j < T) : (j <= i);
        if (!vis) x = -INFINITY;
        s[nt][e] = x;
        mx[e >> 1] = fmaxf(mx[e >> 1], x);
      }
    }
    float alpha[2], neg_mc[2];
#pragma unroll
    for (int r = 0; r < 2; r++) {
      float m = mx[r];
      m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, 1));
      m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, 2));
      const float m_new = fmaxf(m_run[r], m);
      alpha[r] = (m_new == -INFINITY) ? 1.f : ex2_fast((m_run[r] - m_new) * c);
      neg_mc[r] = (m_new == -INFINITY) ? 0.f : -m_new * c;
      m_run[r] = m_new;
    }
    float rs[2] = {0.f, 0.f};
    uint32_t pa[4][4];
#pragma unroll
    for (int nt = 0; nt < 8; nt++) {
      float p[4];
#pragma unroll
      for (int e = 0; e < 4; e++) {
        p[e] = ex2_fast(fmaf(s[nt][e], c, neg_mc[e >> 1]));
        rs[e >> 1] += p[e];
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
  // VARLEN: the sequence index is read again rather than kept in a register across the key loop (52 instead of 12 bytes of spill
  // stores with it kept)
  int bo = b;
  if constexpr (VARLEN) bo = *(volatile const int*)(a.seqs + blockIdx.x / nTb / a.H);
#pragma unroll
  for (int r = 0; r < 2; r++) {
    float l = l_run[r];
    l += __shfl_xor_sync(0xffffffffu, l, 1);
    l += __shfl_xor_sync(0xffffffffu, l, 2);
    if (row_g[r] >= T) continue;
    const float inv = l > 0.f ? 1.f / l : 0.f;
    bf16* orow = a.out + ((long long)bo * a.T + row_g[r]) * HD + h * 64;
#pragma unroll
    for (int nt = 0; nt < 8; nt++)
      *(uint32_t*)(orow + 8 * nt + 2 * t) = pack_bf16x2(o[nt][2 * r] * inv, o[nt][2 * r + 1] * inv);
  }
}

}  // namespace

// qkv: bf16 [B*T, 3*H*64]; rd: the inference rel-pos key cache [H][Dcap][64] (bf16); out: bf16 [B*T, H*64]
int attn_flash(const bf16* qkv, const bf16* rd, int Dcap, const float* u, const float* v, bf16* out, int B, int T, int H, int bert,
               float scale, cudaStream_t st) {
  DMG_CHECK(T >= 1 && Dcap >= T, "attn_flash: rel-pos cache too small (T=%d, Dcap=%d)", T, Dcap);   // distances 0 .. T-1 are live
  FlashArgs a;
  a.qkv = qkv; a.rk = rd; a.rk_hs = (long long)Dcap * 64; a.rk_ld = 64; a.rk_rows = Dcap; a.u = u; a.v = v; a.out = out;
  a.B = B; a.T = T; a.H = H; a.scale = scale;
  a.lens = nullptr; a.seqs = nullptr; a.nTg = 0;
  static bool configured = false;
  if (!configured) {
    DMG_CUDA_OK(cudaFuncSetAttribute(attn_flash_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, FL_SMEM));
    DMG_CUDA_OK(cudaFuncSetAttribute(attn_flash_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, FL_SMEM));
    configured = true;
  }
  const dim3 grid(B * H * ((T + 63) / 64));
  if (bert) return launch_k(attn_flash_kernel<true, false>, grid, dim3(128), (size_t)FL_SMEM, st, 1, a);
  return launch_k(attn_flash_kernel<false, false>, grid, dim3(128), (size_t)FL_SMEM, st, 1, a);
}

// BERT encoder over the n_seqs sequences seqs_dev[] of a padded batch (qkv rows b*T_max + i, lengths lens_dev[b]); max_len = the longest
// of them (sizes the grid).  Writes only rows < lens[b].
int attn_flash_varlen(const bf16* qkv, const bf16* rd, int Dcap, const float* u, const float* v, bf16* out, const int* lens_dev,
                      const int* seqs_dev, int n_seqs, int max_len, int T_max, int H, float scale, cudaStream_t st) {
  DMG_CHECK(max_len >= 1 && max_len <= T_max && Dcap >= max_len, "attn_flash_varlen: length %d outside [1, T_max=%d] or past the rel-pos cache (%d)",
            max_len, T_max, Dcap);
  if (n_seqs <= 0) return 0;
  FlashArgs a;
  a.qkv = qkv; a.rk = rd; a.rk_hs = (long long)Dcap * 64; a.rk_ld = 64; a.rk_rows = Dcap; a.u = u; a.v = v; a.out = out;
  a.B = n_seqs; a.T = T_max; a.H = H; a.scale = scale;
  a.lens = lens_dev; a.seqs = seqs_dev; a.nTg = (max_len + 63) / 64;
  static bool configured = false;
  if (!configured) {
    DMG_CUDA_OK(cudaFuncSetAttribute(attn_flash_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, FL_SMEM));
    configured = true;
  }
  return launch_k(attn_flash_kernel<true, true>, dim3(n_seqs * H * a.nTg), dim3(128), (size_t)FL_SMEM, st, 1, a);
}

}  // namespace dmg
