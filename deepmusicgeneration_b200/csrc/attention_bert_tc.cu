// Attention of the masked-BERT remix encoder on tcgen05 / TMEM / TMA (inference, bf16), for sequences of at least 128 tokens.
//
// Replaces MemMultiHeadRelativeAttentionKV._apply_attention (deep_music_remix.py:2078-2104; a14-a18 of SURVEY.md section 8):
//   softmax(((q+u) K^T + _line_shift((q+v) Rk^T, mask=False)) / sqrt(Dh)) V        - no mask, no dropout, no out-projection
// where the unmasked _line_shift keeps all three "lines" of the padded reshape alive:
//   j <= i   : BD[i, j] = (q_i + v)     . Rk[i - j]                (line 1)
//   j == i+1 : BD[i, j] = 0                                        (line 2, the zero pad)
//   j >  i+1 : BD[i, j] = (q_{i+1} + v) . Rk[T + 1 + i - j]        (line 3: the NEXT query row, wrapped distance)
// Same scheme as attn_train_fwd_tc_kernel (attention_train_tc.cu) per work item (stream, head, 128-query tile) - but the grid is
// PERSISTENT: one CTA per SM walks its items, barriers / buffers / TMEM carry over, the next item's operands are prepared under the
// current item's last tile (attention_bert_tc_common.cuh).  Row-per-thread
// softmax warps, AC and a 256-column position strip in TMEM, skew through thread-private shared-memory lines, P as the A operand
// of the PV MMA.  The strip is strip[r][c] = BD[r, jj] with c = 128 + r - jj; below the diagonal both 128-column halves come from
// (q+v) and two consecutive 128-row blocks of Rk, above it from (q_next+v) and blocks of Rk3[x] = Rk[x + T + 1 - 128 nT] (nT key tiles;
// a TMA box may start at any row), and ON the diagonal tile line 1 only ever reads the upper half (r - jj >= 0) and line 3 only the
// lower half (r - jj <= -2), so one half of each fits the same 256 columns.  Consecutive key tiles share a block (upper half of tile
// n+1 = lower half of tile n), also across the diagonal.  A ragged last tile (T not a multiple of 128) masks its keys >= T and does
// not store its rows >= T; the boxes that reach past the sequence bring finite rows of the neighbouring sequence / head or zeros.
#include "attention_bert_tc_common.cuh"

namespace dmg {

namespace {

using namespace bert_tc;

// 2^x for x <= 0 on the FMA pipe: Cody-Waite split around the nearest integer + degree-3 polynomial on [-0.5, 0.5] (relative error
// 7.7e-5, far below the bf16 rounding of the probability it feeds).  Both softmax warps of a scheduler reach their 64 exponentials per
// row at the same time and the MUFU unit retires 4 lanes per cycle: a quarter of them computed here shortens that phase.
__device__ __forceinline__ float bt_ex2_poly(float x) {
  x = fmaxf(x, -125.f);
  const float r = x + 12582912.f;                      // 1.5 * 2^23: the nearest integer n sits in the low mantissa bits
  const float f = x - (r - 12582912.f);
  float p = fmaf(0.05508868f, f, 0.24260405f);
  p = fmaf(p, f, 0.69327624f);
  p = fmaf(p, f, 0.99992894f);
  return __int_as_float(__float_as_int(p) + (__float_as_int(r) << 23));   // p * 2^n through the exponent field
}

constexpr int BT_SOFT_WARPS = 8;
constexpr int BT_THREADS = (BT_SOFT_WARPS + 4) * 32;   // + one auxiliary warpgroup: TMA warp, MMA warp, two q-transform warps
constexpr int BT_STRIP_LD = 68;
constexpr int BO_BAR = BO_STRIP + BT_SOFT_WARPS * 32 * BT_STRIP_LD * 4;
constexpr int BT_SMEM = BO_BAR + 256 + 1024;
static_assert(BT_SMEM <= 227 * 1024, "shared memory budget");
static_assert(BO_V2 + BT16K <= BO_BAR && BO_V2 % 1024 == 0, "second V stage of the fp16-strip kernel");
static_assert(BT_SOFT_WARPS * 32 * BT_LINE16 <= BT_SOFT_WARPS * 32 * BT_STRIP_LD * 4 && 34 * 4 <= BT_LINE16, "fp16 lines fit; a line holds the merge record");

// H16: the position strip goes through shared memory as fp16 (|BD| < 65504 saturates; 11 bits of mantissa against the 8 of the bf16
// operands): the thread's two 64-column windows overlap in 32 columns, so it reads 96 distinct columns once (three tcgen05.ld.x32
// instead of four), stores 12 instead of 32 16-byte chunks and reads its 64 scores back as 33 aligned words + funnel shifts - 40 % of
// the shared-memory wavefronts of the fp32 line (the kernel sits on the shared-memory pipe, profiles/r1g_attn_bert_tc_ncu.txt).
//
// VARLEN: a padded batch of sequences of their own lengths (a.lens, each >= 128) walked through the host-built item list a.items; every
// item is computed as it would be with T = its sequence's length, at row stride a.T.  Keys past the end are masked by a select and
// the V rows there are zeroed in shared memory, so the padding rows may hold anything (NaN included).
template <bool H16, bool VARLEN>
__global__ void __launch_bounds__(BT_THREADS, 1)
attn_bert_tc_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmR, const BertTcArgs a) {
  extern __shared__ __align__(1024) uint8_t bt_smem_raw[];
  uint8_t* smem = bt_smem_raw + ((1024u - (smem_u32(bt_smem_raw) & 1023u)) & 1023u);
  uint64_t* bar = (uint64_t*)(smem + BO_BAR);
  uint32_t* tmem_holder = (uint32_t*)(bar + Q_COUNT);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int NT_all = (a.T + 127) / 128;              // a ragged last tile: keys >= T are masked, rows >= T are not stored
  const int n_items = VARLEN ? a.n_items : a.B * a.H * NT_all;   // every query tile sees all NT key tiles: uniform work
  const int HD = a.H * 64;

  if (warp == BT_SOFT_WARPS && lane == 0) {
    tma_prefetch_desc(&tmX);
    tma_prefetch_desc(&tmR);
    bt_init_barriers(bar, BT_SOFT_WARPS);
  }
  if (warp == BT_SOFT_WARPS + 1) tmem_alloc<512>(tmem_holder);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;
  pdl_launch_dependents();

  if (warp >= BT_SOFT_WARPS) {
    // register pool of the CTA: 384 threads x 168 at launch; 128 auxiliary threads give back 104 each (13312), the 256 softmax threads
    // take 48 each (12288) - an increase beyond what was given back would wait forever
    asm volatile("setmaxnreg.dec.sync.aligned.u32 64;");
    if (warp == BT_SOFT_WARPS) {
      // =========================================== TMA producer ===========================================
      if (lane == 0) bt_producer<H16 ? 2 : 1, VARLEN>(smem, bar, tmX, tmR, a, NT_all, n_items);
    } else if (warp == BT_SOFT_WARPS + 1) {
      // =========================================== MMA issuer ===========================================
      bt_mma_issuer<H16 ? 2 : 1, VARLEN>(smem, bar, tmem_base, NT_all, n_items, a, a.dbg);   // the whole warp: uniform control flow
    } else {
      // =========================================== transform warps ===========================================
      bt_transform<VARLEN>(smem, bar, a, NT_all, n_items, threadIdx.x - 32 * (BT_SOFT_WARPS + 2));
    }
  } else {
    // =========================================== softmax warps ===========================================
    asm volatile("setmaxnreg.inc.sync.aligned.u32 216;");
    const int hf = warp >> 2, q4 = warp & 3;
    const int r = q4 * 32 + lane;                   // query row of this thread inside the tile
    const uint32_t t_lane = tmem_base + ((uint32_t)(q4 * 32) << 16);
    float* strip = (float*)(smem + BO_STRIP) + (size_t)(warp * 32 + lane) * BT_STRIP_LD;
    const float c = a.scale * BT_LOG2E;
    uint8_t* prow = smem + BO_P + hf * BT16K + (r >> 3) * 1024 + (r & 7) * 128;

    int kit = 0, gsum = 0;                          // items this CTA has finished: the barriers count on across items
    for (int item = blockIdx.x; item < n_items; item += gridDim.x, kit++) {
    int b, h, it, T, NT;
    if constexpr (VARLEN) {
      const BtVarItem wi = bt_var_item(a, item);
      b = wi.b; h = wi.h; it = wi.it; T = wi.T; NT = wi.NT;
    } else {
      const BtItem wi = bt_item(item, NT_all, a.H);
      b = wi.b; h = wi.h; it = wi.it; T = a.T; NT = NT_all;
    }
    const int i0 = it * 128, row = i0 + r;
    const int g0 = VARLEN ? gsum : kit * NT;
    if constexpr (VARLEN) gsum += NT;

    float o[64];
#pragma unroll
    for (int i = 0; i < 64; i++) o[i] = 0.f;
    float m_run = -INFINITY, l_run = 0.f, alpha_prev = 1.f;
    // the zero pad of _line_shift: key j = i + 1 (tile (row+1)/128, local key (row+1)%128; for the last row of a tile that is key 0
    // of the NEXT tile)
    const int zero_tile = (row + 1) >> 7, zero_jj = ((((row + 1) & 127) >> 6) == hf) ? ((row + 1) & 63) : -1000;

    for (int n = 0; n < NT; n++) {
      float s[64];
      const int mslot = 256 * hf + 48 * kit + 5 * n;
      const bool mk = q4 == 0 && lane == 0 && NT <= 8;
      if (mk) bt_mark(a.dbg, mslot, kit);
      bt_wait(&bar[Q_SFULL], (g0 + n) & 1);
      tc_fence_after();
      if (mk) bt_mark(a.dbg, mslot + 1, kit);
      const int zj = n == zero_tile ? zero_jj : -1000;
      if constexpr (H16) {
        // strip columns [wbase, wbase + 96) -> fp16 -> this thread's line; score of local key jj (0..63) = line[64 + lane - jj]
        const uint32_t wbase = (uint32_t)(64 - 64 * hf + 32 * q4);
        uint8_t* line = smem + BO_STRIP + (size_t)(warp * 32 + lane) * BT_LINE16;
        {
          uint32_t x0[32], x1[32];
          tmem_ld_32x32(t_lane + BTM_STRIP + wbase, x0);
          tmem_ld_32x32(t_lane + BTM_STRIP + wbase + 32, x1);
          tmem_ld_wait();
#pragma unroll
          for (int k = 0; k < 4; k++)
            *(uint4*)(line + 16 * k) = make_uint4(bt_f16x2_sat(__uint_as_float(x0[8 * k]), __uint_as_float(x0[8 * k + 1])),
                                                  bt_f16x2_sat(__uint_as_float(x0[8 * k + 2]), __uint_as_float(x0[8 * k + 3])),
                                                  bt_f16x2_sat(__uint_as_float(x0[8 * k + 4]), __uint_as_float(x0[8 * k + 5])),
                                                  bt_f16x2_sat(__uint_as_float(x0[8 * k + 6]), __uint_as_float(x0[8 * k + 7])));
          tmem_ld_32x32(t_lane + BTM_STRIP + wbase + 64, x0);
#pragma unroll
          for (int k = 0; k < 4; k++)
            *(uint4*)(line + 64 + 16 * k) = make_uint4(bt_f16x2_sat(__uint_as_float(x1[8 * k]), __uint_as_float(x1[8 * k + 1])),
                                                       bt_f16x2_sat(__uint_as_float(x1[8 * k + 2]), __uint_as_float(x1[8 * k + 3])),
                                                       bt_f16x2_sat(__uint_as_float(x1[8 * k + 4]), __uint_as_float(x1[8 * k + 5])),
                                                       bt_f16x2_sat(__uint_as_float(x1[8 * k + 6]), __uint_as_float(x1[8 * k + 7])));
          tmem_ld_32x32(t_lane + BTM_AC + 64 * hf, x1);
          tmem_ld_wait();
#pragma unroll
          for (int k = 0; k < 4; k++)
            *(uint4*)(line + 128 + 16 * k) = make_uint4(bt_f16x2_sat(__uint_as_float(x0[8 * k]), __uint_as_float(x0[8 * k + 1])),
                                                        bt_f16x2_sat(__uint_as_float(x0[8 * k + 2]), __uint_as_float(x0[8 * k + 3])),
                                                        bt_f16x2_sat(__uint_as_float(x0[8 * k + 4]), __uint_as_float(x0[8 * k + 5])),
                                                        bt_f16x2_sat(__uint_as_float(x0[8 * k + 6]), __uint_as_float(x0[8 * k + 7])));
          tmem_ld_32x32(t_lane + BTM_AC + 64 * hf + 32, x0);
          tmem_ld_wait();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&bar[Q_SFREE]);
          if (mk) bt_mark(a.dbg, mslot + 2, kit);
#pragma unroll
          for (int i = 0; i < 32; i++) { s[i] = __uint_as_float(x1[i]); s[32 + i] = __uint_as_float(x0[i]); }
        }
        const int S_h = 64 + lane;                   // half index of local key 0
        if ((unsigned)zj < 64u) ((__half*)line)[S_h - zj] = __float2half(0.f);   // the zero pad: one slot of the line
        asm volatile("" ::: "memory");              // the word reads below alias the stores above
        const uint32_t* rdw = (const uint32_t*)line + (S_h >> 1);   // word k back holds halves S' - 2k - 1 (low), S' - 2k (high), S' = S_h | 1
        const uint32_t sh = (S_h & 1) ? 0u : 16u;   // lanes with an even S_h shift the word chain by one half
        uint32_t wprev = rdw[0];
#pragma unroll
        for (int k = 0; k < 32; k++) {
          const uint32_t wnext = rdw[-(k + 1)];
          const uint32_t x = __funnelshift_l(wnext, wprev, sh);
          const __half2 h2 = *reinterpret_cast<const __half2*>(&x);
          s[2 * k] += __high2float(h2);
          s[2 * k + 1] += __low2float(h2);
          wprev = wnext;
        }
      } else {
      {
        uint32_t x0[32], x1[32];
        tmem_ld_32x32(t_lane + BTM_AC + 64 * hf, x0);
        tmem_ld_32x32(t_lane + BTM_AC + 64 * hf + 32, x1);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 32; i++) { s[i] = __uint_as_float(x0[i]); s[32 + i] = __uint_as_float(x1[i]); }
      }
#pragma unroll
      for (int sp = 0; sp < 2; sp++) {
        const uint32_t base = (uint32_t)(96 - 64 * hf - 32 * sp + 32 * q4);
        {
          uint32_t x0[32], x1[32];
          tmem_ld_32x32(t_lane + BTM_STRIP + base, x0);
          tmem_ld_32x32(t_lane + BTM_STRIP + base + 32, x1);
          tmem_ld_wait();
          if (sp == 1) {
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&bar[Q_SFREE]);
          }
#pragma unroll
          for (int k = 0; k < 8; k++) {
            *(float4*)(strip + 4 * k) = make_float4(__uint_as_float(x0[4 * k]), __uint_as_float(x0[4 * k + 1]),
                                                    __uint_as_float(x0[4 * k + 2]), __uint_as_float(x0[4 * k + 3]));
            *(float4*)(strip + 32 + 4 * k) = make_float4(__uint_as_float(x1[4 * k]), __uint_as_float(x1[4 * k + 1]),
                                                         __uint_as_float(x1[4 * k + 2]), __uint_as_float(x1[4 * k + 3]));
          }
        }
        const float* sk = strip + 32 + lane;
        if ((unsigned)(zj - 32 * sp) < 32u) strip[32 + lane - (zj - 32 * sp)] = 0.f;   // the zero pad: one slot of the line, no select per key
#pragma unroll
        for (int jj = 0; jj < 32; jj++) s[32 * sp + jj] += sk[-jj];
      }

      }

      if (n == NT - 1 && (T & 127)) {                // ragged last tile: keys past the sequence end
        const int jlim = T - n * 128 - 64 * hf;
#pragma unroll
        for (int jj = 0; jj < 64; jj++) s[jj] = jj < jlim ? s[jj] : -INFINITY;
      }

      if (n > 0) {                                   // fold the previous tile's P V into the running output
        bt_wait(&bar[Q_OFULL0 + hf], (g0 + n - 1) & 1);
        tc_fence_after();
#pragma unroll
        for (int ch = 0; ch < 2; ch++) {
          uint32_t x[32];
          tmem_ld_32x32(t_lane + BTM_O + 64 * hf + 32 * ch, x);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 32; i++) o[32 * ch + i] = fmaf(o[32 * ch + i], alpha_prev, __uint_as_float(x[i]));
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bar[Q_OFREE0 + hf]);
      }
      if (mk) bt_mark(a.dbg, mslot + 3, kit);

      float mx = -INFINITY;
#pragma unroll
      for (int jj = 0; jj < 64; jj++) mx = fmaxf(mx, s[jj]);
      const float m_new = fmaxf(m_run, mx);
      const float alpha = ex2_fast((m_run - m_new) * c);        // exp2(-inf) = 0 on the first tile
      const float neg_mc = -m_new * c;
      m_run = m_new;
      float rs = 0.f;
#pragma unroll
      for (int ck = 0; ck < 8; ck++) {
        uint32_t pk[4];
#pragma unroll
        for (int e = 0; e < 4; e++) {
          const int pp = 4 * ck + e;
          const float p0 = ex2_fast(fmaf(s[2 * pp], c, neg_mc));
          const float p1 = (e & 1) ? bt_ex2_poly(fmaf(s[2 * pp + 1], c, neg_mc)) : ex2_fast(fmaf(s[2 * pp + 1], c, neg_mc));
          rs += p0 + p1;
          pk[e] = pack_bf16x2(p0, p1);
        }
        *(uint4*)(prow + ((ck ^ (r & 7)) << 4)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
      }
      l_run = l_run * alpha + rs;
      alpha_prev = alpha;
      bt_fence_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar[Q_PFULL0 + hf]);
      if (mk) bt_mark(a.dbg, mslot + 4, kit);
      if (lane == 0 && NT <= 8) bt_mark(a.dbg, 1024 + 64 * kit + 8 * n + warp, kit);
    }
    bt_wait(&bar[Q_OFULL0 + hf], (g0 + NT - 1) & 1);
    if (q4 == 0 && lane == 0 && NT <= 8) bt_mark(a.dbg, 256 * hf + 48 * kit + 40, kit);
    tc_fence_after();
#pragma unroll
    for (int ch = 0; ch < 2; ch++) {
      uint32_t x[32];
      tmem_ld_32x32(t_lane + BTM_O + 64 * hf + 32 * ch, x);
      tmem_ld_wait();
#pragma unroll
      for (int i = 0; i < 32; i++) o[32 * ch + i] = fmaf(o[32 * ch + i], alpha_prev, __uint_as_float(x[i]));
    }
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(&bar[Q_OFREE0 + hf]);   // the next item's first P V may overwrite the accumulator

    // merge the two key halves of every row, both halves at work: half 0 finishes output columns 0-31, half 1 columns 32-63; each
    // leaves the 32 accumulators the other one needs, its maximum and its row sum in ITS OWN strip line (dead since the last skew; 136
    // of its 208 / 272 bytes) and reads the line of the same row's thread in the other half (same lane, warp +- 4)
    float* wr_o; const float* rd_o;
    if constexpr (H16) {
      uint8_t* line = smem + BO_STRIP + (size_t)(warp * 32 + lane) * BT_LINE16;
      wr_o = (float*)line;
      rd_o = (const float*)(hf ? line - (size_t)4 * 32 * BT_LINE16 : line + (size_t)4 * 32 * BT_LINE16);
    } else {
      wr_o = strip;
      rd_o = hf ? strip - (size_t)4 * 32 * BT_STRIP_LD : strip + (size_t)4 * 32 * BT_STRIP_LD;
    }
    float* wr_s = wr_o + 32;
    const float* rd_s = rd_o + 32;
#pragma unroll
    for (int k = 0; k < 8; k++)
      *(float4*)(wr_o + 4 * k) = make_float4(hf ? o[4 * k] : o[32 + 4 * k], hf ? o[4 * k + 1] : o[32 + 4 * k + 1],
                                             hf ? o[4 * k + 2] : o[32 + 4 * k + 2], hf ? o[4 * k + 3] : o[32 + 4 * k + 3]);
    wr_s[0] = m_run;
    wr_s[1] = l_run;
    asm volatile("bar.sync 1, 256;" ::: "memory");
    if (row < T) {
      const float m1 = rd_s[0], l1 = rd_s[1];
      const float m = fmaxf(m_run, m1);
      const float w0 = ex2_fast((m_run - m) * c), w1 = ex2_fast((m1 - m) * c);
      const float inv = 1.f / (l_run * w0 + l1 * w1);
      bf16* orow = a.out + ((long long)b * a.T + row) * HD + h * 64 + 32 * hf;
#pragma unroll
      for (int k = 0; k < 4; k++) {
        uint32_t w[4];
#pragma unroll
        for (int e = 0; e < 4; e++) {
          const int d0 = 8 * k + 2 * e;
          const float mine0 = hf ? o[32 + d0] : o[d0], mine1 = hf ? o[32 + d0 + 1] : o[d0 + 1];
          w[e] = pack_bf16x2((mine0 * w0 + rd_o[d0] * w1) * inv, (mine1 * w0 + rd_o[d0 + 1] * w1) * inv);
        }
        *(uint4*)(orow + 8 * k) = make_uint4(w[0], w[1], w[2], w[3]);
      }
    }
    asm volatile("bar.sync 1, 256;" ::: "memory");   // the partner has read this line before the next item's first skew overwrites it
    if (q4 == 0 && lane == 0 && NT <= 8) bt_mark(a.dbg, 256 * hf + 48 * kit + 41, kit);
    }   // items
  }
  tc_fence_before();
  __syncthreads();
  if (warp == BT_SOFT_WARPS + 1) tmem_dealloc<512>(tmem_base);
}

}  // namespace

bool attn_bert_tc_supported(int T, int H, int Dcap) {
  return T >= 128 && Dcap >= T && H >= 1;   // T >= 128: every row has seen a full tile before the ragged one (finite running maximum)
}

// qkv: bf16 [B*T, 3*H*64] (q | k | v); rd: the inference rel-pos key cache [H][Dcap][64] (bf16, row = distance); out: bf16 [B*T, H*64]
int attn_bert_tc(const bf16* qkv, const bf16* rd, int Dcap, const float* u, const float* v, bf16* out, int B, int T, int H, float scale,
                 int fp32_strip, cudaStream_t st) {
  static bool configured = false;
  if (!configured) {
    DMG_CUDA_OK(cudaFuncSetAttribute(attn_bert_tc_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, BT_SMEM));
    DMG_CUDA_OK(cudaFuncSetAttribute(attn_bert_tc_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, BT_SMEM));
    configured = true;
  }
  const int HD = H * 64;
  const TensorMap2D *tx = nullptr, *tr = nullptr;
  if (train_get_tmap(qkv, 3 * HD, (long long)B * T, 3 * HD, 128, &tx)) return -1;
  if (train_get_tmap(rd, 64, (long long)H * Dcap, 64, 128, &tr)) return -1;
  BertTcArgs a;
  a.u = u; a.v = v; a.out = out; a.B = B; a.T = T; a.H = H; a.Dcap = Dcap; a.scale = scale;
  a.dbg = nullptr;
  a.lens = nullptr; a.items = nullptr; a.n_items = 0;
  // persistent: one CTA per SM (shared memory and all 512 TMEM columns allow one), items dealt round-robin.  DMG_BERT_TC_ONE_ITEM=1
  // (measurement only) launches one CTA per item, the schedule of rounds 1 and 2.
  static int num_sms = 0, one_item = -1;
  if (num_sms == 0) {
    int dev = 0;
    DMG_CUDA_OK(cudaGetDevice(&dev));
    DMG_CUDA_OK(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev));
    const char* e = getenv("DMG_BERT_TC_ONE_ITEM");
    one_item = e && e[0] == '1';
  }
  const int n_items = B * H * ((T + 127) / 128);
  const dim3 grid(one_item || n_items < num_sms ? n_items : num_sms);
  // DMG_BERT_TC_TIMELINE=<file> (measurement only, scripts/probe_bert_tc.py): marks of CTA 0 of every launch, the last one is kept
  static const char* tl_path = getenv("DMG_BERT_TC_TIMELINE");
  static unsigned long long* tl_dev = nullptr;
  if (tl_path && tl_path[0]) {
    if (!tl_dev) DMG_CUDA_OK(cudaMalloc(&tl_dev, 2048 * sizeof(unsigned long long)));
    DMG_CUDA_OK(cudaMemsetAsync(tl_dev, 0, 2048 * sizeof(unsigned long long), st));
    a.dbg = tl_dev;
    const int rc = fp32_strip ? launch_k(attn_bert_tc_kernel<false, false>, grid, dim3(BT_THREADS), (size_t)BT_SMEM, st, 1, *(const CUtensorMap*)tx->bytes,
                                         *(const CUtensorMap*)tr->bytes, a)
                              : launch_k(attn_bert_tc_kernel<true, false>, grid, dim3(BT_THREADS), (size_t)BT_SMEM, st, 1, *(const CUtensorMap*)tx->bytes,
                                         *(const CUtensorMap*)tr->bytes, a);
    if (rc) return rc;
    static unsigned long long host[2048];
    DMG_CUDA_OK(cudaStreamSynchronize(st));
    DMG_CUDA_OK(cudaMemcpy(host, tl_dev, sizeof(host), cudaMemcpyDeviceToHost));
    FILE* f = fopen(tl_path, "wb");
    if (f) { fwrite(host, sizeof(host), 1, f); fclose(f); }
    return 0;
  }
  if (fp32_strip)
    return launch_k(attn_bert_tc_kernel<false, false>, grid, dim3(BT_THREADS), (size_t)BT_SMEM, st, 1, *(const CUtensorMap*)tx->bytes,
                    *(const CUtensorMap*)tr->bytes, a);
  return launch_k(attn_bert_tc_kernel<true, false>, grid, dim3(BT_THREADS), (size_t)BT_SMEM, st, 1, *(const CUtensorMap*)tx->bytes,
                  *(const CUtensorMap*)tr->bytes, a);
}

// Padded batch of B sequences (qkv rows b*T_max + i): the n_items work items items_dev[] (see BertTcArgs) of the sequences with
// lens_dev[b] >= 128.  Writes only rows < lens[b].
int attn_bert_tc_varlen(const bf16* qkv, const bf16* rd, int Dcap, const float* u, const float* v, bf16* out, const int* lens_dev,
                        const int* items_dev, int n_items, int B, int T_max, int H, float scale, int fp32_strip, cudaStream_t st) {
  DMG_CHECK(T_max >= 128 && Dcap >= T_max && H <= 256 && B <= 32768, "attn_bert_tc_varlen: T_max %d / H %d / B %d outside the kernel's range", T_max, H, B);
  if (n_items <= 0) return 0;
  static bool configured = false;
  if (!configured) {
    DMG_CUDA_OK(cudaFuncSetAttribute(attn_bert_tc_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, BT_SMEM));
    DMG_CUDA_OK(cudaFuncSetAttribute(attn_bert_tc_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, BT_SMEM));
    configured = true;
  }
  const int HD = H * 64;
  const TensorMap2D *tx = nullptr, *tr = nullptr;
  if (train_get_tmap(qkv, 3 * HD, (long long)B * T_max, 3 * HD, 128, &tx)) return -1;
  if (train_get_tmap(rd, 64, (long long)H * Dcap, 64, 128, &tr)) return -1;
  BertTcArgs a;
  a.u = u; a.v = v; a.out = out; a.B = B; a.T = T_max; a.H = H; a.Dcap = Dcap; a.scale = scale;
  a.dbg = nullptr;
  a.lens = lens_dev; a.items = items_dev; a.n_items = n_items;
  int dev = 0, num_sms = 0;
  DMG_CUDA_OK(cudaGetDevice(&dev));
  DMG_CUDA_OK(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev));
  const dim3 grid(n_items < num_sms ? n_items : num_sms);
  if (fp32_strip)
    return launch_k(attn_bert_tc_kernel<false, true>, grid, dim3(BT_THREADS), (size_t)BT_SMEM, st, 1, *(const CUtensorMap*)tx->bytes,
                    *(const CUtensorMap*)tr->bytes, a);
  return launch_k(attn_bert_tc_kernel<true, true>, grid, dim3(BT_THREADS), (size_t)BT_SMEM, st, 1, *(const CUtensorMap*)tx->bytes,
                  *(const CUtensorMap*)tr->bytes, a);
}

}  // namespace dmg
