// Persistent tcgen05 GEMM for the training path (forward, input-gradient and weight-gradient contractions).
//
//   C[M,N] = A * B, reduction over K, bf16 operands, fp32 accumulation in TMEM.
//   One CTA per SM loops over 128 x BN output tiles (x split-K slices).  Warp 0 = TMA producer, warp 1 = single-thread
//   tcgen05.mma issuer, warps 2..9 = epilogue (TMEM -> registers -> fused epilogue -> global).  Two accumulator stages
//   in TMEM (2 x BN columns) let the epilogue of tile i overlap the main loop of tile i+1.
//
//   Both operands can be "K-major" (reduction index contiguous in memory: activations [rows, features] as A, nn.Linear
//   weights [out, in] as B) or "MN-major" (reduction index is the slow one: dY^T X weight gradients take both operands
//   that way, dX = dY W takes W that way), so no transposed copy of an activation or a weight is ever made.  MN-major
//   tiles are fetched as 64(mn) x 64(k) TMA boxes with the 128B swizzle; the UMMA descriptor walks them with
//   LBO = 8192 B (next 64-wide mn block) and SBO = 1024 B (next group of 8 k rows).
//
// Replaces, for training, the nn.Linear forward/backward calls of fastai's MultiHeadRelativeAttention / feed_forward /
// LinearDecoder under autograd (SURVEY.md App. A.3, 3.3).
#include <cuda.h>
#include <map>
#include <tuple>
#include "kernels.cuh"
#include "launch.cuh"
#include "train_kernels.cuh"

namespace dmg {

namespace {

constexpr int GT_BM = 128;
constexpr int GT_EPI_WARPS = 8;
constexpr int GT_THREADS = 64 + GT_EPI_WARPS * 32;

// CG = CTAs per MMA (tcgen05 cta_group): with CG = 2 a CTA pair computes one 256 x BN tile - every CTA stages its own
// 128 rows of A and only HALF of the B tile (the pair's tensor cores read both halves), which cuts the L2 -> SM operand
// traffic per flop by a third and is what lifts a K = 512 GEMM off the L2 bandwidth ceiling.
__host__ __device__ constexpr int gt_stage_bytes(int BN, int CG) { return GT_BM * 64 * 2 + (BN / CG) * 64 * 2; }
constexpr int GT_STRIP_BYTES = 6144;                           // per epilogue warp: fp32 32x32 transposition strip, or 3 bf16 boxes
constexpr int GT_EPI_STAGE_BYTES = GT_EPI_WARPS * GT_STRIP_BYTES;
__host__ __device__ constexpr int gt_stages(int BN, int CG) {
  return (176 * 1024) / gt_stage_bytes(BN, CG) > 8 ? 8 : (176 * 1024) / gt_stage_bytes(BN, CG);
}
__host__ __device__ constexpr int gt_smem_bytes(int BN, int CG) {
  return gt_stages(BN, CG) * gt_stage_bytes(BN, CG) + 1024 /*alignment*/ + 1024 /*barriers*/ + GT_EPI_STAGE_BYTES;
}

// shared-memory matrix descriptor, 128B swizzle, sm_100 version bit; lbo/sbo in bytes
__device__ __forceinline__ uint64_t umma_desc(uint32_t smem_addr, uint32_t lbo, uint32_t sbo) {
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo >> 4) << 16) | ((uint64_t)(sbo >> 4) << 32) | (1ull << 46) |
         (2ull << 61);
}

// ---- cta_group::2 forms (the CTA pair of a 2-CTA cluster; rank 0 = leader issues the MMAs)
constexpr uint32_t PEER_MASK = 0xFEFFFFFFu;   // clears the pair-rank bit of a shared-window address -> the leader CTA's copy
__device__ __forceinline__ uint32_t cluster_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// TMA load into THIS CTA's shared memory, transaction bytes reported to the LEADER's mbarrier
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const void* tmap, int c0, int c1, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(smem_dst)),
      "l"(tmap), "r"(smem_u32(bar) & PEER_MASK), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrives on the mbarrier at this offset in BOTH CTAs of the pair once the MMAs issued so far have completed
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
               "h"((uint16_t)3)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive_leader(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & PEER_MASK) : "memory");
}
// TMA store shared -> global (bulk async group), 2-D tile
__device__ __forceinline__ void tma_store_2d(const void* tmap, const void* smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(tmap), "r"(smem_u32(smem_src)),
               "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

template <int COLS>
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_holder) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_holder)), "n"(COLS) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(COLS) : "memory");
}

struct GemmTParams {
  int M, N, K;
  int a_mn, b_mn;
  int splitk, kb_per_split, num_kb;
  int num_m, num_n;
  const float* bias;
  int act;
  const void* aux; long long ld_aux; int aux_mode;
  void* out; long long ldc; int out_mode;
  bf16* out2; long long ld2;
  uint32_t drop_thresh, drop_seed; float drop_scale;
  int groups; int a_gs, b_gs; long long c_gs;
  int tma_store;   // bf16 output(s) leave through TMA stores (tmC / tmC2)
  int aux_tma;     // the bf16 aux operand arrives as 32x32 TMA boxes (tmX), prefetched one chunk ahead
};

template <int BN, int CG>
__global__ void __launch_bounds__(GT_THREADS, 1)
gemm_train_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                  const __grid_constant__ CUtensorMap tmC, const __grid_constant__ CUtensorMap tmC2,
                  const __grid_constant__ CUtensorMap tmX, const GemmTParams p) {
  constexpr int STAGES = gt_stages(BN, CG);
  constexpr int STAGE_BYTES = gt_stage_bytes(BN, CG);
  constexpr int A_BYTES = GT_BM * 64 * 2;
  constexpr int BN_CTA = BN / CG;     // B rows (N) staged by one CTA
  constexpr int TMEM_COLS = 2 * BN;   // 128 / 256 / 512: powers of two
  extern __shared__ uint8_t gt_smem_raw[];
  uint8_t* tiles = (uint8_t*)(((uintptr_t)gt_smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* full = (uint64_t*)(tiles + STAGES * STAGE_BYTES);
  uint64_t* empty = full + STAGES;
  uint64_t* tmem_full = empty + STAGES;     // [2]
  uint64_t* tmem_empty = tmem_full + 2;     // [2]
  uint32_t* tmem_holder = (uint32_t*)(tmem_empty + 2);
  uint64_t* aux_bar = (uint64_t*)(tiles + STAGES * STAGE_BYTES + 512);  // [8 epilogue warps][2 buffers]
  uint8_t* stage_all = tiles + STAGES * STAGE_BYTES + 1024;             // 8 epilogue warps x 6 KB, 2048-byte aligned strips

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int rank = CG == 2 ? (int)cluster_rank() : 0;          // position in the CTA pair
  const int unit = blockIdx.x / CG, num_units = gridDim.x / CG; // a "unit" (CTA or CTA pair) owns whole tiles
  const int tiles_mn = p.num_m * p.num_n;
  const int tiles_g = tiles_mn * p.splitk;
  const int total = tiles_g * p.groups;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    if (p.tma_store) {
      tma_prefetch_desc(&tmC);
      if (p.out2) tma_prefetch_desc(&tmC2);
      if (p.aux_tma) tma_prefetch_desc(&tmX);
    }
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; s++) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int s = 0; s < 2 * GT_EPI_WARPS; s++) mbar_init(&aux_bar[s], 1);
    for (int s = 0; s < 2; s++) {
      mbar_init(&tmem_full[s], 1);
      mbar_init(&tmem_empty[s], GT_EPI_WARPS * CG);   // the leader's barrier collects the epilogue warps of both CTAs
    }
    mbar_fence_init();
  }
  if (warp == 2) {
    if (CG == 2) tmem_alloc_pair<TMEM_COLS>(tmem_holder);
    else tmem_alloc<TMEM_COLS>(tmem_holder);
  }
  tc_fence_before();
  if (CG == 2) cluster_sync();
  else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      uint32_t it = 0;
      for (int t = unit; t < total; t += num_units) {
        const int grp = t / tiles_g, tg = t - grp * tiles_g;
        const int ks = tg / tiles_mn, r = tg - ks * tiles_mn;
        const int m0 = (r % p.num_m) * (GT_BM * CG) + rank * GT_BM + grp * p.a_gs;
        const int n0 = (r / p.num_m) * BN + rank * BN_CTA + grp * p.b_gs;
        const int kb_lo = ks * p.kb_per_split;
        const int kb_hi = min(p.num_kb, kb_lo + p.kb_per_split);
        for (int kb = kb_lo; kb < kb_hi; kb++, it++) {
          const int s = it % STAGES;
          const uint32_t ph = (it / STAGES) & 1;
          mbar_wait(&empty[s], ph ^ 1);
          if (rank == 0) mbar_expect_tx(&full[s], STAGE_BYTES * CG);   // the pair's bytes all land on the leader's barrier
          uint8_t* a_dst = tiles + s * STAGE_BYTES;
          uint8_t* b_dst = a_dst + A_BYTES;
          if (CG == 2) {
            if (!p.a_mn) {
              tma_load_2d_pair(a_dst, &tmA, kb * 64, m0, &full[s]);
            } else {
#pragma unroll
              for (int j = 0; j < GT_BM / 64; j++) tma_load_2d_pair(a_dst + j * 8192, &tmA, m0 + j * 64, kb * 64, &full[s]);
            }
            if (!p.b_mn) {
              tma_load_2d_pair(b_dst, &tmB, kb * 64, n0, &full[s]);
            } else {
#pragma unroll
              for (int j = 0; j < BN_CTA / 64; j++) tma_load_2d_pair(b_dst + j * 8192, &tmB, n0 + j * 64, kb * 64, &full[s]);
            }
          } else {
            if (!p.a_mn) {
              tma_load_2d(a_dst, &tmA, kb * 64, m0, &full[s]);
            } else {
#pragma unroll
              for (int j = 0; j < GT_BM / 64; j++) tma_load_2d(a_dst + j * 8192, &tmA, m0 + j * 64, kb * 64, &full[s]);
            }
            if (!p.b_mn) {
              tma_load_2d(b_dst, &tmB, kb * 64, n0, &full[s]);
            } else {
#pragma unroll
              for (int j = 0; j < BN_CTA / 64; j++) tma_load_2d(b_dst + j * 8192, &tmB, n0 + j * 64, kb * 64, &full[s]);
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA of the pair only) =====================
    if (rank == 0) {
      const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)p.a_mn << 15) | ((uint32_t)p.b_mn << 16) |
                             ((uint32_t)(BN >> 3) << 17) | ((uint32_t)((GT_BM * CG) >> 4) << 24);
      const uint32_t a_lbo = p.a_mn ? 8192u : 16u, a_kstep = p.a_mn ? 2048u : 32u;
      const uint32_t b_lbo = p.b_mn ? 8192u : 16u, b_kstep = p.b_mn ? 2048u : 32u;
      uint32_t it = 0, tile_i = 0;
      for (int t = unit; t < total; t += num_units, tile_i++) {
        const int ks = (t % tiles_g) / tiles_mn;
        const int kb_lo = ks * p.kb_per_split;
        const int kb_hi = min(p.num_kb, kb_lo + p.kb_per_split);
        const uint32_t acc = tile_i & 1, acc_ph = (tile_i >> 1) & 1;
        mbar_wait(&tmem_empty[acc], acc_ph ^ 1);     // the epilogue (of both CTAs) has drained this accumulator stage
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
        for (int kb = kb_lo; kb < kb_hi; kb++, it++) {
          const int s = it % STAGES;
          const uint32_t ph = (it / STAGES) & 1;
          mbar_wait(&full[s], ph);
          tc_fence_after();
          // descriptors in uniform control flow, issue under elect_one: the operands of tcgen05.mma live in uniform registers, and behind
          // an `if (lane == 0)` ptxas wraps every MMA in a vector-to-uniform move loop (5 R2UR + elect + predicate shuffles + branch) and
          // rebuilds both descriptors - ~19 instructions per MMA of one thread against the 128 cycles a 256 x 256 x 16 pair MMA takes
          const uint32_t a_addr = smem_u32(tiles + s * STAGE_BYTES);
          const uint64_t da0 = umma_desc(a_addr, a_lbo, 1024u), db0 = umma_desc(a_addr + A_BYTES, b_lbo, 1024u);
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < 4; k++) {
              const uint64_t da = da0 + (uint64_t)(k * (a_kstep >> 4)), db = db0 + (uint64_t)(k * (b_kstep >> 4));
              const uint32_t accum = (uint32_t)((kb > kb_lo) || k > 0);
              if (CG == 2) umma_bf16_pair(d_tmem, da, db, idesc, accum);
              else umma_bf16(d_tmem, da, db, idesc, accum);
            }
            if (CG == 2) {
              umma_commit_pair(&empty[s]);                     // frees the stage in both CTAs
              if (kb == kb_hi - 1) umma_commit_pair(&tmem_full[acc]);
            } else {
              umma_commit(&empty[s]);
              if (kb == kb_hi - 1) umma_commit(&tmem_full[acc]);
            }
          }
          __syncwarp();
        }
      }
    }
  } else {
    // ===================== epilogue =====================
    const int ew = warp - 2;
    const int q = warp & 3;                  // TMEM lane quarter this warp may read
    const int half = ew >> 2;                // column half of the tile
    float4* stg = (float4*)(stage_all + ew * GT_STRIP_BYTES);
    uint64_t* xbar = aux_bar + 2 * ew;
    uint32_t xcnt = 0;                       // aux boxes consumed so far by this warp (buffer = xcnt & 1, parity = (xcnt >> 1) & 1)
    constexpr int HALF_COLS = BN / 2;
    uint32_t tile_i = 0;
    for (int t = unit; t < total; t += num_units, tile_i++) {
      const int grp = t / tiles_g, tg = t - grp * tiles_g;
      const int ks = tg / tiles_mn, r = tg - ks * tiles_mn;
      const int m0 = (r % p.num_m) * (GT_BM * CG) + rank * GT_BM, n0 = (r / p.num_m) * BN;
      const long long c_off = (long long)grp * p.c_gs;
      const uint32_t acc = tile_i & 1, acc_ph = (tile_i >> 1) & 1;
      if (p.aux_tma && lane == 0) {          // first aux box of the tile: in flight while the MMAs of this tile finish
        mbar_expect_tx(&xbar[xcnt & 1], 2048);
        tma_load_2d((uint8_t*)stg + 2048 + (xcnt & 1) * 2048, &tmX, n0 + half * HALF_COLS, m0 + q * 32, &xbar[xcnt & 1]);
      }
      mbar_wait(&tmem_full[acc], acc_ph);
      tc_fence_after();
      const bool first_split = ks == 0;
#pragma unroll 1
      for (int c = 0; c < HALF_COLS; c += 32) {
        uint32_t rr[32];
        const int ccol = half * HALF_COLS + c;
        tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + acc * BN + (uint32_t)ccol, rr);
        tmem_ld_wait();
        if (c + 32 >= HALF_COLS) {            // last read of this accumulator stage by this warp: hand it back
          tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            if (CG == 2) mbar_arrive_leader(&tmem_empty[acc]);
            else mbar_arrive(&tmem_empty[acc]);
          }
        }
        if (p.tma_store) {
          // ---- bf16 output: row-per-lane math in registers, 32x32 bf16 box staged in shared memory (64B-swizzled rows),
          // one TMA store per box; out-of-range rows / columns are clipped by the tensor map
          const int col0 = n0 + ccol, row = m0 + q * 32 + lane;
          float v[32];
#pragma unroll
          for (int j = 0; j < 32; j++) v[j] = __uint_as_float(rr[j]);
          if (p.bias && first_split) {
#pragma unroll
            for (int j = 0; j < 8; j++) {
              const float4 bq = (col0 + 4 * j < p.N) ? __ldg((const float4*)(p.bias + col0) + j) : make_float4(0.f, 0.f, 0.f, 0.f);
              v[4 * j] += bq.x; v[4 * j + 1] += bq.y; v[4 * j + 2] += bq.z; v[4 * j + 3] += bq.w;
            }
          }
          uint8_t* strip = (uint8_t*)stg;             // 4 KB per warp: two 2 KB boxes
          const uint32_t sw = (uint32_t)((lane >> 1) & 3);
          if (lane == 0) tma_store_wait_read<0>();     // the boxes of the previous chunk have been read out
          __syncwarp();
          float g2[32];                               // act = 2: the saved backward factor gelu'(pre) (dropout applied below)
          if (p.act == GEMM_ACT_GELU_GRADSAVE) {
#pragma unroll
            for (int j = 0; j < 32; j++) {
              const float x = v[j], kk = 0.7978845608028654f, cc = 0.044715f;
              const float x2 = x * x;
              const float t = tanh_fast(x * fmaf(kk * cc, x2, kk));
              const float hx = 0.5f * x;
              v[j] = fmaf(hx, t, hx);
              g2[j] = fmaf(hx * (1.f - t * t), fmaf(3.f * kk * cc, x2, kk), fmaf(0.5f, t, 0.5f));
            }
          } else if (p.act) {
#pragma unroll
            for (int j = 0; j < 32; j++) v[j] = gelu_tanh_fast(v[j]);
          }
          if (p.aux_tma) {
            if (lane == 0 && c + 32 < HALF_COLS) {     // prefetch the next chunk's box into the other buffer
              mbar_expect_tx(&xbar[(xcnt + 1) & 1], 2048);
              tma_load_2d(strip + 2048 + ((xcnt + 1) & 1) * 2048, &tmX, col0 + 32, m0 + q * 32, &xbar[(xcnt + 1) & 1]);
            }
            mbar_wait(&xbar[xcnt & 1], (xcnt >> 1) & 1);
            const uint8_t* xb = strip + 2048 + (xcnt & 1) * 2048 + lane * 64;
#pragma unroll
            for (int j = 0; j < 4; j++) {
              const uint4 w = *(const uint4*)(xb + ((j ^ sw) << 4));
              const float a8[8] = {bf16lo(w.x), bf16hi(w.x), bf16lo(w.y), bf16hi(w.y), bf16lo(w.z), bf16hi(w.z), bf16lo(w.w), bf16hi(w.w)};
#pragma unroll
              for (int e = 0; e < 8; e++) {
                if (p.aux_mode == GEMM_AUX_MUL_BF16) v[8 * j + e] *= a8[e];
                else v[8 * j + e] += a8[e];
              }
            }
            xcnt++;
          } else if (p.aux_mode == GEMM_AUX_ADD_BF16 || p.aux_mode == GEMM_AUX_MUL_BF16) {
            if (row < p.M) {
              const bf16* ax = (const bf16*)p.aux + (size_t)row * p.ld_aux + col0;
#pragma unroll
              for (int j = 0; j < 4; j++) {
                if (col0 + 8 * j < p.N) {
                  const uint4 w = __ldg((const uint4*)ax + j);
                  const float a8[8] = {bf16lo(w.x), bf16hi(w.x), bf16lo(w.y), bf16hi(w.y), bf16lo(w.z), bf16hi(w.z), bf16lo(w.w), bf16hi(w.w)};
#pragma unroll
                  for (int e = 0; e < 8; e++) {
                    if (p.aux_mode == GEMM_AUX_MUL_BF16) v[8 * j + e] *= a8[e];
                    else v[8 * j + e] += a8[e];
                  }
                }
              }
            }
          }
          if (p.drop_thresh) {
            const uint32_t e0 = ((uint32_t)row * (uint32_t)p.N + (uint32_t)col0) >> 1;
#pragma unroll
            for (int j = 0; j < 32; j += 2) {
              const uint32_t h = drop_pair_bits(p.drop_seed, e0 + (j >> 1));
              v[j] = ((h & 0xFFFFu) >= p.drop_thresh) ? v[j] * p.drop_scale : 0.f;
              v[j + 1] = ((h >> 16) >= p.drop_thresh) ? v[j + 1] * p.drop_scale : 0.f;
              if (p.act == GEMM_ACT_GELU_GRADSAVE) {
                g2[j] = ((h & 0xFFFFu) >= p.drop_thresh) ? g2[j] * p.drop_scale : 0.f;
                g2[j + 1] = ((h >> 16) >= p.drop_thresh) ? g2[j + 1] * p.drop_scale : 0.f;
              }
            }
          }
          if (p.act == GEMM_ACT_GELU_GRADSAVE) {
#pragma unroll
            for (int j = 0; j < 4; j++)
              *(uint4*)(strip + 2048 + lane * 64 + ((j ^ sw) << 4)) =
                  make_uint4(pack_bf16x2(g2[8 * j], g2[8 * j + 1]), pack_bf16x2(g2[8 * j + 2], g2[8 * j + 3]),
                             pack_bf16x2(g2[8 * j + 4], g2[8 * j + 5]), pack_bf16x2(g2[8 * j + 6], g2[8 * j + 7]));
          }
#pragma unroll
          for (int j = 0; j < 4; j++)
            *(uint4*)(strip + lane * 64 + ((j ^ sw) << 4)) =
                make_uint4(pack_bf16x2(v[8 * j], v[8 * j + 1]), pack_bf16x2(v[8 * j + 2], v[8 * j + 3]),
                           pack_bf16x2(v[8 * j + 4], v[8 * j + 5]), pack_bf16x2(v[8 * j + 6], v[8 * j + 7]));
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0 && col0 < p.N && m0 + q * 32 < p.M) {
            tma_store_2d(&tmC, strip, col0 + (int)c_off, m0 + q * 32);
            if (p.out2) tma_store_2d(&tmC2, strip + 2048, col0, m0 + q * 32);
            tma_store_commit();
          }
          continue;
        }
        // ---- transpose through the warp's staging strip so that every global access of a warp instruction covers
        // 4 rows x 128 contiguous bytes (the 32x32b TMEM layout alone gives one row per lane = 32 lines per instruction)
        const int col0 = n0 + ccol;
#pragma unroll
        for (int jq = 0; jq < 8; jq++)
          stg[lane * 8 + (jq ^ (lane & 7))] = make_float4(__uint_as_float(rr[4 * jq]), __uint_as_float(rr[4 * jq + 1]),
                                                          __uint_as_float(rr[4 * jq + 2]), __uint_as_float(rr[4 * jq + 3]));
        __syncwarp();
        const int cq = lane & 7, rsub = lane >> 3;
        const int col = col0 + 4 * cq;                // this lane's 4 columns (N % 4 == 0)
        if (col < p.N) {
          float4 bias4 = make_float4(0.f, 0.f, 0.f, 0.f);
          if (p.bias && first_split) bias4 = __ldg((const float4*)(p.bias + col));
#pragma unroll 2
          for (int k = 0; k < 8; k++) {
            const int rloc = 4 * k + rsub;
            const int row = m0 + q * 32 + rloc;
            if (row >= p.M) continue;
            const float4 sv = stg[rloc * 8 + (cq ^ (rloc & 7))];
            float v[4] = {sv.x + bias4.x, sv.y + bias4.y, sv.z + bias4.z, sv.w + bias4.w};
            if (p.act) {
#pragma unroll
              for (int e = 0; e < 4; e++) v[e] = gelu_tanh_fast(v[e]);
            }
            if (p.aux_mode == GEMM_AUX_ADD_BF16) {
              const uint2 w = __ldg((const uint2*)((const bf16*)p.aux + (size_t)row * p.ld_aux + col));
              const float a[4] = {bf16lo(w.x), bf16hi(w.x), bf16lo(w.y), bf16hi(w.y)};
#pragma unroll
              for (int e = 0; e < 4; e++) v[e] += a[e];
            } else if (p.aux_mode == GEMM_AUX_ADD_F32) {
              const float4 w = *((const float4*)((const float*)p.aux + (size_t)row * p.ld_aux + col));
              v[0] += w.x; v[1] += w.y; v[2] += w.z; v[3] += w.w;
            }
            if (p.drop_thresh) {
              // element index = row * N + col (a multiple of 4): two pair hashes
              const uint32_t e0 = ((uint32_t)row * (uint32_t)p.N + (uint32_t)col) >> 1;
              const uint32_t h0 = drop_pair_bits(p.drop_seed, e0), h1 = drop_pair_bits(p.drop_seed, e0 + 1);
              v[0] = ((h0 & 0xFFFFu) >= p.drop_thresh) ? v[0] * p.drop_scale : 0.f;
              v[1] = ((h0 >> 16) >= p.drop_thresh) ? v[1] * p.drop_scale : 0.f;
              v[2] = ((h1 & 0xFFFFu) >= p.drop_thresh) ? v[2] * p.drop_scale : 0.f;
              v[3] = ((h1 >> 16) >= p.drop_thresh) ? v[3] * p.drop_scale : 0.f;
            }
            if (p.out_mode == GEMM_OUT_BF16) {
              *(uint2*)((bf16*)p.out + (size_t)row * p.ldc + col + c_off) = make_uint2(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]));
            } else if (p.out_mode == GEMM_OUT_F32) {
              *(float4*)((float*)p.out + (size_t)row * p.ldc + col + c_off) = make_float4(v[0], v[1], v[2], v[3]);
            } else {
              float* o = (float*)p.out + (size_t)row * p.ldc + col + c_off;
              asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(o), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]) : "memory");
            }
          }
        }
        __syncwarp();                                 // the strip is rewritten by the next chunk
      }
    }
  }
  if (warp >= 2 && lane == 0 && p.tma_store) tma_store_wait_all();   // staged boxes must be out before the CTA retires
  tc_fence_before();
  if (CG == 2) cluster_sync();      // the leader's MMAs read the peer's shared memory: nobody leaves early
  else __syncthreads();
  if (warp == 2) {
    if (CG == 2) tmem_dealloc_pair<TMEM_COLS>(tmem_base);
    else tmem_dealloc<TMEM_COLS>(tmem_base);
  }
}

// ---- tensor-map cache: the training step re-issues the same few hundred (buffer, shape) pairs every iteration
typedef std::tuple<const void*, long long, long long, long long, int> TmKey;
std::map<TmKey, TensorMap2D>& tm_cache() {
  static std::map<TmKey, TensorMap2D> c;
  return c;
}
int get_tmap(const void* base, long long inner, long long rows, long long ld, int box_rows, const TensorMap2D** out) {
  TmKey k(base, inner, rows, ld, box_rows);
  auto& c = tm_cache();
  auto it = c.find(k);
  if (it == c.end()) {
    TensorMap2D tm;
    if (box_rows < 0) { if (make_tmap_bf16_store(&tm, base, inner, rows, ld)) return -1; }   // box_rows = -1: output (store) map
    else if (make_tmap_bf16_ex(&tm, base, inner, rows, ld, box_rows)) return -1;
    if (c.size() > 8192) c.clear();
    it = c.emplace(k, tm).first;
  }
  *out = &it->second;
  return 0;
}

template <int BN, int CG>
int launch_gt(const TensorMap2D* ta, const TensorMap2D* tb, const TensorMap2D* tc, const TensorMap2D* tc2, const TensorMap2D* tx,
              const GemmTParams& p, int grid, cudaStream_t st) {
  static bool configured = false;
  if (!configured) {
    DMG_CUDA_OK(cudaFuncSetAttribute(gemm_train_kernel<BN, CG>, cudaFuncAttributeMaxDynamicSharedMemorySize, gt_smem_bytes(BN, CG)));
    configured = true;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(GT_THREADS);
  cfg.dynamicSmemBytes = (size_t)gt_smem_bytes(BN, CG);
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CG; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = CG > 1 ? 1 : 0;
  DMG_CUDA_OK(cudaLaunchKernelEx(&cfg, gemm_train_kernel<BN, CG>, *(const CUtensorMap*)ta->bytes, *(const CUtensorMap*)tb->bytes,
                                 *(const CUtensorMap*)tc->bytes, *(const CUtensorMap*)tc2->bytes, *(const CUtensorMap*)tx->bytes, p));
  g_launch_count++;
  return 0;
}

}  // namespace

// tensor-map cache for the other training kernels (attention_train_tc.cu): [rows, inner] bf16, 64-column x box_rows boxes
int train_get_tmap(const void* base, long long inner, long long rows, long long ld, int box_rows, const TensorMap2D** out) {
  return get_tmap(base, inner, rows, ld, box_rows, out);
}

int gemm_bf16_tc(const bf16* A, int a_mn, long long lda, const bf16* B, int b_mn, long long ldb, int M, int N, int K,
                 int splitk, const GemmEpi& e, int num_sms, cudaStream_t st) {
  if (M <= 0 || N <= 0) return 0;
  DMG_CHECK(K > 0, "gemm_bf16_tc: K=%d", K);
  DMG_CHECK(A && B && e.out, "gemm_bf16_tc: null operand");
  DMG_CHECK(lda % 8 == 0 && ldb % 8 == 0, "gemm_bf16_tc: operand row strides must be multiples of 8 (lda=%lld ldb=%lld)", lda, ldb);
  DMG_CHECK(splitk >= 1 && (splitk == 1 || e.out_mode == GEMM_OUT_ATOMIC), "gemm_bf16_tc: split-K needs the atomic output mode");
  DMG_CHECK(e.out_mode == GEMM_OUT_BF16 ? e.ldc % 8 == 0 : e.ldc % 4 == 0, "gemm_bf16_tc: output row stride %lld misaligned", e.ldc);
  DMG_CHECK((e.out2 != nullptr) == (e.act == GEMM_ACT_GELU_GRADSAVE),
            "gemm_bf16_tc: a second output goes with the gradient-saving GeLU epilogue (act 2) and only with it (act=%d)", e.act);
  DMG_CHECK(!e.out2 || e.ld2 % 8 == 0, "gemm_bf16_tc: second output row stride misaligned");
  DMG_CHECK(e.aux_mode == GEMM_AUX_NONE || e.aux_mode == GEMM_AUX_ADD_BF16 || e.aux_mode == GEMM_AUX_ADD_F32 || e.aux_mode == GEMM_AUX_MUL_BF16,
            "gemm_bf16_tc: unknown aux_mode %d", e.aux_mode);
  DMG_CHECK(e.aux_mode == GEMM_AUX_NONE || (e.aux && (e.aux_mode == GEMM_AUX_ADD_F32 ? e.ld_aux % 4 == 0 : e.ld_aux % 8 == 0)),
            "gemm_bf16_tc: aux operand missing or misaligned");
  DMG_CHECK(N % 4 == 0, "gemm_bf16_tc: N=%d must be a multiple of 4 (16-byte epilogue accesses)", N);
  // CTA pairs (256-row tiles) whenever there are at least two 128-row blocks; tile width: the widest that still yields
  // about one wave of tiles
  const int CG = (M > GT_BM && N > 64 && num_sms >= 2) ? 2 : 1;   // a pair stages N/2 >= 64 columns of B per CTA
  const int units = num_sms / CG;
  const int num_m = (M + GT_BM * CG - 1) / (GT_BM * CG);
  // tile width: the candidate with the smallest estimated time = waves x (k-blocks x (MMA + fixed cost) + epilogue); a
  // narrower tile only pays when it removes a (partly idle) wave
  const int groups = e.groups < 1 ? 1 : e.groups;
  const int BN_min = 64 * CG;
  const long long kb_tile = ((K + 63) / 64 + splitk - 1) / splitk;
  int BN = 256;
  long long best = -1;
  for (int cand = 256; cand >= BN_min; cand >>= 1) {
    if (cand > 64 * CG && N <= cand / 2) continue;                       // mostly padding
    const long long tiles = (long long)num_m * ((N + cand - 1) / cand) * splitk * groups;
    const long long waves = (tiles + units - 1) / units;
    const long long cost = waves * (kb_tile * (cand + 768) + 8ll * cand);   // measured: a k-block of a 128-wide tile costs ~0.85 of a 256-wide one
    if (best < 0 || cost < best) { best = cost; BN = cand; }
  }
  const int num_n = (N + BN - 1) / BN;
  GemmTParams p;
  p.M = M; p.N = N; p.K = K; p.a_mn = a_mn ? 1 : 0; p.b_mn = b_mn ? 1 : 0;
  p.num_kb = (K + 63) / 64;
  if (splitk > p.num_kb) splitk = p.num_kb;
  p.kb_per_split = (p.num_kb + splitk - 1) / splitk;
  p.splitk = (p.num_kb + p.kb_per_split - 1) / p.kb_per_split;
  p.num_m = num_m; p.num_n = num_n;
  p.bias = e.bias; p.act = e.act; p.aux = e.aux; p.ld_aux = e.ld_aux; p.aux_mode = e.aux_mode;
  p.out = e.out; p.ldc = e.ldc; p.out_mode = e.out_mode; p.out2 = e.out2; p.ld2 = e.ld2;
  p.drop_thresh = e.drop_thresh; p.drop_seed = e.drop_seed; p.drop_scale = e.drop_scale;
  p.groups = e.groups < 1 ? 1 : e.groups; p.a_gs = (int)e.a_gs; p.b_gs = (int)e.b_gs; p.c_gs = e.c_gs;
  DMG_CHECK(p.groups == 1 || (!e.out2 && e.aux_mode == GEMM_AUX_NONE && !e.bias && !e.drop_thresh), "gemm_bf16_tc: grouped launches take the plain epilogue only");
  const TensorMap2D *ta = nullptr, *tb = nullptr;
  const long long Mext = M + (long long)(groups - 1) * e.a_gs, Next = N + (long long)(groups - 1) * e.b_gs;   // tensor extents
  if (!a_mn) { if (get_tmap(A, K, Mext, lda, GT_BM, &ta)) return -1; }
  else       { if (get_tmap(A, Mext, K, lda, 64, &ta)) return -1; }
  if (!b_mn) { if (get_tmap(B, K, Next, ldb, BN / CG, &tb)) return -1; }
  else       { if (get_tmap(B, Next, K, ldb, 64, &tb)) return -1; }
  // bf16 outputs leave through TMA stores (dense boxes; the map clips at M and N); needs N-extent columns in a group-free launch
  p.tma_store = (e.out_mode == GEMM_OUT_BF16 && groups == 1 && e.aux_mode != GEMM_AUX_ADD_F32) ? 1 : 0;
  p.aux_tma = (p.tma_store && !e.out2 && (e.aux_mode == GEMM_AUX_ADD_BF16 || e.aux_mode == GEMM_AUX_MUL_BF16)) ? 1 : 0;
  DMG_CHECK(e.act != GEMM_ACT_GELU_GRADSAVE || p.tma_store, "gemm_bf16_tc: the gradient-saving GeLU epilogue needs bf16 TMA-store outputs");
  const TensorMap2D *tc = ta, *tc2 = ta, *tx = ta;   // placeholders when unused
  if (p.tma_store) {
    if (get_tmap(e.out, N, M, e.ldc, -1, &tc)) return -1;
    if (e.out2 && get_tmap(e.out2, N, M, e.ld2, -1, &tc2)) return -1;
    if (p.aux_tma && get_tmap(e.aux, N, M, e.ld_aux, -1, &tx)) return -1;
  }
  const long long total = (long long)num_m * num_n * p.splitk * groups;
  const int grid = (int)(total < units ? total : units) * CG;
  if (CG == 2) {
    if (BN == 256) return launch_gt<256, 2>(ta, tb, tc, tc2, tx, p, grid, st);
    if (BN == 128) return launch_gt<128, 2>(ta, tb, tc, tc2, tx, p, grid, st);
    return launch_gt<64, 2>(ta, tb, tc, tc2, tx, p, grid, st);
  }
  if (BN == 256) return launch_gt<256, 1>(ta, tb, tc, tc2, tx, p, grid, st);
  if (BN == 128) return launch_gt<128, 1>(ta, tb, tc, tc2, tx, p, grid, st);
  return launch_gt<64, 1>(ta, tb, tc, tc2, tx, p, grid, st);
}

}  // namespace dmg
