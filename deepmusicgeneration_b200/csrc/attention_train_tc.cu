// Training attention FORWARD on the 5th-generation tensor cores (tcgen05.mma, accumulators in TMEM, operands staged by TMA).
//
// Same contract as attn_train_fwd_kernel (attention_train.cu; fastai MultiHeadRelativeAttention._apply_attention, SURVEY.md
// App. A.3/A.4): out = dropout(softmax(((q+u) K^T + _line_shift((q+v) Rk^T)) / sqrt(Dh) + mask)) V, plus the row
// log-sum-exp for the backward.  Used when T, M and mem_count are multiples of 128 (the mma.sync kernel serves the rest).
//
// One CTA = one (stream, head, 128-query tile); 12 warps (the auxiliary warpgroup gives its registers away: setmaxnreg):
//   warps 0-7  softmax: warp w owns TMEM lanes 32*(w%4).. (= query rows) and the key half w/4 of every 128-key tile, so a
//              thread owns ONE query row x 64 keys - row max / row sum need no shuffles; the two halves keep independent
//              online-softmax states (m, l, O[64]) that are merged once at the end
//   warp 8     TMA producer: Q once; per key tile K (2 stages), V, one new 128-distance block of Rk (2 slots)
//   warp 9     one thread issues every tcgen05.mma
// TMEM (512 columns): [0,128) AC = (q+u) K^T | [128,384) position strip (q+v) Rk[D0-128 .. D0+127]^T | [384,448) and
//   [448,512) P_half V of the current tile (the running O lives in registers: o = o * alpha + PV).
// _line_shift is index arithmetic: BD[r, j] = strip[r][128 + r - j] (D0 = M + i0 - j0 is a multiple of 128, so a window is
// two aligned 128-row blocks of Rk and consecutive key tiles share one).  A thread needs 64 consecutive strip columns of
// ITS OWN row at a lane-dependent offset; TMEM loads take warp-uniform column addresses, so the row passes through a
// thread-private shared-memory line (written with 16-byte stores, read back at offset `lane` - no synchronisation at all).
// P goes to shared memory as bf16 in the canonical K-major 128B-swizzled layout and is the A operand of the PV MMA; V is
// used as it lies (MN-major B operand).  The softmax of tile n overlaps the score MMAs of tile n+1 (issued as soon as every
// softmax warp has copied tile n out of TMEM) and the PV MMA of tile n-1.
#include <cuda.h>
#include "kernels.cuh"
#include "launch.cuh"
#include "mma_sync.cuh"
#include "train_kernels.cuh"

namespace dmg {

namespace {

constexpr float LOG2E = 1.4426950408889634f;
constexpr float LN2 = 0.6931471805599453f;

constexpr int TC_SOFT_WARPS = 8;
constexpr int TC_THREADS = (TC_SOFT_WARPS + 4) * 32;   // + one auxiliary warpgroup: TMA warp, MMA warp, two idle warps
constexpr int T16K = 128 * 64 * 2;                 // one [128 rows][64 bf16] tile, 128B swizzle
constexpr int STRIP_LD = 68;                        // floats per thread-private strip line (64 used; 68: conflict-free v4 stores)
constexpr int OFF_QU = 0;
constexpr int OFF_QV = OFF_QU + T16K;
constexpr int OFF_K = OFF_QV + T16K;                // 2 stages
constexpr int OFF_V = OFF_K + 2 * T16K;
constexpr int OFF_R = OFF_V + T16K;                 // 2 slots (slot = block & 1)
constexpr int OFF_P = OFF_R + 2 * T16K;             // 2 key halves; half 0 doubles as the raw-Q landing buffer
constexpr int OFF_STRIP = OFF_P + 2 * T16K;
constexpr int STRIP_WARP_BYTES = 9 * 1024;          // 32 lines of 272 B, padded to a 1024-byte multiple: the region doubles as a swizzled
                                                    // [32 rows][128 B] tile for the TMA store of the saved probabilities
static_assert(32 * STRIP_LD * 4 <= STRIP_WARP_BYTES, "strip lines must fit");
constexpr int OFF_BAR = OFF_STRIP + TC_SOFT_WARPS * STRIP_WARP_BYTES;
constexpr int TC_SMEM = OFF_BAR + 256 + 1024 /*alignment slack*/;
static_assert(TC_SMEM <= 227 * 1024, "shared memory budget");

enum { B_QFULL = 0, B_QREADY, B_KFULL0, B_KFULL1, B_KEMPTY0, B_KEMPTY1, B_RFULL0, B_RFULL1, B_REMPTY0, B_REMPTY1, B_VFULL, B_VEMPTY,
       B_SFULL, B_SFREE, B_PFULL0, B_PFULL1, B_OFULL0, B_OFULL1, B_OFREE0, B_OFREE1, B_COUNT };

constexpr uint32_t TM_AC = 0, TM_STRIP = 128, TM_O = 384;

// shared-memory matrix descriptors (sm_100 version bit 46, SWIZZLE_128B)
// bounded wait without the printf of mbar_wait, for the MMA-issuing warps: they run the issue loop as a WHOLE warp in uniform control flow
// (waits by all lanes, tcgen05.mma / commit by the elected lane), so that descriptors and barrier addresses stay in uniform registers.
// As the body of an `if (lane == 0)` branch every tcgen05.mma cost ~20 instructions (vector-to-uniform move loop, elect, predicate
// shuffles, descriptor rebuild): ~0.1 us per MMA of one thread's time, 2 us per tile in the attention kernels
// (profiles/r2h_attn_bert_tc_timeline_single_v.txt, profiles/r2g_attn_bwd_dq_tc_timeline.txt).
__device__ __forceinline__ void tc_wait(uint64_t* bar, uint32_t parity) {
  uint32_t n = 0;
  while (!mbar_try_wait(bar, parity))
    if (++n > (1u << 26)) __trap();
}
__device__ __forceinline__ uint64_t desc_kmajor(uint32_t addr) {          // rows of 128 B, 8-row groups 1024 B apart
  return (uint64_t)((addr & 0x3FFFFu) >> 4) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
__device__ __forceinline__ uint64_t desc_mnmajor(uint32_t addr) {         // [k rows][64 mn] boxes: LBO 8192 (next mn block), SBO 1024 (next 8 k rows)
  return (uint64_t)((addr & 0x3FFFFu) >> 4) | ((uint64_t)(8192u >> 4) << 16) | ((uint64_t)(1024u >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void softmax_bar_sync() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

// SAVE: also write the undropped probabilities / block maxima for the backward (AttnTrainArgs::p_save, m_save)
// RING: the inference engine's layout - the memory keys / values are the per-head K/V RINGS ([stream][head][slot][64]; tmM = K ring,
//       tmP = V ring, logical memory row j = slot (ring_head + j) % M, ring_head a multiple of 128) and the relative-position keys the
//       per-head cache Rd ([head][Dcap][64], tmR); multi-token segments over a warm memory (chunked prefill, validation passes)
template <bool SAVE, bool RING>
__global__ void __launch_bounds__(TC_THREADS, 1)
attn_train_fwd_tc_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmM,
                         const __grid_constant__ CUtensorMap tmR, const __grid_constant__ CUtensorMap tmP,
                         const __grid_constant__ CUtensorMap tmQU, const __grid_constant__ CUtensorMap tmQV, const AttnTrainArgs a) {
  extern __shared__ __align__(1024) uint8_t tc_smem_raw[];
  uint8_t* smem = tc_smem_raw + ((1024u - (smem_u32(tc_smem_raw) & 1023u)) & 1023u);
  uint64_t* bar = (uint64_t*)(smem + OFF_BAR);
  uint32_t* tmem_holder = (uint32_t*)(bar + B_COUNT);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nT = a.T / 128;
  const int it = nT - 1 - (blockIdx.x % nT);        // heavy (late) query tiles first
  const int bh = blockIdx.x / nT, b = bh / a.H, h = bh % a.H;
  const int i0 = it * 128, HD = a.H * 64, S = a.M + a.T;
  const int jt_lo = (a.M - a.mem_count) / 128, jt_hi = (a.M + i0) / 128;
  const int NT = jt_hi - jt_lo + 1;                 // key tiles of this CTA
  const int blk0 = (a.M + i0) / 128 - jt_lo;        // upper Rk block of the first tile (block = distance / 128)

  if (warp == TC_SOFT_WARPS && lane == 0) {
    tma_prefetch_desc(&tmX);
    tma_prefetch_desc(&tmM);
    tma_prefetch_desc(&tmR);
    if (SAVE || RING) tma_prefetch_desc(&tmP);
    for (int i = 0; i < B_COUNT; i++) {
      uint32_t cnt = 1;
      if (i == B_QREADY || i == B_SFREE) cnt = TC_SOFT_WARPS;
      if (i == B_PFULL0 || i == B_PFULL1 || i == B_OFREE0 || i == B_OFREE1) cnt = TC_SOFT_WARPS / 2;
      mbar_init(&bar[i], cnt);
    }
    mbar_fence_init();
  }
  if (warp == TC_SOFT_WARPS + 1) tmem_alloc<512>(tmem_holder);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  // register budget: 384 threads start with 168 registers each; the auxiliary warpgroup hands its share to the softmax warpgroups
  if (warp >= TC_SOFT_WARPS) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 64;");
    if (warp == TC_SOFT_WARPS) {
    // =========================================== TMA producer ===========================================
    if (lane == 0) {
      mbar_expect_tx(&bar[B_QFULL], T16K);
      tma_load_2d(smem + OFF_P, &tmX, h * 64, b * a.T + i0, &bar[B_QFULL]);
      auto load_k = [&](int n) {
        const int s = n & 1, j0 = (jt_lo + n) * 128;
        mbar_wait(&bar[B_KEMPTY0 + s], ((n >> 1) & 1) ^ 1);
        mbar_expect_tx(&bar[B_KFULL0 + s], T16K);
        if (j0 < a.M) {
          if (RING) tma_load_2d(smem + OFF_K + s * T16K, &tmM, 0, ((a.ring_b0 + b) * a.H + h) * a.M + (a.ring_head + j0) % a.M, &bar[B_KFULL0 + s]);
          else tma_load_2d(smem + OFF_K + s * T16K, &tmM, h * 64, b * a.M + j0, &bar[B_KFULL0 + s]);
        } else {
          tma_load_2d(smem + OFF_K + s * T16K, &tmX, HD + h * 64, b * a.T + (j0 - a.M), &bar[B_KFULL0 + s]);
        }
      };
      auto load_r = [&](int k) {                    // k-th block load: block blk0 - k (may be -1: all rows out of bounds -> zeros)
        const int blk = blk0 - k, s = blk & 1;
        mbar_wait(&bar[B_REMPTY0 + s], ((k >> 1) & 1) ^ 1);
        mbar_expect_tx(&bar[B_RFULL0 + s], T16K);
        // RING: block -1 of head h > 0 reads the previous head's rows instead of zeros - only masked (future) keys ever meet it
        if (RING) tma_load_2d(smem + OFF_R + s * T16K, &tmR, 0, h * a.ring_dcap + blk * 128, &bar[B_RFULL0 + s]);
        else tma_load_2d(smem + OFF_R + s * T16K, &tmR, h * 64, blk * 128, &bar[B_RFULL0 + s]);
      };
      auto load_v = [&](int n) {
        const int j0 = (jt_lo + n) * 128;
        mbar_wait(&bar[B_VEMPTY], (n & 1) ^ 1);
        mbar_expect_tx(&bar[B_VFULL], T16K);
        if (j0 < a.M) {
          if (RING) tma_load_2d(smem + OFF_V, &tmP, 0, ((a.ring_b0 + b) * a.H + h) * a.M + (a.ring_head + j0) % a.M, &bar[B_VFULL]);
          else tma_load_2d(smem + OFF_V, &tmM, HD + h * 64, b * a.M + j0, &bar[B_VFULL]);
        } else {
          tma_load_2d(smem + OFF_V, &tmX, 2 * HD + h * 64, b * a.T + (j0 - a.M), &bar[B_VFULL]);
        }
      };
      load_k(0);
      load_r(0);
      load_r(1);
      if (NT > 1) load_k(1);
      load_v(0);
      // waits in the order the MMAs retire: S(n-1) is issued half a tile before PV(n-2), so the V requests trail the K / R requests by
      // one tile (a V request waiting for PV(n-1) in front of them would hold the operands of S(n+1) back until half a tile before use)
      for (int n = 1; n < NT; n++) {
        load_r(n + 1);
        if (n + 1 < NT) load_k(n + 1);
        if (n >= 2) load_v(n - 1);
      }
      if (NT >= 2) load_v(NT - 1);
    }
  } else if (warp == TC_SOFT_WARPS + 1) {
    // =========================================== MMA issuer (whole warp, elected lane issues) ===========================================
    {
      // instruction descriptors: D fp32, A/B bf16, N>>3 @17, M>>4 @24; bit 16: B is MN-major
      constexpr uint32_t idesc_s = (1u << 4) | (1u << 7) | (1u << 10) | ((128u >> 3) << 17) | ((128u >> 4) << 24);
      constexpr uint32_t idesc_pv = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 16) | ((64u >> 3) << 17) | ((128u >> 4) << 24);
      const uint32_t qu = smem_u32(smem + OFF_QU), qv = smem_u32(smem + OFF_QV);
      // operand descriptors; a 16-element K step is +32 bytes (K-major) / +2048 bytes (MN-major V) in the address field
      const uint64_t d_qu = desc_kmajor(qu), d_qv = desc_kmajor(qv), d_k0 = desc_kmajor(smem_u32(smem + OFF_K)),
                     d_k1 = desc_kmajor(smem_u32(smem + OFF_K + T16K)), d_r0 = desc_kmajor(smem_u32(smem + OFF_R)),
                     d_r1 = desc_kmajor(smem_u32(smem + OFF_R + T16K)), d_p0 = desc_kmajor(smem_u32(smem + OFF_P)),
                     d_p1 = desc_kmajor(smem_u32(smem + OFF_P + T16K)), d_v = desc_mnmajor(smem_u32(smem + OFF_V));
      auto issue_pv = [&](int m) {
        tc_wait(&bar[B_VFULL], m & 1);
#pragma unroll
        for (int hf = 0; hf < 2; hf++) {
          tc_wait(&bar[B_PFULL0 + hf], m & 1);
          if (m > 0) tc_wait(&bar[B_OFREE0 + hf], (m - 1) & 1);
          tc_fence_after();
          if (elect_one()) {
            const uint64_t dp = hf ? d_p1 : d_p0, dv = d_v + (uint64_t)(hf * (8192 >> 4));
#pragma unroll
            for (int k = 0; k < 4; k++)
              umma_bf16(tmem_base + TM_O + 64 * hf, dp + (uint64_t)(2 * k), dv + (uint64_t)(128 * k), idesc_pv, (uint32_t)(k > 0));
            umma_commit(&bar[B_OFULL0 + hf]);
            if (hf == 1) umma_commit(&bar[B_VEMPTY]);
          }
          __syncwarp();
        }
      };
      tc_wait(&bar[B_QREADY], 0);
      if (SAVE && a.qu_save) {                       // the biased query tiles are the backward's operands as well: store them as they lie
        if (elect_one()) {
          asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(&tmQU), "r"(qu), "r"(h * 64),
                       "r"(b * a.T + i0)
                       : "memory");
          asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(&tmQV), "r"(qv), "r"(h * 64),
                       "r"(b * a.T + i0)
                       : "memory");
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
        __syncwarp();
      }
      for (int n = 0; n < NT; n++) {
        const int s = n & 1, blkU = blk0 - n, blkL = blkU - 1;
        tc_wait(&bar[B_KFULL0 + s], (n >> 1) & 1);
        tc_wait(&bar[B_RFULL0 + (blkU & 1)], (n >> 1) & 1);
        tc_wait(&bar[B_RFULL0 + (blkL & 1)], ((n + 1) >> 1) & 1);
        if (n > 0) tc_wait(&bar[B_SFREE], (n - 1) & 1);
        tc_fence_after();
        if (elect_one()) {
          const uint64_t ks = s ? d_k1 : d_k0, rl = (blkL & 1) ? d_r1 : d_r0, ru = (blkU & 1) ? d_r1 : d_r0;
#pragma unroll
          for (int k = 0; k < 4; k++) umma_bf16(tmem_base + TM_AC, d_qu + (uint64_t)(2 * k), ks + (uint64_t)(2 * k), idesc_s, (uint32_t)(k > 0));
#pragma unroll
          for (int k = 0; k < 4; k++) umma_bf16(tmem_base + TM_STRIP, d_qv + (uint64_t)(2 * k), rl + (uint64_t)(2 * k), idesc_s, (uint32_t)(k > 0));
#pragma unroll
          for (int k = 0; k < 4; k++)
            umma_bf16(tmem_base + TM_STRIP + 128, d_qv + (uint64_t)(2 * k), ru + (uint64_t)(2 * k), idesc_s, (uint32_t)(k > 0));
          umma_commit(&bar[B_SFULL]);
          umma_commit(&bar[B_KEMPTY0 + s]);
          umma_commit(&bar[B_REMPTY0 + (blkU & 1)]);   // the upper block is dead after this tile; the lower one serves the next
        }
        __syncwarp();
        if (n > 0) issue_pv(n - 1);
      }
      issue_pv(NT - 1);
      // the bulk group belongs to the lane that issued it
      if (SAVE && a.qu_save) {
        if (elect_one()) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        __syncwarp();
      }
    }
    }
  } else {
    // =========================================== softmax warps ===========================================
    asm volatile("setmaxnreg.inc.sync.aligned.u32 216;");
    const int hf = warp >> 2, q4 = warp & 3;
    const int r = q4 * 32 + lane;                   // query row of this thread inside the tile
    const int row = i0 + r;                         // ... inside the segment
    const uint32_t t_lane = tmem_base + ((uint32_t)(q4 * 32) << 16);
    uint8_t* strip_warp = smem + OFF_STRIP + warp * STRIP_WARP_BYTES;
    float* strip = (float*)strip_warp + (size_t)lane * STRIP_LD;
    uint8_t* psave_row = strip_warp + (lane >> 3) * 1024 + (lane & 7) * 128;   // this lane's row of the warp's [32][128 B] swizzled tile
    const int vis_lim = a.k == 1 ? row + 1 : max((row / a.win) * a.win, 1);
    const float c = a.scale * LOG2E;

    // ---- q + u and q + v in the canonical swizzled layout.  Eight consecutive threads take the eight 16-byte chunks of one row (128
    // contiguous bytes: no bank conflicts); a thread's rows are 32 apart, so its physical chunk maps to the same logical columns in all
    // of them and it needs one 8-wide slice of u and v only (requested before the wait for q).
    {
      const int tid = threadIdx.x, pc = tid & 7, rb = tid >> 3;
      const int col = 8 * (pc ^ (rb & 7));
      const float4 ua = __ldg((const float4*)(a.u + h * 64 + col)), ub = __ldg((const float4*)(a.u + h * 64 + col + 4));
      const float4 va = __ldg((const float4*)(a.v + h * 64 + col)), vb = __ldg((const float4*)(a.v + h * 64 + col + 4));
      const float uu[8] = {ua.x, ua.y, ua.z, ua.w, ub.x, ub.y, ub.z, ub.w}, vv8[8] = {va.x, va.y, va.z, va.w, vb.x, vb.y, vb.z, vb.w};
      mbar_wait(&bar[B_QFULL], 0);
#pragma unroll
      for (int k = 0; k < 4; k++) {
        const int qr = rb + 32 * k;
        const uint32_t off = (uint32_t)((qr >> 3) * 1024 + (qr & 7) * 128 + pc * 16);
        const uint4 raw = *(const uint4*)(smem + OFF_P + off);
        const uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
        uint32_t ou[4], ov[4];
#pragma unroll
        for (int e = 0; e < 4; e++) {
          const float lo = bf16lo(w[e]), hi = bf16hi(w[e]);
          ou[e] = pack_bf16x2(lo + uu[2 * e], hi + uu[2 * e + 1]);
          ov[e] = pack_bf16x2(lo + vv8[2 * e], hi + vv8[2 * e + 1]);
        }
        *(uint4*)(smem + OFF_QU + off) = make_uint4(ou[0], ou[1], ou[2], ou[3]);
        *(uint4*)(smem + OFF_QV + off) = make_uint4(ov[0], ov[1], ov[2], ov[3]);
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar[B_QREADY]);
    }

    float o[64];
#pragma unroll
    for (int i = 0; i < 64; i++) o[i] = 0.f;
    float m_run = -INFINITY, l_run = 0.f, alpha_prev = 1.f;
    // dropout pair index of (row, key j) = ((bh*T + row)*S + j) / 2 (S and this thread's first key of a tile are even)
    const uint32_t drop_base = (uint32_t)((((long long)bh * a.T + row) * S) >> 1);
    uint8_t* prow = smem + OFF_P + hf * T16K + (r >> 3) * 1024 + (r & 7) * 128;

    for (int n = 0; n < NT; n++) {
      const int j0 = (jt_lo + n) * 128 + 64 * hf;    // full-context index of this thread's first key
      float s[64];
      mbar_wait(&bar[B_SFULL], n & 1);
      tc_fence_after();
      {   // content term (both loads in flight before the wait)
        uint32_t x0[32], x1[32];
        tmem_ld_32x32(t_lane + TM_AC + 64 * hf, x0);
        tmem_ld_32x32(t_lane + TM_AC + 64 * hf + 32, x1);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 32; i++) { s[i] = __uint_as_float(x0[i]); s[32 + i] = __uint_as_float(x1[i]); }
      }
      if (SAVE) {                                    // last tile's saved-P tile has left the strip region
        if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        __syncwarp();
      }
      // position term: keys 32*sp .. 32*sp+31 of this half need strip columns base + (32 + lane - jj), base warp-uniform
#pragma unroll
      for (int sp = 0; sp < 2; sp++) {
        const uint32_t base = (uint32_t)(96 - 64 * hf - 32 * sp + 32 * q4);
        {
          uint32_t x0[32], x1[32];
          tmem_ld_32x32(t_lane + TM_STRIP + base, x0);
          tmem_ld_32x32(t_lane + TM_STRIP + base + 32, x1);
          tmem_ld_wait();
          if (sp == 1) {                             // last TMEM read of this tile: the score MMAs of the next tile may overwrite it
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&bar[B_SFREE]);
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
#pragma unroll
        for (int jj = 0; jj < 32; jj++) s[32 * sp + jj] += sk[-jj];
      }
      __syncwarp();                                  // every lane is done with its strip line (the SAVE tile reuses the region)

      if (n > 0) {                                   // fold the previous tile's P V into the running output
        mbar_wait(&bar[B_OFULL0 + hf], (n - 1) & 1);
        tc_fence_after();
#pragma unroll
        for (int ch = 0; ch < 2; ch++) {
          uint32_t x[32];
          tmem_ld_32x32(t_lane + TM_O + 64 * hf + 32 * ch, x);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 32; i++) o[32 * ch + i] = fmaf(o[32 * ch + i], alpha_prev, __uint_as_float(x[i]));
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bar[B_OFREE0 + hf]);
      }

      // mask: x-region tiles only; causal (1,1) tiles strictly below the diagonal are fully visible.  Key jx (segment
      // coordinates) is visible from this row iff jx < vis_lim (window_mask: (1,1) -> jx <= row; (w,0) -> jx < (row/w)*w or jx == 0)
      const int jx0 = j0 - a.M;
      const bool need_mask = jx0 + 63 >= 1 && !(a.k == 1 && jx0 + 63 <= i0);
      if (need_mask) {
        const int lim = vis_lim - jx0;              // local keys jj < lim stay
#pragma unroll
        for (int jj = 0; jj < 64; jj++) s[jj] = jj < lim ? s[jj] : -INFINITY;
      }
      float mx = -INFINITY;
#pragma unroll
      for (int jj = 0; jj < 64; jj++) mx = fmaxf(mx, s[jj]);
      const float m_new = fmaxf(m_run, mx);
      const float alpha = (m_new == -INFINITY) ? 1.f : ex2_fast((m_run - m_new) * c);
      const float neg_mc = (m_new == -INFINITY) ? 0.f : -m_new * c;
      m_run = m_new;
      float rs = 0.f;
      // P (unscaled dropout: the 1/(1-p) factor is applied to the output) -> canonical K-major swizzled bf16 tile
#pragma unroll
      for (int ck = 0; ck < 8; ck++) {
        uint32_t pk[4], pu[4];
#pragma unroll
        for (int e = 0; e < 4; e++) {
          const int pp = 4 * ck + e;
          float p0 = ex2_fast(fmaf(s[2 * pp], c, neg_mc)), p1 = ex2_fast(fmaf(s[2 * pp + 1], c, neg_mc));
          rs += p0 + p1;
          if (SAVE) pu[e] = pack_bf16x2(p0, p1);
          if (a.drop_thresh) {
            const uint32_t hb = drop_pair_bits(a.drop_seed, drop_base + (uint32_t)(j0 >> 1) + pp);
            p0 = ((hb & 0xFFFFu) >= a.drop_thresh) ? p0 : 0.f;
            p1 = ((hb >> 16) >= a.drop_thresh) ? p1 : 0.f;
          }
          pk[e] = (a.drop_thresh || !SAVE) ? pack_bf16x2(p0, p1) : pu[e];
        }
        *(uint4*)(prow + ((ck ^ (r & 7)) << 4)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        if (SAVE) *(uint4*)(psave_row + ((ck ^ (lane & 7)) << 4)) = make_uint4(pu[0], pu[1], pu[2], pu[3]);   // the strip lines are free after the skew
      }
      l_run = l_run * alpha + rs;
      alpha_prev = alpha;
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar[B_PFULL0 + hf]);
      if (SAVE) {   // the warp's 32 rows x 64 undropped probabilities leave through one TMA store
        if (lane == 0) {
          asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(&tmP), "r"(smem_u32(strip_warp)),
                       "r"(j0), "r"(bh * a.T + i0 + q4 * 32)
                       : "memory");
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
        a.m_save[((long long)bh * a.T + row) * (S >> 6) + (j0 >> 6)] = m_new;
      }
    }
    if (SAVE) {
      if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
      __syncwarp();
    }
    // last tile's P V
    mbar_wait(&bar[B_OFULL0 + hf], (NT - 1) & 1);
    tc_fence_after();
#pragma unroll
    for (int ch = 0; ch < 2; ch++) {
      uint32_t x[32];
      tmem_ld_32x32(t_lane + TM_O + 64 * hf + 32 * ch, x);
      tmem_ld_wait();
#pragma unroll
      for (int i = 0; i < 32; i++) o[32 * ch + i] = fmaf(o[32 * ch + i], alpha_prev, __uint_as_float(x[i]));
    }
    tc_fence_before();

    // ---- merge the two key halves of every row (half 1 hands its state over through its strip line), write out / lse
    if (hf == 1) {
#pragma unroll
      for (int k = 0; k < 16; k++) *(float4*)(strip + 4 * k) = make_float4(o[4 * k], o[4 * k + 1], o[4 * k + 2], o[4 * k + 3]);
      strip[64] = m_run;
      strip[65] = l_run;
    }
    softmax_bar_sync();
    if (hf == 0) {
      const float* other = (const float*)(strip_warp + 4 * STRIP_WARP_BYTES) + (size_t)lane * STRIP_LD;   // same lane of warp + 4
      const float m1 = other[64], l1 = other[65];
      const float m = fmaxf(m_run, m1);
      const float w0 = (m_run == -INFINITY) ? 0.f : ex2_fast((m_run - m) * c);
      const float w1 = (m1 == -INFINITY) ? 0.f : ex2_fast((m1 - m) * c);
      const float l = l_run * w0 + l1 * w1;
      const float inv = l > 0.f ? (a.drop_thresh ? a.drop_scale : 1.f) / l : 0.f;
      bf16* orow = a.out + ((long long)b * a.T + row) * HD + h * 64;
#pragma unroll
      for (int k = 0; k < 8; k++) {
        uint32_t w[4];
#pragma unroll
        for (int e = 0; e < 4; e++) {
          const int d0 = 8 * k + 2 * e;
          w[e] = pack_bf16x2((o[d0] * w0 + other[d0] * w1) * inv, (o[d0 + 1] * w0 + other[d0 + 1] * w1) * inv);
        }
        *(uint4*)(orow + 8 * k) = make_uint4(w[0], w[1], w[2], w[3]);
      }
      if (a.lse) a.lse[(long long)bh * a.T + row] = (m * c + log2f(l)) * LN2;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == TC_SOFT_WARPS + 1) tmem_dealloc<512>(tmem_base);
}

// =============================================================================================
// dK / dV on tcgen05 from the tiles the dQ kernel spilled (no softmax work left: a pure contraction, HBM-bound):
//   dV[keys, :] = sum_i Pd[i, keys]^T dO[i, :]        dK[keys, :] = sum_i dS[i, keys]^T (q_i + u)
// One CTA = (stream, head, 128-key tile); the reduction runs over the query rows that see the tile, 64 per pipeline stage.
// Pd / dS lie row-major [query][key], i.e. with the reduction index as the slow one: they are MN-major A operands (64 x 64
// TMA boxes, LBO 8192 / SBO 1024, as in gemm_train.cu), dO and (q+u) are MN-major B operands.  Accumulators: TMEM columns
// [0,64) dV, [64,128) dK.  Warp 0 = TMA producer, warp 1 = MMA issuer, warps 2-5 = epilogue.
// The dQ kernel works on 64 x 64 tiles and never touches tiles above the diagonal, so for a key tile inside the current
// segment the upper key half of the FIRST stage was never written: it is not loaded, its shared-memory boxes are zero-filled.
// =============================================================================================
constexpr int DKV_STAGES = 2;                                      // 2 x 48 KB -> two CTAs per SM: one CTA's prologue / epilogue hides under the other's stream
constexpr int DKV_BOX = 64 * 64 * 2;                                  // one 64 x 64 bf16 box
constexpr int DKV_STAGE_BYTES = 6 * DKV_BOX;                          // Pd (2 key halves), dS (2), dO, q+u
constexpr int DKV_SMEM = DKV_STAGES * DKV_STAGE_BYTES + 1024 + 256;
enum { DB_FULL0 = 0, DB_EMPTY0 = DKV_STAGES, DB_ACC = 2 * DKV_STAGES, DB_ZERO, DB_COUNT };

__device__ __forceinline__ uint64_t desc_mn64(uint32_t addr) { return desc_mnmajor(addr); }   // LBO 8192 (next 64-wide block), SBO 1024

__global__ void __launch_bounds__(192)
attn_bwd_dkv_tc_kernel(const __grid_constant__ CUtensorMap tmPd, const __grid_constant__ CUtensorMap tmdS,
                       const __grid_constant__ CUtensorMap tmdO, const __grid_constant__ CUtensorMap tmQu, const AttnTrainBwdArgs ba) {
  const AttnTrainArgs& a = ba.f;
  extern __shared__ __align__(1024) uint8_t dk_smem_raw[];
  uint8_t* smem = dk_smem_raw + ((1024u - (smem_u32(dk_smem_raw) & 1023u)) & 1023u);
  uint64_t* bar = (uint64_t*)(smem + DKV_STAGES * DKV_STAGE_BYTES);
  uint32_t* tmem_holder = (uint32_t*)(bar + DB_COUNT);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nS = (a.M + a.T) / 128;
  const int jt = (int)(blockIdx.x % nS);            // memory tiles (most query rows) first
  // (stream, head) pairs in the REVERSE of the dQ kernel's order: the Pd / dS tiles it wrote last are still in L2 (the 537 MB of a layer's
  // tiles do not fit, the most recent ~100 MB do)
  const int bh = a.B * a.H - 1 - (int)(blockIdx.x / nS), b = bh / a.H, h = bh % a.H;
  const int j0 = jt * 128, HD = a.H * 64;
  const bool in_x = j0 >= a.M;
  bf16 *dk_dst, *dv_dst;
  long long ldd;
  if (!in_x) {
    ldd = a.ldm;
    dk_dst = ba.dkv_m + ((long long)b * a.M + j0) * a.ldm + h * 64;
    dv_dst = dk_dst + HD;
  } else {
    ldd = a.ldx;
    dk_dst = ba.dqkv_x + ((long long)b * a.T + (j0 - a.M)) * a.ldx + HD + h * 64;
    dv_dst = dk_dst + HD;
  }
  if (j0 < a.M - a.mem_count) {                     // memory rows that hold nothing yet: zero gradient
    for (int i = threadIdx.x; i < 128 * 8; i += 192) {
      const int r = i >> 3, c8 = (i & 7) * 8;
      *(uint4*)(dk_dst + (long long)r * ldd + c8) = make_uint4(0u, 0u, 0u, 0u);
      *(uint4*)(dv_dst + (long long)r * ldd + c8) = make_uint4(0u, 0u, 0u, 0u);
    }
    return;
  }
  const int it_lo = in_x ? (j0 - a.M) / 64 : 0;    // first 64-row query chunk that sees the tile's first key half
  const int NI = a.T / 64 - it_lo;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmPd); tma_prefetch_desc(&tmdS); tma_prefetch_desc(&tmdO); tma_prefetch_desc(&tmQu);
    for (int i = 0; i < DB_COUNT; i++) mbar_init(&bar[i], i == DB_ZERO ? 4u : 1u);
    mbar_fence_init();
  }
  if (warp == 1) tmem_alloc<128>(tmem_holder);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  if (warp == 0) {
    if (lane == 0) {
      for (int n = 0; n < NI; n++) {
        const int s = n % DKV_STAGES, i0 = (it_lo + n) * 64;
        mbar_wait(&bar[DB_EMPTY0 + s], ((n / DKV_STAGES) & 1) ^ 1);
        const bool half_only = in_x && n == 0;       // the upper key half of the diagonal chunk was never written
        uint8_t* st = smem + s * DKV_STAGE_BYTES;
        mbar_expect_tx(&bar[DB_FULL0 + s], (half_only ? 4 : 6) * DKV_BOX);
        tma_load_2d(st, &tmPd, j0, bh * a.T + i0, &bar[DB_FULL0 + s]);
        tma_load_2d(st + 2 * DKV_BOX, &tmdS, j0, bh * a.T + i0, &bar[DB_FULL0 + s]);
        if (!half_only) {
          tma_load_2d(st + DKV_BOX, &tmPd, j0 + 64, bh * a.T + i0, &bar[DB_FULL0 + s]);
          tma_load_2d(st + 3 * DKV_BOX, &tmdS, j0 + 64, bh * a.T + i0, &bar[DB_FULL0 + s]);
        }
        tma_load_2d(st + 4 * DKV_BOX, &tmdO, h * 64, b * a.T + i0, &bar[DB_FULL0 + s]);
        tma_load_2d(st + 5 * DKV_BOX, &tmQu, h * 64, b * a.T + i0, &bar[DB_FULL0 + s]);
      }
    }
  } else if (warp == 1) {
    {   // whole warp in uniform control flow, the elected lane issues (see tc_wait)
      // D fp32, A / B bf16, both MN-major (bits 15, 16), N = 64, M = 128
      constexpr uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((64u >> 3) << 17) | ((128u >> 4) << 24);
      if (in_x) tc_wait(&bar[DB_ZERO], 0);
      for (int n = 0; n < NI; n++) {
        const int s = n % DKV_STAGES;
        tc_wait(&bar[DB_FULL0 + s], (n / DKV_STAGES) & 1);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t st = smem_u32(smem + s * DKV_STAGE_BYTES);
          const uint64_t d0 = desc_mn64(st), d2 = desc_mn64(st + 2 * DKV_BOX), d4 = desc_mn64(st + 4 * DKV_BOX), d5 = desc_mn64(st + 5 * DKV_BOX);
#pragma unroll
          for (int k = 0; k < 4; k++) {
            umma_bf16(tmem_base, d0 + (uint64_t)(128 * k), d4 + (uint64_t)(128 * k), idesc, (uint32_t)(n > 0 || k > 0));
            umma_bf16(tmem_base + 64, d2 + (uint64_t)(128 * k), d5 + (uint64_t)(128 * k), idesc, (uint32_t)(n > 0 || k > 0));
          }
          umma_commit(&bar[DB_EMPTY0 + s]);
          if (n == NI - 1) umma_commit(&bar[DB_ACC]);
        }
        __syncwarp();
      }
    }
  } else {
    const int q4 = warp & 3;
    if (in_x) {                                      // zero the never-written upper key half of the first stage (Pd and dS boxes)
      for (int i = (warp - 2) * 32 + lane; i < DKV_BOX / 16; i += 128) {
        *(uint4*)(smem + DKV_BOX + i * 16) = make_uint4(0u, 0u, 0u, 0u);
        *(uint4*)(smem + 3 * DKV_BOX + i * 16) = make_uint4(0u, 0u, 0u, 0u);
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar[DB_ZERO]);
    }
    mbar_wait(&bar[DB_ACC], 0);
    tc_fence_after();
    const int key = q4 * 32 + lane;
    const uint32_t t_lane = tmem_base + ((uint32_t)(q4 * 32) << 16);
#pragma unroll
    for (int which = 0; which < 2; which++) {
      bf16* dst = (which == 0 ? dv_dst : dk_dst) + (long long)key * ldd;
#pragma unroll
      for (int ch = 0; ch < 2; ch++) {
        uint32_t x[32];
        tmem_ld_32x32(t_lane + 64 * which + 32 * ch, x);
        tmem_ld_wait();
#pragma unroll
        for (int k = 0; k < 4; k++)
          *(uint4*)(dst + 32 * ch + 8 * k) =
              make_uint4(pack_bf16x2(__uint_as_float(x[8 * k]), __uint_as_float(x[8 * k + 1])),
                         pack_bf16x2(__uint_as_float(x[8 * k + 2]), __uint_as_float(x[8 * k + 3])),
                         pack_bf16x2(__uint_as_float(x[8 * k + 4]), __uint_as_float(x[8 * k + 5])),
                         pack_bf16x2(__uint_as_float(x[8 * k + 6]), __uint_as_float(x[8 * k + 7])));
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc<128>(tmem_base);
}


// =============================================================================================
// dQ on tcgen05 (replaces attn_bwd_dq_kernel<true> of attention_train.cu when T, M and mem_count are multiples of 128): the autograd of
// fastai's _apply_attention with respect to the query side, from the probabilities the forward saved.
//   dPd = dO V^T                         (tcgen05, TMEM, double-buffered)
//   P = p_save * exp(m_save*scale - lse),  Pd = dropout(P),  dS = P * (dropout'(dPd) - delta) * scale       (softmax warps, one row each)
//   dQ  = dS K  +  dS_dist Rk            (tcgen05; dS_dist = dS in (row, distance) coordinates = the transpose of _line_shift)
// and, for the kernels downstream, Pd and dS tiles (dK/dV kernel) and dS_dist (dRk GEMM) leave through TMA stores.
// One CTA = (stream, head, 128-query tile), key tiles of 128 from the oldest visible key up to the diagonal, 20 warps:
//   warps 0-15 tile math: thread = one query row x 32 keys (key quarter = warp / 4)
//   warp 16    TMA loads: dO once; per tile the saved probabilities (2 buffers), K, one 128-distance block of Rk
//   warp 19    TMA loads: V (its own thread: it runs two tiles ahead of the other streams)
//   warp 17    one thread issues every tcgen05.mma
//   warp 18    TMA stores: dS tile, Pd tile (written in place over the saved probabilities), finished dS_dist blocks
// The distance of (row r, key jl) inside a tile is D0 + r - jl (D0 = M + i0 - j0, a multiple of 128), so a tile touches two aligned
// 128-distance blocks: the upper one (shared with the previous, older key tile) becomes complete with this tile, the lower one is
// started.  A block lives in one of two [128 rows][128 distances] bf16 buffers (canonical K-major swizzled layout): every entry is
// written exactly once by the two tiles that share the block, a finished block is the A operand of  dQ_bd += block . Rk[block]
// and is stored to ds_dist as it lies.  The first (largest-distance) block only gets its upper-tile part: its buffer starts zeroed;
// the blocks beyond it (distances no visible key produces) are stored as zeros from that buffer before the first tile.
// TMEM: [0,128) / [128,256) dPd of even / odd tiles | [256,320) dQ content part | [320,384) dQ position part.
// =============================================================================================
constexpr int DQT_MATH_WARPS = 16;                // thread = one query row x 32 keys: four warps per scheduler hide the tile math's latencies
constexpr int DQT_THREADS = (DQT_MATH_WARPS + 4) * 32;
constexpr int DQO_DO = 0;
constexpr int DQO_K = DQO_DO + T16K;
constexpr int DQO_V = DQO_K + T16K;
constexpr int DQO_R = DQO_V + T16K;
constexpr int DQO_P = DQO_R + T16K;                  // 2 buffers x 2 key halves
constexpr int DQO_DS = DQO_P + 4 * T16K;             // 2 key halves
constexpr int DQO_STRIP = DQO_DS + 2 * T16K;         // 2 block buffers x 2 distance halves
constexpr int DQO_BAR = DQO_STRIP + 4 * T16K;
constexpr int DQT_SMEM = DQO_BAR + 512 + 1024 /*alignment slack*/;
static_assert(DQT_SMEM <= 227 * 1024, "shared memory budget");
enum { D_DOFULL = 0, D_KFULL, D_KEMPTY, D_VFULL, D_VEMPTY, D_RFULL, D_REMPTY, D_PFULL0, D_PFULL1, D_PFREE0, D_PFREE1, D_DPFULL0, D_DPFULL1,
       D_DPFREE0, D_DPFREE1, D_DSFULL, D_DSFREE, D_SFREE0, D_SFREE1, D_ZINIT, D_ZDONE, D_DQFULL, D_COUNT };
constexpr uint32_t DTM_DP = 0, DTM_AC = 256, DTM_BD = 320;

__device__ __forceinline__ void tma_store_2d(const CUtensorMap* tm, uint32_t smem_addr, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(tm), "r"(smem_addr), "r"(c0), "r"(c1)
               : "memory");
}

__global__ void __launch_bounds__(DQT_THREADS, 1)
attn_bwd_dq_tc_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmM, const __grid_constant__ CUtensorMap tmR,
                      const __grid_constant__ CUtensorMap tmDO, const __grid_constant__ CUtensorMap tmP, const __grid_constant__ CUtensorMap tmPB,
                      const __grid_constant__ CUtensorMap tmDS, const __grid_constant__ CUtensorMap tmDD, const AttnTrainBwdArgs ba) {
  const AttnTrainArgs& a = ba.f;
  extern __shared__ __align__(1024) uint8_t dq_smem_raw[];
  uint8_t* smem = dq_smem_raw + ((1024u - (smem_u32(dq_smem_raw) & 1023u)) & 1023u);
  uint64_t* bar = (uint64_t*)(smem + DQO_BAR);
  uint32_t* tmem_holder = (uint32_t*)(bar + D_COUNT);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nT = a.T / 128;
  const int it = nT - 1 - (blockIdx.x % nT);        // heavy (late) query tiles first
  const int bh = blockIdx.x / nT, b = bh / a.H, h = bh % a.H;
  const int i0 = it * 128, HD = a.H * 64, S = a.M + a.T;
  const int jt_lo = (a.M - a.mem_count) / 128, jt_hi = (a.M + i0) / 128;
  const int NT = jt_hi - jt_lo + 1;                 // key tiles of this CTA
  const int blk0 = (a.M + i0) / 128 - jt_lo;        // upper distance block of the first (oldest) tile; tile n completes block blk0 - n

  if (warp == DQT_MATH_WARPS && lane == 0) {
    tma_prefetch_desc(&tmX); tma_prefetch_desc(&tmM); tma_prefetch_desc(&tmR); tma_prefetch_desc(&tmDO);
    tma_prefetch_desc(&tmP); tma_prefetch_desc(&tmPB); tma_prefetch_desc(&tmDS); tma_prefetch_desc(&tmDD);
    for (int i = 0; i < D_COUNT; i++) {
      uint32_t cnt = 1;
      if (i == D_DPFREE0 || i == D_DPFREE1 || i == D_DSFULL || i == D_ZINIT) cnt = DQT_MATH_WARPS;
      if (i == D_DSFREE || i == D_SFREE0 || i == D_SFREE1) cnt = 2;       // the MMA that read the buffer + the TMA store that read it
      mbar_init(&bar[i], cnt);
    }
    mbar_fence_init();
  }
  if (warp == DQT_MATH_WARPS + 1) tmem_alloc<512>(tmem_holder);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  if (warp >= DQT_MATH_WARPS) {
    if (warp == DQT_MATH_WARPS) {
      // =========================================== TMA loads ===========================================
      if (lane == 0) {
        mbar_expect_tx(&bar[D_DOFULL], T16K);
        tma_load_2d(smem + DQO_DO, &tmDO, h * 64, b * a.T + i0, &bar[D_DOFULL]);
        auto load_kv = [&](int n, int which) {      // which: 0 = K, 1 = V
          const int j0 = (jt_lo + n) * 128;
          mbar_wait(&bar[which ? D_VEMPTY : D_KEMPTY], (n & 1) ^ 1);
          uint64_t* full = &bar[which ? D_VFULL : D_KFULL];
          mbar_expect_tx(full, T16K);
          uint8_t* dst = smem + (which ? DQO_V : DQO_K);
          if (j0 < a.M) tma_load_2d(dst, &tmM, which * HD + h * 64, b * a.M + j0, full);
          else tma_load_2d(dst, &tmX, (1 + which) * HD + h * 64, b * a.T + (j0 - a.M), full);
        };
        auto load_r = [&](int n) {
          mbar_wait(&bar[D_REMPTY], (n & 1) ^ 1);
          mbar_expect_tx(&bar[D_RFULL], T16K);
          tma_load_2d(smem + DQO_R, &tmR, h * 64, (blk0 - n) * 128, &bar[D_RFULL]);
        };
        auto load_p = [&](int n) {
          const int s = n & 1, j0 = (jt_lo + n) * 128;
          mbar_wait(&bar[D_PFREE0 + s], ((n >> 1) & 1) ^ 1);
          mbar_expect_tx(&bar[D_PFULL0 + s], 2 * T16K);
          tma_load_2d(smem + DQO_P + s * 2 * T16K, &tmP, j0, bh * a.T + i0, &bar[D_PFULL0 + s]);
          tma_load_2d(smem + DQO_P + s * 2 * T16K + T16K, &tmP, j0 + 64, bh * a.T + i0, &bar[D_PFULL0 + s]);
        };
        // V has its own producer thread (warp 19): dPd runs two tiles ahead of the tile math, so V(n+2)'s buffer is free long before
        // the buffers of this thread's streams are, and a request queued behind their waits arrived microseconds late
        // (profiles/r2g_attn_bwd_dq_tc_timeline.txt).  The waits below come in the order their conditions become true: K (after dS K of
        // tile n-1), the probability buffer (after the first TMA store group of n-1 has read it), Rk (after the position MMA of n-1).
        load_p(0);
        load_kv(0, 0);
        load_r(0);
        if (NT > 1) load_p(1);
        for (int n = 1; n < NT; n++) {
          load_kv(n, 0);
          if (n + 1 < NT) load_p(n + 1);
          load_r(n);
        }
      }
    } else if (warp == DQT_MATH_WARPS + 3) {
      // =========================================== TMA loads: V ===========================================
      if (lane == 0) {
        for (int n = 0; n < NT; n++) {
          const int j0 = (jt_lo + n) * 128;
          mbar_wait(&bar[D_VEMPTY], (n & 1) ^ 1);
          mbar_expect_tx(&bar[D_VFULL], T16K);
          if (j0 < a.M) tma_load_2d(smem + DQO_V, &tmM, HD + h * 64, b * a.M + j0, &bar[D_VFULL]);
          else tma_load_2d(smem + DQO_V, &tmX, 2 * HD + h * 64, b * a.T + (j0 - a.M), &bar[D_VFULL]);
        }
      }
    } else if (warp == DQT_MATH_WARPS + 1) {
      // =========================================== MMA issuer (whole warp, elected lane issues) ===========================================
      {
        constexpr uint32_t idesc_s = (1u << 4) | (1u << 7) | (1u << 10) | ((128u >> 3) << 17) | ((128u >> 4) << 24);
        constexpr uint32_t idesc_n64 = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 16) | ((64u >> 3) << 17) | ((128u >> 4) << 24);
        const uint64_t d_do = desc_kmajor(smem_u32(smem + DQO_DO)), d_v = desc_kmajor(smem_u32(smem + DQO_V)),
                       d_k = desc_mnmajor(smem_u32(smem + DQO_K)), d_r = desc_mnmajor(smem_u32(smem + DQO_R)),
                       d_ds = desc_kmajor(smem_u32(smem + DQO_DS)), d_st0 = desc_kmajor(smem_u32(smem + DQO_STRIP)),
                       d_st1 = desc_kmajor(smem_u32(smem + DQO_STRIP + 2 * T16K));
        auto m1 = [&](int n) {                       // dPd(n) = dO V(n)^T
          const int s = n & 1;
          tc_wait(&bar[D_VFULL], n & 1);
          if (n >= 2) tc_wait(&bar[D_DPFREE0 + s], ((n >> 1) & 1) ^ 1);
          tc_fence_after();
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < 4; k++) umma_bf16(tmem_base + DTM_DP + 128 * s, d_do + (uint64_t)(2 * k), d_v + (uint64_t)(2 * k), idesc_s, (uint32_t)(k > 0));
            umma_commit(&bar[D_DPFULL0 + s]);
            umma_commit(&bar[D_VEMPTY]);
          }
          __syncwarp();
        };
        tc_wait(&bar[D_DOFULL], 0);
        m1(0);
        if (NT > 1) m1(1);
        for (int n = 0; n < NT; n++) {
          const int sb = (blk0 - n) & 1;
          tc_wait(&bar[D_DSFULL], n & 1);
          tc_wait(&bar[D_KFULL], n & 1);
          tc_fence_after();
          if (elect_one()) {
#pragma unroll
            for (int hf = 0; hf < 2; hf++)
#pragma unroll
              for (int k = 0; k < 4; k++)
                umma_bf16(tmem_base + DTM_AC, d_ds + (uint64_t)(hf * (T16K >> 4) + 2 * k), d_k + (uint64_t)(hf * (8192 >> 4) + 128 * k), idesc_n64,
                          (uint32_t)(n > 0 || hf > 0 || k > 0));
            umma_commit(&bar[D_DSFREE]);
            umma_commit(&bar[D_KEMPTY]);
          }
          __syncwarp();
          tc_wait(&bar[D_RFULL], n & 1);
          tc_fence_after();
          if (elect_one()) {
            const uint64_t d_st = sb ? d_st1 : d_st0;
#pragma unroll
            for (int hf = 0; hf < 2; hf++)
#pragma unroll
              for (int k = 0; k < 4; k++)
                umma_bf16(tmem_base + DTM_BD, d_st + (uint64_t)(hf * (T16K >> 4) + 2 * k), d_r + (uint64_t)(hf * (8192 >> 4) + 128 * k),
                          idesc_n64, (uint32_t)(n > 0 || hf > 0 || k > 0));
            umma_commit(&bar[D_SFREE0 + sb]);
            umma_commit(&bar[D_REMPTY]);
            if (n == NT - 1) umma_commit(&bar[D_DQFULL]);
          }
          __syncwarp();
          if (n + 2 < NT) m1(n + 2);
        }
      }
    } else if (warp == DQT_MATH_WARPS + 2) {
      // =========================================== TMA stores ===========================================
      if (lane == 0) {
        const uint32_t ds = smem_u32(smem + DQO_DS), st = smem_u32(smem + DQO_STRIP), pp = smem_u32(smem + DQO_P);
        const int row_bh = bh * a.T + i0, row_b = b * a.T + i0;
        mbar_wait(&bar[D_ZINIT], 0);
        for (int blk = blk0 + 1; blk < S / 128; blk++) {   // distances beyond the oldest visible key: zeros for the dRk GEMM
          tma_store_2d(&tmDD, st + (blk0 & 1) * 2 * T16K, h * S + blk * 128, row_b);
          tma_store_2d(&tmDD, st + (blk0 & 1) * 2 * T16K + T16K, h * S + blk * 128 + 64, row_b);
        }
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        mbar_arrive(&bar[D_ZDONE]);
        for (int n = 0; n < NT; n++) {
          const int j0 = (jt_lo + n) * 128, U = blk0 - n, sb = U & 1;
          mbar_wait(&bar[D_DSFULL], n & 1);
          // three bulk groups, released in the order the pipeline needs the buffers back: the probability buffer first - its reload for
          // tile n + 2 comes from HBM (~2 us) and must be requested before tile n + 1 is half done (the timeline in
          // profiles/r2g_attn_bwd_dq_tc_timeline.txt: as the last group its read finished 2 us after the tile) - then the dS tile, then the
          // distance block
          tma_store_2d(&tmPB, pp + (n & 1) * 2 * T16K, j0, row_bh);
          tma_store_2d(&tmPB, pp + (n & 1) * 2 * T16K + T16K, j0 + 64, row_bh);
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          tma_store_2d(&tmDS, ds, j0, row_bh);
          tma_store_2d(&tmDS, ds + T16K, j0 + 64, row_bh);
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          tma_store_2d(&tmDD, st + sb * 2 * T16K, h * S + U * 128, row_b);
          tma_store_2d(&tmDD, st + sb * 2 * T16K + T16K, h * S + U * 128 + 64, row_b);
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          asm volatile("cp.async.bulk.wait_group.read 2;" ::: "memory");
          mbar_arrive(&bar[D_PFREE0 + (n & 1)]);
          asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
          mbar_arrive(&bar[D_DSFREE]);
          asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
          mbar_arrive(&bar[D_SFREE0 + sb]);
        }
        asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
      }
    }
  } else {
    // =========================================== tile math ===========================================
    const int qk = warp >> 2, q4 = warp & 3;        // key quarter (32 keys) of every tile, TMEM lane quarter
    const int hf = qk >> 1, sub = qk & 1;           // ... = 64-key half tile hf, 16-byte chunks 4 sub .. 4 sub + 3 of its rows
    const int r = q4 * 32 + lane;                   // query row of this thread inside the tile
    const int row = i0 + r;
    const uint32_t t_lane = tmem_base + ((uint32_t)(q4 * 32) << 16);
    const uint32_t rowoff = (uint32_t)((r >> 3) * 1024 + (r & 7) * 128);
    const int rsw = r & 7;
    {   // both distance-block buffers start as zeros
      uint4* z = (uint4*)(smem + DQO_STRIP) + threadIdx.x;
#pragma unroll
      for (int i = 0; i < 4 * T16K / 16 / (DQT_MATH_WARPS * 32); i++) z[i * DQT_MATH_WARPS * 32] = make_uint4(0u, 0u, 0u, 0u);
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar[D_ZINIT]);
    }
    const long long bhrow = (long long)bh * a.T + row;
    const float lse2 = a.lse[bhrow] * LOG2E, dl = ba.delta[bhrow];
    const float c2 = a.scale * LOG2E;
    const uint32_t drop_base = (uint32_t)((bhrow * S) >> 1);
    const float* mrow = a.m_save + bhrow * (S >> 6);
    const int C0 = 128 + r - 32 * qk;               // strip column of this thread's first key: c = C0 - jj
    uint8_t* const strip = smem + DQO_STRIP;

    float mnext = __ldg(mrow + ((jt_lo * 128 + 32 * qk) >> 6));
    for (int n = 0; n < NT; n++) {
      const int j0q = (jt_lo + n) * 128 + 32 * qk;   // full-context index of this thread's first key
      const float mblk = mnext;
      if (n + 1 < NT) mnext = __ldg(mrow + ((j0q + 128) >> 6));
      const int s = n & 1, U = blk0 - n, sbU = U & 1;
      const bool has_L = n + 1 < NT;                 // the diagonal tile's lower block would hold negative distances (masked keys)
      mbar_wait(&bar[D_PFULL0 + s], (n >> 1) & 1);
      mbar_wait(&bar[D_DPFULL0 + s], (n >> 1) & 1);
      tc_fence_after();
      uint32_t dpd[32];
      tmem_ld_32x32(t_lane + DTM_DP + 128 * s + 32 * qk, dpd);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar[D_DPFREE0 + s]);
      const float fac = ex2_fast(mblk * c2 - lse2);
      uint8_t* const prow = smem + DQO_P + s * 2 * T16K + hf * T16K + rowoff;
      uint8_t* const dsrow = smem + DQO_DS + hf * T16K + rowoff;
      uint8_t* const bufU = strip + sbU * 2 * T16K + rowoff;
      uint8_t* const bufL = strip + (sbU ^ 1) * 2 * T16K + rowoff;
      uint32_t dsw[16];                               // dS of this thread's 32 keys, bf16 pairs (keys 2 i, 2 i + 1)
#pragma unroll
      for (int ck = 0; ck < 4; ck++) {
        const uint32_t choff = (uint32_t)(((4 * sub + ck) ^ rsw) << 4);
        const uint4 raw = *(const uint4*)(prow + choff);
        const uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
        uint32_t pk[4];
#pragma unroll
        for (int e = 0; e < 4; e++) {
          const int pp = 4 * ck + e;
          float keep0 = 1.f, keep1 = 1.f;
          if (a.drop_thresh) {
            const uint32_t hb = drop_pair_bits(a.drop_seed, drop_base + (uint32_t)(j0q >> 1) + pp);
            keep0 = ((hb & 0xFFFFu) >= a.drop_thresh) ? a.drop_scale : 0.f;
            keep1 = ((hb >> 16) >= a.drop_thresh) ? a.drop_scale : 0.f;
          }
          const float p0 = bf16lo(w[e]) * fac, p1 = bf16hi(w[e]) * fac;
          const float s0 = p0 * (__uint_as_float(dpd[2 * pp]) * keep0 - dl) * a.scale;
          const float s1 = p1 * (__uint_as_float(dpd[2 * pp + 1]) * keep1 - dl) * a.scale;
          pk[e] = pack_bf16x2(keep0 * p0, keep1 * p1);
          dsw[pp] = pack_bf16x2(s0, s1);
        }
        *(uint4*)(prow + choff) = make_uint4(pk[0], pk[1], pk[2], pk[3]);      // Pd over the saved probabilities (own row, own chunk)
      }
      // the dS tile and the distance blocks are single buffers: the previous tile's MMAs and TMA stores must have read them (they had the
      // whole tile math above to do so)
      if (n >= 1) mbar_wait(&bar[D_DSFREE], (n - 1) & 1);
#pragma unroll
      for (int ck = 0; ck < 4; ck++)
        *(uint4*)(dsrow + (((4 * sub + ck) ^ rsw) << 4)) = make_uint4(dsw[4 * ck], dsw[4 * ck + 1], dsw[4 * ck + 2], dsw[4 * ck + 3]);
      if (n == 0) mbar_wait(&bar[D_ZDONE], 0);
      if (n >= 1 && has_L) mbar_wait(&bar[D_SFREE0 + (sbU ^ 1)], ((n - 1) >> 1) & 1);
      // ---- the same 32 values in (row, distance) coordinates: key jj sits in column C0 - jj of this tile's [128][256] window, i.e. the
      // run of columns [C0 - 31, C0] in REVERSED key order.  The run starts at a lane-dependent offset sh = (C0 - 31) & 7 inside an aligned
      // 8-column chunk (16 bytes of the swizzled layout), so the reversed run is shifted right by `sh` elements with a three-stage barrel
      // shifter on the packed words (select + byte-permute), which leaves three full chunks (one 16-byte store each) and two partial ones
      // at the ends (element stores: the rest of those chunks belongs to a neighbouring thread or key tile, possibly being written now).
      {
        const int c_lo = C0 - 31, sh = c_lo & 7, cbase = c_lo - sh;
        uint32_t y[20];
#pragma unroll
        for (int i = 0; i < 20; i++) {                // stage 0: reverse (word i = keys 31 - 2 i, 30 - 2 i), shifted by one element if sh & 1
          const uint32_t cur = i < 16 ? __byte_perm(dsw[15 - i], 0u, 0x1032) : 0u;
          const uint32_t prev = (i >= 1 && i <= 16) ? __byte_perm(dsw[16 - i], 0u, 0x1032) : 0u;
          y[i] = (sh & 1) ? __byte_perm(prev, cur, 0x5432) : cur;
        }
        if (sh & 2) {
#pragma unroll
          for (int i = 19; i >= 1; i--) y[i] = y[i - 1];
        }
        if (sh & 4) {
#pragma unroll
          for (int i = 19; i >= 2; i--) y[i] = y[i - 2];
        }
        auto chunk_ptr = [&](int c) -> uint8_t* {     // address of the aligned 8-column chunk at window column c; nullptr: not stored
          if (c >= 128) { const int cc = c - 128; return bufU + (cc >> 6) * T16K + ((((cc & 63) >> 3) ^ rsw) << 4); }
          return has_L ? bufL + (c >> 6) * T16K + ((((c & 63) >> 3) ^ rsw) << 4) : nullptr;
        };
#pragma unroll
        for (int j = 1; j < 4; j++) {
          uint8_t* dst = chunk_ptr(cbase + 8 * j);
          if (dst) *(uint4*)dst = make_uint4(y[4 * j], y[4 * j + 1], y[4 * j + 2], y[4 * j + 3]);
        }
        uint8_t* d0 = chunk_ptr(cbase);
        uint8_t* d4 = chunk_ptr(cbase + 32);
        if (sh == 0) {
          if (d0) *(uint4*)d0 = make_uint4(y[0], y[1], y[2], y[3]);
        } else {
#pragma unroll
          for (int e = 0; e < 8; e++) {
            const uint16_t lo = (uint16_t)((e & 1) ? (y[e >> 1] >> 16) : (y[e >> 1] & 0xFFFFu));
            const uint16_t hi = (uint16_t)((e & 1) ? (y[16 + (e >> 1)] >> 16) : (y[16 + (e >> 1)] & 0xFFFFu));
            if (d0 && e >= sh) *(uint16_t*)(d0 + 2 * e) = lo;
            if (d4 && e < sh) *(uint16_t*)(d4 + 2 * e) = hi;
          }
        }
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar[D_DSFULL]);
    }

    // ---- dq = content part + position part (columns 16 qk .. 16 qk + 15 of this row); du / dv = their column sums over all rows
    mbar_wait(&bar[D_DQFULL], 0);
    tc_fence_after();
    uint32_t xa[32], xb[32];                        // 32-column loads, the first 16 are this thread's
    tmem_ld_32x32(t_lane + DTM_AC + 16 * qk, xa);
    tmem_ld_32x32(t_lane + DTM_BD + 16 * qk, xb);
    tmem_ld_wait();
    tc_fence_before();
    bf16* qrow = ba.dqkv_x + ((long long)b * a.T + row) * a.ldx + h * 64 + 16 * qk;
#pragma unroll
    for (int k = 0; k < 2; k++) {
      uint32_t o[4];
#pragma unroll
      for (int e = 0; e < 4; e++) {
        const int d0 = 8 * k + 2 * e;
        o[e] = pack_bf16x2(__uint_as_float(xa[d0]) + __uint_as_float(xb[d0]), __uint_as_float(xa[d0 + 1]) + __uint_as_float(xb[d0 + 1]));
      }
      *(uint4*)(qrow + 8 * k) = make_uint4(o[0], o[1], o[2], o[3]);
    }
    float* red = (float*)(smem + DQO_K);            // the K tile is dead (every MMA has retired): [16 warps][32] column sums
#pragma unroll
    for (int i = 0; i < 16; i++) {
      const float sa = warp_sum(__uint_as_float(xa[i])), sbv = warp_sum(__uint_as_float(xb[i]));
      if (lane == 0) { red[warp * 32 + i] = sa; red[warp * 32 + 16 + i] = sbv; }
    }
    asm volatile("bar.sync 1, %0;" ::"n"(DQT_MATH_WARPS * 32) : "memory");
    if (threadIdx.x < 128) {
      const int t = threadIdx.x >> 6, cc = threadIdx.x & 63, w0 = (cc >> 4) * 4;
      float sum = 0.f;
#pragma unroll
      for (int q = 0; q < 4; q++) sum += red[(w0 + q) * 32 + t * 16 + (cc & 15)];
      atomicAdd((t ? ba.dv : ba.du) + h * 64 + cc, sum);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == DQT_MATH_WARPS + 1) tmem_dealloc<512>(tmem_base);
}

}  // namespace

bool attn_bwd_dq_tc_supported(const AttnTrainBwdArgs& ba) {
  const AttnTrainArgs& a = ba.f;
  return a.p_save && a.m_save && a.T % 128 == 0 && a.M % 128 == 0 && a.mem_count % 128 == 0 &&
         a.ldx % 8 == 0 && (a.M == 0 || a.ldm % 8 == 0);
}

int attn_bwd_dq_tc(const AttnTrainBwdArgs& ba, cudaStream_t st) {
  const AttnTrainArgs& a = ba.f;
  static bool configured = false;
  if (!configured) {
    DMG_CUDA_OK(cudaFuncSetAttribute(attn_bwd_dq_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, DQT_SMEM));
    configured = true;
  }
  const int HD = a.H * 64;
  const long long S = (long long)a.M + a.T, rows_bh = (long long)a.B * a.H * a.T;
  const TensorMap2D *tx = nullptr, *tm = nullptr, *tr = nullptr, *tdo = nullptr, *tp = nullptr, *tpb = nullptr, *tds = nullptr, *tdd = nullptr;
  if (train_get_tmap(a.qkv_x, 3 * HD, (long long)a.B * a.T, a.ldx, 128, &tx)) return -1;
  if (a.M > 0) { if (train_get_tmap(a.kv_m, 2 * HD, (long long)a.B * a.M, a.ldm, 128, &tm)) return -1; }
  else tm = tx;
  if (train_get_tmap(a.rk, HD, S, HD, 128, &tr)) return -1;
  if (train_get_tmap(ba.dout, HD, (long long)a.B * a.T, HD, 128, &tdo)) return -1;
  if (train_get_tmap(a.p_save, S, rows_bh, S, 128, &tp)) return -1;
  if (train_get_tmap(ba.p_buf, S, rows_bh, S, 128, &tpb)) return -1;
  if (train_get_tmap(ba.ds_buf, S, rows_bh, S, 128, &tds)) return -1;
  if (train_get_tmap(ba.ds_dist, (long long)a.H * S, (long long)a.B * a.T, (long long)a.H * S, 128, &tdd)) return -1;
  return launch_np(attn_bwd_dq_tc_kernel, dim3(a.B * a.H * (a.T / 128)), dim3(DQT_THREADS), (size_t)DQT_SMEM, st, *(const CUtensorMap*)tx->bytes,
                   *(const CUtensorMap*)tm->bytes, *(const CUtensorMap*)tr->bytes, *(const CUtensorMap*)tdo->bytes, *(const CUtensorMap*)tp->bytes,
                   *(const CUtensorMap*)tpb->bytes, *(const CUtensorMap*)tds->bytes, *(const CUtensorMap*)tdd->bytes, ba);
}


bool attn_bwd_dkv_tc_supported(const AttnTrainBwdArgs& ba) {
  const AttnTrainArgs& a = ba.f;
  return ba.qu && a.T % 128 == 0 && a.M % 128 == 0 && a.mem_count % 128 == 0 && a.ldx % 8 == 0 &&
         (a.M == 0 || a.ldm % 8 == 0);
}

int attn_bwd_dkv_tc(const AttnTrainBwdArgs& ba, cudaStream_t st) {
  const AttnTrainArgs& a = ba.f;
  static bool configured = false;
  if (!configured) {
    DMG_CUDA_OK(cudaFuncSetAttribute(attn_bwd_dkv_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, DKV_SMEM));
    configured = true;
  }
  const int HD = a.H * 64;
  const long long S = (long long)a.M + a.T;
  const TensorMap2D *tp = nullptr, *ts = nullptr, *td = nullptr, *tq = nullptr;
  if (train_get_tmap(ba.p_buf, S, (long long)a.B * a.H * a.T, S, 64, &tp)) return -1;
  if (train_get_tmap(ba.ds_buf, S, (long long)a.B * a.H * a.T, S, 64, &ts)) return -1;
  if (train_get_tmap(ba.dout, HD, (long long)a.B * a.T, HD, 64, &td)) return -1;
  if (train_get_tmap(ba.qu, HD, (long long)a.B * a.T, HD, 64, &tq)) return -1;
  return launch_np(attn_bwd_dkv_tc_kernel, dim3(a.B * a.H * (int)(S / 128)), dim3(192), (size_t)DKV_SMEM, st, *(const CUtensorMap*)tp->bytes,
                   *(const CUtensorMap*)ts->bytes, *(const CUtensorMap*)td->bytes, *(const CUtensorMap*)tq->bytes, ba);
}

bool attn_train_fwd_tc_supported(const AttnTrainArgs& a) {
  return a.T % 128 == 0 && a.M % 128 == 0 && a.mem_count % 128 == 0 && a.ldx % 8 == 0 && (a.M == 0 || a.ldm % 8 == 0);
}

int attn_train_fwd_tc(const AttnTrainArgs& a, cudaStream_t st) {
  static bool configured = false;
  if (!configured) {
    DMG_CUDA_OK(cudaFuncSetAttribute(attn_train_fwd_tc_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM));
    DMG_CUDA_OK(cudaFuncSetAttribute(attn_train_fwd_tc_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM));
    configured = true;
  }
  DMG_CHECK((a.p_save == nullptr) == (a.m_save == nullptr), "training attention: p_save and m_save go together");
  const int HD = a.H * 64;
  const TensorMap2D *tx = nullptr, *tm = nullptr, *tr = nullptr;
  if (train_get_tmap(a.qkv_x, 3 * HD, (long long)a.B * a.T, a.ldx, 128, &tx)) return -1;
  if (a.M > 0) { if (train_get_tmap(a.kv_m, 2 * HD, (long long)a.B * a.M, a.ldm, 128, &tm)) return -1; }
  else tm = tx;
  if (train_get_tmap(a.rk, HD, (long long)a.M + a.T, HD, 128, &tr)) return -1;
  const dim3 grid(a.B * a.H * (a.T / 128)), block(TC_THREADS);
  if (a.p_save) {
    const TensorMap2D *tp = nullptr, *tqu = tx, *tqv = tx;   // p_save as [B*H*T rows, S columns], 64 x 32 boxes
    if (train_get_tmap(a.p_save, (long long)a.M + a.T, (long long)a.B * a.H * a.T, (long long)a.M + a.T, 32, &tp)) return -1;
    DMG_CHECK((a.qu_save == nullptr) == (a.qv_save == nullptr), "training attention: qu_save and qv_save go together");
    if (a.qu_save) {
      if (train_get_tmap(a.qu_save, HD, (long long)a.B * a.T, HD, 128, &tqu)) return -1;
      if (train_get_tmap(a.qv_save, HD, (long long)a.B * a.T, HD, 128, &tqv)) return -1;
    }
    return launch_np(attn_train_fwd_tc_kernel<true, false>, grid, block, (size_t)TC_SMEM, st, *(const CUtensorMap*)tx->bytes,
                     *(const CUtensorMap*)tm->bytes, *(const CUtensorMap*)tr->bytes, *(const CUtensorMap*)tp->bytes,
                     *(const CUtensorMap*)tqu->bytes, *(const CUtensorMap*)tqv->bytes, a);
  }
  return launch_np(attn_train_fwd_tc_kernel<false, false>, grid, block, (size_t)TC_SMEM, st, *(const CUtensorMap*)tx->bytes,
                   *(const CUtensorMap*)tm->bytes, *(const CUtensorMap*)tr->bytes, *(const CUtensorMap*)tx->bytes,
                   *(const CUtensorMap*)tx->bytes, *(const CUtensorMap*)tx->bytes, a);
}

// The same kernel over the inference engine's K/V rings and per-head Rd cache (model.cu: bf16 segments of T % 128 == 0 tokens over a
// warm memory with mem_count, the ring position and mem_len multiples of 128).  qkv16: [B*T, 3*H*64] bf16 of the current segment.
bool attn_fwd_tc_ring_supported(int T, int Dh, int M, int mem_count, int pos_total) {
  return Dh == 64 && T % 128 == 0 && M > 0 && M % 128 == 0 && mem_count > 0 && mem_count % 128 == 0 && pos_total % 128 == 0;
}

int attn_fwd_tc_ring(const bf16* qkv16, const bf16* kring, const bf16* vring, const bf16* rd, int Dcap, const float* u, const float* v,
                     bf16* out, int B, int T, int H, int M, int mem_count, int win, int k, int pos_total, int b0, int max_batch, float scale,
                     cudaStream_t st) {
  static bool configured = false;
  if (!configured) {
    DMG_CUDA_OK(cudaFuncSetAttribute(attn_train_fwd_tc_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM));
    configured = true;
  }
  const int HD = H * 64;
  AttnTrainArgs a;
  a.qkv_x = qkv16; a.ldx = 3 * HD; a.kv_m = nullptr; a.ldm = 0; a.rk = rd; a.u = u; a.v = v; a.out = out; a.lse = nullptr;
  a.B = B; a.T = T; a.H = H; a.M = M; a.mem_count = mem_count; a.win = win; a.k = k; a.scale = scale;
  a.drop_thresh = 0; a.drop_seed = 0; a.drop_scale = 1.f;
  a.ring_head = pos_total % M; a.ring_b0 = b0; a.ring_dcap = Dcap;
  const TensorMap2D *tx = nullptr, *tk = nullptr, *tv = nullptr, *tr = nullptr;
  if (train_get_tmap(qkv16, 3 * HD, (long long)B * T, 3 * HD, 128, &tx)) return -1;
  if (train_get_tmap(kring, 64, (long long)max_batch * H * M, 64, 128, &tk)) return -1;
  if (train_get_tmap(vring, 64, (long long)max_batch * H * M, 64, 128, &tv)) return -1;
  if (train_get_tmap(rd, 64, (long long)H * Dcap, 64, 128, &tr)) return -1;
  return launch_np(attn_train_fwd_tc_kernel<false, true>, dim3(B * H * (T / 128)), dim3(TC_THREADS), (size_t)TC_SMEM, st,
                   *(const CUtensorMap*)tx->bytes, *(const CUtensorMap*)tk->bytes, *(const CUtensorMap*)tr->bytes, *(const CUtensorMap*)tv->bytes,
                   *(const CUtensorMap*)tx->bytes, *(const CUtensorMap*)tx->bytes, a);
}

}  // namespace dmg
