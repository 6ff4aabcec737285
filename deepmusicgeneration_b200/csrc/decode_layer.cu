// The one-token step between two attention launches as ONE kernel (SURVEY.md 2.2 K10-K12 + K3 of the next layer):
//
//     x   = LayerNorm(x + out(attn))                     fastai MultiHeadRelativeAttention.forward   (after _apply_attention)
//     x   = LayerNorm(x + W2 gelu(W1 x + b1) + b2)       fastai feed_forward (SequentialEx + MergeLayer + LayerNorm)
//     qkv = Wqkv' x                                      the NEXT layer's fused q|k|v projection (deep_music_genre.py:1641-1644 loop body)
//
// The unfused path runs these as 6 dependent launches per layer (4 split-K GEMMs + 2 LayerNorms, ~6 us each: every one of them
// is bound by its launch-to-launch latency chain, not by bytes or flops - profiles/README.md).  Here a CLUSTER of 8 CTAs owns 32
// generation streams ("rows") for the whole chain, so nothing but those 32 rows ever has to be exchanged:
//
//  * operands are swapped: D[feature, row] = W[feature, k] * X[row, k]^T - the weights are the M = 64 / 128 operand of
//    tcgen05.mma (K-major as nn.Linear stores them), the 32 rows are the N = 32 operand; accumulators live in TMEM, lane = feature.
//    An MMA this small is bound by the latency of its accumulate chain (measured: ~180 cycles per dependent MMA with one
//    accumulator per tile, profiles/README.md r2d), so every tile keeps 4-8 INDEPENDENT partial accumulators (one per 16-wide K
//    step of a k-block, times two alternating k-blocks for single-tile phases; tiles of a phase are interleaved) that the
//    epilogue adds up;
//  * every GEMM's output features are split over the 8 CTAs of the cluster, so each CTA streams 1/8 of the layer's weights
//    (768 KB at C2) through a 10-stage TMA ring - the weight stream never waits for activations and runs ahead across phases;
//  * the exchanges of a layer: out-projection -> LayerNorm 1 stays inside the cluster's shared memory (every CTA normalises the 64
//    features it computed for all 32 rows; only the (mean, M2) pairs of the slices and then the finished bf16 / fp32 slices travel,
//    over distributed shared memory); FFN-up -> FFN-down needs none (a CTA's GeLU slice is its own K slice of the split-K FFN-down);
//    FFN-down -> LayerNorm 2 goes through an L2-resident scratch of partial sums and the second LayerNorm of the 4 rows a CTA owns
//    is broadcast as the bf16 B operand into all 8 CTAs' shared memory (canonical 128B-swizzled K-major layout); four hardware
//    cluster barriers (release / acquire) per layer;
//  * launched with programmatic dependent launch: barrier init, TMEM allocation and the first weight tiles overlap the tail of
//    the attention kernel.
//
// Warp roles: warp 0 = TMA producer (eight lanes per round of stage uses), warps 1-2 = tcgen05.mma issuers (stage uses alternate between
// them; each runs its loop as a whole warp in uniform control flow and its elected lane issues the four K steps of a k-block),
// the last 8 warps = TMEM epilogues + LayerNorm.
// Grid: 8 CTAs per 32 streams - 64 CTAs at the benchmark's 256 streams (at most 15 clusters of 8 are co-resident on a B200, so
// 16-row clusters would run in two waves).
#include <cuda.h>

#include "attention_decode3.cuh"
#include "kernels.cuh"
#include "launch.cuh"

namespace dmg {
namespace {

constexpr int DL_STAGES = 10;                       // weight ring: 10 x 16 KB in flight
constexpr int DL_STAGE = 128 * 128;                 // one stage = one weight tile: up to 128 features x 64 bf16
constexpr int DL_B_BYTES = DL_ROWS * 128;           // activation k-block: 32 rows x 64 bf16
constexpr int DL_D = 512;                           // d_model this kernel is specialised for (LayerNorm thread mapping)
constexpr int DL_XA_BYTES = DL_ROWS * DL_D * 2;     // resident B operand: 32 rows x 512 (attention output, then LayerNorm rows), 8 k-blocks of 4 KB
constexpr int DL_HS_KB = 4;                         // k-blocks of this CTA's GeLU slice (d_inner / 8 / 64)
constexpr int DL_HS_BYTES = DL_HS_KB * DL_B_BYTES;  // resident B operand of the FFN-down phase: 32 rows x 256
constexpr int DL_OWN = DL_ROWS / DL_CLUSTER;        // rows whose second LayerNorm this CTA computes (4)
constexpr int DL_X1_BYTES = DL_OWN * DL_D * 4;      // their LayerNorm-1 output (fp32 residual of LayerNorm 2)
constexpr int DL_MMAW = 2;                          // MMA-issuing warps (round-robin over stage uses)
constexpr int DL_THREADS = 32 * (1 + DL_MMAW + 8);  // producer warp + MMA-issuing warps + 8 epilogue warps
constexpr int DL_EPI0 = 32 * (1 + DL_MMAW);         // first epilogue thread
constexpr int DL_EPI = 256;                         // epilogue / LayerNorm threads
constexpr int DL_LN_BYTES = 4 * DL_D * 4;           // ln1 w, b and ln2 w, b staged in shared memory
constexpr int DL_SMEM = DL_STAGES * DL_STAGE + DL_XA_BYTES + DL_HS_BYTES + DL_X1_BYTES + DL_LN_BYTES + 512 /*barriers + reduction scratch*/ + 1024 /*alignment slack*/;
constexpr int DL_TMEM_COLS = 512;                   // 16 partial accumulators x 32 columns; phases reuse the columns
constexpr int DL_CHAIN = DL_ROWS;                   // TMEM columns of one partial accumulator (N = 32 rows)
static_assert(DL_SMEM <= 227 * 1024, "decode_layer_kernel: shared memory budget");

__device__ __forceinline__ uint64_t dl_desc_sw128(uint32_t smem_addr) {
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
__host__ __device__ constexpr uint32_t dl_idesc(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ uint32_t dl_cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
// split-phase cluster barrier, every thread of the cluster takes part (non-aligned forms: the one-lane roles diverge)
__device__ __forceinline__ void dl_arrive() { asm volatile("barrier.cluster.arrive.release;" ::: "memory"); }
__device__ __forceinline__ void dl_wait() { asm volatile("barrier.cluster.wait.acquire;" ::: "memory"); }
__device__ __forceinline__ void dl_fence_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }
__device__ __forceinline__ void dl_fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
// bounded spin without the printf of mbar_wait (a protocol bug must trap, not hang the GPU box)
__device__ __forceinline__ void dl_spin(uint64_t* bar, uint32_t parity) {
  uint32_t n = 0;
  while (!mbar_try_wait(bar, parity))
    if (++n > (1u << 27)) __trap();
}
__device__ __forceinline__ float4 ldcg4(const float* p) { return __ldcg((const float4*)p); }
// optional per-role timeline (DecodeLayerArgs::dbg, scripts/probe_decode_layer.py): slot = role * 16 + mark, value = %globaltimer ns
__device__ __forceinline__ void dl_mark(unsigned long long* dbg, int role, int mark) {
  if (dbg == nullptr) return;
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  dbg[role * 16 + mark] = t;
}

// tanh-GeLU with the hardware tanh (error ~5e-4, below the bf16 rounding of the value that is stored)
__device__ __forceinline__ float dl_gelu(float x) {
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(0.7978845608028654f * (x + 0.044715f * x * x * x)));
  return 0.5f * x * (1.f + t);
}

// LayerNorm over the 512 features of one row held by 8 consecutive lanes (64 values each); eps 1e-5, two-pass
__device__ __forceinline__ void dl_layernorm(float (&z)[64], const float* __restrict__ w, const float* __restrict__ b, int t) {
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 64; i++) s += z[i];
  s += __shfl_xor_sync(0xffffffffu, s, 1); s += __shfl_xor_sync(0xffffffffu, s, 2); s += __shfl_xor_sync(0xffffffffu, s, 4);
  const float mean = s * (1.f / DL_D);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < 64; i++) { const float c = z[i] - mean; q += c * c; }
  q += __shfl_xor_sync(0xffffffffu, q, 1); q += __shfl_xor_sync(0xffffffffu, q, 2); q += __shfl_xor_sync(0xffffffffu, q, 4);
  const float rstd = rsqrtf(q * (1.f / DL_D) + 1e-5f);
#pragma unroll
  for (int kb = 0; kb < 8; kb++) {
    const int c = 64 * kb + 8 * t;
    const float4 w0 = *(const float4*)(w + c), w1 = *(const float4*)(w + c + 4);      // shared memory
    const float4 b0 = *(const float4*)(b + c), b1 = *(const float4*)(b + c + 4);
    float* v = z + 8 * kb;
    v[0] = (v[0] - mean) * rstd * w0.x + b0.x; v[1] = (v[1] - mean) * rstd * w0.y + b0.y;
    v[2] = (v[2] - mean) * rstd * w0.z + b0.z; v[3] = (v[3] - mean) * rstd * w0.w + b0.w;
    v[4] = (v[4] - mean) * rstd * w1.x + b1.x; v[5] = (v[5] - mean) * rstd * w1.y + b1.y;
    v[6] = (v[6] - mean) * rstd * w1.z + b1.z; v[7] = (v[7] - mean) * rstd * w1.w + b1.w;
  }
}
// the row as the bf16 B operand: k-block kb = columns [64 kb, +64), 32 rows x 128 B, 16-byte chunk index XOR (row & 7)
__device__ __forceinline__ void dl_store_xa(uint8_t* xa_s, const float (&z)[64], int r, int t) {
#pragma unroll
  for (int kb = 0; kb < 8; kb++) {
    const float* v = z + 8 * kb;
    *(uint4*)(xa_s + kb * DL_B_BYTES + r * 128 + ((t ^ (r & 7)) << 4)) =
        make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
  }
}

// Sum of the `nacc` partial accumulators of one tile for this thread's TMEM lane and its 16 rows (columns [16 half, +16) of
// every 32-column chain)
__device__ __forceinline__ void dl_gather(uint32_t taddr, int nacc, float (&out)[16]) {
  uint32_t r[16];
  tmem_ld_32x16(taddr, r);
  tmem_ld_wait();
#pragma unroll
  for (int i = 0; i < 16; i++) out[i] = __uint_as_float(r[i]);
  for (int c = 1; c < nacc; c++) {
    tmem_ld_32x16(taddr + c * DL_CHAIN, r);
    tmem_ld_wait();
#pragma unroll
    for (int i = 0; i < 16; i++) out[i] += __uint_as_float(r[i]);
  }
}

__device__ __forceinline__ uint32_t dl_mapa(uint32_t local_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void dl_st_cluster_v4(uint32_t addr, uint4 v) {
  asm volatile("st.shared::cluster.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// Phases of one launch (body = bit 0 of mode, next = bit 1):
//   A  out-projection        64 features per CTA  x K = HD     B operand: the attention output rows (TMA -> XA)
//      LayerNorm 1           column-sliced: the CTA's 64 features of all 32 rows; statistics merged over DSMEM; the bf16 slice goes to every
//                            CTA's XA, the fp32 slice to the X1 of the row's LayerNorm-2 owner
//   B  FFN-up + GeLU         256 features per CTA x K = 512    B operand: XA;  result stays in this CTA's shared memory (HS)
//   C  FFN-down, split-K     all 512 features     x K = this CTA's 256 GeLU features (HS); partial sums -> global scratch
//      LayerNorm 2           each CTA reduces the 8 partials of its OWN 4 rows, normalises, broadcasts the bf16 rows into the XA
//                            of all 8 CTAs through distributed shared memory
//   D  next layer's q|k|v    192 features per CTA x K = 512    B operand: XA
// Four cluster barriers per launch: #1 slice statistics published, #2 LayerNorm-1 slices in every XA / X1, #3 partial sums published,
// #4 LayerNorm-2 broadcast done.
// `cluster` = index of this CTA's cluster among the clusters of the fused role (the stand-alone kernel: blockIdx.x / 8).
__device__ __forceinline__ void decode_layer_body(const CUtensorMap& tmAttn, const CUtensorMap& tmWo, const CUtensorMap& tmW1,
                                                  const CUtensorMap& tmW2, const CUtensorMap& tmWq, const DecodeLayerArgs& a_in, int cluster,
                                                  uint8_t* dl_smem) {
  DecodeLayerArgs a = a_in;
  if (cluster != 0 || dl_cluster_ctarank() != 0) a.dbg = nullptr;      // the timeline probe follows CTA 0
  uint8_t* tiles = dl_smem + ((1024u - (smem_u32(dl_smem) & 1023u)) & 1023u);
  uint8_t* xa_s = tiles + DL_STAGES * DL_STAGE;
  uint8_t* hs_s = xa_s + DL_XA_BYTES;
  float* x1_s = (float*)(hs_s + DL_HS_BYTES);                // [4][512] fp32: LayerNorm-1 output of the rows this CTA owns
  float* ln_s = x1_s + DL_OWN * DL_D;                        // [4][512]: ln1 w, ln1 b, ln2 w, ln2 b
  uint64_t* full = (uint64_t*)(ln_s + 4 * DL_D);
  uint64_t* empty = full + DL_STAGES;
  uint64_t* tmem_full = empty + DL_STAGES;   // [4]: one per phase, single use
  uint64_t* xa_ready = tmem_full + 4;        // [0]: LayerNorm-1 rows in XA; [1]: embedded rows in XA (first launch of a step)
  uint64_t* hs_ready = xa_ready + 2;         // GeLU slice in HS
  uint64_t* attn_full = hs_ready + 1;        // attention output rows in XA (TMA)
  uint32_t* tmem_holder = (uint32_t*)(attn_full + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int crank = (int)dl_cluster_ctarank();
  const int row0 = a.row_base + cluster * DL_ROWS;
  const bool body = (a.mode & 1) != 0, next = (a.mode & 2) != 0;
  const int nkb_A = a.HD >> 6, nkb_d = DL_D >> 6;
  constexpr int nB = 2, nC = 4, nD = 2;                      // tiles per phase (decode_layer_supported): 2 x 128, 4 x 128, 128 + 64
  const int fB = a.di / DL_CLUSTER, fD = a.n3 / DL_CLUSTER;  // 256 FFN-up features, 192 q|k|v features per CTA
  const int nA_use = body ? nkb_A : 0, nB_use = body ? nB * nkb_d : 0, nC_use = body ? nC * DL_HS_KB : 0, nD_use = next ? nD * nkb_d : 0;
  pdl_launch_dependents();

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmWo); tma_prefetch_desc(&tmW1); tma_prefetch_desc(&tmW2); tma_prefetch_desc(&tmWq); tma_prefetch_desc(&tmAttn);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < DL_STAGES; s++) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }   // the issuing lane commits per stage
    for (int p = 0; p < 4; p++) mbar_init(&tmem_full[p], DL_MMAW);                              // the issuing lane of every MMA warp commits
    mbar_init(&xa_ready[0], DL_EPI); mbar_init(&xa_ready[1], DL_EPI); mbar_init(hs_ready, DL_EPI); mbar_init(attn_full, 1);
    mbar_fence_init();
  }
  if (warp == 1 + DL_MMAW) tmem_alloc<DL_TMEM_COLS>(tmem_holder);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  if (warp == 0) {
    // ================================================================== TMA producer
    // The weights depend on nothing: all stage uses of the launch stream through the ring as fast as stages free up.  Eight lanes
    // issue in lock-step (lane j = use r + j of a round): one thread's scalar issue loop was measured to be a bottleneck.
    if (lane == 0) dl_mark(a.dbg, 0, 0);
    const int total = nA_use + nB_use + nC_use + nD_use;
    int bar_state = 0;                                   // cluster barrier progress of this warp: n = arrived at barrier #n (#1, #2: LayerNorm 1)
    const uint64_t w_policy = l2_policy_evict_last();
    for (int r = 0; r < total; r += 8) {
      // barrier duties first, at round granularity; never block on a stage whose release needs a barrier we have not served
      if (body && bar_state == 0 && r >= nA_use) { dl_arrive(); bar_state = 1; }                                   // #1
      // stages released by the FFN-up MMAs need LayerNorm 1, i.e. barrier #2 with this warp's arrival
      if (body && bar_state == 1 && r + 8 > nA_use + DL_STAGES) { dl_wait(); dl_arrive(); bar_state = 2; }         // #2
      if (body && bar_state == 2 && r >= nA_use + nB_use) { dl_wait(); dl_arrive(); bar_state = 3; }               // #3
      if (body && bar_state == 3 && r + 8 > nA_use + nB_use + nC_use + DL_STAGES) { dl_wait(); dl_arrive(); bar_state = 4; }   // #4
      const int i = r + lane;
      if (lane < 8 && i < total) {
        const int s = i % DL_STAGES;
        if (i >= DL_STAGES) dl_spin(&empty[s], (uint32_t)((i / DL_STAGES) - 1) & 1u);
        uint8_t* dst = tiles + s * DL_STAGE;
        const CUtensorMap* tm; int c0, frow, boxes;
        if (i < nA_use) { tm = &tmWo; c0 = i * 64; frow = 64 * crank; boxes = 1; }
        else if (i < nA_use + nB_use) { const int j = i - nA_use; tm = &tmW1; c0 = (j / nB) * 64; frow = fB * crank + 128 * (j % nB); boxes = 2; }
        else if (i < nA_use + nB_use + nC_use) { const int j = i - nA_use - nB_use; tm = &tmW2; c0 = fB * crank + (j / nC) * 64; frow = 128 * (j % nC); boxes = 2; }
        else { const int j = i - nA_use - nB_use - nC_use; tm = &tmWq; c0 = (j / nD) * 64; frow = fD * crank + 128 * (j % nD); boxes = (j % nD) == 0 ? 2 : 1; }
        mbar_expect_tx(&full[s], (uint32_t)(boxes * 64 * 128));
        // weights: keep them in L2 across steps (101 MB of bf16 weights against a 126 MB L2; the K/V streams are loaded evict-first)
        tma_load_2d_hint(dst, tm, c0, frow, &full[s], w_policy);
        if (boxes == 2) tma_load_2d_hint(dst + 64 * 128, tm, c0, frow + 64, &full[s], w_policy);
      }
      if (r == 0 && body) {                              // the attention output rows: the only load that waits for the predecessor
        pdl_wait();
        if (lane == 0) mbar_expect_tx(attn_full, (uint32_t)(nkb_A * DL_B_BYTES));
        __syncwarp();
        if (lane < nkb_A) tma_load_2d(xa_s + lane * DL_B_BYTES, &tmAttn, lane * 64, row0, attn_full);
      }
      __syncwarp();
    }
    if (lane == 0) dl_mark(a.dbg, 0, 6);
    if (body) {                                          // whatever barrier duty is left (short launches)
      if (bar_state == 0) { dl_arrive(); bar_state = 1; }
      if (bar_state == 1) { dl_wait(); dl_arrive(); bar_state = 2; }
      if (bar_state == 2) { dl_wait(); dl_arrive(); bar_state = 3; }
      if (bar_state == 3) { dl_wait(); dl_arrive(); bar_state = 4; }
      dl_wait();
    }
  } else if (warp <= DL_MMAW) {
    // ================================================================== tcgen05.mma issuers (warp w: stage uses i with i % DL_MMAW == w - 1)
    // The whole warp runs the issue loop in uniform control flow (waits by all lanes); the elected lane issues the four 16-wide K steps of
    // a k-block back to back, each into its own accumulator chain, and commits the stage.  A tensor-core MMA retires every ~63 cycles
    // whatever N <= 128 is (scripts/probes/probe_mma_rate.cu); in uniform control flow the operands of tcgen05.mma stay in uniform registers
    // and an issue costs a 64-bit add, where the body of a divergent `if (lane < 4)` branch paid a vector-to-uniform move loop with elect
    // and predicate shuffles per MMA (profiles/README.md, round 2h).
    int it = 0;
    const int mine = warp - 1;
    const uint32_t xa_addr = smem_u32(xa_s), hs_addr = smem_u32(hs_s), tiles_addr = smem_u32(tiles);
    constexpr uint64_t DHI = (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
    // k-block `kb` of a tile whose 4 (or, kbx = 1, 8) partial accumulators start at column `col`
    auto kblock = [&](int i, uint32_t col, uint32_t idesc, uint32_t b_addr, int kb, int kbx) {
      if ((i & (DL_MMAW - 1)) != mine) return;
      const int s = i % DL_STAGES;
      dl_spin(&full[s], (uint32_t)(i / DL_STAGES) & 1u);
      tc_fence_after();
      if (elect_one()) {
        const uint64_t da = DHI | (uint64_t)(((tiles_addr + s * DL_STAGE) & 0x3FFFFu) >> 4), db = DHI | (uint64_t)((b_addr & 0x3FFFFu) >> 4);
        const uint32_t d = tmem_base + col + (uint32_t)(((kb & kbx) << 2) * DL_CHAIN);
#pragma unroll
        for (int l = 0; l < 4; l++)               // K step l: +32 bytes in both operands, its own accumulator chain
          umma_bf16(d + (uint32_t)(l * DL_CHAIN), da + (uint64_t)(2 * l), db + (uint64_t)(2 * l), idesc, kb > kbx ? 1u : 0u);
        umma_commit(&empty[s]);
      }
      __syncwarp();
    };
    constexpr uint32_t ID64 = dl_idesc(64, DL_ROWS), ID128 = dl_idesc(128, DL_ROWS);
    if (lane == 0 && mine == 0) dl_mark(a.dbg, 1, 0);
    if (body) {
      {
        dl_spin(attn_full, 0);
        tc_fence_after();
        for (int kb = 0; kb < nkb_A; kb++) kblock(it++, 0, ID64, xa_addr + kb * DL_B_BYTES, kb, 1);       // 8 chains (alternating k-blocks)
        if (elect_one()) {
          dl_mark(a.dbg, 1, 1);
          umma_commit(&tmem_full[0]);
        }
      }
      __syncwarp();
      dl_arrive();                                                     // #1
      dl_wait();
      dl_arrive();                                                     // #2 (before waiting for LayerNorm 1: its broadcast needs every thread's arrival)
      {
        dl_spin(&xa_ready[0], 0);                                      // LayerNorm 1 rows are in XA
        tc_fence_after();
        if (lane == 0) dl_mark(a.dbg, 1, 2);
        for (int kb = 0; kb < nkb_d; kb++)
          for (int t = 0; t < nB; t++) kblock(it++, (uint32_t)(t * 4 * DL_CHAIN), ID128, xa_addr + kb * DL_B_BYTES, kb, 0);
        if (elect_one()) {
          dl_mark(a.dbg, 1, 3);
          umma_commit(&tmem_full[1]);
        }
        __syncwarp();
        dl_spin(hs_ready, 0);                                          // this CTA's GeLU slice is in HS (the B accumulators have been read)
        tc_fence_after();
        for (int kb = 0; kb < DL_HS_KB; kb++)
          for (int t = 0; t < nC; t++) kblock(it++, (uint32_t)(t * 4 * DL_CHAIN), ID128, hs_addr + kb * DL_B_BYTES, kb, 0);
        if (elect_one()) {
          dl_mark(a.dbg, 1, 5);
          umma_commit(&tmem_full[2]);
        }
      }
      __syncwarp();
      dl_wait();                                                       // #2
      dl_arrive();                                                     // #3
      dl_wait();
      dl_arrive();                                                     // #4
      dl_wait();                                                       // every CTA's LayerNorm-2 rows have landed in this XA
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // remote generic-proxy stores -> this CTA's tensor-core reads
    }
    if (next) {
      if (!body) dl_spin(&xa_ready[1], 0);
      tc_fence_after();
      if (lane == 0) dl_mark(a.dbg, 1, 6);
      for (int kb = 0; kb < nkb_d; kb++) {
        kblock(it++, 0, ID128, xa_addr + kb * DL_B_BYTES, kb, 0);
        kblock(it++, (uint32_t)(4 * DL_CHAIN), ID64, xa_addr + kb * DL_B_BYTES, kb, 0);
      }
      if (elect_one()) {
        dl_mark(a.dbg, 1, 7);
        umma_commit(&tmem_full[3]);
      }
    }
    __syncwarp();
  } else {
    // ================================================================== epilogues + LayerNorm (256 threads)
    const int q = warp & 3;                               // TMEM lane quarter this warp may read (warp % 4)
    const int half = (warp - 1 - DL_MMAW) >> 2;           // which 16 of the 32 rows (accumulator columns) this warp unloads
    const int te = threadIdx.x - DL_EPI0;
    const int r = te >> 3, t = te & 7;                    // LayerNorm-1 role: row r of the cluster's 32, 16-byte chunk t of every k-block
    const int lr = te >> 6, lc = te & 63;                 // LayerNorm-2 role: own row lr (cluster row 4 crank + lr), columns [8 lc, +8)
    const int row = row0 + r;
    const bool valid = row < a.B;
    const int erow0 = row0 + 16 * half;                   // first row of this warp's epilogue columns
    const uint32_t tq = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(16 * half);
    float z[64];
    const bool mk = te == 0;
    if (body) {                                           // LayerNorm parameters never change: stage them before the dependency wait
      const float* src[4] = {a.ln1w, a.ln1b, a.ln2w, a.ln2b};
#pragma unroll
      for (int i = 0; i < 4; i++) *(float2*)(ln_s + i * DL_D + 2 * te) = __ldg((const float2*)(src[i] + 2 * te));
      asm volatile("bar.sync 1, 256;" ::: "memory");     // the 256 epilogue threads only
    }
    if (mk) dl_mark(a.dbg, 2, 0);
    pdl_wait();                                           // the residual stream comes from the predecessors
    if (mk) dl_mark(a.dbg, 2, 1);
    float rs[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};   // body: this CTA's 64-feature slice of the residual row (LayerNorm 1 is column-sliced)
    if (body) {
      if (valid) {
        const float4 x0 = ldcg4(a.x32 + (size_t)row * DL_D + 64 * crank + 8 * t), x1 = ldcg4(a.x32 + (size_t)row * DL_D + 64 * crank + 8 * t + 4);
        rs[0] = x0.x; rs[1] = x0.y; rs[2] = x0.z; rs[3] = x0.w; rs[4] = x1.x; rs[5] = x1.y; rs[6] = x1.z; rs[7] = x1.w;
      }
    } else {
#pragma unroll
      for (int kb = 0; kb < 8; kb++) {
        float4 x0 = make_float4(0.f, 0.f, 0.f, 0.f), x1 = x0;
        if (valid) { x0 = ldcg4(a.x32 + (size_t)row * DL_D + 64 * kb + 8 * t); x1 = ldcg4(a.x32 + (size_t)row * DL_D + 64 * kb + 8 * t + 4); }
        float* v = z + 8 * kb;
        v[0] = x0.x; v[1] = x0.y; v[2] = x0.z; v[3] = x0.w; v[4] = x1.x; v[5] = x1.y; v[6] = x1.z; v[7] = x1.w;
      }
    }
    float acc[16];
    if (body) {
      // ---- out-projection slice
      mbar_wait(&tmem_full[0], 0);
      tc_fence_after();
      if (mk) dl_mark(a.dbg, 2, 2);
      dl_gather(tq, 4 * nkb_A < 8 ? 4 * nkb_A : 8, acc);
      // ---- out-projection slice + bias -> T[row][feature of this CTA] (fp32, in the not yet used HS buffer)
      float* T = (float*)hs_s;                            // [32][64]
      float4* stats = (float4*)(hs_s + DL_ROWS * 64 * 4); // [8 CTAs][32 rows]: (mean, M2) of the CTA's 64-feature slice of the row
      if (lane < 16) {                                    // M = 64: feature 16 q + lane sits in TMEM lane 32 q + lane
        const int fl = 16 * q + lane;
        const float bias = a.bo ? __ldg(a.bo + 64 * crank + fl) : 0.f;
#pragma unroll
        for (int rr = 0; rr < 16; rr++) T[(16 * half + rr) * 64 + fl] = acc[rr] + bias;
      }
      tc_fence_before();
      asm volatile("bar.sync 1, 256;" ::: "memory");
      if (mk) dl_mark(a.dbg, 2, 3);
      // ---- LayerNorm 1, column-sliced: this CTA normalises ITS 64 features of all 32 rows.  Row statistics: every CTA's (mean, M2) of
      // its slice goes to all 8 CTAs through distributed shared memory, the slices are merged exactly (Chan et al.); then the bf16 slice
      // goes into k-block `crank` of every CTA's XA and the fp32 slice to the CTA that owns the row in LayerNorm 2.
      float v[8];
      {
        const float4 t0 = *(const float4*)(T + r * 64 + 8 * t), t1 = *(const float4*)(T + r * 64 + 8 * t + 4);
        v[0] = t0.x + rs[0]; v[1] = t0.y + rs[1]; v[2] = t0.z + rs[2]; v[3] = t0.w + rs[3];
        v[4] = t1.x + rs[4]; v[5] = t1.y + rs[5]; v[6] = t1.z + rs[6]; v[7] = t1.w + rs[7];
      }
      float s1 = 0.f;
#pragma unroll
      for (int i = 0; i < 8; i++) s1 += v[i];
      s1 += __shfl_xor_sync(0xffffffffu, s1, 1); s1 += __shfl_xor_sync(0xffffffffu, s1, 2); s1 += __shfl_xor_sync(0xffffffffu, s1, 4);
      const float mj = s1 * (1.f / 64.f);
      float s2 = 0.f;
#pragma unroll
      for (int i = 0; i < 8; i++) { const float c = v[i] - mj; s2 += c * c; }
      s2 += __shfl_xor_sync(0xffffffffu, s2, 1); s2 += __shfl_xor_sync(0xffffffffu, s2, 2); s2 += __shfl_xor_sync(0xffffffffu, s2, 4);
      {   // lane t of the row's 8 sends the pair to CTA t
        const uint32_t off = smem_u32(stats + crank * DL_ROWS + r);
        dl_st_cluster_v4(dl_mapa(off, (uint32_t)t), make_uint4(__float_as_uint(mj), __float_as_uint(s2), 0u, 0u));
      }
      dl_arrive();                                                     // #1: slice statistics published; every CTA is done reading its attention rows
      dl_wait();
      if (mk) dl_mark(a.dbg, 2, 4);
      {
        float ms[DL_CLUSTER], qs[DL_CLUSTER], mean = 0.f;
#pragma unroll
        for (int p = 0; p < DL_CLUSTER; p++) { const float4 st = stats[p * DL_ROWS + r]; ms[p] = st.x; qs[p] = st.y; mean += st.x; }
        mean *= (1.f / DL_CLUSTER);
        float m2 = 0.f;
#pragma unroll
        for (int p = 0; p < DL_CLUSTER; p++) { const float dm = ms[p] - mean; m2 += qs[p] + 64.f * dm * dm; }
        const float rstd = rsqrtf(m2 * (1.f / DL_D) + 1e-5f);
        const float* w = ln_s + 64 * crank + 8 * t;
        const float* bb = ln_s + DL_D + 64 * crank + 8 * t;
#pragma unroll
        for (int i = 0; i < 8; i++) v[i] = (v[i] - mean) * rstd * w[i] + bb[i];
      }
      {
        // fp32 slice -> X1 of the row's LayerNorm-2 owner (CTA r / 4, its row r % 4)
        const uint32_t xoff = smem_u32(x1_s + (r & 3) * DL_D + 64 * crank + 8 * t);
        const uint32_t xo = dl_mapa(xoff, (uint32_t)(r >> 2));
        dl_st_cluster_v4(xo, make_uint4(__float_as_uint(v[0]), __float_as_uint(v[1]), __float_as_uint(v[2]), __float_as_uint(v[3])));
        dl_st_cluster_v4(xo + 16, make_uint4(__float_as_uint(v[4]), __float_as_uint(v[5]), __float_as_uint(v[6]), __float_as_uint(v[7])));
        // bf16 slice -> k-block `crank` of every CTA's XA (row r, 16-byte chunk t, swizzled)
        const uint4 packed = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
        const uint32_t off = smem_u32(xa_s) + (uint32_t)(crank * DL_B_BYTES + r * 128 + ((t ^ (r & 7)) << 4));
#pragma unroll
        for (int p = 0; p < DL_CLUSTER; p++) dl_st_cluster_v4(dl_mapa(off, (uint32_t)p), packed);
      }
      dl_arrive();                                                     // #2: the LayerNorm-1 rows (XA of all CTAs) and residual rows (X1 of the owners) are published
      dl_wait();
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // remote generic-proxy stores -> this CTA's tensor-core reads
      mbar_arrive(&xa_ready[0]);
      if (mk) dl_mark(a.dbg, 2, 5);
      // ---- FFN-up slice: + b1, tanh-GeLU, bf16 -> HS (this CTA's K slice of the FFN-down GEMM), K-major 128B-swizzled k-blocks
      mbar_wait(&tmem_full[1], 0);
      tc_fence_after();
      if (mk) dl_mark(a.dbg, 2, 6);
#pragma unroll
      for (int tt = 0; tt < nB; tt++) {
        dl_gather(tq + tt * 4 * DL_CHAIN, 4, acc);
        const int fl = 128 * tt + 32 * q + lane;          // local feature = K index of the next GEMM
        const float bias = a.b1 ? __ldg(a.b1 + fB * crank + fl) : 0.f;
        uint8_t* base = hs_s + (fl >> 6) * DL_B_BYTES + (fl & 7) * 2;
        const int ch = (fl & 63) >> 3;
#pragma unroll
        for (int rr = 0; rr < 16; rr++) {
          const int rw = 16 * half + rr;
          *(bf16*)(base + rw * 128 + ((ch ^ (rw & 7)) << 4)) = __float2bfloat16_rn(dl_gelu(acc[rr] + bias));
        }
      }
      tc_fence_before();
      dl_fence_async_smem();
      mbar_arrive(hs_ready);
      if (mk) dl_mark(a.dbg, 2, 7);
      // ---- FFN-down partial sums over this CTA's K slice -> scratch PP[crank][row][feature]
      mbar_wait(&tmem_full[2], 0);
      tc_fence_after();
      if (mk) dl_mark(a.dbg, 2, 9);
      float* pp = a.PP + (size_t)crank * a.pp_stride;
#pragma unroll
      for (int tt = 0; tt < nC; tt++) {
        dl_gather(tq + tt * 4 * DL_CHAIN, 4, acc);
        const int f = 128 * tt + 32 * q + lane;
#pragma unroll
        for (int rr = 0; rr < 16; rr++) pp[(size_t)(erow0 + rr) * DL_D + f] = acc[rr];
      }
      tc_fence_before();
      __syncwarp();
      if (mk) dl_mark(a.dbg, 2, 10);
      dl_arrive();                                                     // #3: partial sums published
      dl_wait();
      if (mk) dl_mark(a.dbg, 2, 11);
      // ---- LayerNorm 2 of the 4 rows this CTA owns: x1 + b2 + the 8 partial sums, 64 threads per row, 8 columns each
      {
        const int crow = DL_OWN * crank + lr;             // row inside the cluster
        const int grow = row0 + crow;
        const int c0 = 8 * lc;
        float v[8];
        const float4 xa0 = *(const float4*)(x1_s + lr * DL_D + c0), xa1 = *(const float4*)(x1_s + lr * DL_D + c0 + 4);
        v[0] = xa0.x; v[1] = xa0.y; v[2] = xa0.z; v[3] = xa0.w; v[4] = xa1.x; v[5] = xa1.y; v[6] = xa1.z; v[7] = xa1.w;
        if (a.b2) {
          const float4 b0 = __ldg((const float4*)(a.b2 + c0)), b1 = __ldg((const float4*)(a.b2 + c0 + 4));
          v[0] += b0.x; v[1] += b0.y; v[2] += b0.z; v[3] += b0.w; v[4] += b1.x; v[5] += b1.y; v[6] += b1.z; v[7] += b1.w;
        }
#pragma unroll
        for (int p = 0; p < DL_CLUSTER; p++) {
          const float* src = a.PP + (size_t)p * a.pp_stride + (size_t)grow * DL_D + c0;
          const float4 p0 = ldcg4(src), p1 = ldcg4(src + 4);
          v[0] += p0.x; v[1] += p0.y; v[2] += p0.z; v[3] += p0.w; v[4] += p1.x; v[5] += p1.y; v[6] += p1.z; v[7] += p1.w;
        }
        // row statistics: 64 threads = 2 warps of the row; two-pass like every LayerNorm of the path
        float* red = (float*)(tmem_holder + 4);           // 16 floats of scratch behind the barriers
        float s1 = 0.f;
#pragma unroll
        for (int i = 0; i < 8; i++) s1 += v[i];
        s1 = warp_sum(s1);
        if (lane == 0) red[(te >> 5)] = s1;
        asm volatile("bar.sync 1, 256;" ::: "memory");
        const float mean = (red[2 * lr] + red[2 * lr + 1]) * (1.f / DL_D);
        float s2 = 0.f;
#pragma unroll
        for (int i = 0; i < 8; i++) { const float c = v[i] - mean; s2 += c * c; }
        s2 = warp_sum(s2);
        if (lane == 0) red[8 + (te >> 5)] = s2;
        asm volatile("bar.sync 1, 256;" ::: "memory");
        const float rstd = rsqrtf((red[8 + 2 * lr] + red[8 + 2 * lr + 1]) * (1.f / DL_D) + 1e-5f);
        const float* w = ln_s + 2 * DL_D + c0;
        const float* bb = ln_s + 3 * DL_D + c0;
#pragma unroll
        for (int i = 0; i < 8; i++) v[i] = (v[i] - mean) * rstd * w[i] + bb[i];
        const uint4 packed = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
        if (grow < a.B) {                                 // the residual stream of the next layer: one writer per row
          float* dst = a.x32 + (size_t)grow * DL_D + c0;
          *(float4*)dst = make_float4(v[0], v[1], v[2], v[3]);
          *(float4*)(dst + 4) = make_float4(v[4], v[5], v[6], v[7]);
          if (a.xa_out) *(uint4*)(a.xa_out + (size_t)grow * DL_D + c0) = packed;
        }
        if (next) {                                       // the bf16 row chunk into the XA of all 8 CTAs (k-block lc / 8, chunk lc % 8, swizzled)
          const uint32_t off = smem_u32(xa_s) + (uint32_t)((lc >> 3) * DL_B_BYTES + crow * 128 + (((lc & 7) ^ (crow & 7)) << 4));
#pragma unroll
          for (int p = 0; p < DL_CLUSTER; p++) dl_st_cluster_v4(dl_mapa(off, (uint32_t)p), packed);
        }
      }
      if (mk) dl_mark(a.dbg, 2, 12);
      dl_arrive();                                                     // #4: the broadcast rows are published (release)
      dl_wait();
    } else if (next) {
      dl_store_xa(xa_s, z, r, t);                         // first launch of a step: the embedded rows, every CTA for itself
      dl_fence_async_smem();
      mbar_arrive(&xa_ready[1]);
    }
    if (next) {
      // ---- next layer's q|k|v slice -> fp32 [row][3 HD] (the input of the decode-attention kernel)
      mbar_wait(&tmem_full[3], 0);
      tc_fence_after();
      if (mk) dl_mark(a.dbg, 2, 13);
#pragma unroll
      for (int tt = 0; tt < nD; tt++) {
        dl_gather(tq + tt * 4 * DL_CHAIN, 4, acc);
        const bool h64 = tt == 1;
        const int f = fD * crank + (h64 ? 128 + 16 * q + lane : 32 * q + lane);
        if (!h64 || lane < 16) {
          const float bias = a.bq ? __ldg(a.bq + f) : 0.f;
#pragma unroll
          for (int rr = 0; rr < 16; rr++)
            if (erow0 + rr < a.B) a.qkv[(size_t)(erow0 + rr) * a.n3 + f] = acc[rr] + bias;
        }
      }
      tc_fence_before();
      if (mk) dl_mark(a.dbg, 2, 14);
    }
  }
  __syncthreads();
  if (warp == 1 + DL_MMAW) tmem_dealloc<DL_TMEM_COLS>(tmem_base);
}

__global__ void __launch_bounds__(DL_THREADS, 1)
decode_layer_kernel(const __grid_constant__ CUtensorMap tmAttn, const __grid_constant__ CUtensorMap tmWo,
                    const __grid_constant__ CUtensorMap tmW1, const __grid_constant__ CUtensorMap tmW2,
                    const __grid_constant__ CUtensorMap tmWq, const DecodeLayerArgs a) {
  extern __shared__ __align__(1024) uint8_t dyn_smem[];
  decode_layer_body(tmAttn, tmWo, tmW1, tmW2, tmWq, a, (int)blockIdx.x / DL_CLUSTER, dyn_smem);
}

// Dual-role launch: the first `n_fused` clusters run the fused layer step of ONE half of the streams, the other clusters are the
// persistent CTAs of the decode attention of the OTHER half (a different layer phase of the software pipeline over the two halves,
// model.cu).  The latency-bound layer step occupies 32 SMs and hardly any bandwidth; the HBM-bound attention gets the rest of the
// machine; one launch instead of two streams, so the co-residency does not depend on the scheduler.
static_assert(D3_THREADS <= DL_THREADS, "the attention role runs on the first D3_THREADS threads of the block");
__global__ void __launch_bounds__(DL_THREADS, 1)
decode_dual_kernel(const __grid_constant__ CUtensorMap tmAttn, const __grid_constant__ CUtensorMap tmWo,
                   const __grid_constant__ CUtensorMap tmW1, const __grid_constant__ CUtensorMap tmW2,
                   const __grid_constant__ CUtensorMap tmWq, const DecodeLayerArgs fa, const __grid_constant__ CUtensorMap tmK,
                   const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmR, const AttnDecodeArgs aa, int n_stages,
                   int b0, int n_fused) {
  extern __shared__ __align__(1024) uint8_t dyn_smem[];
  const int cluster = (int)blockIdx.x / DL_CLUSTER;
  if (cluster < n_fused) {
    decode_layer_body(tmAttn, tmWo, tmW1, tmW2, tmWq, fa, cluster, dyn_smem);
  } else if (threadIdx.x < D3_THREADS) {
    attn_decode3_body<D3_TEAMS>(tmK, tmV, tmR, aa, n_stages, b0, (int)blockIdx.x - n_fused * DL_CLUSTER,
                                (int)gridDim.x - n_fused * DL_CLUSTER, dyn_smem);
  }
}

}  // namespace

bool decode_layer_supported(int d, int HD, int di, int n3) {
  // the C2 geometry class: d_model 512, K of the out-projection a multiple of 64 (at most 8 k-blocks: XA holds the attention rows),
  // d_inner 2048 (256 FFN-up features = 4 k-blocks per CTA), 3 HD = 1536 (128 + 64 q|k|v features per CTA); others: unfused launches
  return d == DL_D && HD % 64 == 0 && HD >= 64 && HD <= DL_D && di == DL_CLUSTER * 64 * DL_HS_KB && n3 == DL_CLUSTER * 192;
}

int decode_layer(const TensorMap2D* tmAttn, const TensorMap2D* tmWo, const TensorMap2D* tmW1, const TensorMap2D* tmW2,
                 const TensorMap2D* tmWq, const DecodeLayerArgs& a, cudaStream_t st) {
  DMG_CHECK(decode_layer_supported(a.d, a.HD, a.di, a.n3), "decode_layer: geometry d=%d HD=%d di=%d n3=%d not supported", a.d, a.HD, a.di, a.n3);
  static bool configured = false;
  if (!configured) {
    DMG_CUDA_OK(cudaFuncSetAttribute(decode_layer_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, DL_SMEM));
    configured = true;
  }
  const int clusters = (a.B - a.row_base + DL_ROWS - 1) / DL_ROWS;
  if (clusters <= 0) return 0;
  return launch_k(decode_layer_kernel, dim3(clusters * DL_CLUSTER), dim3(DL_THREADS), (size_t)DL_SMEM, st, DL_CLUSTER,
                  *(const CUtensorMap*)tmAttn->bytes, *(const CUtensorMap*)tmWo->bytes, *(const CUtensorMap*)tmW1->bytes,
                  *(const CUtensorMap*)tmW2->bytes, *(const CUtensorMap*)tmWq->bytes, a);
}


bool decode_dual_supported(int M) { return attn_decode3_supported(64, M); }
int decode_dual_max_items(int attn_clusters) { return attn_clusters * DL_CLUSTER * D3_CAP; }   // (stream, head) items of the attention role

int decode_dual_max_clusters() {
  static int cached = -1;
  if (cached >= 0) return cached;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(DL_CLUSTER * 32); cfg.blockDim = dim3(DL_THREADS); cfg.dynamicSmemBytes = 227 * 1024;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = DL_CLUSTER; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  int n = 0;
  if (cudaFuncSetAttribute(decode_dual_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess ||
      cudaOccupancyMaxActiveClusters(&n, decode_dual_kernel, &cfg) != cudaSuccess) {
    cudaGetLastError();
    n = 0;
  }
  cached = n;
  return cached;
}

// fa: the fused layer step over rows [fa.row_base, fa.B); aa / b0: the decode attention of the other half (chunk-local pointers, ring
// offset b0), on `attn_clusters` clusters of 8 persistent CTAs
int decode_dual(const TensorMap2D* tmAttn, const TensorMap2D* tmWo, const TensorMap2D* tmW1, const TensorMap2D* tmW2, const TensorMap2D* tmWq,
                const DecodeLayerArgs& fa, const TensorMap2D* tmK, const TensorMap2D* tmV, const TensorMap2D* tmR, const AttnDecodeArgs& aa,
                int b0, int attn_clusters, cudaStream_t st) {
  DMG_CHECK(decode_layer_supported(fa.d, fa.HD, fa.di, fa.n3) && decode_dual_supported(aa.M), "decode_dual: geometry not supported");
  DMG_CHECK(aa.Dcap >= aa.M + 1, "decode_dual: rel-pos cache too small (%d < %d)", aa.Dcap, aa.M + 1);
  DMG_CHECK((long long)aa.B * aa.H <= decode_dual_max_items(attn_clusters), "decode_dual: %d x %d items do not fit %d attention clusters",
            aa.B, aa.H, attn_clusters);
  const int ns = d3_pick_stages(aa.M);
  const D3Layout L = d3_layout(aa.M, ns);
  const int smem = L.total > DL_SMEM ? L.total : DL_SMEM;
  static int configured = 0;
  if (configured < smem) {
    DMG_CUDA_OK(cudaFuncSetAttribute(decode_dual_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    configured = smem;
  }
  const int n_fused = (fa.B - fa.row_base + DL_ROWS - 1) / DL_ROWS;
  DMG_CHECK(n_fused >= 1 && attn_clusters >= 1, "decode_dual: empty role");
  return launch_k(decode_dual_kernel, dim3((n_fused + attn_clusters) * DL_CLUSTER), dim3(DL_THREADS), (size_t)smem, st, DL_CLUSTER,
                  *(const CUtensorMap*)tmAttn->bytes, *(const CUtensorMap*)tmWo->bytes, *(const CUtensorMap*)tmW1->bytes,
                  *(const CUtensorMap*)tmW2->bytes, *(const CUtensorMap*)tmWq->bytes, fa, *(const CUtensorMap*)tmK->bytes,
                  *(const CUtensorMap*)tmV->bytes, *(const CUtensorMap*)tmR->bytes, aa, ns, b0, n_fused);
}

}  // namespace dmg
