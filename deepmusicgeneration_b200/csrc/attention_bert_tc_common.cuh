// The roles around the softmax warps of the tcgen05 attention kernel of the masked-BERT remix encoder (attention_bert_tc.cu): the operand
// tiles in shared memory, the TMEM columns, the mbarriers, the TMA producer, the q-transform warps and the MMA issuer.  Replaces MemMultiHeadRelativeAttentionKV._apply_attention (deep_music_remix.py:2078-2104); the scheme is described at the
// top of attention_bert_tc.cu.
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include "kernels.cuh"
#include "launch.cuh"
#include "mma_sync.cuh"
#include "train_kernels.cuh"

namespace dmg {
namespace bert_tc {

constexpr float BT_LOG2E = 1.4426950408889634f;
constexpr int BT16K = 128 * 64 * 2;
constexpr int BO_QU = 0;
constexpr int BO_QV = BO_QU + BT16K;
constexpr int BO_QVN = BO_QV + BT16K;
constexpr int BO_K = BO_QVN + BT16K;                   // one stage
constexpr int BO_V = BO_K + BT16K;
constexpr int BO_R = BO_V + BT16K;                     // 2 slots (slot = load index & 1): per item the raw q and q_next tiles, then the position-key blocks
constexpr int BO_P = BO_R + 2 * BT16K;                 // 2 key halves
constexpr int BO_STRIP = BO_P + 2 * BT16K;             // the kernels' own strip lines, exchange buffers and barriers follow

enum { Q_QFULL = 0, Q_QREADY, Q_KFULL, Q_KEMPTY, Q_RFULL0, Q_RFULL1, Q_REMPTY0, Q_REMPTY1, Q_VFULL, Q_VEMPTY, Q_SFULL, Q_SFREE,
       Q_PFULL0, Q_PFULL1, Q_OFULL0, Q_OFULL1, Q_OFREE0, Q_OFREE1, Q_VFULL1, Q_VEMPTY1, Q_COUNT };
constexpr uint32_t BTM_AC = 0, BTM_STRIP = 128, BTM_O = 384;
constexpr int BT_LINE16 = 208;                         // bytes of an fp16 strip line: 96 halves + 16 (16-byte stores of 8 lanes hit 8 bank groups)
constexpr int BO_V2 = BO_STRIP + 256 * BT_LINE16;      // second V stage of the fp16-strip kernel: the 16 KB its lines leave of the fp32 lines' space

__device__ __forceinline__ uint64_t bt_desc_k(uint32_t addr) {          // K-major, 128B swizzle: rows of 128 B, 8-row groups 1024 B apart
  return (uint64_t)((addr & 0x3FFFFu) >> 4) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
__device__ __forceinline__ uint64_t bt_desc_mn(uint32_t addr) {         // MN-major: LBO 8192, SBO 1024
  return (uint64_t)((addr & 0x3FFFFu) >> 4) | ((uint64_t)(8192u >> 4) << 16) | ((uint64_t)(1024u >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
__device__ __forceinline__ void bt_fence_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ uint32_t bt_f16x2_sat(float lo, float hi) {
  uint32_t w;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(w) : "f"(hi), "f"(lo));
  return w;
}

struct BertTcArgs {
  const float* u; const float* v;   // [H*64]
  bf16* out;                        // [B*T, H*64]
  int B, T, H, Dcap;
  float scale;
  unsigned long long* dbg;          // measurement only (DMG_BERT_TC_TIMELINE): %globaltimer marks of CTA 0, nullptr in the product path
  // per-sequence lengths (the VARLEN kernels): T is the padded length (row stride of a sequence), sequence b has lens[b] >= 128 tokens,
  // items[0, n_items) lists the work items as (b << 16) | (h << 8) | query tile
  const int* lens;
  const int* items;
  int n_items;
};
// timeline slots: softmax warp 0 / 4 at [256 hf + 48 item + 5 tile + mark], issuer at [512 + 48 item + 6 tile + mark], transform warps at
// [768 + 4 item + mark], producer at [832 + 4 item + mark]; the first four items of CTA 0
__device__ __forceinline__ void bt_mark(unsigned long long* dbg, int slot, int item) {
  if (dbg == nullptr || blockIdx.x != 0 || item >= 4) return;
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  dbg[slot] = t;
}

// mbarrier arrival counts: soft_warps = number of softmax warps (half of them per key half)
__device__ __forceinline__ void bt_init_barriers(uint64_t* bar, int soft_warps) {
  for (int i = 0; i < Q_COUNT; i++) {
    uint32_t cnt = 1;
    if (i == Q_SFREE) cnt = soft_warps;
    if (i == Q_PFULL0 || i == Q_PFULL1 || i == Q_OFREE0 || i == Q_OFREE1) cnt = soft_warps / 2;
    mbar_init(&bar[i], cnt);
  }
  mbar_fence_init();
}

// bounded wait without the printf of mbar_wait (its argument buffer and call cost the 64-register one-lane roles a dozen spills): a
// protocol bug still traps (-> CUDA error on the host) instead of hanging the GPU box
__device__ __forceinline__ void bt_wait(uint64_t* bar, uint32_t parity) {
  uint32_t n = 0;
  while (!mbar_try_wait(bar, parity))
    if (++n > (1u << 26)) __trap();
}

// Work decomposition of the persistent kernel: item = (stream, head, query tile), items are dealt round-robin over the CTAs
// (item = blockIdx.x + k * gridDim.x: CTAs that run side by side work on neighbouring query tiles of one (stream, head) and share
// its K / V / position-key tiles in L2).  Every mbarrier keeps counting across items: a role derives the phase parity from the
// number of uses so far (g = k * NT + n for the per-tile barriers, k * (NT + 3) + j for the loads into the two position-key slots:
// j = 0, 1 are the item's raw q and q_next tiles, j = 2 + m is position-key load m).
//
// Item boundary: the slots are released when the last S MMA of an item completes, one tile time before the softmax warps are done with
// the item.  In that time the producer brings the next item's q / q_next into the slots, the two transform warps turn them into the
// q + u / q + v / q_next + v operand tiles (free: every MMA that read them has completed) and release the slots, the first two
// position-key blocks follow, and the issuer runs S(0) of the next item right behind the last P V of this one - the softmax warps
// find their first scores waiting when they return from the item's epilogue.
struct BtItem {
  int b, h, it;
};
__device__ __forceinline__ BtItem bt_item(int item, int nT, int H) {
  const int bh = item / nT;
  return {bh / H, bh % H, item % nT};
}
// VARLEN: the item list and the sequence's own length T / tile count NT.  Every role keeps the running sums of NT and NT + 3 over the
// items it has walked (the barrier use counts g0 / r0 of the fixed-length kernel, k * NT and k * (NT + 3)).
struct BtVarItem {
  int b, h, it, T, NT;
};
__device__ __forceinline__ BtVarItem bt_var_item(const BertTcArgs& a, int item) {
  const int e = __ldg(a.items + item), b = e >> 16, T = __ldg(a.lens + b);
  return {b, (e >> 8) & 255, e & 255, T, (T + 127) / 128};
}

// TMA producer (one thread): per item q / q_next, then per key tile K, the position-key blocks and V
template <int VS, bool VARLEN>
__device__ __forceinline__ void bt_producer(uint8_t* smem, uint64_t* bar, const CUtensorMap& tmX, const CUtensorMap& tmR, const BertTcArgs& a,
                                            int NT_all, int n_items) {
  const int HD = a.H * 64;
  pdl_wait();                                  // q | k | v come from the predecessor kernel (the QKV GEMM)
  int k = 0, gsum = 0, rsum = 0;
  for (int item = blockIdx.x; item < n_items; item += gridDim.x, k++) {
    int b, h, it, T, NT;
    if constexpr (VARLEN) {
      const BtVarItem w = bt_var_item(a, item);
      b = w.b; h = w.h; it = w.it; T = w.T; NT = w.NT;
    } else {
      const BtItem w = bt_item(item, NT_all, a.H);
      b = w.b; h = w.h; it = w.it; T = a.T; NT = NT_all;
    }
    const int i0 = it * 128;
    const int g0 = VARLEN ? gsum : k * NT, r0 = VARLEN ? rsum : k * (NT + 3);  // tiles / slot loads of the earlier items
    if constexpr (VARLEN) { gsum += NT; rsum += NT + 3; }
    auto slot_wait = [&](int j) {               // the slot of load j of this item, once its previous tenant has been released
      const int gl = r0 + j, s = gl & 1;
      bt_wait(&bar[Q_REMPTY0 + s], ((gl >> 1) & 1) ^ 1);
      return s;
    };
    auto load_k = [&](int n) {
      const int g = g0 + n;
      bt_wait(&bar[Q_KEMPTY], (g & 1) ^ 1);
      mbar_expect_tx(&bar[Q_KFULL], BT16K);
      tma_load_2d(smem + BO_K, &tmX, HD + h * 64, b * a.T + n * 128, &bar[Q_KFULL]);
    };
    auto load_r = [&](int j) {                  // load 0 = upper block of tile 0; load j >= 1 = lower block of tile j-1
      // line 1: Rk rows (it-j)*128 ...; line 3: Rk rows T + 1 + (it-j)*128 ... (distance T + 1 + i - j; rows below 0 or past T - 1
      // only meet masked keys or the zero pad)
      const int row = j <= it ? (it - j) * 128 : T + 1 + (it - j) * 128;
      const int s = slot_wait(2 + j);
      mbar_expect_tx(&bar[Q_RFULL0 + s], BT16K);
      tma_load_2d(smem + BO_R + s * BT16K, &tmR, 0, h * a.Dcap + row, &bar[Q_RFULL0 + s]);
    };
    auto load_v = [&](int n) {                  // VS stages: stage g % VS, its use g / VS
      const int g = g0 + n, vs = g % VS, vu = g / VS;
      uint64_t* full = &bar[vs ? Q_VFULL1 : Q_VFULL];
      bt_wait(&bar[vs ? Q_VEMPTY1 : Q_VEMPTY], (vu & 1) ^ 1);
      mbar_expect_tx(full, BT16K);
      tma_load_2d(smem + (vs ? BO_V2 : BO_V), &tmX, 2 * HD + h * 64, b * a.T + n * 128, full);
    };
    {   // the raw q tiles complete on their own barrier (one phase per item): a waiter on RFULL that skips the position-key phases in
        // between would find the parity of an older phase and walk through
      const int s0 = slot_wait(0), s1 = slot_wait(1);
      bt_mark(a.dbg, 832 + 4 * k, k);
      mbar_expect_tx(&bar[Q_QFULL], 2 * BT16K);
      tma_load_2d(smem + BO_R + s0 * BT16K, &tmX, h * 64, b * a.T + i0, &bar[Q_QFULL]);
      tma_load_2d(smem + BO_R + s1 * BT16K, &tmX, h * 64, b * a.T + i0 + 1, &bar[Q_QFULL]);   // rows i+1 (the last row of the last tile is never used)
    }
    load_k(0);
    load_r(0);
    load_r(1);
    bt_mark(a.dbg, 832 + 4 * k + 1, k);
    load_v(0);
    bt_mark(a.dbg, 832 + 4 * k + 2, k);
    // One V stage: the request for V(n) can only go out when P V(n-1) has retired, and P V(n) cannot be issued before it lands - the
    // kernel then runs at one TMA latency + one P V per tile (2.05 us measured, profiles/r2h_attn_bert_tc_timeline_single_v.txt),
    // and the requests trail the K / R requests by one tile so that they do not hold those back as well (70.8 -> 64.5 ms per C4
    // forward).  Two stages: V(n) waits for P V(n-2), a whole tile before it is needed.
    for (int n = 1; n < NT; n++) {
      load_k(n);
      load_r(n + 1);
      if (VS == 2) load_v(n);
      else if (n >= 2) load_v(n - 1);
    }
    if (VS == 1 && NT >= 2) load_v(NT - 1);
  }
}

// Transform warps (64 threads): the item's raw q / q_next tiles (position-key slots) -> q + u, q + v and q_next + v in the canonical
// swizzled layout.  Eight consecutive threads take the eight 16-byte chunks of one row (128 contiguous bytes: no bank conflicts); a
// thread's rows are 8 apart, so its physical chunk maps to the same logical columns in all of them and it needs one 8-wide slice of
// u and v only (requested before the wait for q).
template <bool VARLEN>
__device__ __forceinline__ void bt_transform(uint8_t* smem, uint64_t* bar, const BertTcArgs& a, int NT_all, int n_items, int tid) {
  const int pc = tid & 7, rb = tid >> 3;
  const int col = 8 * (pc ^ rb);
  int k = 0, rsum = 0;
  for (int item = blockIdx.x; item < n_items; item += gridDim.x, k++) {
    int h, NT;
    if constexpr (VARLEN) {
      const BtVarItem w = bt_var_item(a, item);
      h = w.h; NT = w.NT;
    } else {
      h = (item / NT_all) % a.H; NT = NT_all;
    }
    const float4 ua = __ldg((const float4*)(a.u + h * 64 + col)), ub = __ldg((const float4*)(a.u + h * 64 + col + 4));
    const float4 va = __ldg((const float4*)(a.v + h * 64 + col)), vb = __ldg((const float4*)(a.v + h * 64 + col + 4));
    const float uu[8] = {ua.x, ua.y, ua.z, ua.w, ub.x, ub.y, ub.z, ub.w}, vv8[8] = {va.x, va.y, va.z, va.w, vb.x, vb.y, vb.z, vb.w};
    const int g0 = VARLEN ? rsum : k * (NT + 3), g1 = g0 + 1;
    if constexpr (VARLEN) rsum += NT + 3;
    // the slots were released by the last S MMA of the previous item: nothing reads the three operand tiles any more
    bt_wait(&bar[Q_QFULL], k & 1);
    if (tid == 0) bt_mark(a.dbg, 768 + 4 * k, k);
    const uint8_t* q_raw = smem + BO_R + (g0 & 1) * BT16K;
    const uint8_t* qn_raw = smem + BO_R + (g1 & 1) * BT16K;
#pragma unroll 4
    for (int i = 0; i < 16; i++) {
      const int qr = rb + 8 * i;
      const uint32_t off = (uint32_t)((qr >> 3) * 1024 + (qr & 7) * 128 + pc * 16);
      const uint4 raw = *(const uint4*)(q_raw + off);
      const uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
      uint32_t ou[4], ov[4];
#pragma unroll
      for (int e = 0; e < 4; e++) {
        const float u0 = uu[2 * e], u1 = uu[2 * e + 1], v0 = vv8[2 * e], v1 = vv8[2 * e + 1];
        ou[e] = pack_bf16x2(bf16lo(w[e]) + u0, bf16hi(w[e]) + u1);
        ov[e] = pack_bf16x2(bf16lo(w[e]) + v0, bf16hi(w[e]) + v1);
      }
      *(uint4*)(smem + BO_QU + off) = make_uint4(ou[0], ou[1], ou[2], ou[3]);
      *(uint4*)(smem + BO_QV + off) = make_uint4(ov[0], ov[1], ov[2], ov[3]);
      // row qr of q + v is row qr - 1 of q_next + v: same logical chunk, the swizzle of the row above
      if (qr > 0) {
        const int pr = qr - 1;
        *(uint4*)(smem + BO_QVN + (pr >> 3) * 1024 + (pr & 7) * 128 + ((pc ^ (qr & 7) ^ (pr & 7)) << 4)) = make_uint4(ov[0], ov[1], ov[2], ov[3]);
      }
    }
    if (rb == 7) {                             // the last row of q_next + v is the only one the raw q_next tile is needed for
      const uint32_t off = (uint32_t)(15 * 1024 + 7 * 128 + pc * 16);
      const uint4 rawn = *(const uint4*)(qn_raw + off);
      const uint32_t wn[4] = {rawn.x, rawn.y, rawn.z, rawn.w};
      uint32_t on[4];
#pragma unroll
      for (int e = 0; e < 4; e++) on[e] = pack_bf16x2(bf16lo(wn[e]) + vv8[2 * e], bf16hi(wn[e]) + vv8[2 * e + 1]);
      *(uint4*)(smem + BO_QVN + off) = make_uint4(on[0], on[1], on[2], on[3]);
    }
    bt_fence_async();
    asm volatile("bar.sync 2, 64;" ::: "memory");   // the two transform warps
    if (tid == 0) {
      bt_mark(a.dbg, 768 + 4 * k + 1, k);
      mbar_arrive(&bar[Q_REMPTY0]);            // the raw tiles are consumed: the slots go back to the producer
      mbar_arrive(&bar[Q_REMPTY1]);
      mbar_arrive(&bar[Q_QREADY]);
    }
  }
}

// MMA issuer: S(n) = AC | strip, then P V of the previous tile.  Executed by the WHOLE warp in uniform control flow (waits by all
// lanes, tcgen05.mma / commit by the elected lane): descriptors and barrier addresses stay in uniform registers.  As the body of an
// `if (lane == 0)` branch the same loop cost ~400 instructions per tile (per MMA a vector-to-uniform move loop, elect, predicate
// shuffles, descriptor rebuild) = 2 us of one thread's time - and THAT was the tile period of the kernel, with the tensor pipe
// 24 % busy and the softmax warps waiting for scores (profiles/r2h_attn_bert_tc_timeline_single_v.txt).
template <int VS, bool VARLEN>
__device__ __forceinline__ void bt_mma_issuer(uint8_t* smem, uint64_t* bar, uint32_t tmem_base, int NT_all, int n_items, const BertTcArgs& a,
                                              unsigned long long* dbg) {
  constexpr uint32_t idesc_s = (1u << 4) | (1u << 7) | (1u << 10) | ((128u >> 3) << 17) | ((128u >> 4) << 24);
  constexpr uint32_t idesc_pv = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 16) | ((64u >> 3) << 17) | ((128u >> 4) << 24);
  // descriptors of the operand tiles; a 16-element K step is +32 bytes (K-major) / +2048 bytes (MN-major V) in the address field
  const uint64_t d_qu = bt_desc_k(smem_u32(smem + BO_QU)), d_qv = bt_desc_k(smem_u32(smem + BO_QV)), d_qvn = bt_desc_k(smem_u32(smem + BO_QVN)),
                 d_k = bt_desc_k(smem_u32(smem + BO_K)), d_r0 = bt_desc_k(smem_u32(smem + BO_R)), d_r1 = bt_desc_k(smem_u32(smem + BO_R + BT16K)),
                 d_p0 = bt_desc_k(smem_u32(smem + BO_P)), d_p1 = bt_desc_k(smem_u32(smem + BO_P + BT16K)),
                 d_v0 = bt_desc_mn(smem_u32(smem + BO_V)), d_v1 = bt_desc_mn(smem_u32(smem + (VS == 2 ? BO_V2 : BO_V)));
  // g: tile count over all items of this CTA; ms, k: timeline slot / item; vzero (VARLEN): V rows from vzero on lie past the sequence end
  // and are zeroed before the MMA reads them (the probabilities there are 0, but 0 * NaN is not)
  auto issue_pv = [&](int g, int ms, int k, int vzero) {
    const int vs = g % VS, vu = g / VS;
    bt_wait(&bar[vs ? Q_VFULL1 : Q_VFULL], vu & 1);
    if (VARLEN && vzero < 128) {
      uint8_t* vt = smem + (vs ? BO_V2 : BO_V);
      for (int c = vzero * 8 + (int)(threadIdx.x & 31); c < 128 * 8; c += 32) *(uint4*)(vt + 16 * c) = make_uint4(0u, 0u, 0u, 0u);
      bt_fence_async();
      __syncwarp();
    }
#pragma unroll
    for (int hf = 0; hf < 2; hf++) {
      bt_wait(&bar[Q_PFULL0 + hf], g & 1);
      if (g > 0) bt_wait(&bar[Q_OFREE0 + hf], (g - 1) & 1);
      tc_fence_after();
      if (elect_one()) {
        const uint64_t dp = hf ? d_p1 : d_p0, dv = (vs ? d_v1 : d_v0) + (uint64_t)(hf * (8192 >> 4));
#pragma unroll
        for (int k4 = 0; k4 < 4; k4++)
          umma_bf16(tmem_base + BTM_O + 64 * hf, dp + (uint64_t)(2 * k4), dv + (uint64_t)(128 * k4), idesc_pv, (uint32_t)(k4 > 0));
        umma_commit(&bar[Q_OFULL0 + hf]);
        if (hf == 1) {
          umma_commit(&bar[vs ? Q_VEMPTY1 : Q_VEMPTY]);
          bt_mark(dbg, ms + 4, k);
        }
      }
      __syncwarp();
    }
  };
  int k = 0, gsum = 0, rsum = 0;
  for (int item = blockIdx.x; item < n_items; item += gridDim.x, k++) {
    int it, NT, vzero = 128;
    if constexpr (VARLEN) {
      const BtVarItem w = bt_var_item(a, item);
      it = w.it; NT = w.NT; vzero = w.T - (NT - 1) * 128;
    } else {
      it = item % NT_all; NT = NT_all;
    }
    const int g0 = VARLEN ? gsum : k * NT, r0 = (VARLEN ? rsum : k * (NT + 3)) + 2;
    if constexpr (VARLEN) { gsum += NT; rsum += NT + 3; }
    bt_wait(&bar[Q_QREADY], k & 1);
    for (int n = 0; n < NT; n++) {
      const int g = g0 + n, gu = r0 + n, gl = gu + 1;                   // load gu = this tile's upper block, gl = its lower block
      bt_wait(&bar[Q_KFULL], g & 1);
      // RFULL counts position-key loads only: every earlier item and this one put one raw q tile into each slot
      bt_wait(&bar[Q_RFULL0 + (gu & 1)], ((gu >> 1) - (k + 1)) & 1);
      bt_wait(&bar[Q_RFULL0 + (gl & 1)], ((gl >> 1) - (k + 1)) & 1);
      if (g > 0) bt_wait(&bar[Q_SFREE], (g - 1) & 1);
      tc_fence_after();
      if (elect_one()) {
        const uint64_t ru = (gu & 1) ? d_r1 : d_r0, rl = (gl & 1) ? d_r1 : d_r0;
        const uint64_t au = n <= it ? d_qv : d_qvn, al = (n + 1) <= it ? d_qv : d_qvn;   // line 1 below / on the diagonal, line 3 above
        // (separate ready / free barriers for AC and the strip - AC(n+1) issued right after the AC reads of tile n - were measured
        // slower: 68.4 vs 64.4 ms per C4 forward; the extra arrive sits in the softmax warps' critical path)
#pragma unroll
        for (int k4 = 0; k4 < 4; k4++) umma_bf16(tmem_base + BTM_AC, d_qu + (uint64_t)(2 * k4), d_k + (uint64_t)(2 * k4), idesc_s, (uint32_t)(k4 > 0));
#pragma unroll
        for (int k4 = 0; k4 < 4; k4++) umma_bf16(tmem_base + BTM_STRIP, al + (uint64_t)(2 * k4), rl + (uint64_t)(2 * k4), idesc_s, (uint32_t)(k4 > 0));
#pragma unroll
        for (int k4 = 0; k4 < 4; k4++)
          umma_bf16(tmem_base + BTM_STRIP + 128, au + (uint64_t)(2 * k4), ru + (uint64_t)(2 * k4), idesc_s, (uint32_t)(k4 > 0));
        umma_commit(&bar[Q_SFULL]);
        umma_commit(&bar[Q_KEMPTY]);
        umma_commit(&bar[Q_REMPTY0 + (gu & 1)]);   // the upper block is dead after this tile; the lower one serves the next
        if (n == NT - 1) umma_commit(&bar[Q_REMPTY0 + (gl & 1)]);   // ... or nobody: the next item starts with two fresh blocks
        bt_mark(dbg, 512 + 48 * k + 6 * n, k);
      }
      __syncwarp();
      if (n > 0) issue_pv(g - 1, 512 + 48 * k + 6 * (n - 1), k, 128);
    }
    issue_pv(g0 + NT - 1, 512 + 48 * k + 6 * (NT - 1), k, vzero);
  }
}

}  // namespace bert_tc
}  // namespace dmg
