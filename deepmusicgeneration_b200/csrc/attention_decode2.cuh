// Second-generation decode attention (x_len == 1, bf16 ring): persistent, warp-specialised, tensor-core dot products.
//
// Why (profiles/r1a_attn_decode_v1_ncu_full.csv): the first kernel moved the right bytes (270.6 MB DRAM per launch
// vs 271.3 MB algorithmic) but reached only 67 % of the measured HBM peak: 2048 short-lived CTAs, 12 warps/SM,
// 27.8 M warp instructions per launch (FFMA dot products + shuffles + bf16 unpacks), stalls split between mbarrier
// waits, __syncthreads and dependent-issue waits.
//
// This kernel:
//  * one persistent CTA per SM; CTA c owns a contiguous range of the B*H (stream, head) items in head-major order,
//    so the relative-position keys Rd[head] (M+1 rows, 64 KB) stay RESIDENT in shared memory (reloaded only when
//    the head changes, at most once per CTA) instead of being re-fetched from L2 for every stream;
//  * a producer warp streams 64-key K tiles then V tiles (8 KB, 2-D TMA, 128B swizzle) through an N-stage ring of
//    full/empty mbarriers, running up to one whole item ahead of the consumers, plus the new token's q/k/v rows
//    (3 x 256 B bulk copies): the consumers never issue a global load;
//  * four consumer warps do the math with mma.sync.m16n8k16 (bf16 in, fp32 accumulate): scores = K.(q+u) + Rd.(q+v)
//    with the key tile as the A operand (ldmatrix from the swizzled tile, Rd rows addressed per key by distance =
//    rel_shift by index arithmetic) and the query replicated over the 8 B columns, so every key's score lands
//    replicated in its quad without a shuffle; exact two-pass softmax over the M+1 scores in shared memory;
//    out = V^T.p with V^T fragments from ldmatrix.trans and each warp owning 16 of the 64 output dims;
//  * ~10x fewer issued instructions than v1; the CTA appends the new token's K/V to the ring slot it has finished with.
#pragma once
#include <cuda.h>
#include <cstdlib>
#include "kernels.cuh"
#include "launch.cuh"

namespace dmg {

constexpr int D2_ROWS = 64;      // keys per consumer group per tile
constexpr float D2_LOG2E = 1.4426950408889634f;

// G consumer groups of 4 warps; a tile holds 64*G keys (8 KB * G); NS (power of two) tiles in flight.
struct D2Layout {
  int r_boxes, n_stages, tile_bytes;
  int off_r, off_stage, off_q, off_sc, off_pw, off_red, off_bar, total;
};

__host__ __device__ inline D2Layout d2_layout(int M, int G, int n_stages) {
  D2Layout L;
  L.r_boxes = (M + 1 + 63) / 64;
  L.n_stages = n_stages;
  L.tile_bytes = G * 8192;
  L.off_r = 0;
  L.off_stage = L.off_r + L.r_boxes * 8192;
  L.off_q = L.off_stage + n_stages * L.tile_bytes;
  L.off_sc = L.off_q + 2 * 768;
  L.off_pw = L.off_sc + 2 * (M + 8) * 4;
  L.off_red = (L.off_pw + (M + 16) * 2 + 15) & ~15;        // [G][64] partial outputs + [4G] partial sums
  L.off_bar = L.off_red + G * 64 * 4 + 4 * G * 4 + 16;
  L.total = L.off_bar + (2 * n_stages + 6) * 8 + 1024 /*alignment slack*/;
  return L;
}

static inline int d2_pick_stages(int M, int G) {
  for (int s = 16; s >= 2; s >>= 1)
    if (d2_layout(M, G, s).total <= 227 * 1024) return s;
  return 0;
}
static inline int d2_pick_groups(int M) {
  static const int want = getenv("DMG_DECODE_GROUPS") ? atoi(getenv("DMG_DECODE_GROUPS")) : 2;   // timing experiments; read once
  for (int G = want; G >= 1; G >>= 1)
    if ((G == 1 || G == 2 || G == 4) && M % (64 * G) == 0 && d2_pick_stages(M, G) >= 2) return G;
  return 0;
}

__device__ __forceinline__ void ldmatrix_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void mma_bf16_16816(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3,
                                               uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

#ifdef D2_PROFILE   // scripts/probes/probe_attn_decode.cu: cycles consumer warp 0 spends waiting, per CTA [total, q, K tiles, V tiles, barriers, items]
__device__ unsigned long long* d2_prof_ptr;
#define D2_MARK(k) do { if (warp == 0 && lane == 0) { const long long _n = clock64(); sec[k] += _n - t_last; t_last = _n; } } while (0)
#define D2_T0() const long long _t0 = clock64()
#define D2_ACC(k) do { if (warp == 0 && lane == 0) prof[k] += clock64() - _t0; } while (0)
#else
#define D2_MARK(k) do {} while (0)
#define D2_T0() do {} while (0)
#define D2_ACC(k) do {} while (0)
#endif

// {pos_total, mem_count} of the stream of (stream, head) item `it` (head-major: stream b0 + it mod B): the streams of a batch may hold
// memories of different lengths.  The producer fetches it one item ahead and stores it beside the item's q slot before the arrive that
// releases the slot, so the consumers read it from shared memory.
__device__ __forceinline__ int2 item_ring_state(const AttnDecodeArgs& a, int b0, int it) {
  return *(const int2*)(a.state + a.state_stride * (b0 + it % a.B));
}

// The kernel body as a device function: `cta` of `ncta` persistent CTAs (the stand-alone kernel passes blockIdx.x / gridDim.x; the
// dual-role decode kernel of decode_layer.cu gives it the CTAs that are not busy with the fused layer step of the other half of the
// streams).  Runs on the first (4 G + 1) * 32 threads of the block; `d2_smem` is the block's dynamic shared memory.
template <int G>
__device__ __forceinline__ void attn_decode2_body(const CUtensorMap& tmK, const CUtensorMap& tmV, const CUtensorMap& tmR, const AttnDecodeArgs& a,
                                                  int n_stages, int b0, int cta, int ncta, uint8_t* d2_smem) {
  constexpr int NW = 4 * G;                 // consumer warps
  constexpr int TR = D2_ROWS * G;           // keys per tile
  uint8_t* base = d2_smem + ((1024u - (smem_u32(d2_smem) & 1023u)) & 1023u);   // keeps the shared address space
  const int M = a.M, H = a.H, B = a.B, HD = H * 64;
  const D2Layout L = d2_layout(M, G, n_stages);
  uint8_t* Rres = base + L.off_r;
  uint8_t* stages = base + L.off_stage;
  float* qbuf = (float*)(base + L.off_q);
  float* sc = (float*)(base + L.off_sc);
  bf16* pw = (bf16*)(base + L.off_pw);
  float* ored = (float*)(base + L.off_red);     // [G][64]
  float* psum = ored + G * 64;                  // [NW]
  uint64_t* full = (uint64_t*)(base + L.off_bar);
  uint64_t* empty = full + n_stages;
  uint64_t* q_full = empty + n_stages;    // [2]
  uint64_t* q_empty = q_full + 2;         // [2]
  uint64_t* r_full = q_empty + 2;
  uint64_t* r_free = r_full + 1;
  int2* qstate = (int2*)(psum + NW);      // [2] ring state of the item in q slot 0 / 1

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int nT = M / TR;                  // K tiles (= V tiles) per item
  pdl_launch_dependents();
  const long long NI = (long long)B * H;
  const int lo = (int)(NI * cta / ncta), hi = (int)(NI * (cta + 1) / ncta);
  const uint32_t smask = (uint32_t)n_stages - 1;
  int sshift = 0;
  while ((1 << sshift) < n_stages) sshift++;

  if (tid == 0) {
    for (int s = 0; s < n_stages; s++) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], NW);
    }
    for (int s = 0; s < 2; s++) {
      mbar_init(&q_full[s], 1);
      mbar_init(&q_empty[s], NW);
    }
    mbar_init(r_full, 1);
    mbar_init(r_free, NW);
    mbar_fence_init();
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmV);
    tma_prefetch_desc(&tmR);
  }
  named_bar_sync(4, (NW + 1) * 32);           // the threads of this role only

  if (warp == NW) {
    // ============================== producer: every byte arrives through the TMA engine ==============================
    if (lane == 0) {
      int cur_h = -1;
      uint32_t tile_cnt = 0;
      if (lo < hi) {   // the rel-pos keys derive from weights only: fetch them while the predecessor kernel drains
        cur_h = lo / B;
        mbar_expect_tx(r_full, (uint32_t)(L.r_boxes * 8192));
        for (int bx = 0; bx < L.r_boxes; bx++) tma_load_2d(Rres + bx * 8192, &tmR, 0, cur_h * a.Dcap + bx * 64, r_full);
      }
      // The K/V ring of this layer was last written by this layer's attention kernel of the PREVIOUS step (116 launches
      // back: long retired - at most a handful of kernels of the chain can be resident at once), so the first item's tiles
      // do not depend on the predecessor kernel either: fill the stage ring while the QKV GEMM drains (the HBM pipe is idle
      // then), and only the current token's q / k / v wait for it.
      int pre = 0;                                   // tiles of the first item already requested
      if (lo < hi && !a.no_early_kv) {
        const int h = lo / B, b = lo - h * B;
        const int row0 = ((b0 + b) * H + h) * M;
        const int npre = min(n_stages, 2 * nT);
        for (int t = 0; t < npre; ++t, ++tile_cnt, ++pre) {
          const int s = tile_cnt & smask;
          mbar_expect_tx(&full[s], (uint32_t)L.tile_bytes);
          uint8_t* dst = stages + s * L.tile_bytes;
          const CUtensorMap* tm = t < nT ? &tmK : &tmV;
          const int r0 = row0 + (t < nT ? t : t - nT) * TR;
#pragma unroll
          for (int gq = 0; gq < G; gq++) tma_load_2d(dst + gq * 8192, tm, 0, r0 + gq * 64, &full[s]);
        }
      }
      pdl_wait();
      int2 rs = lo < hi ? item_ring_state(a, b0, lo) : make_int2(0, 0);
      for (int it = lo, n = 0; it < hi; ++it, ++n) {
        const int h = it / B, b = it - h * B;
        const int qs = n & 1;
        // q slot first: it means the consumers are done with item n - 2, so r_free's phase n - 1 is the only phase of that parity
        // that can still be open.  (Waiting on r_free first, with the consumers still scoring item n - 2, the finished phase n - 3
        // has the parity of phase n - 1 and passed: the next head's Rd overwrote the keys of items n - 2 and n - 1.)
        mbar_wait(&q_empty[qs], (uint32_t)(((n >> 1) & 1) ^ 1));
        if (h != cur_h) {
          if (cur_h >= 0) mbar_wait(r_free, (uint32_t)((n - 1) & 1));   // previous item's score phase is done with Rd
          mbar_expect_tx(r_full, (uint32_t)(L.r_boxes * 8192));
          for (int bx = 0; bx < L.r_boxes; bx++) tma_load_2d(Rres + bx * 8192, &tmR, 0, h * a.Dcap + bx * 64, r_full);
          cur_h = h;
        }
        qstate[qs] = rs;                             // the item's ring state goes with its q|k|v: released by the arrive below
        if (it + 1 < hi) rs = item_ring_state(a, b0, it + 1);
        mbar_expect_tx(&q_full[qs], 768);
        const float* qrow = a.qkv + (size_t)b * 3 * HD + h * 64;
        bulk_g2s(qbuf + qs * 192, qrow, 256, &q_full[qs]);
        bulk_g2s(qbuf + qs * 192 + 64, qrow + HD, 256, &q_full[qs]);
        bulk_g2s(qbuf + qs * 192 + 128, qrow + 2 * HD, 256, &q_full[qs]);
        const int row0 = ((b0 + b) * H + h) * M;
        for (int t = (it == lo ? pre : 0); t < 2 * nT; ++t, ++tile_cnt) {
          const int s = tile_cnt & smask;
          const uint32_t ph = (tile_cnt >> sshift) & 1;
          mbar_wait(&empty[s], ph ^ 1);
          mbar_expect_tx(&full[s], (uint32_t)L.tile_bytes);
          uint8_t* dst = stages + s * L.tile_bytes;
          const CUtensorMap* tm = t < nT ? &tmK : &tmV;
          const int r0 = row0 + (t < nT ? t : t - nT) * TR;
#pragma unroll
          for (int gq = 0; gq < G; gq++) tma_load_2d(dst + gq * 8192, tm, 0, r0 + gq * 64, &full[s]);
        }
      }
    }
    return;
  }

  // ============================== consumers ==============================
#ifdef D2_PROFILE
  long long prof[6] = {0, 0, 0, 0, 0, 0}, sec[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  const long long t_begin = clock64();
  long long t_last = t_begin;
#endif
  pdl_wait();
  const int grp = warp >> 2, w = warp & 3;      // group: which 64 keys of a tile; w: 16-key block / 16-dim block
  const int g = lane >> 2, t4 = lane & 3;
  const float sscale = a.scale * D2_LOG2E;
  const uint32_t r_base = smem_u32(Rres);
  uint32_t tile_cnt = 0;
  int cur_h = -1, r_epoch = 0;
  // per-lane constants of the fragment addressing
  const int krow_l = 16 * w + (lane & 15);                       // K phase: row inside the group's 64 keys
  const int hi16 = lane >> 4;
  const int vrow_l = (lane >> 4) * 8 + (lane & 7);               // V phase: key row inside a 16-key step
  const int vchunk = 2 * w + ((lane >> 3) & 1);

  for (int it = lo, n = 0; it < hi; ++it, ++n) {
    const int h = it / B, b = it - h * B;
    if (h != cur_h) {
      mbar_wait(r_full, (uint32_t)(r_epoch & 1));
      r_epoch++;
      cur_h = h;
    }
    const int qs = n & 1;
    D2_MARK(7);
    { D2_T0(); mbar_wait(&q_full[qs], (uint32_t)((n >> 1) & 1)); D2_ACC(1); }
    const int2 rs = qstate[qs];                  // this item's stream: its memory may differ from the other streams'
    const int mc = rs.y, head = rs.x % M;
    D2_MARK(0);
    const float* qb = qbuf + qs * 192;
    // B fragments of the query (replicated over the 8 columns): k = 16*ks + {2t, 2t+1} and {2t+8, 2t+9}
    uint32_t quf[4][2], qvf[4][2];
#pragma unroll
    for (int ks = 0; ks < 4; ks++) {
#pragma unroll
      for (int hh = 0; hh < 2; hh++) {
        const int d = ks * 16 + 2 * t4 + 8 * hh;
        const float q0 = qb[d], q1 = qb[d + 1];
        const float2 uu = *(const float2*)(a.u + h * 64 + d), vv = *(const float2*)(a.v + h * 64 + d);
        quf[ks][hh] = pack_bf16x2(q0 + uu.x, q1 + uu.y);
        qvf[ks][hh] = pack_bf16x2(q0 + vv.x, q1 + vv.y);
      }
    }
    float* scb = sc + (n & 1) * (M + 8);
    D2_MARK(1);

    // ---------------- phase 1: scores; group grp owns keys [TR j + 64 grp, +64) of tile j, warp w a 16-key block ----------------
    for (int j = 0; j < nT; ++j, ++tile_cnt) {
      const int s = tile_cnt & smask;
      { D2_T0(); mbar_wait(&full[s], (tile_cnt >> sshift) & 1); D2_ACC(2); }
      const uint32_t kt = smem_u32(stages + s * L.tile_bytes) + grp * 8192;
      const int p = TR * j + 64 * grp + krow_l;          // ring slot of this lane's ldmatrix row
      const int dist = p < head ? head - p : M + head - p;
      const uint32_t k_row = kt + krow_l * 128, r_row = r_base + dist * 128;
      const int ksw = krow_l & 7, rsw = dist & 7;
      float accK[4] = {0.f, 0.f, 0.f, 0.f}, accR[4] = {0.f, 0.f, 0.f, 0.f};   // two independent mma chains
#pragma unroll
      for (int ks = 0; ks < 4; ks++) {
        uint32_t a0, a1, a2, a3, c0, c1, c2, c3;
        ldmatrix_x4(k_row + (((2 * ks + hi16) ^ ksw) << 4), a0, a1, a2, a3);
        ldmatrix_x4(r_row + (((2 * ks + hi16) ^ rsw) << 4), c0, c1, c2, c3);
        mma_bf16_16816(accK, a0, a1, a2, a3, quf[ks][0], quf[ks][1]);
        mma_bf16_16816(accR, c0, c1, c2, c3, qvf[ks][0], qvf[ks][1]);
      }
      if (t4 == 0) {   // element 0 = key (16w + g), element 2 = key (16w + g + 8); both replicated over the quad
        const int p0 = TR * j + 64 * grp + 16 * w + g, p1 = p0 + 8;
        const int d0 = p0 < head ? head - p0 : M + head - p0;
        const int d1 = p1 < head ? head - p1 : M + head - p1;
        scb[p0] = d0 <= mc ? (accK[0] + accR[0]) * sscale : -INFINITY;
        scb[p1] = d1 <= mc ? (accK[2] + accR[2]) * sscale : -INFINITY;
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty[s]);
    }
    D2_MARK(2);
    if (warp == 0) {   // the new token itself (distance 0): fp32 q and k from the staged row, Rd[0] from the resident table
      const bf16* r0 = (const bf16*)Rres;   // row 0 is not permuted by the swizzle
      float acc = 0.f;
#pragma unroll
      for (int e = 0; e < 2; e++) {
        const int d = lane + 32 * e;
        const float q = qb[d];
        acc += (q + a.u[h * 64 + d]) * qb[64 + d] + (q + a.v[h * 64 + d]) * __bfloat162float(r0[d]);
      }
      acc = warp_sum(acc);
      if (lane == 0) scb[M] = acc * sscale;
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(r_free);
    { D2_T0(); named_bar_sync(1, NW * 32); D2_ACC(4); }
    D2_MARK(3);

    // ---------------- exact softmax over M+1 scores: max redundantly per warp, p = exp2(s - max) shared as bf16 ----------------
    float mx = -INFINITY;
    for (int jj = lane; jj <= M; jj += 32) mx = fmaxf(mx, scb[jj]);
    mx = warp_max(mx);
    float part = 0.f;
    for (int jj = 2 * (warp * 32 + lane); jj < M; jj += 2 * NW * 32) {
      const float2 s2 = *(const float2*)(scb + jj);
      const uint32_t pk = pack_bf16x2(exp2f(s2.x - mx), exp2f(s2.y - mx));
      *(uint32_t*)(pw + jj) = pk;
      part += bf16lo(pk) + bf16hi(pk);
    }
    part = warp_sum(part);
    if (lane == 0) psum[warp] = part;
    const float p_cur = exp2f(scb[M] - mx);
    { D2_T0(); named_bar_sync(2, NW * 32); D2_ACC(4); }
    float sum = p_cur;
#pragma unroll
    for (int ww = 0; ww < NW; ww++) sum += psum[ww];
    D2_MARK(4);

    // ---------------- phase 2: partial out[16 w .. 16 w + 16) over the group's 64 keys of every V tile ----------------
    float oA[4] = {0.f, 0.f, 0.f, 0.f}, oB[4] = {0.f, 0.f, 0.f, 0.f};
    for (int j = 0; j < nT; ++j, ++tile_cnt) {
      const int s = tile_cnt & smask;
      { D2_T0(); mbar_wait(&full[s], (tile_cnt >> sshift) & 1); D2_ACC(3); }
      const uint32_t vt = smem_u32(stages + s * L.tile_bytes) + grp * 8192;
      const bf16* pj = pw + TR * j + 64 * grp + 2 * t4;
#pragma unroll
      for (int ks = 0; ks < 4; ks++) {
        const int r = 16 * ks + vrow_l;
        uint32_t a0, a1, a2, a3;
        ldmatrix_x4_trans(vt + r * 128 + ((vchunk ^ (r & 7)) << 4), a0, a1, a2, a3);
        const uint32_t b0r = *(const uint32_t*)(pj + 16 * ks), b1r = *(const uint32_t*)(pj + 16 * ks + 8);
        if (ks & 1) mma_bf16_16816(oB, a0, a1, a2, a3, b0r, b1r);
        else mma_bf16_16816(oA, a0, a1, a2, a3, b0r, b1r);
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty[s]);
    }
    D2_MARK(5);
    // ---------------- epilogue: combine the groups, add the new token's own value, normalise, store; ring append ----------------
    if (G > 1) {
      if (t4 == 0) {
        ored[grp * 64 + 16 * w + g] = oA[0] + oB[0];
        ored[grp * 64 + 16 * w + g + 8] = oA[2] + oB[2];
      }
      { D2_T0(); named_bar_sync(3, NW * 32); D2_ACC(4); }
    }
    if (grp == 0 && t4 == 0) {
      const float inv = 1.f / sum;
      const int dA = 16 * w + g, dB = dA + 8;
      float vA = oA[0] + oB[0], vB = oA[2] + oB[2];
      if (G > 1) {
        vA = 0.f; vB = 0.f;
#pragma unroll
        for (int gg = 0; gg < G; gg++) { vA += ored[gg * 64 + dA]; vB += ored[gg * 64 + dB]; }
      }
      bf16* o = a.out + (size_t)b * HD + h * 64;
      o[dA] = __float2bfloat16_rn((vA + p_cur * qb[128 + dA]) * inv);
      o[dB] = __float2bfloat16_rn((vB + p_cur * qb[128 + dB]) * inv);
    }
    if (warp == 1 || warp == 2) {   // ring append (K13): slot `head` has been fully read for this (stream, head)
      bf16* ring = (warp == 1 ? a.kring : a.vring) + (((size_t)b * H + h) * M + head) * 64;
      const float* src = qb + (warp == 1 ? 64 : 128);
      *(uint32_t*)(ring + 2 * lane) = pack_bf16x2(src[2 * lane], src[2 * lane + 1]);
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&q_empty[qs]);
    D2_MARK(6);
  }
#ifdef D2_PROFILE
  if (warp == 0 && lane == 0 && d2_prof_ptr) {
    prof[0] = clock64() - t_begin; prof[5] = hi - lo;
    for (int k = 0; k < 6; k++) d2_prof_ptr[cta * 14 + k] = prof[k];
    for (int k = 0; k < 8; k++) d2_prof_ptr[cta * 14 + 6 + k] = sec[k];
  }
#endif
}


}  // namespace dmg
