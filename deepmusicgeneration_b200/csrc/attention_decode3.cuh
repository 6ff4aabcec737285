// Third-generation decode attention (x_len == 1, bf16 K/V ring, mem_len a multiple of 128).
//
// What the second kernel (attention_decode2.cuh) turned out to be bound by (scripts/probes/probe_attn_decode.cu,
// profiles/r2e_probe_attn_decode.txt): not HBM and not the ring depth (4 or 8 stages: same time) but the SM itself - 6400 cycles
// per (stream, head) item, the same at 37, 88 and 148 CTAs.  2500 of them are shared-memory bandwidth (per item the consumers
// ldmatrix 64 KB of K, 64 KB of rel-pos keys and 64 KB of V while TMA writes 128 KB), the other 3900 are the serial part of an item
// (query fragments, softmax with two block barriers, epilogue) during which the memory pipe of the SM sits idle, because all eight
// consumer warps walk through the same item in lock step.
//
// This kernel
//  * takes the rel-pos keys out of the per-item work: (q + v) . Rd[dist] is a real GEMM once the items of a CTA are put side by
//    side (the CTA's <= 16 items are consecutive streams of one or two heads), so a prologue computes PosTab[item][dist] with the
//    EIGHT mma columns holding eight different streams' queries - Rd is read once per 8 items instead of once per item - and
//    the main loop only adds a table entry to every key's score;
//  * splits the consumers into TEAMS of four warps that work on different items out of phase, each with its own producer warp, TMA
//    ring and query slots: while one team is in its softmax / epilogue the other one streams K or V;
//  * keeps a thread's scores in registers from the K phase to the exponentials (one score per lane per 128-key tile, running
//    maximum on the way), so the score array in shared memory, its 17-load maximum scan and one barrier-separated pass are gone;
//  * a team's four warps cover all 64 output dims over the whole 128-key V tile: no cross-group reduction of the output;
//  * the rel-pos keys are only needed in the prologue: their 72 KB are the tail stages of the K/V rings afterwards (the producers
//    use the head stages for the early prefetch and wait for `prologue_done` before their first use of a tail stage).
#pragma once
#include "attention_decode2.cuh"

namespace dmg {

constexpr int D3_TEAMS = 2;
constexpr int D3_CAP = 16;          // items per CTA (two mma column blocks)
constexpr int D3_KEYS = 128;        // keys per tile
constexpr int D3_TILE = D3_KEYS * 128;
constexpr int D3_THREADS = D3_TEAMS * 5 * 32;

struct D3Layout {
  int r_boxes, n_stages, tab_stride, free_bytes;
  int off_ring, off_r, off_tab, off_team, team_bytes, off_bar, total;
};

__host__ __device__ inline D3Layout d3_layout(int M, int n_stages, int teams = D3_TEAMS) {
  D3Layout L;
  L.r_boxes = (M + 1 + 63) / 64;
  L.n_stages = n_stages;
  L.tab_stride = M + 4;                        // = 4 mod 32: the mma C fragments scatter into it without bank conflicts
  const int ring = teams * n_stages * D3_TILE;
  L.off_ring = 0;
  L.off_r = ring - L.r_boxes * 8192;           // the rel-pos keys alias the tail of the ring region
  L.free_bytes = L.off_r;
  L.off_tab = ring;
  L.off_team = L.off_tab + D3_CAP * L.tab_stride * 4;
  L.team_bytes = 2 * 768 + (((M + 16) * 2 + 15) & ~15) + 64;   // q/k/v slots, bf16 probabilities, warp maxima / sums / own score
  L.off_bar = (L.off_team + teams * L.team_bytes + 15) & ~15;
  L.total = L.off_bar + (teams * (2 * n_stages + 4) + 2) * 8 + 1024 /*alignment slack*/;
  return L;
}

static inline int d3_pick_stages(int M, int teams = D3_TEAMS) {
  for (int s = 6; s >= 2; s--) {
    const D3Layout L = d3_layout(M, s, teams);
    if (L.off_r >= 0 && L.total <= 227 * 1024) return s;
  }
  return 0;
}

template <int T>
__device__ __forceinline__ void attn_decode3_body(const CUtensorMap& tmK, const CUtensorMap& tmV, const CUtensorMap& tmR, const AttnDecodeArgs& a,
                                                  int n_stages, int b0, int cta, int ncta, uint8_t* d3_smem) {
  constexpr int CW = 4 * T;                 // consumer warps [0, CW); producer warps [CW, CW + T)
  uint8_t* base = d3_smem + ((1024u - (smem_u32(d3_smem) & 1023u)) & 1023u);
  const int M = a.M, H = a.H, B = a.B, HD = H * 64;
  const D3Layout L = d3_layout(M, n_stages, T);
  uint8_t* Rres = base + L.off_r;
  float* tab = (float*)(base + L.off_tab);
  const int S = L.tab_stride;
  uint64_t* bars = (uint64_t*)(base + L.off_bar);
  uint64_t* r_full = bars;
  uint64_t* prologue_done = bars + 1;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int nT = M / D3_KEYS;               // K tiles (= V tiles) per item
  pdl_launch_dependents();
  const long long NI = (long long)B * H;
  const int lo = (int)(NI * cta / ncta), hi = (int)(NI * (cta + 1) / ncta);
  const int n_items = hi - lo;              // <= D3_CAP (the launcher sizes the chunks)

  if (tid == 0) {
    for (int t = 0; t < T; t++) {
      uint64_t* tb = bars + 2 + t * (2 * n_stages + 4);
      for (int s = 0; s < n_stages; s++) {
        mbar_init(&tb[s], 1);                       // full
        mbar_init(&tb[n_stages + s], 4);            // empty: one arrival per consumer warp of the team
      }
      for (int s = 0; s < 2; s++) {
        mbar_init(&tb[2 * n_stages + s], 1);        // q_full
        mbar_init(&tb[2 * n_stages + 2 + s], 4);    // q_empty
      }
    }
    mbar_init(r_full, 1);
    mbar_init(prologue_done, CW);
    mbar_fence_init();
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmV);
    tma_prefetch_desc(&tmR);
    if (n_items > 0) {   // the rel-pos keys derive from weights only: fetch them while the predecessor kernel drains
      mbar_expect_tx(r_full, (uint32_t)(L.r_boxes * 8192));
      for (int bx = 0; bx < L.r_boxes; bx++) tma_load_2d(Rres + bx * 8192, &tmR, 0, (lo / B) * a.Dcap + bx * 64, r_full);
    }
  }
  named_bar_sync(4, (CW + T) * 32);           // the threads of this role only

  if (warp >= CW) {
    // ============================== producers: one warp per team, every byte arrives through the TMA engine ==============================
    if (lane == 0) {
      const int team = warp - CW;
      uint64_t* tb = bars + 2 + team * (2 * n_stages + 4);
      uint64_t *full = tb, *empty = tb + n_stages, *q_full = tb + 2 * n_stages, *q_empty = q_full + 2;
      uint8_t* ring = base + L.off_ring;
      float* qbuf = (float*)(base + L.off_team + team * L.team_bytes);
      int2* qstate = (int2*)(base + L.off_team + team * L.team_bytes + 2 * 768 + (((M + 16) * 2 + 15) & ~15) + 40);   // = consumers' wmax + 10
      // stage s of team t lives at slot s * T + t of the ring region: the first stages of every team are outside the rel-pos alias
      int s = 0, use = 0, pre = 0;
      bool alias_ok = false;
      const uint64_t kv_policy = l2_policy_evict_first();
      // The K/V ring of this layer was last written by this layer's attention kernel of the PREVIOUS step (long retired), so the
      // first item's tiles do not depend on the predecessor kernel: request them while it drains.
      if (team < n_items && !a.no_early_kv) {
        const int it = lo + team, h = it / B, b = it - h * B;
        const int row0 = ((b0 + b) * H + h) * M;
        while (pre < 2 * nT && s < n_stages && (s * T + team + 1) * D3_TILE <= L.free_bytes) {
          mbar_expect_tx(&full[s], (uint32_t)D3_TILE);
          uint8_t* dst = ring + (s * T + team) * D3_TILE;
          const CUtensorMap* tm = pre < nT ? &tmK : &tmV;
          const int r0 = row0 + (pre < nT ? pre : pre - nT) * D3_KEYS;
          tma_load_2d_hint(dst, tm, 0, r0, &full[s], kv_policy);          // read once per step: evict-first, the weights stay in L2
          tma_load_2d_hint(dst + 8192, tm, 0, r0 + 64, &full[s], kv_policy);
          ++pre; ++s;
        }
        if (s == n_stages) { s = 0; use = 1; }
      }
      pdl_wait();
      int2 rs = team < n_items ? item_ring_state(a, b0, lo + team) : make_int2(0, 0);
      for (int i = team, k = 0; i < n_items; i += T, ++k) {
        const int it = lo + i, h = it / B, b = it - h * B;
        const int qs = k & 1;
        mbar_wait(&q_empty[qs], (uint32_t)(((k >> 1) & 1) ^ 1));
        qstate[qs] = rs;                            // the item's ring state goes with its q|k|v: released by the arrive below
        if (i + T < n_items) rs = item_ring_state(a, b0, it + T);
        mbar_expect_tx(&q_full[qs], 768);
        const float* qrow = a.qkv + (size_t)b * 3 * HD + h * 64;
        bulk_g2s(qbuf + qs * 192, qrow, 256, &q_full[qs]);
        bulk_g2s(qbuf + qs * 192 + 64, qrow + HD, 256, &q_full[qs]);
        bulk_g2s(qbuf + qs * 192 + 128, qrow + 2 * HD, 256, &q_full[qs]);
        const int row0 = ((b0 + b) * H + h) * M;
        for (int t = (k == 0 ? pre : 0); t < 2 * nT; ++t) {
          if (!alias_ok && (s * T + team + 1) * D3_TILE > L.free_bytes) {   // first use of a stage that overlaps the rel-pos keys
            mbar_wait(prologue_done, 0);
            alias_ok = true;
          }
          mbar_wait(&empty[s], (uint32_t)((use & 1) ^ 1));
          mbar_expect_tx(&full[s], (uint32_t)D3_TILE);
          uint8_t* dst = ring + (s * T + team) * D3_TILE;
          const CUtensorMap* tm = t < nT ? &tmK : &tmV;
          const int r0 = row0 + (t < nT ? t : t - nT) * D3_KEYS;
          tma_load_2d_hint(dst, tm, 0, r0, &full[s], kv_policy);          // read once per step: evict-first, the weights stay in L2
          tma_load_2d_hint(dst + 8192, tm, 0, r0 + 64, &full[s], kv_policy);
          if (++s == n_stages) { s = 0; ++use; }
        }
      }
    }
    return;
  }

  // ============================== consumers ==============================
  if (a.dbg && cta == 0 && tid == 0) { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); a.dbg[48] = t; }
#ifdef D2_PROFILE
  long long prof[6] = {0, 0, 0, 0, 0, 0}, sec[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  const long long t_begin = clock64();
  long long t_last = t_begin;
#endif
  pdl_wait();
  const int team = warp >> 2, w = warp & 3;
  const int g = lane >> 2, t4 = lane & 3;
  const int hi16 = lane >> 4;
  const float sscale = a.scale * D2_LOG2E;

  // ---------------- prologue: PosTab[item][dist] = (q_item + v) . Rd[head][dist], eight items per mma column block ----------------
  {
    const uint32_t r_base = smem_u32(Rres);
    const int nblk = (M + 1 + 15) / 16;
    int seg = 0, r_epoch = 0;
    while (seg < n_items) {
      const int h = (lo + seg) / B;
      const int seg_end = min(n_items, (h + 1) * B - lo);
      mbar_wait(r_full, (uint32_t)(r_epoch & 1));
      r_epoch++;
      // both column blocks (2 x 8 items, D3_CAP = 16) in one pass over the keys: the A fragments are loaded once
      uint32_t qvf[2][4][2];
#pragma unroll
      for (int nb = 0; nb < 2; nb++) {
        const int item = min(seg + 8 * nb + g, seg_end - 1);   // column g of the block (a repeated column past the end is never stored)
        const float* qrow = a.qkv + (size_t)(lo + item - h * B) * 3 * HD + h * 64;
#pragma unroll
        for (int ks = 0; ks < 4; ks++) {
#pragma unroll
          for (int hh = 0; hh < 2; hh++) {
            const int d = ks * 16 + 2 * t4 + 8 * hh;
            const float2 qq = *(const float2*)(qrow + d), vv = *(const float2*)(a.v + h * 64 + d);
            qvf[nb][ks][hh] = pack_bf16x2(qq.x + vv.x, qq.y + vv.y);
          }
        }
      }
      const bool two = seg_end - seg > 8;
      for (int blk = warp; blk < nblk; blk += CW) {
        const int dr = 16 * blk + (lane & 15);
        const uint32_t r_row = r_base + dr * 128;
        const int rsw = dr & 7;
        float acc0[4] = {0.f, 0.f, 0.f, 0.f}, acc1[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int ks = 0; ks < 4; ks++) {
          uint32_t c0, c1, c2, c3;
          ldmatrix_x4(r_row + (((2 * ks + hi16) ^ rsw) << 4), c0, c1, c2, c3);
          mma_bf16_16816(acc0, c0, c1, c2, c3, qvf[0][ks][0], qvf[0][ks][1]);
          if (two) mma_bf16_16816(acc1, c0, c1, c2, c3, qvf[1][ks][0], qvf[1][ks][1]);
        }
        // C fragment: [0] (dist g, item 2 t4), [1] (dist g, item 2 t4 + 1), [2] / [3] the same for dist g + 8
        const int d0 = 16 * blk + g, d1 = d0 + 8;
#pragma unroll
        for (int nb = 0; nb < 2; nb++) {
          const float* acc = nb ? acc1 : acc0;
          const int i0 = seg + 8 * nb + 2 * t4;
          if (i0 < seg_end) {
            if (d0 <= M) tab[i0 * S + d0] = acc[0];
            if (d1 <= M) tab[i0 * S + d1] = acc[2];
          }
          if (i0 + 1 < seg_end) {
            if (d0 <= M) tab[(i0 + 1) * S + d0] = acc[1];
            if (d1 <= M) tab[(i0 + 1) * S + d1] = acc[3];
          }
        }
      }
      seg = seg_end;
      named_bar_sync(5, CW * 32);              // every warp is done with this head's keys; the table rows are visible
      if (seg < n_items && tid == 0) {
        mbar_expect_tx(r_full, (uint32_t)(L.r_boxes * 8192));
        for (int bx = 0; bx < L.r_boxes; bx++) tma_load_2d(Rres + bx * 8192, &tmR, 0, ((lo + seg) / B) * a.Dcap + bx * 64, r_full);
      }
    }
    if (lane == 0) mbar_arrive(prologue_done);   // the ring stages under the rel-pos keys may be filled now
  }

  D2_MARK(7);   // prologue
  if (a.dbg && cta == 0 && tid == 0) { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); a.dbg[49] = t; }
  // ---------------- main loop: the team's items ----------------
  uint64_t* tb = bars + 2 + team * (2 * n_stages + 4);
  uint64_t *full = tb, *empty = tb + n_stages, *q_full = tb + 2 * n_stages, *q_empty = q_full + 2;
  uint8_t* ring = base + L.off_ring;
  uint8_t* tmem_base = base + L.off_team + team * L.team_bytes;
  float* qbuf = (float*)tmem_base;
  bf16* pw = (bf16*)(tmem_base + 2 * 768);
  float* wmax = (float*)(tmem_base + 2 * 768 + (((M + 16) * 2 + 15) & ~15));   // [4] warp maxima, [4] warp sums, [1] own score
  float* psum = wmax + 4;
  float* own_s = wmax + 8;
  const int2* qstate = (const int2*)(wmax + 10);   // [2] ring state of the item in q slot 0 / 1 (written by the producer)
  const int bar_a = 6 + 2 * team, bar_b = 7 + 2 * team;
  // per-lane constants of the fragment addressing
  const int krowA = 32 * w + (lane & 15), krowB = krowA + 16;     // K phase: the lane's ldmatrix rows inside the 128-key tile
  const uint32_t koffA = (krowA >> 6) * 8192 + (krowA & 63) * 128, koffB = (krowB >> 6) * 8192 + (krowB & 63) * 128;
  const int kswA = krowA & 7, kswB = krowB & 7;
  const int my_row = 32 * w + 16 * (t4 >> 1) + 8 * (t4 & 1) + g;  // the key whose score this lane finishes
  const int vrow_l = (lane >> 4) * 8 + (lane & 7);                // V phase: key row inside a 16-key step
  const int vchunk = 2 * w + ((lane >> 3) & 1);
  int s = 0, use = 0, cur_h = -1;
  float2 uu[4][2];
#pragma unroll
  for (int ks = 0; ks < 4; ks++) uu[ks][0] = uu[ks][1] = make_float2(0.f, 0.f);

  for (int i = team, k = 0; i < n_items; i += T, ++k) {
    const int it = lo + i, h = it / B, b = it - h * B;
    if (h != cur_h) {
#pragma unroll
      for (int ks = 0; ks < 4; ks++) {
        uu[ks][0] = *(const float2*)(a.u + h * 64 + ks * 16 + 2 * t4);
        uu[ks][1] = *(const float2*)(a.u + h * 64 + ks * 16 + 2 * t4 + 8);
      }
      cur_h = h;
    }
    const int qs = k & 1;
    mbar_wait(&q_full[qs], (uint32_t)((k >> 1) & 1));
    const int2 rs = qstate[qs];                 // this item's stream: its memory may differ from the other streams'
    const int mc = rs.y, head = rs.x % M;
    D2_MARK(0);
    const float* qb = qbuf + qs * 192;
    const float* tabrow = tab + i * S;
    uint32_t quf[4][2];     // B fragments of the query (replicated over the 8 columns): k = 16*ks + {2t, 2t+1} and {2t+8, 2t+9}
#pragma unroll
    for (int ks = 0; ks < 4; ks++) {
#pragma unroll
      for (int hh = 0; hh < 2; hh++) {
        const float2 qq = *(const float2*)(qb + ks * 16 + 2 * t4 + 8 * hh);
        quf[ks][hh] = pack_bf16x2(qq.x + uu[ks][hh].x, qq.y + uu[ks][hh].y);
      }
    }
    if (w == 0) {   // the new token itself (distance 0): fp32 q and k from the staged row
      float acc = 0.f;
#pragma unroll
      for (int e = 0; e < 2; e++) {
        const int d = lane + 32 * e;
        acc += (qb[d] + a.u[h * 64 + d]) * qb[64 + d];
      }
      acc = warp_sum(acc);
      if (lane == 0) own_s[0] = (acc + tabrow[0]) * sscale;
    }

    D2_MARK(1);
    // ---------------- K phase: warp w owns keys [32 w, 32 w + 32) of every 128-key tile; one finished score per lane per tile ----------------
    float sv[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
    float mx = -INFINITY;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (j < nT) {
        { D2_T0(); mbar_wait(&full[s], (uint32_t)(use & 1)); D2_ACC(2); }
        const uint32_t kt = smem_u32(ring + (s * T + team) * D3_TILE);
        float accA[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}}, accB[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
#pragma unroll
        for (int ks = 0; ks < 4; ks++) {                    // four independent mma chains of depth two
          uint32_t a0, a1, a2, a3, c0, c1, c2, c3;
          ldmatrix_x4(kt + koffA + (((2 * ks + hi16) ^ kswA) << 4), a0, a1, a2, a3);
          ldmatrix_x4(kt + koffB + (((2 * ks + hi16) ^ kswB) << 4), c0, c1, c2, c3);
          mma_bf16_16816(accA[ks & 1], a0, a1, a2, a3, quf[ks][0], quf[ks][1]);
          mma_bf16_16816(accB[ks & 1], c0, c1, c2, c3, quf[ks][0], quf[ks][1]);
        }
        // every column of the accumulator holds the same score: lane t4 of a quad finishes key 16 (t4 >> 1) + 8 (t4 & 1) + g
        const float val = t4 == 0 ? accA[0][0] + accA[1][0] : t4 == 1 ? accA[0][2] + accA[1][2] : t4 == 2 ? accB[0][0] + accB[1][0] : accB[0][2] + accB[1][2];
        const int p = D3_KEYS * j + my_row;                 // ring slot
        const int dist = p < head ? head - p : M + head - p;
        const float sc = dist <= mc ? (val + tabrow[dist]) * sscale : -INFINITY;
        sv[j] = sc;
        mx = fmaxf(mx, sc);
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[s]);
        if (++s == n_stages) { s = 0; ++use; }
      }
    }
    D2_MARK(2);
    // ---------------- exact softmax over the M + 1 scores (scores stay in registers) ----------------
    mx = warp_max(mx);
    if (lane == 0) wmax[w] = mx;
    named_bar_sync(bar_a, 128);
    const float own = own_s[0];
    mx = fmaxf(fmaxf(fmaxf(wmax[0], wmax[1]), fmaxf(wmax[2], wmax[3])), own);
    float part = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (j < nT) {
        const bf16 pb = __float2bfloat16_rn(exp2f(sv[j] - mx));
        pw[D3_KEYS * j + my_row] = pb;
        part += __bfloat162float(pb);
      }
    }
    part = warp_sum(part);
    if (lane == 0) psum[w] = part;
    const float p_cur = exp2f(own - mx);
    named_bar_sync(bar_b, 128);
    const float sum = p_cur + psum[0] + psum[1] + psum[2] + psum[3];
    D2_MARK(4);

    // ---------------- V phase: warp w owns out[16 w .. 16 w + 16) over all 128 keys of every tile ----------------
    float oA[4] = {0.f, 0.f, 0.f, 0.f}, oB[4] = {0.f, 0.f, 0.f, 0.f}, oC[4] = {0.f, 0.f, 0.f, 0.f}, oD[4] = {0.f, 0.f, 0.f, 0.f};
    for (int j = 0; j < nT; ++j) {
      { D2_T0(); mbar_wait(&full[s], (uint32_t)(use & 1)); D2_ACC(3); }
      const uint32_t vt = smem_u32(ring + (s * T + team) * D3_TILE);
      const bf16* pj = pw + D3_KEYS * j + 2 * t4;
#pragma unroll
      for (int ks = 0; ks < 8; ks++) {
        const int r = 16 * ks + vrow_l;
        uint32_t a0, a1, a2, a3;
        ldmatrix_x4_trans(vt + (r >> 6) * 8192 + (r & 63) * 128 + ((vchunk ^ (r & 7)) << 4), a0, a1, a2, a3);
        const uint32_t b0r = *(const uint32_t*)(pj + 16 * ks), b1r = *(const uint32_t*)(pj + 16 * ks + 8);
        if (ks & 1) mma_bf16_16816(oB, a0, a1, a2, a3, b0r, b1r);
        else mma_bf16_16816(oA, a0, a1, a2, a3, b0r, b1r);
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty[s]);
      if (++s == n_stages) { s = 0; ++use; }
    }
    D2_MARK(5);
    // ---------------- epilogue: add the new token's own value, normalise, store; ring append ----------------
    if (t4 == 0) {
      const float inv = 1.f / sum;
      const int dA = 16 * w + g, dB = dA + 8;
      bf16* o = a.out + (size_t)b * HD + h * 64;
      o[dA] = __float2bfloat16_rn(((oA[0] + oB[0]) + (oC[0] + oD[0]) + p_cur * qb[128 + dA]) * inv);
      o[dB] = __float2bfloat16_rn(((oA[2] + oB[2]) + (oC[2] + oD[2]) + p_cur * qb[128 + dB]) * inv);
    }
    if (w == 1 || w == 2) {   // ring append (K13): slot `head` has been fully read for this (stream, head)
      bf16* rg = (w == 1 ? a.kring : a.vring) + (((size_t)b * H + h) * M + head) * 64;
      const float* src = qb + (w == 1 ? 64 : 128);
      *(uint32_t*)(rg + 2 * lane) = pack_bf16x2(src[2 * lane], src[2 * lane + 1]);
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&q_empty[qs]);
    D2_MARK(6);
  }
  if (a.dbg && tid == 0 && (cta == 0 || cta == ncta - 1)) { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); a.dbg[cta == 0 ? 50 : 51] = t; }
#ifdef D2_PROFILE
  if (warp == 0 && lane == 0 && d2_prof_ptr) {
    prof[0] = clock64() - t_begin; prof[5] = (n_items + T - 1) / T;
    for (int k = 0; k < 6; k++) d2_prof_ptr[cta * 14 + k] = prof[k];
    for (int k = 0; k < 8; k++) d2_prof_ptr[cta * 14 + 6 + k] = sec[k];
  }
#endif
}

}  // namespace dmg
