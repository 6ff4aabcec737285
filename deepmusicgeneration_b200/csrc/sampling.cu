// Fused per-stream sampling step: temperature (+repeat penalty), grammar mask, top-k, top-p, softmax, multinomial
// and the loop bookkeeping of MusicLearner.predict - one CTA per generation stream, no host round trip.
//
// Reference being replaced (SURVEY.md 2.2 K15, App. C.3): deep_music_genre.py:1895-1967 (loop body),
// top_k_top_p :1679-1706, filter_invalid_indexes :1984-2018 (remix variant deep_music_remix.py:2394-2437),
// predict_mask's sampling deep_music_remix.py:2586-2609.
#include "kernels.cuh"
#include "sampling.cuh"
#include "launch.cuh"

namespace dmg {

// ---- Philox4x32-10 (counter-based; one draw per (stream, step)) ----
__device__ __forceinline__ uint32_t mulhilo(uint32_t a, uint32_t b, uint32_t* hi) {
  const uint64_t p = (uint64_t)a * b;
  *hi = (uint32_t)(p >> 32);
  return (uint32_t)p;
}
__device__ float philox_uniform(uint64_t seed, uint64_t offset, uint32_t stream) {
  uint32_t c0 = (uint32_t)offset, c1 = (uint32_t)(offset >> 32), c2 = stream, c3 = 0x9E3779B9u;
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
  for (int i = 0; i < 10; i++) {
    uint32_t hi0, hi1;
    const uint32_t lo0 = mulhilo(0xD2511F53u, c0, &hi0);
    const uint32_t lo1 = mulhilo(0xCD9E8D57u, c2, &hi1);
    c0 = hi1 ^ c1 ^ k0;
    c1 = lo1;
    c2 = hi0 ^ c3 ^ k1;
    c3 = lo0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return (float)(c0 >> 8) * (1.0f / 16777216.0f);   // [0, 1)
}

// order-preserving float -> uint32 (larger float = larger key)
__device__ __forceinline__ uint32_t float_key(float f) {
  const uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key_float(uint32_t k) {
  const uint32_t u = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
  return __uint_as_float(u);
}

constexpr int SAMP_THREADS = 256;
constexpr int SAMP_MAXV = 1024;

// inclusive scan of vals[0..n) by warp 0 (chunked shuffle scan); result in place. Returns total via vals[n-1].
__device__ void warp0_inclusive_scan(float* vals, int n) {
  if (threadIdx.x >= 32) return;
  const int lane = threadIdx.x;
  float carry = 0.f;
  for (int base = 0; base < n; base += 32) {
    const int i = base + lane;
    float x = i < n ? vals[i] : 0.f;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const float y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    x += carry;
    if (i < n) vals[i] = x;
    carry = __shfl_sync(0xffffffffu, x, 31);
  }
}

__device__ float block_max(float v, float* scratch) {
  v = warp_max(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = scratch[0];
  for (int w = 1; w < SAMP_THREADS / 32; w++) r = fmaxf(r, scratch[w]);
  return r;
}
__device__ float block_sum(float v, float* scratch) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = 0.f;
  for (int w = 0; w < SAMP_THREADS / 32; w++) r += scratch[w];
  return r;
}

__device__ __forceinline__ bool in_range(int x, int lo, int hi) { return x >= lo && x < hi; }

__global__ void __launch_bounds__(SAMP_THREADS) sample_kernel(SampleArgs a) {
  __shared__ float l[SAMP_MAXV];                 // working logits, vocab order
  __shared__ unsigned long long keys[SAMP_MAXV]; // (float key << 32) | (~index): descending sort = value desc, index asc
  __shared__ unsigned long long kin[SAMP_MAXV];  // the same keys in vocabulary order (input of the rank sort)
  __shared__ float pr[SAMP_MAXV];                // probabilities (sorted order, then vocab order)
  __shared__ float scratch[SAMP_THREADS / 32];
  __shared__ int sh_int[4];

  const int sidx = blockIdx.x, tid = threadIdx.x;
  pdl_launch_dependents();
  pdl_wait();
  const int V = a.V;
  const dmg_vocab_layout vl = a.vocab;
  const dmg_sampler_params sp = a.params;
  const float NEG = -INFINITY;

  // ---------------- per-stream scalar state ----------------
  int prev, repeat_count, last_xxsep = 0, status = 0, step = 0;
  long long last_pos = 0, start_pos = 0;
  if (a.loop_mode == 2) {   // one step of the predict loop on caller-provided state (nothing is written back)
    prev = a.prev_idx[sidx];
    repeat_count = a.repeat_count[sidx];
    last_xxsep = a.last_xxsep[sidx];
    last_pos = a.last_pos[sidx];
  } else if (a.loop_mode) {
    status = a.status[sidx];
    prev = a.prev_idx[sidx];
    repeat_count = a.repeat_count[sidx];
    last_xxsep = a.last_xxsep[sidx];
    last_pos = a.last_pos[sidx];
    start_pos = a.start_pos[sidx];
    step = a.step[sidx];
    if (status != 0) {   // stopped / errored stream: keep the batch in lock-step on a harmless token
      if (tid == 0) {
        if (a.out_tokens) a.out_tokens[sidx] = status == 1 ? -1 : -2;
        a.next_ids[sidx] = vl.pad;
        if (a.next_pos) a.next_pos[sidx] = last_pos;
      }
      return;
    }
  } else {
    prev = a.prev_idx[sidx];
    repeat_count = a.repeat_count[sidx];
  }
  const bool prev_dur = in_range(prev, vl.dur_lo, vl.dur_hi);
  const bool prev_note = prev == vl.sep || in_range(prev, vl.note_lo, vl.note_hi);
  const bool prev_ins = prev == vl.ni || in_range(prev, vl.ins_lo, vl.ins_hi);
  const bool remix = (sp.flags & DMG_SAMPLE_REMIX_FILTER) != 0;

  double temperature;
  if (a.loop_mode) {
    if (prev == vl.sep) last_xxsep = 1;
    else if (prev_ins && prev == vl.ni) last_xxsep = 0;
    if (prev_dur) temperature = sp.temperatures[2];
    else if (prev_note) temperature = sp.temperatures[1];
    else if (prev_ins || prev == vl.pad) temperature = sp.temperatures[0];
    else {   // reference: `assert temperature is not None` -> AssertionError (deep_music_genre.py:1920-1925)
      if (tid == 0) {
        if (a.out_tokens) a.out_tokens[sidx] = -2;
        if (a.loop_mode == 1) {
          a.status[sidx] = 2;
          a.next_ids[sidx] = vl.pad;
          if (a.next_pos) a.next_pos[sidx] = last_pos;
        }
      }
      return;
    }
  } else {
    temperature = (prev == vl.pad || prev_dur) ? sp.temperatures[0] : sp.temperatures[1];   // is_duration_or_pad
  }
  {
    double pen = log(((double)repeat_count + 1.0) / 4.0) / 5.0;
    if (pen < 0.0) pen = 0.0;
    temperature += pen * temperature;
  }
  const float tf = (float)temperature;
  const bool forbid_bos = a.loop_mode && (((last_pos - start_pos) / 16) <= (long long)sp.min_bars);

  // ---------------- temperature + grammar mask ----------------
  const float* lg = a.logits + (size_t)sidx * V;
  for (int i = tid; i < V; i += SAMP_THREADS) {
    float x = lg[i];
    if (temperature != 1.0) x = x / tf;
    bool kill = false;
    const bool is_special = in_range(i, vl.special_lo, vl.special_hi);
    const bool is_note = in_range(i, vl.note_lo, vl.note_hi);
    const bool is_dur = in_range(i, vl.dur_lo, vl.dur_hi);
    const bool is_ins = in_range(i, vl.ins_lo, vl.ins_hi);
    if (forbid_bos && i == vl.bos) kill = true;
    if (!a.loop_mode) {   // predict_mask: no special tokens at all (pad and mask excepted), deep_music_remix.py:2595-2596
      if (is_special && i != vl.pad && i != vl.mask) kill = true;
    }
    if (sp.allowed_ins_mask != 0 && is_ins && !((sp.allowed_ins_mask >> (i - vl.ins_lo)) & 1u)) kill = true;
    if (last_xxsep) { if (is_ins) kill = true; }
    else if (i == vl.ni) kill = true;
    if (remix && prev == vl.pad) {
      if (is_dur || is_ins || (is_special && i != vl.sep)) kill = true;
    } else if (prev_dur) {
      if (is_dur || is_note || (is_special && i != vl.ni)) kill = true;
    } else if (prev_ins || (!remix && prev == vl.pad)) {
      if (is_ins || is_dur || (is_special && i != vl.sep)) kill = true;
    } else {
      if (is_note || is_ins || is_special) kill = true;
    }
    if ((sp.flags & DMG_SAMPLE_MASK_UNUSED) && i >= vl.ins_hi) kill = true;
    l[i] = kill ? NEG : x;
  }
  __syncthreads();

  // ---------------- sort (value desc, index asc) ----------------
  // The keys are distinct (the index is part of the key), so the sorted position of an element is the number of larger keys: every
  // thread counts for its elements (V broadcast reads each) and scatters - two block barriers instead of the 45 of a bitonic network
  // over 512 keys, which were most of this kernel's 21 us.
  for (int i = tid; i < V; i += SAMP_THREADS)
    kin[i] = ((unsigned long long)float_key(l[i]) << 32) | (unsigned long long)(0xFFFFFFFFu - (uint32_t)i);
  __syncthreads();
  for (int i = tid; i < V; i += SAMP_THREADS) {
    const unsigned long long me = kin[i];
    int r = 0;
#pragma unroll 4
    for (int j = 0; j < V; j++) r += kin[j] > me ? 1 : 0;
    keys[r] = me;
  }
  __syncthreads();

  // ---------------- top-k: drop everything strictly below the k-th largest ----------------
  int top_k = sp.top_k < V ? sp.top_k : V;
  float kth = NEG;
  if (top_k > 0) {
    kth = key_float((uint32_t)(keys[top_k - 1] >> 32));
    for (int i = tid; i < V; i += SAMP_THREADS)
      if (l[i] < kth) l[i] = NEG;
  }
  __syncthreads();

  // ---------------- top-p over the sorted, top-k-filtered logits ----------------
  if (sp.top_p > 0.0f) {
    const float smax = key_float((uint32_t)(keys[0] >> 32));
    float part = 0.f;
    for (int i = tid; i < V; i += SAMP_THREADS) {
      float x = key_float((uint32_t)(keys[i] >> 32));
      if (top_k > 0 && x < kth) x = NEG;
      const float e = (smax == NEG) ? 0.f : expf(x - smax);
      pr[i] = e;
      part += e;
    }
    const float tot = block_sum(part, scratch);
    for (int i = tid; i < V; i += SAMP_THREADS) pr[i] = pr[i] / tot;
    __syncthreads();
    warp0_inclusive_scan(pr, V);
    __syncthreads();
    // sorted position i (>= 1) is removed iff cumulative_probs[i-1] > top_p
    for (int i = tid + 1; i < V; i += SAMP_THREADS) {
      if (pr[i - 1] > sp.top_p) {
        const int idx = (int)(0xFFFFFFFFu - (uint32_t)(keys[i] & 0xFFFFFFFFull));
        l[idx] = NEG;
      }
    }
    __syncthreads();
  }

  // ---------------- softmax + multinomial ----------------
  float part = NEG;
  for (int i = tid; i < V; i += SAMP_THREADS) part = fmaxf(part, l[i]);
  const float mx = block_max(part, scratch);
  float ps = 0.f;
  for (int i = tid; i < V; i += SAMP_THREADS) {
    const float e = (mx == NEG) ? 0.f : expf(l[i] - mx);
    pr[i] = e;
    ps += e;
  }
  const float tot = block_sum(ps, scratch);
  int nz = 0;
  for (int i = tid; i < V; i += SAMP_THREADS) {
    const float p = pr[i] / tot;
    pr[i] = p;
    if (a.probs) a.probs[(size_t)sidx * V + i] = p;
    nz += p > 0.f ? 1 : 0;
  }
  const int num_choices = (int)(block_sum((float)nz, scratch) + 0.5f);
  __syncthreads();
  warp0_inclusive_scan(pr, V);
  __syncthreads();
  if (tid == 0) sh_int[0] = V;
  __syncthreads();
  const uint64_t draw = a.offset + (a.loop_mode ? (uint64_t)step : 0ull) + (a.dev_offset ? (uint64_t)*a.dev_offset : 0ull);
  const float u = philox_uniform(sp.seed, draw, a.stream_ids ? (uint32_t)a.stream_ids[sidx] : (uint32_t)sidx);
  const float target = u * pr[V - 1];
  for (int i = tid; i < V; i += SAMP_THREADS) {
    const float prevc = i > 0 ? pr[i - 1] : 0.f;
    if (pr[i] > target && pr[i] > prevc) atomicMin(&sh_int[0], i);   // first index whose cdf exceeds the draw
  }
  __syncthreads();
  int idx = sh_int[0];
  if (idx >= V) {   // numerical corner (target == total): take the last index with mass
    __syncthreads();
    if (tid == 0) sh_int[1] = -1;
    __syncthreads();
    for (int i = tid; i < V; i += SAMP_THREADS) {
      const float prevc = i > 0 ? pr[i - 1] : 0.f;
      if (pr[i] > prevc) atomicMax(&sh_int[1], i);
    }
    __syncthreads();
    idx = sh_int[1] >= 0 ? sh_int[1] : vl.pad;
  }

  // ---------------- bookkeeping ----------------
  if (tid != 0) return;
  if (a.num_choices) a.num_choices[sidx] = num_choices;
  if (a.loop_mode != 1) {
    a.out_tokens[sidx] = idx;
    return;
  }
  if (num_choices <= 2) repeat_count += 1;
  else repeat_count = repeat_count / 2;
  bool stop = false;
  if (prev == vl.sep) {
    last_pos += (long long)(idx - vl.dur_lo);
    const long long abs_bar = last_pos / 16;
    if ((sp.flags & DMG_SAMPLE_EARLY_STOP) && ((double)step / (double)sp.n_words > 0.80) && (abs_bar % 4 == 0)) stop = true;
  }
  if (!stop && (sp.flags & DMG_SAMPLE_EARLY_STOP) && idx == vl.bos) stop = true;
  a.repeat_count[sidx] = repeat_count;
  a.last_xxsep[sidx] = last_xxsep;
  a.last_pos[sidx] = last_pos;
  a.step[sidx] = step + 1;
  if (stop) {
    a.status[sidx] = 1;
    if (a.out_tokens) a.out_tokens[sidx] = -1;
    a.next_ids[sidx] = vl.pad;
  } else {
    a.prev_idx[sidx] = idx;
    if (a.out_tokens) a.out_tokens[sidx] = idx;
    a.next_ids[sidx] = idx;
  }
  if (a.next_pos) a.next_pos[sidx] = last_pos;
}

// ---------------------------------------------------------------------------------------------------------------------------
// One step of MusicLearner.beam_search (deep_music_genre.py:1834-1847) for all live beams, one CTA:
//   out = log_softmax(logits[:, -1]); values, indices = out.topk(top_k); scores = (-values + scores[:, None]).view(-1)
//   sort_idx = scores.argsort()[:beam_sz]  ->  new scores, parent beam (sort_idx // top_k), appended token
// Ties are broken towards the lower candidate index (a stable argsort; torch leaves the order of exact ties unspecified - and the
// reference creates exact ties itself by starting from top_k identical copies of the seed).
__device__ void block_arg_best(float v, int idx, bool want_max, float* sval, int* sidx, float& best_v, int& best_i) {
  // (value, index) reduction: larger (want_max) or smaller value wins, lower index on ties
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, v, o);
    const int oi = __shfl_xor_sync(0xffffffffu, idx, o);
    const bool better = want_max ? (ov > v || (ov == v && oi < idx)) : (ov < v || (ov == v && oi < idx));
    if (better) { v = ov; idx = oi; }
  }
  __syncthreads();
  if ((threadIdx.x & 31) == 0) { sval[threadIdx.x >> 5] = v; sidx[threadIdx.x >> 5] = idx; }
  __syncthreads();
  best_v = sval[0]; best_i = sidx[0];
  for (int w = 1; w < SAMP_THREADS / 32; w++) {
    const float ov = sval[w]; const int oi = sidx[w];
    const bool better = want_max ? (ov > best_v || (ov == best_v && oi < best_i)) : (ov < best_v || (ov == best_v && oi < best_i));
    if (better) { best_v = ov; best_i = oi; }
  }
}

__global__ void __launch_bounds__(SAMP_THREADS) beam_step_kernel(BeamArgs a) {
  __shared__ float lp[SAMP_MAXV];
  __shared__ float cand_score[SAMP_MAXV];
  __shared__ int cand_tok[SAMP_MAXV];
  __shared__ float scratch[SAMP_THREADS / 32];
  __shared__ float sval[SAMP_THREADS / 32];
  __shared__ int sidx[SAMP_THREADS / 32];
  const int tid = threadIdx.x, V = a.V, K = a.top_k;
  const float INF = INFINITY;
  pdl_launch_dependents();
  pdl_wait();                                  // the logits come from the head GEMM launched just before
  for (int row = 0; row < a.nb; row++) {
    const float* lg = a.logits + (size_t)row * V;
    float part = -INF;
    for (int i = tid; i < V; i += SAMP_THREADS) { lp[i] = lg[i]; part = fmaxf(part, lg[i]); }
    const float mx = block_max(part, scratch);
    float ps = 0.f;
    for (int i = tid; i < V; i += SAMP_THREADS) ps += expf(lp[i] - mx);
    const float lse = mx + logf(block_sum(ps, scratch));
    __syncthreads();
    for (int i = tid; i < V; i += SAMP_THREADS) lp[i] -= lse;        // log_softmax
    __syncthreads();
    const float prev = a.scores_in[a.n_scores == 1 ? 0 : row];
    for (int j = 0; j < K; j++) {                                     // topk: K passes of a block argmax
      float v = -INF; int idx = 0x7fffffff;
      for (int i = tid; i < V; i += SAMP_THREADS)
        if (lp[i] > v || (lp[i] == v && i < idx)) { v = lp[i]; idx = i; }
      float bv; int bi;
      block_arg_best(v, idx, true, sval, sidx, bv, bi);
      if (tid == 0) { cand_score[row * K + j] = -bv + prev; cand_tok[row * K + j] = bi; lp[bi] = -INF; }
      __syncthreads();
    }
  }
  const int NC = a.nb * K;
  for (int j = 0; j < a.beam_sz; j++) {                               // argsort()[:beam_sz]: beam_sz passes of a block argmin
    float v = INF; int idx = 0x7fffffff;
    for (int i = tid; i < NC; i += SAMP_THREADS)
      if (cand_score[i] < v || (cand_score[i] == v && i < idx)) { v = cand_score[i]; idx = i; }
    float bv; int bi;
    block_arg_best(v, idx, false, sval, sidx, bv, bi);
    if (tid == 0) {
      if (j < NC) { a.scores_out[j] = bv; a.parents[j] = bi / K; a.tokens[j] = cand_tok[bi]; cand_score[bi] = INF; }
    }
    __syncthreads();
  }
}

int beam_step_launch(const BeamArgs& a, cudaStream_t st) {
  DMG_CHECK(a.V <= SAMP_MAXV && a.nb >= 1 && a.top_k >= 1 && a.top_k <= a.V && a.nb * a.top_k <= SAMP_MAXV && a.beam_sz >= 1 &&
                a.beam_sz <= a.nb * a.top_k,
            "beam step: nb %d x top_k %d (beam_sz %d, vocab %d) outside the kernel's limits", a.nb, a.top_k, a.beam_sz, a.V);
  return launch_k(beam_step_kernel, dim3(1), dim3(SAMP_THREADS), 0, st, 1, a);
}

int sample_launch(const SampleArgs& a, int n, cudaStream_t st) {
  DMG_CHECK(a.V <= SAMP_MAXV, "sampler: vocab %d exceeds %d", a.V, SAMP_MAXV);
  if (n <= 0) return 0;
  return launch_k(sample_kernel, dim3(n), dim3(SAMP_THREADS), 0, st, 1, a);
}

}  // namespace dmg
