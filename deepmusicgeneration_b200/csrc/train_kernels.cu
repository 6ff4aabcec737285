// Elementwise / reduction kernels of the training step: embedding (+dropout), dropout-residual-LayerNorm forward and
// backward, cross-entropy loss + logit gradient, RNN (time-shared) dropout of the head input, AR/TAR regularisers,
// bias-gradient column sums, embedding gradient, memory update, fused Adam.  All HBM-bound: 16-byte accesses,
// one warp per row where a row statistic is needed, grids sized in multiples of the SM count for the reductions.
// Replaces the autograd graph fastai builds around MusicTransformerXL.forward (SURVEY.md 3.3, App. A.3, A.7).
#include "kernels.cuh"
#include "launch.cuh"
#include "train_kernels.cuh"

namespace dmg {

uint32_t drop_seed(uint64_t base, uint64_t step, int site, int layer) {
  uint64_t z = base + 0x9E3779B97F4A7C15ull * (step * 4096ull + (uint64_t)site * 64ull + (uint64_t)layer + 1ull);
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  z ^= z >> 31;
  return (uint32_t)(z ^ (z >> 32));
}

namespace {

__device__ __forceinline__ void keep4(uint32_t seed, uint32_t e0, uint32_t thresh, float scale, float (&k)[4]) {
  // e0 is a multiple of 4: two pair hashes
  const uint32_t h0 = drop_pair_bits(seed, e0 >> 1), h1 = drop_pair_bits(seed, (e0 >> 1) + 1);
  k[0] = ((h0 & 0xFFFFu) >= thresh) ? scale : 0.f;
  k[1] = ((h0 >> 16) >= thresh) ? scale : 0.f;
  k[2] = ((h1 & 0xFFFFu) >= thresh) ? scale : 0.f;
  k[3] = ((h1 >> 16) >= thresh) ? scale : 0.f;
}

// ------------------------------------------------------------------ embedding
__global__ void __launch_bounds__(256) train_embed_kernel(const long long* __restrict__ ids, const long long* __restrict__ pos,
                                                          const float* __restrict__ emb, const float* __restrict__ beat,
                                                          const float* __restrict__ bar, float* __restrict__ x32,
                                                          bf16* __restrict__ xa, int rows, int d, int vocab, uint32_t thresh,
                                                          uint32_t seed, float scale) {
  const int d4 = d >> 2;
  const long long n = (long long)rows * d4;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256) {
    const int row = (int)(i / d4), c = (int)(i % d4) * 4;
    long long id = ids[row];
    id = id < 0 ? 0 : (id >= vocab ? vocab - 1 : id);
    float4 v = *(const float4*)(emb + id * d + c);
    if (pos) {
      const long long p = pos[row];
      const long long bt = p & 31, br = (p >> 5) & 1023;   // p mod 32, floor(p / 32) mod 1024 (Python floor semantics, also for p < 0)
      const float4 x = *(const float4*)(beat + bt * d + c), y = *(const float4*)(bar + br * d + c);
      v.x += x.x + y.x; v.y += x.y + y.y; v.z += x.z + y.z; v.w += x.w + y.w;
    }
    if (thresh) {
      float k[4];
      keep4(seed, (uint32_t)(row * d + c), thresh, scale, k);
      v.x *= k[0]; v.y *= k[1]; v.z *= k[2]; v.w *= k[3];
    }
    *(float4*)(x32 + (long long)row * d + c) = v;
    *(uint2*)(xa + (long long)row * d + c) = make_uint2(pack_bf16x2(v.x, v.y), pack_bf16x2(v.z, v.w));
  }
}

__global__ void __launch_bounds__(256) train_embed_bwd_kernel(const long long* __restrict__ ids, const long long* __restrict__ pos,
                                                              const float* __restrict__ dx, const bf16* __restrict__ dbr, float* __restrict__ demb,
                                                              float* __restrict__ dbeat, float* __restrict__ dbar, int rows, int d,
                                                              int vocab, long long pad_idx, uint32_t thresh, uint32_t seed, float scale) {
  const int d4 = d >> 2;
  const long long n = (long long)rows * d4;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256) {
    const int row = (int)(i / d4), c = (int)(i % d4) * 4;
    long long id = ids[row];
    id = id < 0 ? 0 : (id >= vocab ? vocab - 1 : id);
    float4 g = *(const float4*)(dx + (long long)row * d + c);
    if (dbr) {
      const uint2 b2 = *(const uint2*)(dbr + (long long)row * d + c);
      g.x += bf16lo(b2.x); g.y += bf16hi(b2.x); g.z += bf16lo(b2.y); g.w += bf16hi(b2.y);
    }
    if (thresh) {
      float k[4];
      keep4(seed, (uint32_t)(row * d + c), thresh, scale, k);
      g.x *= k[0]; g.y *= k[1]; g.z *= k[2]; g.w *= k[3];
    }
    if (id != pad_idx) {   // nn.Embedding(padding_idx): lookups of the pad token contribute no gradient
      float* e = demb + id * d + c;
      atomicAdd(e, g.x); atomicAdd(e + 1, g.y); atomicAdd(e + 2, g.z); atomicAdd(e + 3, g.w);
    }
    if (pos) {
      const long long p = pos[row];
      const long long bt = p & 31, br = (p >> 5) & 1023;   // as train_embed_kernel
      if (bt != 0) {   // padding_idx = 0 rows receive no gradient
        float* q = dbeat + bt * d + c;
        atomicAdd(q, g.x); atomicAdd(q + 1, g.y); atomicAdd(q + 2, g.z); atomicAdd(q + 3, g.w);
      }
      if (br != 0) {
        float* q = dbar + br * d + c;
        atomicAdd(q, g.x); atomicAdd(q + 1, g.y); atomicAdd(q + 2, g.z); atomicAdd(q + 3, g.w);
      }
    }
  }
}

// ------------------------------------------------------------------ dropout + residual + LayerNorm (one warp per row)
template <int NV>   // NV = d / 128 float4 chunks per lane
__global__ void __launch_bounds__(256) train_res_ln_fwd_kernel(float* __restrict__ x32, const bf16* __restrict__ add,
                                                               const float* __restrict__ w, const float* __restrict__ b,
                                                               bf16* __restrict__ xa, bf16* __restrict__ zsave,
                                                               float2* __restrict__ stats, int rows, uint32_t thresh, uint32_t seed,
                                                               float scale) {
  constexpr int d = NV * 128;
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= rows) return;
  float z[NV][4];
  float sum = 0.f;
#pragma unroll
  for (int k = 0; k < NV; k++) {
    const int c = (lane + 32 * k) * 4;
    const float4 x = *(const float4*)(x32 + (long long)row * d + c);
    const uint2 a2 = *(const uint2*)(add + (long long)row * d + c);
    float av[4] = {bf16lo(a2.x), bf16hi(a2.x), bf16lo(a2.y), bf16hi(a2.y)};
    if (thresh) {
      float kp[4];
      keep4(seed, (uint32_t)(row * d + c), thresh, scale, kp);
      av[0] *= kp[0]; av[1] *= kp[1]; av[2] *= kp[2]; av[3] *= kp[3];
    }
    z[k][0] = x.x + av[0]; z[k][1] = x.y + av[1]; z[k][2] = x.z + av[2]; z[k][3] = x.w + av[3];
    sum += z[k][0] + z[k][1] + z[k][2] + z[k][3];
  }
  const float mean = warp_sum(sum) * (1.f / d);
  float var = 0.f;
#pragma unroll
  for (int k = 0; k < NV; k++)
#pragma unroll
    for (int e = 0; e < 4; e++) { const float t = z[k][e] - mean; var += t * t; }
  const float rstd = rsqrtf(warp_sum(var) * (1.f / d) + 1e-5f);
  if (lane == 0 && stats) stats[row] = make_float2(mean, rstd);
#pragma unroll
  for (int k = 0; k < NV; k++) {
    const int c = (lane + 32 * k) * 4;
    if (zsave) *(uint2*)(zsave + (long long)row * d + c) = make_uint2(pack_bf16x2(z[k][0], z[k][1]), pack_bf16x2(z[k][2], z[k][3]));
    const float4 ww = *(const float4*)(w + c), bb = *(const float4*)(b + c);
    float4 y;
    y.x = (z[k][0] - mean) * rstd * ww.x + bb.x; y.y = (z[k][1] - mean) * rstd * ww.y + bb.y;
    y.z = (z[k][2] - mean) * rstd * ww.z + bb.z; y.w = (z[k][3] - mean) * rstd * ww.w + bb.w;
    *(float4*)(x32 + (long long)row * d + c) = y;
    *(uint2*)(xa + (long long)row * d + c) = make_uint2(pack_bf16x2(y.x, y.y), pack_bf16x2(y.z, y.w));
  }
}

// LayerNorm backward; dy is overwritten by dz.  Each block walks rows with stride gridDim.x*8 and keeps per-lane column
// partials of dw / db, reduced over the block's 8 warps at the end and added to dw_out / db_out (one atomic per column and block).
template <int NV>
__global__ void __launch_bounds__(256) train_ln_bwd_kernel(float* __restrict__ dy, const bf16* __restrict__ dbr, const bf16* __restrict__ zsave,
                                                           const float2* __restrict__ stats, const float* __restrict__ w,
                                                           bf16* __restrict__ dadd, float* __restrict__ dw_out,
                                                           float* __restrict__ db_out, float* __restrict__ dsum_out, int rows,
                                                           uint32_t thresh, uint32_t seed, float scale) {
  constexpr int d = NV * 128;
  __shared__ float red[8][128];
  const int wp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float dw[NV][4], db[NV][4], ds[NV][4], wv[NV][4];   // ds: column sums of dadd = the bias gradient of the Linear whose output was added
#pragma unroll
  for (int k = 0; k < NV; k++) {
    const float4 ww = *(const float4*)(w + (lane + 32 * k) * 4);
    wv[k][0] = ww.x; wv[k][1] = ww.y; wv[k][2] = ww.z; wv[k][3] = ww.w;
#pragma unroll
    for (int e = 0; e < 4; e++) { dw[k][e] = 0.f; db[k][e] = 0.f; ds[k][e] = 0.f; }
  }
  for (int row = blockIdx.x * 8 + wp; row < rows; row += gridDim.x * 8) {
    const float2 st = stats[row];
    float g[NV][4], xh[NV][4];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int k = 0; k < NV; k++) {
      const int c = (lane + 32 * k) * 4;
      float4 y = *(const float4*)(dy + (long long)row * d + c);
      if (dbr) {   // branch gradient produced in bf16 by the preceding input-gradient GEMM
        const uint2 b2 = *(const uint2*)(dbr + (long long)row * d + c);
        y.x += bf16lo(b2.x); y.y += bf16hi(b2.x); y.z += bf16lo(b2.y); y.w += bf16hi(b2.y);
      }
      const uint2 z2 = *(const uint2*)(zsave + (long long)row * d + c);
      const float zz[4] = {bf16lo(z2.x), bf16hi(z2.x), bf16lo(z2.y), bf16hi(z2.y)};
      const float yy[4] = {y.x, y.y, y.z, y.w};
#pragma unroll
      for (int e = 0; e < 4; e++) {
        xh[k][e] = (zz[e] - st.x) * st.y;
        g[k][e] = yy[e] * wv[k][e];
        dw[k][e] += yy[e] * xh[k][e];
        db[k][e] += yy[e];
        s1 += g[k][e];
        s2 += g[k][e] * xh[k][e];
      }
    }
    s1 = warp_sum(s1) * (1.f / d);
    s2 = warp_sum(s2) * (1.f / d);
#pragma unroll
    for (int k = 0; k < NV; k++) {
      const int c = (lane + 32 * k) * 4;
      float dz[4];
#pragma unroll
      for (int e = 0; e < 4; e++) dz[e] = st.y * (g[k][e] - s1 - xh[k][e] * s2);
      *(float4*)(dy + (long long)row * d + c) = make_float4(dz[0], dz[1], dz[2], dz[3]);
      if (thresh) {
        float kp[4];
        keep4(seed, (uint32_t)(row * d + c), thresh, scale, kp);
        dz[0] *= kp[0]; dz[1] *= kp[1]; dz[2] *= kp[2]; dz[3] *= kp[3];
      }
      ds[k][0] += dz[0]; ds[k][1] += dz[1]; ds[k][2] += dz[2]; ds[k][3] += dz[3];
      *(uint2*)(dadd + (long long)row * d + c) = make_uint2(pack_bf16x2(dz[0], dz[1]), pack_bf16x2(dz[2], dz[3]));
    }
  }
  // block reduction of the column partials, 128 columns (one k) at a time
#pragma unroll
  for (int which = 0; which < 3; which++) {
    float* dst = which == 0 ? dw_out : (which == 1 ? db_out : dsum_out);
    if (dst == nullptr) continue;
#pragma unroll
    for (int k = 0; k < NV; k++) {
      __syncthreads();
#pragma unroll
      for (int e = 0; e < 4; e++) red[wp][lane * 4 + e] = which == 0 ? dw[k][e] : (which == 1 ? db[k][e] : ds[k][e]);
      __syncthreads();
      if (threadIdx.x < 128) {
        float s = 0.f;
#pragma unroll
        for (int q = 0; q < 8; q++) s += red[q][threadIdx.x];
        atomicAdd(dst + k * 128 + threadIdx.x, s);
      }
    }
  }
}

// column sums of a bf16 matrix: block = 256 threads x 2 columns, blockIdx.y = row chunk
__global__ void __launch_bounds__(256) train_colsum_kernel(const bf16* __restrict__ x, long long ld, int rows, int n,
                                                           float* __restrict__ dst) {
  const int c = (blockIdx.x * 256 + threadIdx.x) * 2;
  if (c >= n) return;
  const int chunk = (rows + gridDim.y - 1) / gridDim.y;
  const int r0 = blockIdx.y * chunk, r1 = min(rows, r0 + chunk);
  float s0 = 0.f, s1 = 0.f;
  for (int r = r0; r < r1; r++) {
    const uint32_t v = *(const uint32_t*)(x + (long long)r * ld + c);
    s0 += bf16lo(v); s1 += bf16hi(v);
  }
  atomicAdd(dst + c, s0);
  if (c + 1 < n) atomicAdd(dst + c + 1, s1);
}

// ------------------------------------------------------------------ loss
// MASKED: rows whose target is `ignore` get zero gradient and no loss; the others are scaled by 1 / count[0] (read on the device)
template <bool MASKED>
__global__ void __launch_bounds__(256) train_ce_kernel(const float* __restrict__ logits, long long ldl,
                                                       const long long* __restrict__ targets, bf16* __restrict__ dlogits,
                                                       float* __restrict__ loss_acc, int rows, int V, float gscale, long long ignore,
                                                       const float* __restrict__ count) {
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= rows) return;
  if (MASKED) {
    if (targets[row] == ignore) {
      bf16* dr = dlogits + (long long)row * ldl;
      for (int c = lane; c < (int)ldl; c += 32) dr[c] = __float2bfloat16_rn(0.f);
      return;
    }
    gscale = 1.f / count[0];                        // >= 1: this row counts
  }
  const float* lr = logits + (long long)row * ldl;
  float mx = -INFINITY;
  for (int c = lane; c < V; c += 32) mx = fmaxf(mx, lr[c]);
  mx = warp_max(mx);
  float se = 0.f;
  for (int c = lane; c < V; c += 32) se += __expf(lr[c] - mx);
  se = warp_sum(se);
  long long tg = targets[row];
  tg = tg < 0 ? 0 : (tg >= V ? V - 1 : tg);
  const float inv = 1.f / se;
  bf16* dr = dlogits + (long long)row * ldl;
  for (int c = lane; c < (int)ldl; c += 32) {
    float gq = 0.f;
    if (c < V) gq = (__expf(lr[c] - mx) * inv - (c == tg ? 1.f : 0.f)) * gscale;
    dr[c] = __float2bfloat16_rn(gq);
  }
  if (lane == 0) atomicAdd(loss_acc, mx + logf(se) - lr[tg]);
}

// number of targets != ignore, written to *count (one block)
__global__ void __launch_bounds__(256) train_count_kernel(const long long* __restrict__ targets, int rows, long long ignore,
                                                          float* __restrict__ count) {
  __shared__ int red[8];
  int n = 0;
  for (int r = threadIdx.x; r < rows; r += 256) n += targets[r] != ignore;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) n += __shfl_xor_sync(0xffffffffu, n, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = n;
  __syncthreads();
  if (threadIdx.x == 0) {
    int t = 0;
    for (int q = 0; q < 8; q++) t += red[q];
    *count = (float)t;
  }
}

// ------------------------------------------------------------------ validation metrics
// (value, index) order of torch.argmax: NaN above everything, then the larger value, then the lower index
__device__ __forceinline__ bool argmax_better(float v, int i, float bv, int bi) {
  const bool vn = isnan(v), bn = isnan(bv);
  if (vn != bn) return vn;
  if (vn || v == bv) return i < bi;
  return v > bv;
}

// One warp per row (rows strided over the grid in a fixed assignment): the first maximal index, then logsumexp.  Lane 0 of
// each warp sums its rows in row order; the block adds its 8 warps in order and writes (ce_sum, kept, correct) to part[block].
// No floating-point atomics: the result depends on the grid size only, which depends on `rows` only.
__global__ void __launch_bounds__(256) train_eval_metrics_kernel(const float* __restrict__ logits, long long ldl,
                                                                 const long long* __restrict__ targets, long long ignore, int rows,
                                                                 int V, double* __restrict__ part) {
  __shared__ double red[8][3];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double ce = 0.0, kept = 0.0, correct = 0.0;
  for (int row = blockIdx.x * 8 + warp; row < rows; row += gridDim.x * 8) {
    long long tg = targets[row];
    if (ignore >= 0 && tg == ignore) continue;
    tg = tg < 0 ? 0 : (tg >= V ? V - 1 : tg);      // as train_ce_kernel
    const float* lr = logits + (long long)row * ldl;
    float mx = -INFINITY;
    int am = 0x7fffffff;
#pragma unroll 4
    for (int c = lane; c < V; c += 32) {
      const float x = lr[c];
      if (argmax_better(x, c, mx, am)) { mx = x; am = c; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float omx = __shfl_xor_sync(0xffffffffu, mx, o);
      const int oam = __shfl_xor_sync(0xffffffffu, am, o);
      if (argmax_better(omx, oam, mx, am)) { mx = omx; am = oam; }
    }
    float se = 0.f;
#pragma unroll 4
    for (int c = lane; c < V; c += 32) se += expf(lr[c] - mx);
    se = warp_sum(se);
    if (lane == 0) {
      ce += (double)(mx - lr[tg]) + (double)logf(se);
      kept += 1.0;
      correct += am == (int)tg ? 1.0 : 0.0;
    }
  }
  if (lane == 0) { red[warp][0] = ce; red[warp][1] = kept; red[warp][2] = correct; }
  __syncthreads();
  if (threadIdx.x < 3) {
    double s = 0.0;
    for (int w = 0; w < 8; w++) s += red[w][threadIdx.x];
    part[blockIdx.x * 3 + threadIdx.x] = s;
  }
}

// out3 = the sums of the n partial triples, in a fixed order (one block)
__global__ void __launch_bounds__(96) train_eval_metrics_final_kernel(const double* __restrict__ part, int n, double* __restrict__ out3) {
  __shared__ double red[96];
  const int k = threadIdx.x % 3, j0 = threadIdx.x / 3;     // 32 strided lanes per quantity
  double s = 0.0;
  for (int j = j0; j < n; j += 32) s += part[j * 3 + k];
  red[threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.x < 3) {
    double t = 0.0;
    for (int j = 0; j < 32; j++) t += red[j * 3 + threadIdx.x];
    out3[threadIdx.x] = t;
  }
}

__device__ double g_eval_part[EVAL_PART_SLOTS * 3];   // scratch of the test entry dmg_eval_metrics: one per device, not reentrant

// dst[r, c] += src[r, c] (bf16, fp32 sum), n even
__global__ void __launch_bounds__(256) train_add_bf16_kernel(bf16* __restrict__ dst, long long ldd, const bf16* __restrict__ src,
                                                             long long lds, int rows, int n) {
  const int n2 = n >> 1;
  const long long tot = (long long)rows * n2;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < tot; i += (long long)gridDim.x * 256) {
    const long long r = i / n2;
    const int c = (int)(i % n2) * 2;
    uint32_t* dp = (uint32_t*)(dst + r * ldd + c);
    const uint32_t a = *dp, b = *(const uint32_t*)(src + r * lds + c);
    *dp = pack_bf16x2(bf16lo(a) + bf16lo(b), bf16hi(a) + bf16hi(b));
  }
}

__global__ void __launch_bounds__(256) train_rnn_dropout_kernel(const bf16* __restrict__ x, bf16* __restrict__ y, int B, int T, int d,
                                                                uint32_t thresh, uint32_t seed, float scale) {
  const int d4 = d >> 2;
  const long long n = (long long)B * T * d4;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256) {
    const int c = (int)(i % d4) * 4;
    const long long row = i / d4;
    const int b = (int)(row / T);
    const uint2 v = *(const uint2*)(x + row * d + c);
    float f[4] = {bf16lo(v.x), bf16hi(v.x), bf16lo(v.y), bf16hi(v.y)};
    if (thresh) {
      float k[4];
      keep4(seed, (uint32_t)(b * d + c), thresh, scale, k);
      f[0] *= k[0]; f[1] *= k[1]; f[2] *= k[2]; f[3] *= k[3];
    }
    *(uint2*)(y + row * d + c) = make_uint2(pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]));
  }
}

__global__ void __launch_bounds__(256) train_head_bwd_kernel(const bf16* __restrict__ dxd, const float* __restrict__ core,
                                                             float* __restrict__ dx32, int B, int T, int d, uint32_t thresh,
                                                             uint32_t seed, float scale, float ar_coef) {
  const int d4 = d >> 2;
  const long long n = (long long)B * T * d4;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256) {
    const int c = (int)(i % d4) * 4;
    const long long row = i / d4;
    const int b = (int)(row / T);
    const uint2 v = *(const uint2*)(dxd + row * d + c);
    float f[4] = {bf16lo(v.x), bf16hi(v.x), bf16lo(v.y), bf16hi(v.y)};
    if (thresh) {
      float k[4];
      keep4(seed, (uint32_t)(b * d + c), thresh, scale, k);
      f[0] *= k[0]; f[1] *= k[1]; f[2] *= k[2]; f[3] *= k[3];
    }
    const float4 co = *(const float4*)(core + row * d + c);
    *(float4*)(dx32 + row * d + c) =
        make_float4(f[0] + ar_coef * co.x, f[1] + ar_coef * co.y, f[2] + ar_coef * co.z, f[3] + ar_coef * co.w);
  }
}

__global__ void __launch_bounds__(256) train_sumsq_kernel(const float* __restrict__ x, long long n, float* __restrict__ acc) {
  __shared__ float red[8];
  float s = 0.f;
  const long long n4 = n >> 2;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n4; i += (long long)gridDim.x * 256) {
    const float4 v = ((const float4*)x)[i];
    s += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0)
    for (long long i = n4 * 4; i < n; i++) s += x[i] * x[i];
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float tsum = 0.f;
    for (int i = 0; i < 8; i++) tsum += red[i];
    atomicAdd(acc, tsum);
  }
}

// Deterministic two-stage sum of squares (the gradient norm that scales the Adam update): per-block partials in a fixed slot each,
// then one block adds them in a fixed order - every data-parallel rank derives bit-identical clipping from the same reduced gradient.
__global__ void __launch_bounds__(256) train_sumsq_part_kernel(const float* __restrict__ x, long long n, float* __restrict__ part) {
  __shared__ float red[8];
  float s = 0.f;
  const long long n4 = n >> 2;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n4; i += (long long)gridDim.x * 256) {
    const float4 v = ((const float4*)x)[i];
    s += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0)
    for (long long i = n4 * 4; i < n; i++) s += x[i] * x[i];
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float tsum = 0.f;
    for (int i = 0; i < 8; i++) tsum += red[i];
    part[blockIdx.x] = tsum;
  }
}
__global__ void __launch_bounds__(256) train_sumsq_final_kernel(const float* __restrict__ part, int n, float* __restrict__ out) {
  __shared__ float red[8];
  float s = 0.f;
  for (int i = threadIdx.x; i < n; i += 256) s += part[i];
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float tsum = 0.f;
    for (int i = 0; i < 8; i++) tsum += red[i];
    *out = tsum;
  }
}

__global__ void __launch_bounds__(256) train_tar_kernel(const bf16* __restrict__ h, long long bstride, int B, int n, int d,
                                                        float* __restrict__ acc) {
  __shared__ float red[8];
  float s = 0.f;
  const int d2 = d >> 1;
  const long long tot = (long long)B * (n - 1) * d2;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < tot; i += (long long)gridDim.x * 256) {
    const int c = (int)(i % d2) * 2;
    const long long r = i / d2;
    const int b = (int)(r / (n - 1)), t = (int)(r % (n - 1)) + 1;
    const bf16* p = h + (long long)b * bstride + (long long)t * d + c;
    const uint32_t x = *(const uint32_t*)p, y = *(const uint32_t*)(p - d);
    const float a0 = bf16lo(x) - bf16lo(y), a1 = bf16hi(x) - bf16hi(y);
    s += a0 * a0 + a1 * a1;
  }
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float tsum = 0.f;
    for (int i = 0; i < 8; i++) tsum += red[i];
    atomicAdd(acc, tsum);
  }
}

__global__ void __launch_bounds__(256) train_cast_kernel(const float* __restrict__ src, bf16* __restrict__ dst, long long n) {
  const long long n4 = n >> 2;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n4; i += (long long)gridDim.x * 256) {
    const float4 v = ((const float4*)src)[i];
    ((uint2*)dst)[i] = make_uint2(pack_bf16x2(v.x, v.y), pack_bf16x2(v.z, v.w));
  }
  if (blockIdx.x == 0 && threadIdx.x == 0)
    for (long long i = n4 * 4; i < n; i++) dst[i] = __float2bfloat16_rn(src[i]);
}

// bf16 -> fp32 (the gradient bucket coming back from the bf16 all-reduce)
__global__ void __launch_bounds__(256) train_uncast_kernel(const bf16* __restrict__ src, float* __restrict__ dst, long long n, int vec) {
  const long long n4 = vec ? (n >> 2) : 0;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n4; i += (long long)gridDim.x * 256) {
    const uint2 v = ((const uint2*)src)[i];
    ((float4*)dst)[i] = make_float4(__uint_as_float(v.x << 16), __uint_as_float(v.x & 0xffff0000u), __uint_as_float(v.y << 16),
                                    __uint_as_float(v.y & 0xffff0000u));
  }
  for (long long i = n4 * 4 + (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256)
    dst[i] = __bfloat162float(src[i]);
}
__global__ void __launch_bounds__(256) train_cast_scalar_kernel(const float* __restrict__ src, bf16* __restrict__ dst, long long n) {
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256) dst[i] = __float2bfloat16_rn(src[i]);
}

__global__ void __launch_bounds__(256) train_qpb_kernel(const bf16* __restrict__ qkv, long long ldx, const float* __restrict__ v,
                                                        bf16* __restrict__ out, int rows, int HD) {
  const int h2 = HD >> 1;
  const long long n = (long long)rows * h2;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256) {
    const int c = (int)(i % h2) * 2;
    const long long r = i / h2;
    const uint32_t q = *(const uint32_t*)(qkv + r * ldx + c);
    *(uint32_t*)(out + r * HD + c) = pack_bf16x2(bf16lo(q) + v[c], bf16hi(q) + v[c + 1]);
  }
}

// dst[b, :, :] = cat(src[b, M - keep :, :], x[b, T - take :, :]) with take = min(T, M), keep = M - take  (16-byte chunks)
__global__ void __launch_bounds__(256) train_mem_update_kernel(bf16* __restrict__ dst, const bf16* __restrict__ src,
                                                               const bf16* __restrict__ x, int B, int T, int M, int d) {
  const int d8 = d >> 3;
  const int take = T < M ? T : M, keep = M - take;
  const long long n = (long long)B * M * d8;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256) {
    const int c = (int)(i % d8) * 8;
    const long long r = i / d8;
    const int b = (int)(r / M), s = (int)(r % M);
    const bf16* from = s < keep ? src + ((long long)b * M + s + take) * d + c : x + ((long long)b * T + (T - take) + (s - keep)) * d + c;
    *(uint4*)(dst + r * d + c) = *(const uint4*)from;
  }
}

__global__ void __launch_bounds__(256) train_posenc_kernel(bf16* __restrict__ pe, int n, int d) {
  const int half = d >> 1;
  const long long tot = (long long)n * half;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < tot; i += (long long)gridDim.x * 256) {
    const int k = (int)(i % half), p = (int)(i / half);
    const float f = 1.f / powf(10000.f, (2.f * k) / d);
    const float a = p * f;
    pe[(long long)p * d + k] = __float2bfloat16_rn(sinf(a));
    pe[(long long)p * d + half + k] = __float2bfloat16_rn(cosf(a));
  }
}

// Multi-tensor Adam: one launch for every parameter tensor.  chunk c covers elements [start, start + len) of tensor
// desc[c].t; gradients / moments live in flat buffers at desc.off.
__global__ void __launch_bounds__(256) train_adam_kernel(const AdamTensor* __restrict__ tensors, const AdamChunk* __restrict__ chunks,
                                                         const float* __restrict__ G, float* __restrict__ M1, float* __restrict__ M2,
                                                         float lr, float beta1, float beta2, float eps, float wd, float bc1,
                                                         float bc2, float clip, const float* __restrict__ gnorm2, float gscale) {
  const AdamChunk ch = chunks[blockIdx.x];
  const AdamTensor tn = tensors[ch.t];
  float coef = gscale;
  if (clip > 0.f && gnorm2) {
    const float nrm = sqrtf(gnorm2[0]) * gscale;
    coef *= fminf(1.f, clip / (nrm + 1e-6f));
  }
  float* p = tn.p + ch.start;
  bf16* p16 = tn.p16 ? tn.p16 + ch.start : nullptr;
  const float* g = G + tn.off + ch.start;
  float* m1 = M1 + tn.off + ch.start;
  float* m2 = M2 + tn.off + ch.start;
  const float decay = 1.f - lr * wd, ib1 = 1.f / bc1, ib2 = 1.f / bc2;
  const int n4 = ch.len >> 2;                       // chunk starts are multiples of 4 and tensors are 16-byte aligned
  for (int i = threadIdx.x; i < n4; i += 256) {
    const float4 gr = ((const float4*)g)[i];
    float4 w = ((float4*)p)[i], a = ((float4*)m1)[i], b = ((float4*)m2)[i];
    float wv[4] = {w.x, w.y, w.z, w.w}, av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
    const float gv[4] = {gr.x * coef, gr.y * coef, gr.z * coef, gr.w * coef};
#pragma unroll
    for (int e = 0; e < 4; e++) {
      av[e] = beta1 * av[e] + (1.f - beta1) * gv[e];
      bv[e] = beta2 * bv[e] + (1.f - beta2) * gv[e] * gv[e];
      wv[e] = wv[e] * decay - lr * (av[e] * ib1) / (sqrtf(bv[e] * ib2) + eps);   // fastai true_wd: decay, then Adam
    }
    ((float4*)p)[i] = make_float4(wv[0], wv[1], wv[2], wv[3]);
    ((float4*)m1)[i] = make_float4(av[0], av[1], av[2], av[3]);
    ((float4*)m2)[i] = make_float4(bv[0], bv[1], bv[2], bv[3]);
    if (p16) ((uint2*)p16)[i] = make_uint2(pack_bf16x2(wv[0], wv[1]), pack_bf16x2(wv[2], wv[3]));
  }
  for (int i = n4 * 4 + threadIdx.x; i < ch.len; i += 256) {
    const float gr = g[i] * coef;
    const float a = beta1 * m1[i] + (1.f - beta1) * gr, b = beta2 * m2[i] + (1.f - beta2) * gr * gr;
    const float w = p[i] * decay - lr * (a * ib1) / (sqrtf(b * ib2) + eps);
    m1[i] = a; m2[i] = b; p[i] = w;
    if (p16) p16[i] = __float2bfloat16_rn(w);
  }
}

__global__ void __launch_bounds__(256) train_export_mask_kernel(float* __restrict__ out, long long n, uint32_t thresh, uint32_t seed,
                                                                float scale) {
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256)
    out[i] = drop_keep(seed, (uint32_t)i, thresh) ? scale : 0.f;
}

inline int grid_for(long long work_items, int cap = 148 * 16) {
  long long g = (work_items + 255) / 256;
  if (g < 1) g = 1;
  return (int)(g > cap ? cap : g);
}

}  // namespace

int train_embed(const long long* ids, const long long* pos, const float* emb, const float* beat, const float* bar, float* x32,
                bf16* xa, int rows, int d, int vocab, uint32_t thresh, uint32_t seed, float scale, cudaStream_t st) {
  return launch_np(train_embed_kernel, dim3(grid_for((long long)rows * d / 4)), dim3(256), 0, st, ids, pos, emb, beat, bar, x32, xa,
                   rows, d, vocab, thresh, seed, scale);
}

int train_embed_bwd(const long long* ids, const long long* pos, const float* dx, const bf16* dbr, float* demb, float* dbeat, float* dbar,
                    int rows, int d, int vocab, long long pad_idx, uint32_t thresh, uint32_t seed, float scale, cudaStream_t st) {
  return launch_np(train_embed_bwd_kernel, dim3(grid_for((long long)rows * d / 4)), dim3(256), 0, st, ids, pos, dx, dbr, demb, dbeat, dbar,
                   rows, d, vocab, pad_idx, thresh, seed, scale);
}

int train_residual_ln_fwd(float* x32, const bf16* add, const float* w, const float* b, bf16* xa, bf16* zsave, float2* stats,
                          int rows, int d, uint32_t thresh, uint32_t seed, float scale, cudaStream_t st) {
  const dim3 grid((rows + 7) / 8), block(256);
  switch (d / 128) {
    case 1: return launch_np(train_res_ln_fwd_kernel<1>, grid, block, 0, st, x32, add, w, b, xa, zsave, stats, rows, thresh, seed, scale);
    case 2: return launch_np(train_res_ln_fwd_kernel<2>, grid, block, 0, st, x32, add, w, b, xa, zsave, stats, rows, thresh, seed, scale);
    case 3: return launch_np(train_res_ln_fwd_kernel<3>, grid, block, 0, st, x32, add, w, b, xa, zsave, stats, rows, thresh, seed, scale);
    case 4: return launch_np(train_res_ln_fwd_kernel<4>, grid, block, 0, st, x32, add, w, b, xa, zsave, stats, rows, thresh, seed, scale);
    case 6: return launch_np(train_res_ln_fwd_kernel<6>, grid, block, 0, st, x32, add, w, b, xa, zsave, stats, rows, thresh, seed, scale);
    case 8: return launch_np(train_res_ln_fwd_kernel<8>, grid, block, 0, st, x32, add, w, b, xa, zsave, stats, rows, thresh, seed, scale);
  }
  DMG_CHECK(false, "training LayerNorm: d_model=%d unsupported (128, 256, 384, 512, 768, 1024)", d);
  return -2;
}

int train_ln_bwd(float* dy, const bf16* dbr, const bf16* zsave, const float2* stats, const float* w, bf16* dadd, float* dw, float* db,
                 float* dsum, int rows, int d, uint32_t thresh, uint32_t seed, float scale, cudaStream_t st) {
  int nblk = (rows + 7) / 8;
  if (nblk > 148 * 2) nblk = 148 * 2;
  const dim3 grid(nblk), block(256);
  switch (d / 128) {
    case 1: return launch_np(train_ln_bwd_kernel<1>, grid, block, 0, st, dy, dbr, zsave, stats, w, dadd, dw, db, dsum, rows, thresh, seed, scale);
    case 2: return launch_np(train_ln_bwd_kernel<2>, grid, block, 0, st, dy, dbr, zsave, stats, w, dadd, dw, db, dsum, rows, thresh, seed, scale);
    case 3: return launch_np(train_ln_bwd_kernel<3>, grid, block, 0, st, dy, dbr, zsave, stats, w, dadd, dw, db, dsum, rows, thresh, seed, scale);
    case 4: return launch_np(train_ln_bwd_kernel<4>, grid, block, 0, st, dy, dbr, zsave, stats, w, dadd, dw, db, dsum, rows, thresh, seed, scale);
    case 6: return launch_np(train_ln_bwd_kernel<6>, grid, block, 0, st, dy, dbr, zsave, stats, w, dadd, dw, db, dsum, rows, thresh, seed, scale);
    case 8: return launch_np(train_ln_bwd_kernel<8>, grid, block, 0, st, dy, dbr, zsave, stats, w, dadd, dw, db, dsum, rows, thresh, seed, scale);
  }
  DMG_CHECK(false, "training LayerNorm backward: d_model=%d unsupported", d);
  return -2;
}

int train_colsum_bf16(const bf16* x, long long ld, int rows, int n, float* dst, cudaStream_t st) {
  const int gx = (n + 511) / 512;
  int gy = (148 * 4 + gx - 1) / gx;
  if (gy > rows) gy = rows;
  if (gy < 1) gy = 1;
  return launch_np(train_colsum_kernel, dim3(gx, gy), dim3(256), 0, st, x, ld, rows, n, dst);
}

int train_ce_loss(const float* logits, long long ldl, const long long* targets, bf16* dlogits, float* loss_acc, int rows, int V,
                  float gscale, cudaStream_t st) {
  return launch_np(train_ce_kernel<false>, dim3((rows + 7) / 8), dim3(256), 0, st, logits, ldl, targets, dlogits, loss_acc, rows, V, gscale,
                   -1ll, (const float*)nullptr);
}

int train_ce_loss_masked(const float* logits, long long ldl, const long long* targets, long long ignore, bf16* dlogits, float* loss_acc,
                         float* count, int rows, int V, cudaStream_t st) {
  if (launch_np(train_count_kernel, dim3(1), dim3(256), 0, st, targets, rows, ignore, count)) return -1;
  return launch_np(train_ce_kernel<true>, dim3((rows + 7) / 8), dim3(256), 0, st, logits, ldl, targets, dlogits, loss_acc, rows, V, 0.f,
                   ignore, (const float*)count);
}

int train_eval_metrics(const float* logits, long long ldl, const long long* targets, long long ignore, int rows, int V, double* part,
                       double* out3, cudaStream_t st) {
  DMG_CHECK(logits && targets && out3 && rows >= 0 && V >= 1 && ldl >= V, "eval metrics: bad arguments (rows %d, V %d, ldl %lld)", rows,
            V, ldl);
  if (part == nullptr) DMG_CUDA_OK(cudaGetSymbolAddress((void**)&part, g_eval_part));
  int g = (rows + 7) / 8;
  if (g > EVAL_PART_SLOTS) g = EVAL_PART_SLOTS;
  if (g < 1) g = 1;
  if (launch_np(train_eval_metrics_kernel, dim3(g), dim3(256), 0, st, logits, ldl, targets, ignore, rows, V, part)) return -1;
  return launch_np(train_eval_metrics_final_kernel, dim3(1), dim3(96), 0, st, (const double*)part, g, out3);
}

int train_add_bf16(bf16* dst, long long ldd, const bf16* src, long long lds, int rows, int n, cudaStream_t st) {
  return launch_np(train_add_bf16_kernel, dim3(grid_for((long long)rows * n / 2)), dim3(256), 0, st, dst, ldd, src, lds, rows, n);
}

int train_rnn_dropout(const bf16* x, bf16* y, int B, int T, int d, uint32_t thresh, uint32_t seed, float scale, cudaStream_t st) {
  return launch_np(train_rnn_dropout_kernel, dim3(grid_for((long long)B * T * d / 4)), dim3(256), 0, st, x, y, B, T, d, thresh, seed, scale);
}

int train_head_bwd(const bf16* dxd, const float* core_out, float* dx32, int B, int T, int d, uint32_t thresh, uint32_t seed,
                   float scale, float ar_coef, cudaStream_t st) {
  return launch_np(train_head_bwd_kernel, dim3(grid_for((long long)B * T * d / 4)), dim3(256), 0, st, dxd, core_out, dx32, B, T, d,
                   thresh, seed, scale, ar_coef);
}

int train_sumsq(const float* x, long long n, float* acc, cudaStream_t st) {
  return launch_np(train_sumsq_kernel, dim3(grid_for(n / 4, 148 * 4)), dim3(256), 0, st, x, n, acc);
}

int train_sumsq_det(const float* x, long long n, float* part, int part_cap, float* out, cudaStream_t st) {
  int g = grid_for(n / 4, 148 * 4);
  if (g > part_cap) g = part_cap;
  if (launch_np(train_sumsq_part_kernel, dim3(g), dim3(256), 0, st, x, n, part)) return -1;
  return launch_np(train_sumsq_final_kernel, dim3(1), dim3(256), 0, st, (const float*)part, g, out);
}

int train_tar(const bf16* h, long long bstride, int B, int n, int d, float* acc, cudaStream_t st) {
  if (n < 2) return 0;
  return launch_np(train_tar_kernel, dim3(grid_for((long long)B * (n - 1) * d / 2, 148 * 4)), dim3(256), 0, st, h, bstride, B, n, d, acc);
}

int train_cast_bf16(const float* src, bf16* dst, long long n, cudaStream_t st) {
  return launch_np(train_cast_kernel, dim3(grid_for(n / 4)), dim3(256), 0, st, src, dst, n);
}

int train_grad_pack(const float* src, bf16* dst, long long n, cudaStream_t st) {
  if (n <= 0) return 0;
  if ((((uintptr_t)src) & 15) == 0 && (((uintptr_t)dst) & 7) == 0) return train_cast_bf16(src, dst, n, st);
  return launch_np(train_cast_scalar_kernel, dim3(grid_for(n)), dim3(256), 0, st, src, dst, n);
}
int train_grad_unpack(const bf16* src, float* dst, long long n, cudaStream_t st) {
  if (n <= 0) return 0;
  const int vec = (((uintptr_t)dst) & 15) == 0 && (((uintptr_t)src) & 7) == 0;
  return launch_np(train_uncast_kernel, dim3(grid_for(vec ? n / 4 + 1 : n)), dim3(256), 0, st, src, dst, n, vec);
}

int train_q_plus_bias(const bf16* qkv_x, long long ldx, const float* v, bf16* out, int rows, int HD, cudaStream_t st) {
  return launch_np(train_qpb_kernel, dim3(grid_for((long long)rows * HD / 2)), dim3(256), 0, st, qkv_x, ldx, v, out, rows, HD);
}

int train_mem_update(bf16* mem, const bf16* x, int B, int T, int M, int d, cudaStream_t st) {
  // in-place only when the whole memory is replaced (T >= M); train.cu double-buffers otherwise
  return launch_np(train_mem_update_kernel, dim3(grid_for((long long)B * M * d / 8)), dim3(256), 0, st, mem, (const bf16*)mem, x, B, T, M, d);
}
int train_mem_update2(bf16* dst, const bf16* src, const bf16* x, int B, int T, int M, int d, cudaStream_t st) {
  return launch_np(train_mem_update_kernel, dim3(grid_for((long long)B * M * d / 8)), dim3(256), 0, st, dst, src, x, B, T, M, d);
}

int train_posenc(bf16* pe, int n, int d, cudaStream_t st) {
  return launch_np(train_posenc_kernel, dim3(grid_for((long long)n * d / 2)), dim3(256), 0, st, pe, n, d);
}

int train_adam(const AdamTensor* tensors_dev, const AdamChunk* chunks_dev, int nchunks, const float* G, float* M1, float* M2, float lr,
               float beta1, float beta2, float eps, float wd, int step, float clip, const float* gnorm2, float gscale, cudaStream_t st) {
  const float bc1 = 1.f - powf(beta1, (float)step), bc2 = 1.f - powf(beta2, (float)step);
  return launch_np(train_adam_kernel, dim3(nchunks), dim3(256), 0, st, tensors_dev, chunks_dev, G, M1, M2, lr, beta1, beta2, eps, wd,
                   bc1, bc2, clip, gnorm2, gscale);
}

int train_export_mask(float* out, long long n, uint32_t thresh, uint32_t seed, float scale, cudaStream_t st) {
  return launch_np(train_export_mask_kernel, dim3(grid_for(n)), dim3(256), 0, st, out, n, thresh, seed, scale);
}

}  // namespace dmg
