// Small HBM-bound kernels around the GEMMs: embedding gather (+beat/bar), residual + LayerNorm, positional
// encoding table, memory-ring appends.  Vectorised 16-byte accesses, one warp per row, warp-shuffle reductions.
//
// Replaces (reference citations): self.encoder(x) + BeatPositionEncoder (deep_music_genre.py:1630, 1651-1665),
// TransformerEmbedding.forward (deep_music_remix.py:1926-1932), self.ln(x + ...) of the attention and FFN blocks
// (fastai MultiHeadAttention.forward / feed_forward; deep_music_remix.py:2052), PositionalEncoding (fastai),
// TransformerXL._update_mems (fastai; cat + slice every step -> ring append).
#include "kernels.cuh"
#include "launch.cuh"

namespace dmg {

// ------------------------------------------------------------------ embedding
template <class T>
__global__ void embed_kernel(const long long* __restrict__ ids, const long long* __restrict__ pos,
                             const float* __restrict__ emb, const float* __restrict__ beat,
                             const float* __restrict__ bar, float* __restrict__ x32, T* __restrict__ xa, int rows, int d,
                             int vocab) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  pdl_launch_dependents();
  pdl_wait();
  if (row >= rows) return;
  long long id = ids[row];
  if (id < 0) id = 0;
  if (id >= vocab) id = vocab - 1;
  const float4* e = (const float4*)(emb + (size_t)id * d);
  const float4 *be = nullptr, *ba = nullptr;
  if (pos != nullptr && beat != nullptr) {
    const long long p = pos[row];
    const long long bp = p & 31, br = (p >> 5) & 1023;   // p mod 32, floor(p / 32) mod 1024 (Python floor semantics, also for p < 0)
    be = (const float4*)(beat + (size_t)bp * d);
    ba = (const float4*)(bar + (size_t)br * d);
  }
  for (int c = lane; c < d / 4; c += 32) {
    float4 v = e[c];
    if (be) {
      float4 a = be[c], b = ba[c];
      v.x += a.x + b.x; v.y += a.y + b.y; v.z += a.z + b.z; v.w += a.w + b.w;
    }
    ((float4*)(x32 + (size_t)row * d))[c] = v;
    if ((void*)xa != (void*)x32) {
      T* o = xa + (size_t)row * d + c * 4;
      o[0] = from_f32<T>(v.x); o[1] = from_f32<T>(v.y); o[2] = from_f32<T>(v.z); o[3] = from_f32<T>(v.w);
    }
  }
}

template <class T>
int embed(const long long* ids, const long long* pos, const float* emb, const float* beat, const float* bar, float* x32,
          T* xa, int rows, int d, int vocab, cudaStream_t st) {
  if (rows <= 0) return 0;
  const int wpb = 8;
  return launch_k(embed_kernel<T>, dim3((rows + wpb - 1) / wpb), dim3(wpb * 32), 0, st, 1, ids, pos, emb, beat, bar, x32, xa, rows, d, vocab);
}
template int embed<float>(const long long*, const long long*, const float*, const float*, const float*, float*, float*,
                          int, int, int, cudaStream_t);
template int embed<bf16>(const long long*, const long long*, const float*, const float*, const float*, float*, bf16*, int,
                         int, int, cudaStream_t);

// ------------------------------------------------------------------ residual + LayerNorm (eps 1e-5), one warp per row
// d <= 1024, d % 128 == 0  (each lane owns d/128 float4 chunks, strided by 32)
template <class T, class TAdd, int NV>
__global__ void __launch_bounds__(256) residual_ln_kernel(float* __restrict__ x32, const TAdd* __restrict__ add,
                                                          const float* __restrict__ w, const float* __restrict__ b,
                                                          T* __restrict__ xa, int rows, int d) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  pdl_launch_dependents();
  pdl_wait();
  if (row >= rows) return;
  float v[NV * 4];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; i++) {
    const int c = (lane + 32 * i) * 4;
    float4 x = *(const float4*)(x32 + (size_t)row * d + c);
    const TAdd* ap = add + (size_t)row * d + c;
    v[4 * i + 0] = x.x + to_f32(ap[0]);
    v[4 * i + 1] = x.y + to_f32(ap[1]);
    v[4 * i + 2] = x.z + to_f32(ap[2]);
    v[4 * i + 3] = x.w + to_f32(ap[3]);
    s += v[4 * i] + v[4 * i + 1] + v[4 * i + 2] + v[4 * i + 3];
  }
  const float mean = warp_sum(s) / (float)d;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < NV * 4; i++) {
    const float t = v[i] - mean;
    q += t * t;
  }
  const float rstd = rsqrtf(warp_sum(q) / (float)d + 1e-5f);
#pragma unroll
  for (int i = 0; i < NV; i++) {
    const int c = (lane + 32 * i) * 4;
    const float4 ww = *(const float4*)(w + c), bb = *(const float4*)(b + c);
    float4 o;
    o.x = (v[4 * i + 0] - mean) * rstd * ww.x + bb.x;
    o.y = (v[4 * i + 1] - mean) * rstd * ww.y + bb.y;
    o.z = (v[4 * i + 2] - mean) * rstd * ww.z + bb.z;
    o.w = (v[4 * i + 3] - mean) * rstd * ww.w + bb.w;
    *(float4*)(x32 + (size_t)row * d + c) = o;
    if ((void*)xa != (void*)x32) {
      T* op = xa + (size_t)row * d + c;
      op[0] = from_f32<T>(o.x); op[1] = from_f32<T>(o.y); op[2] = from_f32<T>(o.z); op[3] = from_f32<T>(o.w);
    }
  }
}

template <class T, class TAdd>
int residual_layernorm(float* x32, const TAdd* add, const float* w, const float* b, T* xa, int rows, int d,
                       cudaStream_t st) {
  if (rows <= 0) return 0;
  DMG_CHECK(d % 128 == 0 && d <= 1024, "residual_layernorm: d_model=%d must be a multiple of 128 and <= 1024", d);
  const int wpb = 8;
  dim3 grid((rows + wpb - 1) / wpb), block(wpb * 32);
  switch (d / 128) {
#define DMG_LN_CASE(NV)                                                                                    \
  case NV:                                                                                                 \
    return launch_k(residual_ln_kernel<T, TAdd, NV>, grid, block, 0, st, 1, x32, add, w, b, xa, rows, d);
    DMG_LN_CASE(1) DMG_LN_CASE(2) DMG_LN_CASE(3) DMG_LN_CASE(4) DMG_LN_CASE(5) DMG_LN_CASE(6) DMG_LN_CASE(7) DMG_LN_CASE(8)
#undef DMG_LN_CASE
  }
  return 0;
}
template int residual_layernorm<float, float>(float*, const float*, const float*, const float*, float*, int, int, cudaStream_t);
template int residual_layernorm<bf16, float>(float*, const float*, const float*, const float*, bf16*, int, int, cudaStream_t);
template int residual_layernorm<bf16, bf16>(float*, const bf16*, const float*, const float*, bf16*, int, int, cudaStream_t);

// ------------------------------------------------------------------ positional encoding table
template <class T>
__global__ void posenc_kernel(T* __restrict__ pe, int n, int d) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const int half = d / 2;
  if (idx >= n * half) return;
  const int dist = idx / half, k = idx % half;
  // fastai: freq = 1 / (10000 ** (arange(0., d, 2.) / d)) in fp32; inp = outer(pos, freq)
  const float freq = 1.f / powf(10000.f, (float)(2 * k) / (float)d);
  const float x = (float)dist * freq;
  pe[(size_t)dist * d + k] = from_f32<T>(sinf(x));
  pe[(size_t)dist * d + half + k] = from_f32<T>(cosf(x));
}
template <class T>
int posenc_table(T* pe, int n, int d, cudaStream_t st) {
  const int total = n * (d / 2);
  posenc_kernel<T><<<(total + 255) / 256, 256, 0, st>>>(pe, n, d);
  g_launch_count++;
  DMG_CUDA_OK(cudaGetLastError());
  return 0;
}
template int posenc_table<float>(float*, int, int, cudaStream_t);
template int posenc_table<bf16>(bf16*, int, int, cudaStream_t);

template <class T>
__global__ void rd_relayout_kernel(const float* __restrict__ src, T* __restrict__ dst, int n, int H, int Dh) {
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t total = (size_t)n * H * Dh;
  if (idx >= total) return;
  const int e = idx % Dh;
  const int dist = (idx / Dh) % n;
  const int h = idx / ((size_t)Dh * n);
  dst[idx] = from_f32<T>(src[(size_t)dist * H * Dh + h * Dh + e]);
}
template <class T>
int rd_relayout(const float* src, T* dst, int n, int H, int Dh, cudaStream_t st) {
  const size_t total = (size_t)n * H * Dh;
  rd_relayout_kernel<T><<<(unsigned)((total + 255) / 256), 256, 0, st>>>(src, dst, n, H, Dh);
  g_launch_count++;
  DMG_CUDA_OK(cudaGetLastError());
  return 0;
}
template int rd_relayout<float>(const float*, float*, int, int, int, cudaStream_t);
template int rd_relayout<bf16>(const float*, bf16*, int, int, int, cudaStream_t);

template <class T>
__global__ void cast_kernel(const float* __restrict__ src, T* __restrict__ dst, long long n) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < n; i += stride) dst[i] = from_f32<T>(src[i]);
}
template <class T>
int cast_f32(const float* src, T* dst, long long n, cudaStream_t st) {
  if (n <= 0) return 0;
  long long blocks = (n + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  cast_kernel<T><<<(unsigned)blocks, 256, 0, st>>>(src, dst, n);
  g_launch_count++;
  DMG_CUDA_OK(cudaGetLastError());
  return 0;
}
template int cast_f32<float>(const float*, float*, long long, cudaStream_t);
template int cast_f32<bf16>(const float*, bf16*, long long, cudaStream_t);

template <class T>
__global__ void gather_rows_kernel(const T* __restrict__ src, T* __restrict__ dst, int rows, int d, int stride, int offset,
                                   const int* __restrict__ lens) {
  const int r = blockIdx.x;
  pdl_launch_dependents();
  pdl_wait();
  const T* s = src + ((size_t)r * stride + (lens ? lens[r] - 1 : offset)) * d;
  T* o = dst + (size_t)r * d;
  for (int c = threadIdx.x; c < d; c += blockDim.x) o[c] = s[c];
}
template <class T>
int gather_rows(const T* src, T* dst, int rows, int d, int stride, int offset, cudaStream_t st, const int* lens) {
  if (rows <= 0) return 0;
  return launch_k(gather_rows_kernel<T>, dim3(rows), dim3(128), 0, st, 1, src, dst, rows, d, stride, offset, lens);
}
template int gather_rows<float>(const float*, float*, int, int, int, int, cudaStream_t, const int*);
template int gather_rows<bf16>(const bf16*, bf16*, int, int, int, int, cudaStream_t, const int*);

// ------------------------------------------------------------------ memory rings
// K/V of the last min(len_b, M) new tokens of every stream -> ring slot (token index mod M).  Block x = the x-th of those tokens
// (blocks past min(len_b, M) of a shorter stream of a padded batch do nothing: padding rows never reach the ring).
// qkv row layout: [q (H*Dh) | k (H*Dh) | v (H*Dh)], ring layout [Bcap][H][M][Dh].
template <class T, class TS>
__global__ void ring_append_kv_kernel(const TS* __restrict__ qkv, T* __restrict__ kring, T* __restrict__ vring, int T_len,
                                      int H, int Dh, int M, const int* __restrict__ state, int state_stride,
                                      const int* __restrict__ lens, int b0) {
  // grid: (min(T_len, M), B); block: H*Dh/4 threads (each 4 elements)
  const int b = blockIdx.y;
  const int len = lens ? lens[b] : T_len;
  const int first = len > M ? len - M : 0;
  const int i = first + blockIdx.x;
  if (i >= len) return;
  const int HD = H * Dh;
  const int slot = (int)(((long long)state[(size_t)state_stride * (b0 + b)] + i) % M);
  const TS* row = qkv + ((size_t)b * T_len + i) * 3 * HD;
  for (int e = threadIdx.x * 4; e < HD; e += blockDim.x * 4) {
    const int h = e / Dh, c = e % Dh;
    const TS* kp = row + HD + e;
    const TS* vp = row + 2 * HD + e;
    const size_t o = (((size_t)(b0 + b) * H + h) * M + slot) * Dh + c;
#pragma unroll
    for (int q = 0; q < 4; q++) {
      kring[o + q] = from_f32<T>(to_f32(kp[q]));
      vring[o + q] = from_f32<T>(to_f32(vp[q]));
    }
  }
}
template <class T, class TS>
int ring_append_kv(const TS* qkv, T* kring, T* vring, int B, int T_len, int H, int Dh, int M, const int* state, int state_stride,
                   const int* lens, int b0, cudaStream_t st) {
  if (M <= 0 || B <= 0 || T_len <= 0) return 0;
  int threads = H * Dh / 4;
  if (threads > 256) threads = 256;
  ring_append_kv_kernel<T, TS><<<dim3(T_len < M ? T_len : M, B), threads, 0, st>>>(qkv, kring, vring, T_len, H, Dh, M, state,
                                                                                    state_stride, lens, b0);
  g_launch_count++;
  DMG_CUDA_OK(cudaGetLastError());
  return 0;
}
template int ring_append_kv<float, float>(const float*, float*, float*, int, int, int, int, int, const int*, int, const int*, int,
                                          cudaStream_t);
template int ring_append_kv<bf16, float>(const float*, bf16*, bf16*, int, int, int, int, int, const int*, int, const int*, int,
                                         cudaStream_t);
template int ring_append_kv<bf16, bf16>(const bf16*, bf16*, bf16*, int, int, int, int, int, const int*, int, const int*, int,
                                        cudaStream_t);

__global__ void ring_append_hidden_kernel(const float* __restrict__ x32, float* __restrict__ hring, int T_len, int d, int M,
                                          const int* __restrict__ state, int state_stride, const int* __restrict__ lens, int b0) {
  const int b = blockIdx.y;
  const int len = lens ? lens[b] : T_len;
  const int first = len > M ? len - M : 0;
  const int i = first + blockIdx.x;
  if (i >= len) return;
  const int slot = (int)(((long long)state[(size_t)state_stride * (b0 + b)] + i) % M);
  const float4* s = (const float4*)(x32 + ((size_t)b * T_len + i) * d);
  float4* o = (float4*)(hring + ((size_t)(b0 + b) * M + slot) * d);
  for (int c = threadIdx.x; c < d / 4; c += blockDim.x) o[c] = s[c];
}
int ring_append_hidden(const float* x32, float* hring, int B, int T_len, int d, int M, const int* state, int state_stride,
                       const int* lens, int b0, cudaStream_t st) {
  if (M <= 0 || B <= 0 || T_len <= 0) return 0;
  ring_append_hidden_kernel<<<dim3(T_len < M ? T_len : M, B), 128, 0, st>>>(x32, hring, T_len, d, M, state, state_stride, lens, b0);
  g_launch_count++;
  DMG_CUDA_OK(cudaGetLastError());
  return 0;
}

// out[b][j][:] = ring[b][slot(pos_total_b - mem_count + j)][:], j = 0..mem_count-1  (oldest first, like the reference)
__global__ void ring_export_hidden_kernel(const float* __restrict__ hring, float* __restrict__ out, int d, int M, int mem_count,
                                          const int* __restrict__ state, int state_stride) {
  const int j = blockIdx.x, b = blockIdx.y;
  const int slot = (int)(((long long)state[(size_t)state_stride * b] - mem_count + j) % M);
  const float4* s = (const float4*)(hring + ((size_t)b * M + slot) * d);
  float4* o = (float4*)(out + ((size_t)b * mem_count + j) * d);
  for (int c = threadIdx.x; c < d / 4; c += blockDim.x) o[c] = s[c];
}
int ring_export_hidden(const float* hring, float* out, int B, int d, int M, int mem_count, const int* state, int state_stride,
                       cudaStream_t st) {
  if (mem_count <= 0 || B <= 0) return 0;
  ring_export_hidden_kernel<<<dim3(mem_count, B), 128, 0, st>>>(hring, out, d, M, mem_count, state, state_stride);
  g_launch_count++;
  DMG_CUDA_OK(cudaGetLastError());
  return 0;
}

__global__ void state_advance_kernel(int* st, int n, int T_len, const int* __restrict__ lens, int M) {
  pdl_launch_dependents();
  pdl_wait();
  for (int b = threadIdx.x; b < n; b += blockDim.x) {
    const int len = lens ? lens[b] : T_len;
    st[2 * b] += len;
    const int m = st[2 * b + 1] + len;
    st[2 * b + 1] = m > M ? M : m;
  }
}
int state_advance(int* state, int n, int T_len, const int* lens, int M, cudaStream_t st) {
  if (n <= 0) return 0;
  return launch_k(state_advance_kernel, dim3(1), dim3(n < 256 ? (n + 31) / 32 * 32 : 256), 0, st, 1, state, n, T_len, lens, M);
}

}  // namespace dmg
