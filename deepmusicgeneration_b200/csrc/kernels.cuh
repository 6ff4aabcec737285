// Internal launcher declarations shared by the .cu files of libdmg_b200.so.
#pragma once
#include <vector>

#include "common.cuh"

namespace dmg {

extern long long g_launch_count;   // kernels launched by this library (process-wide)

// ------------------------------------------------------------------ GEMM: C[M,N] = A[M,K] * W[N,K]^T (+bias)(gelu)
// nn.Linear layout: both operands are K-major, which is what tcgen05 wants.
struct TensorMap2D {
  alignas(64) unsigned char bytes[128];   // CUtensorMap
};
// bf16 row-major [rows, cols] (row stride `ld` elements); box = [box_rows, 64 cols], 128B swizzle.
int make_tmap_bf16(TensorMap2D* out, const void* base, long long cols, long long rows, long long ld, int box_rows);
// same, any inner length (OOB box elements read as zero)
int make_tmap_bf16_ex(TensorMap2D* out, const void* base, long long inner, long long rows, long long ld, int box_rows);
// output map for TMA stores: 32 x 32 boxes, 64B swizzle
int make_tmap_bf16_store(TensorMap2D* out, const void* base, long long inner, long long rows, long long ld);

template <class T>
int gemm_simt(const T* A, int lda, const T* W, int ldw, const float* bias, void* C, int ldc, int M, int N, int K,
              int gelu, int out_bf16, cudaStream_t st);

// BN in {32, 128}; tmA box rows = 128, tmW box rows = BN. K % 64 == 0.
int gemm_tc(const TensorMap2D* tmA, const TensorMap2D* tmW, int BN, const float* bias, void* C, int ldc, int M, int N,
            int K, int gelu, int out_bf16, cudaStream_t st);
// Skinny-M variant: split-K over a 4- or 8-CTA cluster, partial tiles reduced through distributed shared memory.
// tmW32 = weight map with 32-row boxes.  gemm_tc_splitk_ways(K) == 0 -> shape not supported.
int gemm_tc_splitk_ways(int K);
int gemm_tc_splitk(const TensorMap2D* tmA, const TensorMap2D* tmW32, const float* bias, void* C, int ldc, int M, int N,
                   int K, int gelu, int out_bf16, cudaStream_t st);

// Fused one-token layer step (decode_layer.cu): out-projection + residual + LayerNorm + FFN (GeLU) + residual + LayerNorm + the
// next layer's q|k|v projection in ONE launch; a cluster of DL_CLUSTER CTAs owns DL_ROWS generation streams.
constexpr int DL_ROWS = 32, DL_CLUSTER = 8;
struct DecodeLayerArgs {
  float* x32;            // [rows, d] fp32 residual stream, in / out
  bf16* xa_out;          // [rows, d] bf16 copy of the final rows (input of the head GEMM) or NULL
  float* qkv;            // [rows, n3] fp32: the next layer's q|k|v (mode & 2)
  float* PP;             // scratch [DL_CLUSTER][pp_stride] fp32: the FFN-down partial sums of the 8 K slices, [row, d] each
  long long pp_stride;   // elements between two slabs of PP
  const float *bo, *b1, *b2, *bq;            // biases (any may be NULL)
  const float *ln1w, *ln1b, *ln2w, *ln2b;
  int row_base, B;       // rows [row_base, B) of the buffers belong to this launch (a stream lane of the step)
  int d, HD, di, n3;     // d_model, n_heads * d_head, d_inner, 3 * n_heads * d_head
  int mode;              // bit 0: the layer body (needs the attention output); bit 1: the next q|k|v projection
  unsigned long long* dbg = nullptr;   // optional timeline of CTA 0 (48 slots), see decode_layer.cu dl_mark
};
bool decode_layer_supported(int d, int HD, int di, int n3);
// tmAttn: DL_ROWS-row boxes over the attention output [rows, HD]; tmWo, tmW1, tmW2, tmWq: 64-row boxes
int decode_layer(const TensorMap2D* tmAttn, const TensorMap2D* tmWo, const TensorMap2D* tmW1, const TensorMap2D* tmW2,
                 const TensorMap2D* tmWq, const DecodeLayerArgs& a, cudaStream_t st);

struct AttnDecodeArgs;
// Dual-role launch (decode_layer.cu): the fused layer step of one half of the streams and the decode attention of the other half in
// ONE kernel (software pipeline over two halves of the batch, model.cu).
bool decode_dual_supported(int M);
int decode_dual_max_items(int attn_clusters);
bool attn_decode3_supported(int Dh, int M);
int decode_dual_max_clusters();      // clusters of 8 CTAs of that kernel that can be co-resident (15 on a B200)
int decode_dual(const TensorMap2D* tmAttn, const TensorMap2D* tmWo, const TensorMap2D* tmW1, const TensorMap2D* tmW2, const TensorMap2D* tmWq,
                const DecodeLayerArgs& fa, const TensorMap2D* tmK, const TensorMap2D* tmV, const TensorMap2D* tmR, const AttnDecodeArgs& aa,
                int b0, int attn_clusters, cudaStream_t st);

// ------------------------------------------------------------------ elementwise / small kernels
// x32[row] = emb[id] (+ beat[pos%32] + bar[min(pos/32 % 1024, 1023)]); xa = T(x32)
template <class T>
int embed(const long long* ids, const long long* pos, const float* emb, const float* beat, const float* bar, float* x32,
          T* xa, int rows, int d, int vocab, cudaStream_t st);

// x32 = LayerNorm(x32 + add) * w + b (eps 1e-5); xa = T(x32).  TAdd = float (GEMM output) or T (BERT: attention output)
template <class T, class TAdd>
int residual_layernorm(float* x32, const TAdd* add, const float* w, const float* b, T* xa, int rows, int d,
                       cudaStream_t st);

// PositionalEncoding table pe[dist][d] = cat(sin(dist*f), cos(dist*f)), f_k = 10000^(-2k/d); dist = 0..n-1
template <class T>
int posenc_table(T* pe, int n, int d, cudaStream_t st);

// [n, H*Dh] fp32 (GEMM output) -> [H][n][Dh] T   (rel-pos key cache layout)
template <class T>
int rd_relayout(const float* src, T* dst, int n, int H, int Dh, cudaStream_t st);

template <class T>
int cast_f32(const float* src, T* dst, long long n, cudaStream_t st);

// gather rows: dst[r] = src[idx(r)] with idx(r) = r*stride + offset, or r*stride + lens[r] - 1 where lens (device [rows]) is
// given   (last position of every stream)
template <class T>
int gather_rows(const T* src, T* dst, int rows, int d, int stride, int offset, cudaStream_t st, const int* lens = nullptr);

// ------------------------------------------------------------------ memory rings
// Device-side ring state, read by graph-captured kernels: one row {pos_total, mem_count} per stream (tokens appended since reset,
// valid memory positions <= M).  Kernels take it as (state, state_stride): stream s (absolute, as the ring index) reads
// state + state_stride * s - the model passes its [max_batch][2] array with stride 2, stride 0 gives every stream the same row.
// lens (device, indexed by the chunk-local stream b like the qkv rows) or NULL: stream b's segment is its first lens[b] of the T_len
// rows (a right-padded batch); NULL = all T_len.
// K/V of the last min(len_b, M) valid tokens of stream b into ring slots (pos_total_b + i) mod M
template <class T, class TS>
int ring_append_kv(const TS* qkv, T* kring, T* vring, int B, int T_len, int H, int Dh, int M, const int* state, int state_stride,
                   const int* lens, int b0, cudaStream_t st);
// hidden-state mems (model[0].hidden): ring [B][M][d] fp32
int ring_append_hidden(const float* x32, float* hring, int B, int T_len, int d, int M, const int* state, int state_stride,
                       const int* lens, int b0, cudaStream_t st);
// the last mem_count tokens of streams [0, B), which all hold that many
int ring_export_hidden(const float* hring, float* out, int B, int d, int M, int mem_count, const int* state, int state_stride,
                       cudaStream_t st);
// rows [0, n) of the model's state: pos_total += len_b, mem_count = min(mem_count + len_b, M); len_b = lens[b] or T_len
int state_advance(int* state, int n, int T_len, const int* lens, int M, cudaStream_t st);

// ------------------------------------------------------------------ attention
struct AttnGeneralArgs {
  const float* qkv;     // [rows, 3*H*Dh] fp32, row = b*T + i
  const void* kring;    // T [Bcap][H][M][Dh]
  const void* vring;
  const void* rd;       // T [H][Dcap][Dh] relative-position keys by distance
  const float* u;       // [H*Dh]
  const float* v;
  void* out;            // T [rows, H*Dh]
  int B, T, H, M, Dcap;
  const int* state;     // ring state of stream b0 + b at state + state_stride * (b0 + b): {pos_total, mem_count} (ring slot = token
  int state_stride;     // index mod M)
  int b0;               // first stream of this chunk (ring offset)
  int bert;             // 1: no mask, _line_shift wrap-around live (deep_music_remix.py:2096, r_mask=False)
  int win, k;           // window_mask (win_size, k); eval = (1, 1)
  float scale;          // 1/sqrt(Dh)
  const int* lens = nullptr;   // BERT only, device [B]: sequence b is rows [b*T, b*T + lens[b]) (T = the padded length); NULL = all T
};
template <class T>
int attn_general(const AttnGeneralArgs& a, cudaStream_t st);

// Tensor-core flash attention for memory-less segments (attention_flash.cu): Transformer-XL prefill after reset() (causal) and
// the BERT remix encoder (no mask, _line_shift wrap-around).  qkv: bf16 [B*T, 3*H*64]; rd: rel-pos key cache [H][Dcap][64].
int attn_flash(const bf16* qkv, const bf16* rd, int Dcap, const float* u, const float* v, bf16* out, int B, int T, int H, int bert,
               float scale, cudaStream_t st);

struct AttnDecodeArgs {
  const float* qkv;     // [B, 3*H*Dh] fp32 (the new token)
  bf16* kring;          // [Bcap][H][M][64]
  bf16* vring;
  const bf16* rd;       // [H][Dcap][64]
  const float* u;
  const float* v;
  bf16* out;            // [B, H*64]
  const int* state;     // ring state {pos_total, mem_count} of stream s (absolute: b0 + row) at state + state_stride * s
  int state_stride;
  int B, H, M, Dcap;
  float scale;
  unsigned long long* dbg = nullptr;   // timeline probe (third kernel, CTA 0 and the last CTA): [48] start, [49] table built, [50] end, [51] last CTA's end
  int force_v2 = 0;     // 1 = the second-generation kernel even where the third one applies (DMG_KF_ATTN_DECODE_V2, parity tests)
  int no_early_kv = 0;  // v2 kernel: 1 = request the first K/V tiles only after the predecessor kernel has finished (DMG_NO_EARLY_KV)
};
// BERT-encoder attention on tcgen05 (attention_bert_tc.cu): T >= 128; same contract as attn_flash(..., bert = 1, ...)
bool attn_bert_tc_supported(int T, int H, int Dcap);
// fp32_strip = 1: the first version of the strip skew (fp32 lines, 2.5 x the shared-memory wavefronts); kept for the parity tests
int attn_bert_tc(const bf16* qkv, const bf16* rd, int Dcap, const float* u, const float* v, bf16* out, int B, int T, int H, float scale,
                 int fp32_strip, cudaStream_t st);
// Per-sequence lengths (the batched remix): qkv / out are a padded batch, rows b*T_max + i, sequence b has lens_dev[b] tokens.  Both
// write only the rows < lens[b] of the sequences they cover.  attn_bert_tc_varlen walks the host-built item list items_dev[n_items]
// ((b << 16) | (h << 8) | 128-row query tile) of the sequences with lens >= 128; attn_flash_varlen the n_seqs sequences seqs_dev[]
// (max_len = the longest of them).
int attn_bert_tc_varlen(const bf16* qkv, const bf16* rd, int Dcap, const float* u, const float* v, bf16* out, const int* lens_dev,
                        const int* items_dev, int n_items, int B, int T_max, int H, float scale, int fp32_strip, cudaStream_t st);
int attn_flash_varlen(const bf16* qkv, const bf16* rd, int Dcap, const float* u, const float* v, bf16* out, const int* lens_dev,
                      const int* seqs_dev, int n_seqs, int max_len, int T_max, int H, float scale, cudaStream_t st);

// remix_batch.cu.  A padded batch of BERT sequences of their own lengths: lens (device [B]) and the host-built routing of
// bert_varlen_plan - the tcgen05 kernel's item list for the sequences of at least 128 tokens (use_tc), the mma.sync flash kernel for
// the others - so that every sequence runs on the kernel it would get alone.
struct VarlenPlan {
  const int* lens = nullptr;
  const int* tc_items = nullptr;
  int n_tc_items = 0;
  const int* fl_seqs = nullptr;
  int n_fl_seqs = 0, fl_max_len = 0;
};
void bert_varlen_plan(const int* lens_host, int B, int H, bool use_tc, std::vector<int>& tc_items, std::vector<int>& fl_seqs,
                      int* fl_max_len);
// both attention launches of the plan, then zeroes the output rows >= lens[b]
int attn_bert_varlen_bf16(const bf16* qkv, const bf16* rd, int Dcap, const float* u, const float* v, bf16* out, const VarlenPlan& p,
                          int B, int T_max, int H, float scale, int fp32_strip, cudaStream_t st);
template <class T>
int varlen_zero_rows(T* out, const int* lens_dev, int B, int T_max, int HD, cudaStream_t st);
// x_len == 1 over the bf16 ring: persistent, TMA-2D swizzled K/V tiles, resident rel-pos keys, mma.sync dot products
// (attention_decode2.cu).  tmK/tmV: ring viewed as [max_batch*H*M rows, 64 cols]; tmR: Rd viewed as [H*Dcap rows, 64 cols];
// 64-row boxes.
int attn_decode2(const TensorMap2D* tmK, const TensorMap2D* tmV, const TensorMap2D* tmR, const AttnDecodeArgs& a, int b0,
                 int num_sms, cudaStream_t st);
bool attn_decode2_supported(int Dh, int M);

}  // namespace dmg
