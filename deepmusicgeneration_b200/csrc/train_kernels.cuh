// Training-side launchers of libdmg_b200.so: persistent tcgen05 GEMM with fused epilogues, flash attention
// forward/backward with the Transformer-XL relative-position term, LayerNorm / dropout / loss / optimiser kernels.
// Replaces fastai's training step around the reference model (SURVEY.md 3.3, App. A.3/A.7): model(x) in train mode,
// CrossEntropyFlat + AR/TAR, backward, Adam.
#pragma once
#include "common.cuh"

namespace dmg {

// ------------------------------------------------------------------ counter-based dropout (all training kernels)
// One 32-bit hash per PAIR of neighbouring elements gives two 16-bit uniforms; keep <=> uniform >= thresh16
// (thresh16 = round(p * 65536)).  `seed` is already a per-(step, site, layer) hash made on the host, so masks are a
// pure function of (seed, element index): the backward pass and the tests regenerate them.
__host__ __device__ __forceinline__ uint32_t mix32(uint32_t x) {
  x ^= x >> 16; x *= 0x7feb352dU; x ^= x >> 15; x *= 0x846ca68bU; x ^= x >> 16;
  return x;
}
__host__ __device__ __forceinline__ uint32_t drop_pair_bits(uint32_t seed, uint32_t pair_idx) {
  return mix32(pair_idx ^ seed);
}
__host__ __device__ __forceinline__ bool drop_keep(uint32_t seed, uint32_t idx, uint32_t thresh16) {
  const uint32_t h = drop_pair_bits(seed, idx >> 1);
  return ((h >> ((idx & 1u) * 16u)) & 0xFFFFu) >= thresh16;
}
inline uint32_t drop_thresh16(float p) {
  int t = (int)(p * 65536.0f + 0.5f);
  return (uint32_t)(t < 0 ? 0 : (t > 65535 ? 65535 : t));
}
inline float drop_scale(float p) { return 1.0f / (1.0f - (float)drop_thresh16(p) / 65536.0f); }   // exact keep probability
uint32_t drop_seed(uint64_t base, uint64_t step, int site, int layer);

// d/dx of fastai's tanh-GeLU
__device__ __forceinline__ float gelu_tanh_grad(float x) {
  const float k = 0.7978845608028654f, c = 0.044715f;
  const float t = tanhf(k * (x + c * x * x * x));
  return 0.5f * (1.f + t) + 0.5f * x * (1.f - t * t) * k * (1.f + 3.f * c * x * x);
}

// single-instruction tanh (MUFU): abs error ~5e-4, used where the result is rounded to bf16 anyway
__device__ __forceinline__ float tanh_fast(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float gelu_tanh_fast(float x) {
  return 0.5f * x * (1.f + tanh_fast(0.7978845608028654f * (x + 0.044715f * x * x * x)));
}
__device__ __forceinline__ float gelu_tanh_grad_fast(float x) {
  const float k = 0.7978845608028654f, c = 0.044715f;
  const float t = tanh_fast(k * (x + c * x * x * x));
  return 0.5f * (1.f + t) + 0.5f * x * (1.f - t * t) * k * (1.f + 3.f * c * x * x);
}

// ------------------------------------------------------------------ persistent tcgen05 GEMM
// C[M,N] = A * B with the reduction over K; operand storage:
//   a_mn = 0: A is [M, K] row-major (K contiguous, "K-major")      a_mn = 1: A is [K, M] row-major ("MN-major")
//   b_mn = 0: B is [N, K] row-major (nn.Linear weight layout)      b_mn = 1: B is [K, N] row-major
// lda / ldb are row strides in elements (multiples of 8).  splitk > 1 requires out_mode = GEMM_OUT_ATOMIC.
enum { GEMM_OUT_F32 = 0, GEMM_OUT_BF16 = 1, GEMM_OUT_ATOMIC = 2 };
// act = 2 (GEMM_ACT_GELU_GRADSAVE): tanh-GeLU after the bias like act = 1, but the second output receives the BACKWARD
// factor gelu'(pre) * keep * drop_scale instead of the pre-activation (it is the only thing the backward needs the
// pre-activation for), so that the input-gradient GEMM's epilogue is one multiply (GEMM_AUX_MUL_BF16): no tanh, no dropout hash.
enum { GEMM_ACT_NONE = 0, GEMM_ACT_GELU = 1, GEMM_ACT_GELU_GRADSAVE = 2 };
enum { GEMM_AUX_NONE = 0,
       GEMM_AUX_GELU_GRAD = 1,   // value *= gelu'(aux[m,n])                 (aux bf16: the saved pre-activation)
       GEMM_AUX_ADD_BF16 = 2,    // value += aux[m,n]                        (bf16 residual)
       GEMM_AUX_ADD_F32 = 3,     // value += aux[m,n]                        (fp32 residual)
       GEMM_AUX_MUL_BF16 = 4 };  // value *= aux[m,n]                        (bf16: a saved gradient factor)
struct GemmEpi {
  const float* bias = nullptr;   // [N]
  int act = 0;                   // 1: tanh-GeLU after the bias
  const void* aux = nullptr;
  long long ld_aux = 0;
  int aux_mode = GEMM_AUX_NONE;
  void* out = nullptr;
  long long ldc = 0;
  int out_mode = GEMM_OUT_F32;
  bf16* out2 = nullptr;          // optional: value before act / aux / dropout (bf16), e.g. the FFN pre-activation
  long long ld2 = 0;
  uint32_t drop_thresh = 0;      // dropout applied last (after act / aux): 0 = none
  uint32_t drop_seed = 0;
  float drop_scale = 1.f;
  // grouped launch: `groups` independent problems of the same shape in one grid; group g reads A at M-coordinate
  // g*a_gs, B at N-coordinate g*b_gs and writes at column offset g*c_gs (the per-head dRk contraction)
  int groups = 1;
  long long a_gs = 0, b_gs = 0, c_gs = 0;
};
int gemm_bf16_tc(const bf16* A, int a_mn, long long lda, const bf16* B, int b_mn, long long ldb, int M, int N, int K,
                 int splitk, const GemmEpi& e, int num_sms, cudaStream_t st);

// ------------------------------------------------------------------ flash attention with the rel-pos term (training)
struct AttnTrainArgs {
  // current-segment projections [B*T rows, ldx] bf16: q at col 0, k at col HD, v at col 2*HD (head h at +h*64)
  const bf16* qkv_x; long long ldx;
  // memory projections [B*M rows, ldm] bf16: k at col 0, v at col HD; only the last mem_count rows of each stream are valid
  const bf16* kv_m; long long ldm;
  const bf16* rk;        // [S = M+T rows, HD] bf16: r_attn(PositionalEncoding(dist)), row = distance
  const float* u;        // [HD]
  const float* v;
  bf16* out;             // [B*T, HD]
  float* lse;            // [B, H, T] log-sum-exp of the scaled, masked scores
  int B, T, H, M, mem_count;
  int win, k;            // window_mask (win_size, k)
  float scale;
  uint32_t drop_thresh, drop_seed; float drop_scale;   // attention dropout (on the probabilities)
  // Optional (tcgen05 forward only; both or neither): the forward saves the UNdropped probabilities of every visited tile,
  // p_save[b*H+h][i][j] = exp((score - m)*scale) in bf16 relative to the running row maximum m of its 64-key column block
  // at that time, m_save[b*H+h][i][j/64] = that maximum (raw score units).  The backward then rebuilds
  // P = p_save * exp(m_save*scale - lse) instead of recomputing AC, BD, the skew and the exponentials.
  bf16* p_save = nullptr;   // [B*H, T, M+T]
  float* m_save = nullptr;  // [B*H, T, (M+T)/64]
  // Optional, with p_save: the forward also stores its (q+u) and (q+v) tiles, [B*T, HD] bf16 each - the operands of the
  // dK contraction (tcgen05 dK/dV kernel) and of the dRk GEMM in the backward
  bf16* qu_save = nullptr;
  bf16* qv_save = nullptr;
  // inference engine (attn_fwd_tc_ring): memory keys / values in per-head rings, relative-position keys in the per-head Rd cache
  int ring_head = 0, ring_b0 = 0, ring_dcap = 0;
};
int attn_train_fwd(const AttnTrainArgs& a, cudaStream_t st);
// tcgen05 / TMEM / TMA forward (attention_train_tc.cu): T, M, mem_count multiples of 128; attn_train_fwd dispatches to it
bool attn_train_fwd_tc_supported(const AttnTrainArgs& a);
int attn_train_fwd_tc(const AttnTrainArgs& a, cudaStream_t st);
bool attn_fwd_tc_ring_supported(int T, int Dh, int M, int mem_count, int pos_total);
int attn_fwd_tc_ring(const bf16* qkv16, const bf16* kring, const bf16* vring, const bf16* rd, int Dcap, const float* u, const float* v,
                     bf16* out, int B, int T, int H, int M, int mem_count, int win, int k, int pos_total, int b0, int max_batch, float scale,
                     cudaStream_t st);
struct AttnTrainBwdArgs;
bool attn_bwd_dkv_tc_supported(const AttnTrainBwdArgs& ba);
// dQ (+ the P / dS tiles and dS in distance coordinates) on tcgen05 from the saved probabilities; same shapes as the dK/dV kernel
bool attn_bwd_dq_tc_supported(const AttnTrainBwdArgs& ba);
int attn_bwd_dq_tc(const AttnTrainBwdArgs& ba, cudaStream_t st);
int attn_bwd_dkv_tc(const AttnTrainBwdArgs& ba, cudaStream_t st);
struct TensorMap2D;
int train_get_tmap(const void* base, long long inner, long long rows, long long ld, int box_rows, const TensorMap2D** out);

struct AttnTrainBwdArgs {
  AttnTrainArgs f;       // the forward arguments (out = the saved forward output)
  const bf16* dout;      // [B*T, HD]
  float* delta;          // [B, H, T] workspace: rowsum(dout * out)
  bf16* dqkv_x;          // [B*T, ldx]: dq | dk | dv of the current segment
  bf16* dkv_m;           // [B*M, ldm]: dk | dv of the memory rows
  bf16* ds_dist;         // [B*T, H*S] bf16: dS in (row, distance) coordinates (zero where masked), for the dRk GEMM
  bf16* qv;              // [B*T, HD] bf16: q + v (operand of the dRk GEMM)
  float* du;             // [HD] accumulated (atomics)
  float* dv;             // [HD]
  const bf16* qu = nullptr; // optional [B*T, HD] bf16: q + u; with p_buf / ds_buf and T, M, mem_count multiples of 128 it selects the
                            // tcgen05 dK/dV kernel (attention_train_tc.cu)
  bf16* p_buf = nullptr;   // optional workspaces [B*H, T, M+T] bf16: when both are set the dQ kernel spills the dropped
  bf16* ds_buf = nullptr;  // probabilities and dS there and dK/dV come from a kernel that does not recompute the scores
};
int attn_train_bwd(const AttnTrainBwdArgs& a, int num_sms, cudaStream_t st);
// pieces of attn_train_bwd that the remix encoder's backward reuses: delta = rowsum(dO * O); dK / dV from the spilled P / dS
// tiles with every query tile seeing every key (M = 0, p_buf and ds_buf set)
int attn_train_delta(const AttnTrainBwdArgs& ba, cudaStream_t st);
int attn_bwd_dkv_all_queries(const AttnTrainBwdArgs& ba, cudaStream_t st);
// remix (masked-BERT) encoder attention for training (attention_bert_train.cu): no memory, no mask, _line_shift wrap-around
// live (lines 1 and 3), T a multiple of 64.  Rk ([T, HD], row = distance) must read as zero for rows -64 .. T+127 and qkv_x
// needs one readable row past the last stream.  The backward writes the content part of dq (+ du), dk, dv, ds_dist and the
// P / dS spill (p_buf / ds_buf, required); the position part of dq is ds_dist . Rk (the trainer's per-head GEMMs).
int attn_bert_train_fwd(const AttnTrainArgs& a, cudaStream_t st);
int attn_bert_train_bwd(const AttnTrainBwdArgs& ba, cudaStream_t st);

// ------------------------------------------------------------------ elementwise / reductions (train_kernels.cu)
// x32 = emb[id] (+beat+bar) with embedding dropout; xa = bf16(x32)
int train_embed(const long long* ids, const long long* pos, const float* emb, const float* beat, const float* bar,
                float* x32, bf16* xa, int rows, int d, int vocab, uint32_t thresh, uint32_t seed, float scale,
                cudaStream_t st);
// z = x32 + dropout(add); save zsave = bf16(z), stats = (mean, rstd); x32 = LN(z)*w+b; xa = bf16(x32)
int train_residual_ln_fwd(float* x32, const bf16* add, const float* w, const float* b, bf16* xa, bf16* zsave,
                          float2* stats, int rows, int d, uint32_t thresh, uint32_t seed, float scale, cudaStream_t st);
// LayerNorm backward: incoming gradient = dy (fp32 [rows,d]) + dbr (bf16 [rows,d] or NULL: the branch gradient a preceding
// input-gradient GEMM produced); dy is overwritten by dz = gradient wrt z, which is also the residual-branch
// gradient); dadd = bf16(dropout_mask * scale * dz) (gradient wrt the GEMM output that was added);
// dw[d] / db[d] += the affine-parameter gradients (one atomic per column and block).
// dsum (may be NULL) += column sums of dadd: the bias gradient of the Linear whose output entered the residual sum.
int train_ln_bwd(float* dy, const bf16* dbr, const bf16* zsave, const float2* stats, const float* w, bf16* dadd, float* dw, float* db,
                 float* dsum, int rows, int d, uint32_t thresh, uint32_t seed, float scale, cudaStream_t st);
int train_partial_finish(const float* partial, int nblk, int n, float* dst0, float* dst1, cudaStream_t st);   // dst += sums
// column sums of a bf16 matrix [rows, n] (row stride ld) added into dst[n] (bias gradients)
int train_colsum_bf16(const bf16* x, long long ld, int rows, int n, float* dst, cudaStream_t st);
// column sums of a fp32 matrix, added into dst (du/dv from dq accumulators are not needed: attention does them)
// head: logits fp32 [rows, ldl] -> per-row CE loss (sum into loss_acc[0]) and dlogits bf16 [rows, ldl] = (softmax - onehot) * gscale
int train_ce_loss(const float* logits, long long ldl, const long long* targets, bf16* dlogits, float* loss_acc,
                  int rows, int V, float gscale, cudaStream_t st);
// CrossEntropyFlat(ignore_index=ignore): *count (device) = number of targets != ignore, counted on the device; rows with the
// ignore target get no loss and zero dlogits, the others (softmax - onehot) / count.  loss_acc / count is the mean (NaN at count 0).
int train_ce_loss_masked(const float* logits, long long ldl, const long long* targets, long long ignore, bf16* dlogits, float* loss_acc,
                         float* count, int rows, int V, cudaStream_t st);
// output (RNN) dropout of the head input: xd[b,t,:] = xa[b,t,:] * mask[b,:]   (one mask per stream and feature)
int train_rnn_dropout(const bf16* x, bf16* y, int B, int T, int d, uint32_t thresh, uint32_t seed, float scale,
                      cudaStream_t st);
// dx32[b,t,:] (fp32) = dxd (bf16) * mask[b,:] + ar_coef * core_out   (head-input gradient + activation regulariser)
int train_head_bwd(const bf16* dxd, const float* core_out, float* dx32, int B, int T, int d, uint32_t thresh,
                   uint32_t seed, float scale, float ar_coef, cudaStream_t st);
// sum of squares of a fp32 buffer into acc[slot] (AR term, gradient norm)
int train_sumsq(const float* x, long long n, float* acc, cudaStream_t st);
// out = sum of squares, summed in a fixed order (part: scratch of part_cap floats)
int train_sumsq_det(const float* x, long long n, float* part, int part_cap, float* out, cudaStream_t st);
// TAR value: sum over b, t>=1 of (h[b,t]-h[b,t-1])^2 for h = bf16 [B, n, d] with stream stride bstride elements
int train_tar(const bf16* h, long long bstride, int B, int n, int d, float* acc, cudaStream_t st);
// embedding backward: demb[id] += mask * scale * (dx + dbr) (atomics) except for id == pad_idx (-1: none); beat/bar likewise
// when pos != NULL (their row 0 is a padding row)
int train_embed_bwd(const long long* ids, const long long* pos, const float* dx, const bf16* dbr, float* demb, float* dbeat, float* dbar,
                    int rows, int d, int vocab, long long pad_idx, uint32_t thresh, uint32_t seed, float scale, cudaStream_t st);
// dst[rows, n] += src (bf16, row strides ldd / lds)
int train_add_bf16(bf16* dst, long long ldd, const bf16* src, long long lds, int rows, int n, cudaStream_t st);
// fp32 [rows, d] -> bf16
int train_cast_bf16(const float* src, bf16* dst, long long n, cudaStream_t st);
// gradient bucket <-> its bf16 wire format (any alignment)
int train_grad_pack(const float* src, bf16* dst, long long n, cudaStream_t st);
int train_grad_unpack(const bf16* src, float* dst, long long n, cudaStream_t st);
// q + v -> bf16 [rows, HD]   (q = qkv_x columns [0, HD))
int train_q_plus_bias(const bf16* qkv_x, long long ldx, const float* v, bf16* out, int rows, int HD, cudaStream_t st);
// memory update of the training state: mem = cat(mem, x)[:, -M:]  (bf16 hidden states, right-aligned)
int train_mem_update(bf16* mem, const bf16* x, int B, int T, int M, int d, cudaStream_t st);
int train_mem_update2(bf16* dst, const bf16* src, const bf16* x, int B, int T, int M, int d, cudaStream_t st);   // dst != src
// PositionalEncoding table in bf16 [n, d]
int train_posenc(bf16* pe, int n, int d, cudaStream_t st);
// fused multi-tensor Adam (decoupled weight decay first - fastai true_wd -, bias correction): ONE launch for all
// parameter tensors; gradients are multiplied by grad_scale * min(1, clip / ||grad_scale * g||) with ||g||^2 read from
// gnorm2[0] on the device; refreshes the bf16 copies.  chunks: <= 16384 elements each, starts multiples of 4.
struct AdamTensor { float* p; bf16* p16; long long off; };
struct AdamChunk { int t; int start; int len; };
int train_adam(const AdamTensor* tensors_dev, const AdamChunk* chunks_dev, int nchunks, const float* G, float* M1, float* M2, float lr,
               float beta1, float beta2, float eps, float wd, int step, float clip, const float* gnorm2, float gscale, cudaStream_t st);
// dropout mask export for the tests: out[i] = keep(seed, i) ? scale : 0
int train_export_mask(float* out, long long n, uint32_t thresh, uint32_t seed, float scale, cudaStream_t st);

}  // namespace dmg
