// libdmg_b200.so: model object, weight registry, forward orchestration, device generation loop, C ABI.
// See include/dmg_b200.h for the contract and the reference call each entry point stands behind.
#include <cstdarg>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "model.cuh"
#include "launch.cuh"
#include "train_kernels.cuh"

namespace dmg {

static thread_local char g_err[1024] = "";
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

}  // namespace dmg

using namespace dmg;

namespace dmg {


static int alloc_weight(dmg_model* m, Weight& w, int rows, int cols, const std::string& name) {
  w.rows = rows;
  w.cols = cols;
  if (dalloc(m, &w.f32, (size_t)rows * cols)) return -1;
  if (m->is_bf16 && dalloc(m, &w.b16, (size_t)rows * cols)) return -1;
  if (!name.empty()) m->reg[name] = {w.f32, (long long)rows * cols};
  return 0;
}
static int alloc_vec(dmg_model* m, float** p, int n, const std::string& name) {
  if (dalloc(m, p, (size_t)n)) return -1;
  m->reg[name] = {*p, n};
  return 0;
}

// C[M,N] = A * W^T (+bias)(gelu) with A one of the model's activation buffers
static int linear(dmg_model* m, int abuf, const void* A, const Weight& w, const float* bias, void* C, int ldc, int M,
                  int gelu, int out_bf16, cudaStream_t st) {
  const int N = w.rows, K = w.cols;
  if (!m->is_bf16) return gemm_simt<float>((const float*)A, K, w.f32, K, bias, C, ldc, M, N, K, gelu, out_bf16, st);
  if (m->use_tc && w.has_tm && K % 64 == 0) {
    const bool skinny = M <= 512;
    // many rows (prefill segments, the BERT encoder): the persistent CTA-pair kernel of the training path (gemm_train.cu) -
    // 256-row tiles, TMA-store epilogue.  Measured at C4 (32768 rows, QKV 512 -> 1536): 307 us with gemm_tc_kernel<128> = 168
    // TFLOP/s; the same shape runs at ~800 TFLOP/s there.
    if (!(m->kflags & DMG_KF_NO_BIG_GEMM) && M >= 1024 && N % 4 == 0 && (out_bf16 ? ldc % 8 == 0 : ldc % 4 == 0)) {
      GemmEpi e;
      e.bias = bias; e.act = gelu ? GEMM_ACT_GELU : GEMM_ACT_NONE; e.out = C; e.ldc = ldc;
      e.out_mode = out_bf16 ? GEMM_OUT_BF16 : GEMM_OUT_F32;
      return gemm_bf16_tc((const bf16*)A, 0, K, w.b16, 0, K, M, N, K, 1, e, m->num_sms, st);
    }
    if (skinny && gemm_tc_splitk_ways(K) && !(m->kflags & DMG_KF_NO_SPLITK))
      return gemm_tc_splitk(&m->tmA[abuf], &w.tm32, bias, C, ldc, M, N, K, gelu, out_bf16, st);
    return gemm_tc(&m->tmA[abuf], skinny ? &w.tm32 : &w.tm128, skinny ? 32 : 128, bias, C, ldc, M, N, K, gelu, out_bf16, st);
  }
  return gemm_simt<bf16>((const bf16*)A, K, w.b16, K, bias, C, ldc, M, N, K, gelu, out_bf16, st);
}

// The launches of the one-token step (product path) over the streams [b0, b0 + nb) of the model: the fused layer step of layer l
// over rows [r0, r1) (l == 0 ... L: body of layer l-1, q|k|v of layer l), the decode attention of layer l over the same kind of row
// range, and the dual-role launch that runs one of each (for different halves of the streams) side by side.
struct DecodeStep {
  dmg_model* m;
  int b0;
  cudaStream_t st;

  DecodeLayerArgs layer_args(int l, int r0, int r1, LayerW** Lb_out, LayerW** Ln_out) const {
    const dmg_config& c = m->cfg;
    const bool body = l > 0, next = l < c.n_layers;
    LayerW& Lb = m->layers[body ? l - 1 : 0];        // the layer whose body runs
    LayerW& Ln = m->layers[next ? l : 0];            // the layer whose q|k|v are produced
    DecodeLayerArgs da;
    da.x32 = m->x32; da.qkv = m->qkv; da.PP = m->dl_PP; da.pp_stride = m->dl_pp_stride;
    da.row_base = r0; da.B = r1; da.d = c.d_model; da.HD = m->HD; da.di = c.d_inner; da.n3 = 3 * m->HD;
    da.mode = (body ? 1 : 0) | (next ? 2 : 0);
    da.dbg = (l == c.n_layers / 2 && r0 == 0) ? m->dl_dbg : nullptr;      // timeline probe: one mid-stack launch
    da.xa_out = next ? nullptr : (bf16*)m->xa;
    da.bo = Lb.bo; da.b1 = Lb.b1; da.b2 = Lb.b2; da.ln1w = Lb.ln1w; da.ln1b = Lb.ln1b; da.ln2w = Lb.ln2w; da.ln2b = Lb.ln2b;
    da.bq = Ln.bqkv;
    *Lb_out = &Lb; *Ln_out = &Ln;
    return da;
  }
  AttnDecodeArgs attn_args(int l, int r0, int r1) const {
    const dmg_config& c = m->cfg;
    const int M = c.mem_len, HD = m->HD;
    LayerW& La = m->layers[l];
    AttnDecodeArgs a;
    a.qkv = m->qkv + (size_t)r0 * 3 * HD;
    a.kring = (bf16*)La.kring + (size_t)(b0 + r0) * c.n_heads * M * 64;
    a.vring = (bf16*)La.vring + (size_t)(b0 + r0) * c.n_heads * M * 64;
    a.rd = (const bf16*)La.rd;
    a.u = m->u; a.v = m->v;
    a.out = (bf16*)m->attn + (size_t)r0 * HD;
    a.dev_state = m->dev_state;
    a.B = r1 - r0; a.H = c.n_heads; a.M = M; a.Dcap = m->Dcap;
    a.scale = 1.f / sqrtf((float)c.d_head);
    a.force_v2 = (m->kflags & DMG_KF_ATTN_DECODE_V2) ? 1 : 0;
    return a;
  }
  int fused_alone(int l, int r0, int r1) const {
    LayerW *Lb, *Ln;
    const DecodeLayerArgs da = layer_args(l, r0, r1, &Lb, &Ln);
    return decode_layer(&m->tmAttn16, &Lb->wo.tm64, &Lb->w1.tm64, &Lb->w2.tm64, &Ln->wqkv.tm64, da, st);
  }
  int attn_alone(int l, int r0, int r1) const {
    LayerW& La = m->layers[l];
    return attn_decode2(&La.tmK, &La.tmV, &La.tmR, attn_args(l, r0, r1), b0 + r0, m->num_sms, st);
  }
  // dual-role launch: fused step `lf` over rows [f0, f1) together with the attention of layer `la` over rows [a0, a1)
  int dual(int lf, int f0, int f1, int la, int a0, int a1) const {
    LayerW *Lb, *Ln;
    const DecodeLayerArgs da = layer_args(lf, f0, f1, &Lb, &Ln);
    LayerW& La = m->layers[la];
    const int n_fused = (f1 - f0 + DL_ROWS - 1) / DL_ROWS;
    int attn_clusters = m->dl_max_clusters - n_fused;
    const long long items = (long long)(a1 - a0) * m->cfg.n_heads;
    if ((long long)attn_clusters * DL_CLUSTER > items) attn_clusters = (int)((items + DL_CLUSTER - 1) / DL_CLUSTER);
    AttnDecodeArgs aa = attn_args(la, a0, a1);
    aa.dbg = da.dbg;                               // the same mid-stack launch carries both roles' timeline marks
    return decode_dual(&m->tmAttn16, &Lb->wo.tm64, &Lb->w1.tm64, &Lb->w2.tm64, &Ln->wqkv.tm64, da, &La.tmK, &La.tmV, &La.tmR,
                       aa, b0 + a0, attn_clusters, st);
  }
  // two-half software pipeline (see forward_chunk): is it on for nb streams, and where the halves split
  bool pipelined(int nb, int* hx) const {
    const int groups = (nb + DL_ROWS - 1) / DL_ROWS, half_groups = (groups + 1) / 2;
    *hx = half_groups * DL_ROWS;
    return m->dl_dual && groups >= 2 && half_groups < m->dl_max_clusters &&
           (long long)half_groups * DL_ROWS * m->cfg.n_heads <= decode_dual_max_items(m->dl_max_clusters - half_groups);
  }
};

// vp (BERT only): the nb sequences have their own lengths (a padded batch, T_len = the padded length; see remix_batch.cu)
template <class T>
static int forward_chunk(dmg_model* m, const long long* ids, const long long* pos, int b0, int nb, int T_len, int win,
                         int k, int logits_mode, float* logits, float* core_out, cudaStream_t st, const VarlenPlan* vp = nullptr) {
  const dmg_config& c = m->cfg;
  const int d = c.d_model, HD = m->HD, rows = nb * T_len, M = c.mem_len;
  const bool bert = c.arch == DMG_ARCH_BERT;
  T* xa = (T*)m->xa;
  if (embed<T>(ids, c.encode_position ? pos : nullptr, m->emb.f32, m->beat, m->bar, m->x32, xa, rows, d, c.vocab, st)) return -1;
  if (c.keep_hidden && M > 0 && ring_append_hidden(m->x32, m->hrings[0], nb, T_len, d, M, m->pos_total, b0, st)) return -1;
  const bool fast_decode = m->is_bf16 && !bert && T_len == 1 && M > 0 && m->layers[0].has_ring_tm &&
                           attn_decode2_supported(c.d_head, M) && !(m->kflags & DMG_KF_NO_DECODE_KERNEL);
  // segments without memory (prefill after reset(), every BERT forward) in bf16: flash attention on the tensor cores
  const bool flash = m->is_bf16 && m->use_tc && T_len > 1 && (bert || (m->mem_count == 0 && win == 1 && k == 1)) &&
                     m->Dcap >= T_len && !(m->kflags & DMG_KF_NO_FLASH);
  // bf16 segments of whole 128-token tiles over a WARM memory (chunked prefill of long seeds, validation passes): the tcgen05 attention of
  // the training forward reading the K/V rings and the per-head Rd cache in place (attention_train_tc.cu)
  const bool tc_warm = m->is_bf16 && m->use_tc && !bert && !flash && !fast_decode && T_len > 1 && !(m->kflags & DMG_KF_NO_FLASH) &&
                       m->qkv16 != nullptr && attn_fwd_tc_ring_supported(T_len, c.d_head, M, m->mem_count, m->pos_total);
  // one-token step, product path: per layer ONE decode-attention launch + ONE fused layer launch (decode_layer.cu)
  const bool fused = fast_decode && m->fused_decode && !c.keep_hidden && m->layers[0].wqkv.has_tm && rows <= m->dl_rows;
  if (fused) {
    const DecodeStep ds{m, b0, st};
    const int L = c.n_layers;
    int hx = 0;
    const bool pipelined = ds.pipelined(nb, &hx);
    if (!pipelined) {
      // Stream lanes (groups of streams on parallel CUDA streams) were measured on top of this path and rejected (profiles/README.md).
      for (int l = 0; l <= L; l++) {
        if (l > 0 && ds.attn_alone(l - 1, 0, nb)) return -1;
        if (ds.fused_alone(l, 0, nb)) return -1;
      }
    } else {
      // Software pipeline over two halves X = [0, hx) and Y = [hx, nb) of the streams: while one half's attention streams its K/V
      // rings (HBM-bound, wants bandwidth, not SMs), the other half runs its latency-bound fused layer step on 8 CTAs per 32 rows -
      // in the SAME launch (decode_dual_kernel), so both really are resident together:
      //   F_0(X+Y) | A_0(X) | A_0(Y)+F_1(X) | A_1(X)+F_1(Y) | A_1(Y)+F_2(X) | ... | A_{L-1}(Y)+F_L(X) | F_L(Y)
      // (F_l = body of layer l-1 + q|k|v of layer l; A_l = attention of layer l).
      if (ds.fused_alone(0, 0, nb)) return -1;
      if (ds.attn_alone(0, 0, hx)) return -1;
      for (int l = 0; l < L; l++) {
        if (ds.dual(l + 1, 0, hx, l, hx, nb)) return -1;                       // A_l(Y) + F_{l+1}(X)
        if (l + 1 < L) { if (ds.dual(l + 1, hx, nb, l + 1, 0, hx)) return -1; }   // A_{l+1}(X) + F_{l+1}(Y)
        else if (ds.fused_alone(L, hx, nb)) return -1;
      }
    }
  }
  for (int l = 0; l < c.n_layers && !fused; l++) {
    LayerW& L = m->layers[l];
    if (flash) {
      // memory-less segment: bf16 q|k|v straight from the GEMM epilogue, tensor-core flash attention (attention_flash.cu)
      if (linear(m, A_XA, xa, L.wqkv, L.bqkv, m->qkv16, 3 * HD, rows, 0, 1, st)) return -1;
      if (vp) {
        if (attn_bert_varlen_bf16(m->qkv16, (const bf16*)L.rd, m->Dcap, m->u, m->v, (bf16*)m->attn, *vp, nb, T_len, c.n_heads,
                                  1.f / sqrtf((float)c.d_head), (m->kflags & DMG_KF_BERT_FP32_STRIP) ? 1 : 0, st)) return -1;
      } else if (bert && !(m->kflags & DMG_KF_BERT_MMA_SYNC) && attn_bert_tc_supported(T_len, c.n_heads, m->Dcap)) {
        // tcgen05 / TMEM / TMA kernel (sequences of at least 128 tokens)
        if (attn_bert_tc(m->qkv16, (const bf16*)L.rd, m->Dcap, m->u, m->v, (bf16*)m->attn, nb, T_len, c.n_heads,
                         1.f / sqrtf((float)c.d_head), (m->kflags & DMG_KF_BERT_FP32_STRIP) ? 1 : 0, st)) return -1;
      } else if (attn_flash(m->qkv16, (const bf16*)L.rd, m->Dcap, m->u, m->v, (bf16*)m->attn, nb, T_len, c.n_heads, bert ? 1 : 0,
                            1.f / sqrtf((float)c.d_head), st)) {
        return -1;
      }
      if (M > 0 && ring_append_kv<bf16, bf16>(m->qkv16, (bf16*)L.kring, (bf16*)L.vring, nb, T_len, c.n_heads, c.d_head, M,
                                               m->pos_total, b0, c.max_batch, st)) return -1;
    } else if (tc_warm) {
      if (linear(m, A_XA, xa, L.wqkv, L.bqkv, m->qkv16, 3 * HD, rows, 0, 1, st)) return -1;
      if (attn_fwd_tc_ring(m->qkv16, (const bf16*)L.kring, (const bf16*)L.vring, (const bf16*)L.rd, m->Dcap, m->u, m->v, (bf16*)m->attn, nb,
                           T_len, c.n_heads, M, m->mem_count, win, k, m->pos_total, b0, c.max_batch, 1.f / sqrtf((float)c.d_head), st)) return -1;
      if (ring_append_kv<bf16, bf16>(m->qkv16, (bf16*)L.kring, (bf16*)L.vring, nb, T_len, c.n_heads, c.d_head, M, m->pos_total, b0,
                                     c.max_batch, st)) return -1;
    } else if (linear(m, A_XA, xa, L.wqkv, L.bqkv, m->qkv, 3 * HD, rows, 0, 0, st)) {
      return -1;
    }
    if (flash || tc_warm) {
    } else if (fast_decode) {
      AttnDecodeArgs a;
      a.qkv = m->qkv;
      a.kring = (bf16*)L.kring + (size_t)b0 * c.n_heads * M * 64;
      a.vring = (bf16*)L.vring + (size_t)b0 * c.n_heads * M * 64;
      a.rd = (const bf16*)L.rd;
      a.u = m->u; a.v = m->v;
      a.out = (bf16*)m->attn;
      a.dev_state = m->dev_state;
      a.B = nb; a.H = c.n_heads; a.M = M; a.Dcap = m->Dcap;
      a.scale = 1.f / sqrtf((float)c.d_head);
      a.force_v2 = (m->kflags & DMG_KF_ATTN_DECODE_V2) ? 1 : 0;
      if (attn_decode2(&L.tmK, &L.tmV, &L.tmR, a, b0, m->num_sms, st)) return -1;
    } else {
      AttnGeneralArgs a;
      a.qkv = m->qkv; a.kring = L.kring; a.vring = L.vring; a.rd = L.rd; a.u = m->u; a.v = m->v; a.out = m->attn;
      a.B = nb; a.T = T_len; a.H = c.n_heads; a.M = M; a.Dcap = m->Dcap;
      a.mem_count = m->mem_count; a.pos_total = m->pos_total; a.b0 = b0; a.bert = bert ? 1 : 0; a.win = win; a.k = k;
      a.scale = 1.f / sqrtf((float)c.d_head);
      a.lens = vp ? vp->lens : nullptr;
      if (attn_general<T>(a, st)) return -1;
      if (vp && varlen_zero_rows<T>((T*)m->attn, vp->lens, nb, T_len, HD, st)) return -1;
      if (M > 0 && ring_append_kv<T, float>(m->qkv, (T*)L.kring, (T*)L.vring, nb, T_len, c.n_heads, c.d_head, M, m->pos_total, b0,
                                            c.max_batch, st)) return -1;
    }
    if (bert) {
      if (residual_layernorm<T, T>(m->x32, (const T*)m->attn, L.ln1w, L.ln1b, xa, rows, d, st)) return -1;
    } else {
      if (linear(m, A_ATTN, m->attn, L.wo, L.bo, m->proj, d, rows, 0, 0, st)) return -1;
      if (residual_layernorm<T, float>(m->x32, m->proj, L.ln1w, L.ln1b, xa, rows, d, st)) return -1;
      if (linear(m, A_XA, xa, L.w1, L.b1, m->hbuf, c.d_inner, rows, 1, m->is_bf16 ? 1 : 0, st)) return -1;
      if (linear(m, A_H, m->hbuf, L.w2, L.b2, m->proj, d, rows, 0, 0, st)) return -1;
      if (residual_layernorm<T, float>(m->x32, m->proj, L.ln2w, L.ln2b, xa, rows, d, st)) return -1;
    }
    if (c.keep_hidden && M > 0 && ring_append_hidden(m->x32, m->hrings[l + 1], nb, T_len, d, M, m->pos_total, b0, st)) return -1;
  }
  if (core_out)
    DMG_CUDA_OK(cudaMemcpyAsync(core_out + (size_t)b0 * T_len * d, m->x32, (size_t)rows * d * 4, cudaMemcpyDeviceToDevice, st));
  if (logits_mode == DMG_LOGITS_ALL && logits) {
    if (linear(m, A_XA, xa, m->emb, m->head_b, logits + (size_t)b0 * T_len * c.vocab, c.vocab, rows, 0, 0, st)) return -1;
  } else if (logits_mode == DMG_LOGITS_LAST && !(T_len == 1 && nb == m->batch)) {
    if (gather_rows<T>(xa, (T*)m->xlast + (size_t)b0 * d, nb, d, T_len, T_len - 1, st)) return -1;
  }
  return 0;
}

static int forward_impl(dmg_model* m, const long long* ids, const long long* pos, int bs, int T_len, int win, int k,
                        int logits_mode, float* logits, float* core_out, cudaStream_t st) {
  const dmg_config& c = m->cfg;
  DMG_CHECK(m->committed, "dmg_forward: weights not committed (call dmg_commit_weights)");
  DMG_CHECK(bs >= 1 && bs <= c.max_batch, "dmg_forward: batch %d outside [1, max_batch=%d]", bs, c.max_batch);
  DMG_CHECK(T_len >= 1 && T_len <= c.max_seq, "dmg_forward: x_len %d outside [1, max_seq=%d]", T_len, c.max_seq);
  DMG_CHECK(T_len <= m->max_rows, "dmg_forward: x_len %d exceeds the activation workspace (%d rows)", T_len, m->max_rows);
  DMG_CHECK(!c.encode_position || pos != nullptr, "dmg_forward: model encodes position but pos is NULL");
  if (c.arch == DMG_ARCH_BERT) { m->mem_count = 0; m->pos_total = 0; }
  if (m->mem_count == 0) m->batch = bs;   // fastai: memory is (re)created by the first forward after reset()
  DMG_CHECK(bs == m->batch, "dmg_forward: batch %d does not match the %d streams held in memory", bs, m->batch);
  const int cb = m->max_rows / T_len;
  for (int b0 = 0; b0 < bs; b0 += cb) {
    const int nb = bs - b0 < cb ? bs - b0 : cb;
    const long long* p = pos ? pos + (size_t)b0 * T_len : nullptr;
    int rc = m->is_bf16 ? forward_chunk<bf16>(m, ids + (size_t)b0 * T_len, p, b0, nb, T_len, win, k, logits_mode, logits, core_out, st)
                        : forward_chunk<float>(m, ids + (size_t)b0 * T_len, p, b0, nb, T_len, win, k, logits_mode, logits, core_out, st);
    if (rc) return rc;
  }
  if (logits_mode == DMG_LOGITS_LAST) {
    const bool direct = T_len == 1 && cb >= bs;   // one-token step in a single chunk: the last rows ARE the rows
    if (linear(m, direct ? A_XA : A_XLAST, direct ? m->xa : m->xlast, m->emb, m->head_b, m->logits_buf, c.vocab, bs, 0, 0, st)) return -1;
    if (logits) DMG_CUDA_OK(cudaMemcpyAsync(logits, m->logits_buf, (size_t)bs * c.vocab * 4, cudaMemcpyDeviceToDevice, st));
    m->logits_valid = true;
  }
  if (c.arch == DMG_ARCH_TXL && c.mem_len > 0) {
    if (state_advance(m->dev_state, T_len, c.mem_len, st)) return -1;
    m->pos_total += T_len;
    m->mem_count = m->mem_count + T_len > c.mem_len ? c.mem_len : m->mem_count + T_len;
  }
  return 0;
}

// A padded batch of bs BERT sequences of their own lengths (lens_host [bs], each in [1, T_max]): validates, uploads the lengths and
// the attention routing (bert_varlen_plan) into the model's buffers.  The plan stays valid until the next call.
static int varlen_setup(dmg_model* m, const int32_t* lens_host, int bs, int T_max, VarlenPlan* p, cudaStream_t st) {
  const dmg_config& c = m->cfg;
  DMG_CHECK(m->committed, "varlen: weights not committed (call dmg_commit_weights)");
  DMG_CHECK(c.arch == DMG_ARCH_BERT, "varlen: per-sequence lengths are for the BERT encoder only");
  DMG_CHECK(bs >= 1 && bs <= c.max_batch, "varlen: batch %d outside [1, max_batch=%d]", bs, c.max_batch);
  DMG_CHECK(T_max >= 1 && T_max <= c.max_seq, "varlen: T_max %d outside [1, max_seq=%d]", T_max, c.max_seq);
  DMG_CHECK((long long)bs * T_max <= m->max_rows, "varlen: %d x %d rows exceed the activation workspace (%d rows)", bs, T_max, m->max_rows);
  for (int b = 0; b < bs; b++)
    DMG_CHECK(lens_host[b] >= 1 && lens_host[b] <= T_max, "varlen: length %d of sequence %d outside [1, T_max=%d]", lens_host[b], b, T_max);
  const bool use_tc = m->is_bf16 && m->use_tc && T_max > 1 && !(m->kflags & (DMG_KF_BERT_MMA_SYNC | DMG_KF_NO_FLASH)) &&
                      attn_bert_tc_supported(T_max, c.n_heads, m->Dcap);
  std::vector<int> items, seqs;
  int fl_max = 0;
  bert_varlen_plan(lens_host, bs, c.n_heads, use_tc, items, seqs, &fl_max);
  DMG_CUDA_OK(cudaMemcpyAsync(m->vl_lens, lens_host, (size_t)bs * 4, cudaMemcpyHostToDevice, st));
  if (!items.empty()) DMG_CUDA_OK(cudaMemcpyAsync(m->vl_items, items.data(), items.size() * 4, cudaMemcpyHostToDevice, st));
  if (!seqs.empty()) DMG_CUDA_OK(cudaMemcpyAsync(m->vl_seqs, seqs.data(), seqs.size() * 4, cudaMemcpyHostToDevice, st));
  p->lens = m->vl_lens;
  p->tc_items = m->vl_items; p->n_tc_items = (int)items.size();
  p->fl_seqs = m->vl_seqs; p->n_fl_seqs = (int)seqs.size(); p->fl_max_len = fl_max;
  m->mem_count = 0; m->pos_total = 0; m->batch = bs;
  return 0;
}

static int forward_varlen(dmg_model* m, const long long* ids, const long long* pos, const VarlenPlan& p, int bs, int T_max,
                          int logits_mode, float* logits, float* core_out, cudaStream_t st) {
  return m->is_bf16 ? forward_chunk<bf16>(m, ids, pos, 0, bs, T_max, 1, 1, logits_mode, logits, core_out, st, &p)
                    : forward_chunk<float>(m, ids, pos, 0, bs, T_max, 1, 1, logits_mode, logits, core_out, st, &p);
}

static int build_rd(dmg_model* m) {
  const dmg_config& c = m->cfg;
  const int d = c.d_model, HD = m->HD, n = m->Dcap;
  float *pe = nullptr, *rp = nullptr;
  DMG_CUDA_OK(cudaMalloc(&pe, (size_t)n * d * 4));
  DMG_CUDA_OK(cudaMalloc(&rp, (size_t)n * HD * 4));
  int rc = posenc_table<float>(pe, n, d, 0);
  for (int l = 0; l < c.n_layers && !rc; l++) {
    LayerW& L = m->layers[l];
    rc = gemm_simt<float>(pe, d, L.wr.f32, d, L.br, rp, HD, n, HD, d, 0, 0, 0);
    if (rc) break;
    rc = m->is_bf16 ? rd_relayout<bf16>(rp, (bf16*)L.rd, n, c.n_heads, c.d_head, 0)
                    : rd_relayout<float>(rp, (float*)L.rd, n, c.n_heads, c.d_head, 0);
  }
  cudaError_t e = cudaDeviceSynchronize();
  cudaFree(pe);
  cudaFree(rp);
  if (rc) return rc;
  DMG_CUDA_OK(e);
  return 0;
}

static int commit_weight(dmg_model* m, Weight& w) {
  if (!m->is_bf16 || w.f32 == nullptr) return 0;
  if (cast_f32<bf16>(w.f32, w.b16, (long long)w.rows * w.cols, 0)) return -1;
  if (m->use_tc && w.cols % 64 == 0) {
    if (make_tmap_bf16(&w.tm32, w.b16, w.cols, w.rows, w.cols, 32)) return -1;
    if (make_tmap_bf16(&w.tm128, w.b16, w.cols, w.rows, w.cols, 128)) return -1;
    if (make_tmap_bf16(&w.tm64, w.b16, w.cols, w.rows, w.cols, 64)) return -1;
    w.has_tm = true;
  }
  return 0;
}

// one generation step on the device: [sample] then the one-token forward
static int decode_forward(dmg_model* m, int bs, cudaStream_t st) {
  return forward_impl(m, m->ids_buf, m->cfg.encode_position ? m->pos_buf : nullptr, bs, 1, 1, 1, DMG_LOGITS_LAST, nullptr,
                      nullptr, st);
}

// The one-token forward as a CUDA graph (all pointers are model-owned and static; the ring position is read from
// dev_state on the device, so replay stays valid while the memory advances).
static int decode_forward_graphed(dmg_model* m, int bs, cudaStream_t st) {
  const bool graph_ok = m->is_bf16 && m->cfg.arch == DMG_ARCH_TXL && !m->cfg.keep_hidden && m->cfg.max_rows >= bs &&
                        attn_decode2_supported(m->cfg.d_head, m->cfg.mem_len) &&
                        !(m->kflags & (DMG_KF_NO_GRAPH | DMG_KF_NO_DECODE_KERNEL));
  if (!graph_ok) return decode_forward(m, bs, st);
  if (m->step_graph == nullptr || m->graph_bs != bs) {
    // first call for this batch size: run eagerly (also performs every one-time cudaFuncSetAttribute), then capture
    if (m->step_graph) { cudaGraphExecDestroy(m->step_graph); m->step_graph = nullptr; }
    if (m->graph_bs != -bs - 1) {   // eager warm-up pass
      m->graph_bs = -bs - 1;
      return decode_forward(m, bs, st);
    }
    const long long before = g_launch_count;
    const long long pt = m->pos_total; const int mc = m->mem_count;
    cudaGraph_t g = nullptr;
    DMG_CUDA_OK(cudaStreamBeginCapture(m->cap_stream, cudaStreamCaptureModeThreadLocal));
    int rc = decode_forward(m, bs, m->cap_stream);
    cudaError_t e = cudaStreamEndCapture(m->cap_stream, &g);
    m->pos_total = pt; m->mem_count = mc;   // capture executed nothing
    if (rc) { if (g) cudaGraphDestroy(g); return rc; }
    DMG_CUDA_OK(e);
    m->graph_launches = g_launch_count - before;
    g_launch_count = before;
    DMG_CUDA_OK(cudaGraphInstantiate(&m->step_graph, g, 0));
    cudaGraphDestroy(g);
    m->graph_bs = bs;
  }
  DMG_CUDA_OK(cudaGraphLaunch(m->step_graph, st));
  g_launch_count += m->graph_launches;
  m->pos_total += 1;
  m->mem_count = m->mem_count + 1 > m->cfg.mem_len ? m->cfg.mem_len : m->mem_count + 1;
  m->logits_valid = true;
  return 0;
}

}  // namespace dmg

// =============================================================================================
// C ABI
// =============================================================================================
extern "C" {

const char* dmg_last_error(void) { return g_err; }
int dmg_abi_version(void) { return 1; }
long long dmg_launch_count_ll(void) { return g_launch_count; }
int64_t dmg_launch_count(void) { return (int64_t)g_launch_count; }
int64_t dmg_device_bytes(dmg_model* m) { return m ? m->bytes : 0; }
int dmg_uses_tcgen05(dmg_model* m) { return m && m->use_tc ? 1 : 0; }
int dmg_mem_count(dmg_model* m) { return m ? m->mem_count : -1; }

void dmg_destroy(dmg_model* m) {
  if (!m) return;
  cudaSetDevice(m->device);
  dmg_train_destroy(m);
  if (m->step_graph) cudaGraphExecDestroy(m->step_graph);
  if (m->cap_stream) cudaStreamDestroy(m->cap_stream);
  for (void* p : m->allocs) cudaFree(p);
  delete m;
}

int dmg_create(const dmg_config* cfg, int device, dmg_model** out) {
  DMG_CHECK(cfg && out, "dmg_create: null argument");
  *out = nullptr;
  int ndev = 0;
  cudaError_t e0 = cudaGetDeviceCount(&ndev);
  DMG_CHECK(e0 == cudaSuccess && ndev > 0, "dmg_create: no CUDA device (%s) - this library has no CPU path",
            cudaGetErrorString(e0));
  DMG_CHECK(device >= 0 && device < ndev, "dmg_create: device %d out of range (%d devices)", device, ndev);
  DMG_CUDA_OK(cudaSetDevice(device));
  cudaDeviceProp prop;
  DMG_CUDA_OK(cudaGetDeviceProperties(&prop, device));
  DMG_CHECK(prop.major == 10, "dmg_create: built for sm_100a (B200), found compute capability %d.%d", prop.major, prop.minor);
  const dmg_config& c = *cfg;
  DMG_CHECK(c.arch == DMG_ARCH_TXL || c.arch == DMG_ARCH_BERT, "dmg_create: unknown arch %d", c.arch);
  DMG_CHECK(c.dtype == DMG_F32 || c.dtype == DMG_BF16, "dmg_create: unknown dtype %d", c.dtype);
  DMG_CHECK(c.d_head == 64, "dmg_create: d_head=%d unsupported (attention kernels are specialised for 64)", c.d_head);
  DMG_CHECK(c.d_model % 128 == 0 && c.d_model <= 1024, "dmg_create: d_model=%d must be a multiple of 128, <= 1024", c.d_model);
  DMG_CHECK(c.vocab > 0 && c.n_layers > 0 && c.n_heads > 0 && c.max_batch > 0 && c.max_seq > 0, "dmg_create: bad sizes");
  DMG_CHECK(c.arch == DMG_ARCH_TXL ? c.d_inner > 0 && c.d_inner % 8 == 0 : true, "dmg_create: bad d_inner");
  DMG_CHECK(c.arch != DMG_ARCH_BERT || c.n_heads * c.d_head == c.d_model, "dmg_create: BERT encoder needs n_heads*d_head == d_model");
  DMG_CHECK(c.arch != DMG_ARCH_BERT || c.mem_len == 0, "dmg_create: BERT encoder has no memory (mem_len must be 0)");

  dmg_model* m = new dmg_model();
  m->cfg = c;
  if (c.arch == DMG_ARCH_BERT) m->cfg.encode_position = 1;   // TransformerEmbedding always adds beat + bar
  m->device = device;
  m->is_bf16 = c.dtype == DMG_BF16;
  // kernel selectors: the config's flags plus the environment variables of the same names, read here and nowhere else
  m->kflags = c.kernel_flags;
  {
    static const struct { const char* env; int flag; } sw[] = {
        {"DMG_NO_DECODE_KERNEL", DMG_KF_NO_DECODE_KERNEL}, {"DMG_NO_FLASH", DMG_KF_NO_FLASH}, {"DMG_NO_GRAPH", DMG_KF_NO_GRAPH},
        {"DMG_BERT_ATTN_MMA_SYNC", DMG_KF_BERT_MMA_SYNC}, {"DMG_BERT_TC_FP32_STRIP", DMG_KF_BERT_FP32_STRIP},
        {"DMG_NO_SPLITK", DMG_KF_NO_SPLITK}, {"DMG_NO_BIG_GEMM", DMG_KF_NO_BIG_GEMM}, {"DMG_GEMM_SIMT", DMG_KF_GEMM_SIMT},
        {"DMG_NO_FUSED_DECODE", DMG_KF_NO_FUSED_DECODE}, {"DMG_NO_DUAL_DECODE", DMG_KF_NO_DUAL_DECODE}, {"DMG_ATTN_DECODE_V2", DMG_KF_ATTN_DECODE_V2}};
    for (const auto& e : sw)
      if (getenv(e.env)) m->kflags |= e.flag;
  }
  m->use_tc = m->is_bf16 && c.gemm_backend != DMG_GEMM_SIMT && !(m->kflags & DMG_KF_GEMM_SIMT);
  m->num_sms = prop.multiProcessorCount;
  m->esz = m->is_bf16 ? 2 : 4;
  m->HD = c.n_heads * c.d_head;
  m->Dcap = c.mem_len + c.max_seq + 1;
  long long mr = c.max_rows > 0 ? c.max_rows : (long long)c.max_batch * c.max_seq;
  if (mr < c.max_seq) mr = c.max_seq;
  m->max_rows = (int)mr;
  const int d = c.d_model, HD = m->HD, V = c.vocab, L = c.n_layers;
  const bool bert = c.arch == DMG_ARCH_BERT;
  int rc = 0;
#define TRY(x) do { if (!rc && (x)) rc = -1; } while (0)
  const std::string enc = bert ? "encoder." : "0.";
  TRY(alloc_weight(m, m->emb, V, d, bert ? "encoder.embed.embed.weight" : "0.encoder.weight"));
  if (!rc) m->reg[bert ? "head.decoder.weight" : "1.decoder.weight"] = {m->emb.f32, (long long)V * d};
  TRY(alloc_vec(m, &m->head_b, V, bert ? "head.decoder.bias" : "1.decoder.bias"));
  TRY(alloc_vec(m, &m->u, HD, enc + "u"));
  TRY(alloc_vec(m, &m->v, HD, enc + "v"));
  if (m->cfg.encode_position) {
    TRY(alloc_vec(m, &m->beat, 32 * d, bert ? "encoder.embed.beat_enc.weight" : "0.beat_enc.beat_enc.weight"));
    TRY(alloc_vec(m, &m->bar, 1024 * d, bert ? "encoder.embed.bar_enc.weight" : "0.beat_enc.bar_enc.weight"));
  }
  m->layers.resize(L);
  for (int l = 0; l < L && !rc; l++) {
    LayerW& W = m->layers[l];
    const std::string p = enc + "layers." + std::to_string(l) + (bert ? ".mha1." : ".mhra.");
    TRY(alloc_weight(m, W.wqkv, 3 * HD, d, bert ? "" : p + "attention.weight"));
    if (bert && !rc) {
      m->reg[p + "q_wgt.weight"] = {W.wqkv.f32, (long long)HD * d};
      m->reg[p + "k_wgt.weight"] = {W.wqkv.f32 + (size_t)HD * d, (long long)HD * d};
      m->reg[p + "v_wgt.weight"] = {W.wqkv.f32 + (size_t)2 * HD * d, (long long)HD * d};
    }
    TRY(alloc_weight(m, W.wr, HD, d, p + "r_attn.weight"));
    TRY(alloc_vec(m, &W.ln1w, d, p + "ln.weight"));
    TRY(alloc_vec(m, &W.ln1b, d, p + "ln.bias"));
    if (c.attn_bias) {
      TRY(dalloc(m, &W.bqkv, (size_t)3 * HD));
      if (!rc) {
        if (bert) {
          m->reg[p + "q_wgt.bias"] = {W.bqkv, HD};
          m->reg[p + "k_wgt.bias"] = {W.bqkv + HD, HD};
          m->reg[p + "v_wgt.bias"] = {W.bqkv + 2 * HD, HD};
        } else {
          m->reg[p + "attention.bias"] = {W.bqkv, 3 * HD};
        }
      }
      TRY(alloc_vec(m, &W.br, HD, p + "r_attn.bias"));
    }
    if (!bert) {
      const std::string f = enc + "layers." + std::to_string(l) + ".ff.layers.";
      TRY(alloc_weight(m, W.wo, d, HD, p + "out.weight"));
      if (c.attn_bias) TRY(alloc_vec(m, &W.bo, d, p + "out.bias"));
      TRY(alloc_weight(m, W.w1, c.d_inner, d, f + "0.weight"));
      TRY(alloc_vec(m, &W.b1, c.d_inner, f + "0.bias"));
      TRY(alloc_weight(m, W.w2, d, c.d_inner, f + "3.weight"));
      TRY(alloc_vec(m, &W.b2, d, f + "3.bias"));
      TRY(alloc_vec(m, &W.ln2w, d, f + "6.weight"));
      TRY(alloc_vec(m, &W.ln2b, d, f + "6.bias"));
    }
    char* p8 = nullptr;
    TRY(dalloc(m, &p8, (size_t)c.n_heads * m->Dcap * c.d_head * m->esz));
    W.rd = p8;
    if (c.mem_len > 0) {
      const size_t rb = (size_t)c.max_batch * c.n_heads * c.mem_len * c.d_head * m->esz;
      p8 = nullptr; TRY(dalloc(m, &p8, rb)); W.kring = p8;
      p8 = nullptr; TRY(dalloc(m, &p8, rb)); W.vring = p8;
      if (!rc && m->is_bf16 && attn_decode2_supported(c.d_head, c.mem_len)) {
        const long long ring_rows = (long long)c.max_batch * c.n_heads * c.mem_len;
        TRY(make_tmap_bf16(&W.tmK, W.kring, 64, ring_rows, 64, 64));
        TRY(make_tmap_bf16(&W.tmV, W.vring, 64, ring_rows, 64, 64));
        TRY(make_tmap_bf16(&W.tmR, W.rd, 64, (long long)c.n_heads * m->Dcap, 64, 64));
        W.has_ring_tm = !rc;
      }
    }
  }
  if (c.keep_hidden && c.mem_len > 0) {
    m->hrings.resize(L + 1, nullptr);
    for (int l = 0; l <= L; l++) TRY(dalloc(m, &m->hrings[l], (size_t)c.max_batch * c.mem_len * d));
  }
  // workspaces
  const size_t R = ((size_t)(m->max_rows < 128 ? 128 : m->max_rows) + 127) / 128 * 128;   // TMA boxes are 128 rows tall
  const size_t RB = (size_t)(c.max_batch < 128 ? 128 : c.max_batch);
  TRY(dalloc(m, &m->x32, R * d));
  if (m->is_bf16) { bf16* t = nullptr; TRY(dalloc(m, &t, R * d)); m->xa = t; } else m->xa = m->x32;
  TRY(dalloc(m, &m->qkv, R * 3 * HD));
  if (m->is_bf16) TRY(dalloc(m, &m->qkv16, R * 3 * HD));
  { char* t = nullptr; TRY(dalloc(m, &t, R * HD * m->esz)); m->attn = t; }
  if (!bert) {
    TRY(dalloc(m, &m->proj, R * d));
    char* t = nullptr; TRY(dalloc(m, &t, R * c.d_inner * m->esz)); m->hbuf = t;
  }
  { char* t = nullptr; TRY(dalloc(m, &t, RB * d * m->esz)); m->xlast = t; }
  TRY(dalloc(m, &m->logits_buf, (size_t)c.max_batch * V));
  TRY(dalloc(m, &m->dev_state, 4));
  TRY(dalloc(m, &m->ids_buf, (size_t)c.max_batch));
  TRY(dalloc(m, &m->pos_buf, (size_t)c.max_batch));
  TRY(dalloc(m, &m->tok_buf, (size_t)c.max_batch));
  memset(&m->samp, 0, sizeof(m->samp));
  TRY(dalloc(m, &m->samp.prev_idx, (size_t)c.max_batch));
  TRY(dalloc(m, &m->samp.repeat_count, (size_t)c.max_batch));
  TRY(dalloc(m, &m->samp.last_xxsep, (size_t)c.max_batch));
  TRY(dalloc(m, &m->samp.last_pos, (size_t)c.max_batch));
  TRY(dalloc(m, &m->samp.start_pos, (size_t)c.max_batch));
  TRY(dalloc(m, &m->samp.step, (size_t)c.max_batch));
  TRY(dalloc(m, &m->samp.status, (size_t)c.max_batch));
  if (!rc && m->use_tc) {
    m->a_rows[A_XA] = (int)R; m->a_cols[A_XA] = d;
    m->a_rows[A_ATTN] = (int)R; m->a_cols[A_ATTN] = HD;
    m->a_rows[A_H] = (int)R; m->a_cols[A_H] = c.d_inner;
    m->a_rows[A_XLAST] = (int)RB; m->a_cols[A_XLAST] = d;
    void* bufs[A_COUNT] = {m->xa, m->attn, m->hbuf, m->xlast};
    for (int i = 0; i < A_COUNT && !rc; i++) {
      if (bufs[i] == nullptr || m->a_cols[i] % 64 != 0) continue;
      TRY(make_tmap_bf16(&m->tmA[i], bufs[i], m->a_cols[i], m->a_rows[i], m->a_cols[i], 128));
    }
    // fused one-token layer step: the FFN-down partial sums get their own [8][rows, d] fp32 scratch; DL_ROWS-row boxes over the
    // attention output
    if (!rc && !bert && c.mem_len > 0 && !(m->kflags & DMG_KF_NO_FUSED_DECODE) && decode_layer_supported(d, HD, c.d_inner, 3 * HD)) {
      m->dl_rows = (int)(R < 512 ? R : 512);                      // one-token steps run max_batch <= 512 rows through this path
      m->dl_pp_stride = (long long)m->dl_rows * d;
      TRY(dalloc(m, &m->dl_PP, (size_t)DL_CLUSTER * m->dl_pp_stride));
      TRY(make_tmap_bf16(&m->tmAttn16, m->attn, HD, (long long)R, HD, DL_ROWS));
      m->fused_decode = !rc;
      m->dl_max_clusters = decode_dual_max_clusters();
      m->dl_dual = m->fused_decode && !(m->kflags & DMG_KF_NO_DUAL_DECODE) && decode_dual_supported(c.mem_len) && m->dl_max_clusters >= 4;
      if (!rc && getenv("DMG_DECODE_TIMELINE")) TRY(dalloc(m, &m->dl_dbg, 64));
    }
  }
  if (bert) {
    const size_t items = (size_t)c.max_batch * c.n_heads * ((c.max_seq + 127) / 128);
    TRY(dalloc(m, &m->vl_lens, (size_t)c.max_batch));
    TRY(dalloc(m, &m->vl_items, items));
    TRY(dalloc(m, &m->vl_seqs, (size_t)c.max_batch));
    TRY(dalloc(m, &m->mk_pos, (size_t)c.max_batch * c.max_seq));
    for (int** p : {&m->mk_n, &m->mk_streams, &m->mk_prev, &m->mk_rc, &m->mk_tok, &m->mk_nc}) TRY(dalloc(m, p, (size_t)c.max_batch));
    TRY(dalloc(m, &m->mk_step, 1));
  }
  if (!rc && cudaStreamCreateWithFlags(&m->cap_stream, cudaStreamNonBlocking) != cudaSuccess) {
    set_error("dmg_create: cudaStreamCreate failed");
    rc = -1;
  }
#undef TRY
  if (rc) {
    dmg_destroy(m);
    return rc;
  }
  *out = m;
  return 0;
}

int dmg_set_weight(dmg_model* m, const char* name, const float* data_host, int64_t numel) {
  DMG_CHECK(m && name && data_host, "dmg_set_weight: null argument");
  auto it = m->reg.find(name);
  if (it == m->reg.end()) return 1;   // strict=False: unknown keys are ignored
  DMG_CHECK(it->second.numel == numel, "dmg_set_weight: %s has %lld elements, expected %lld", name, (long long)numel,
            it->second.numel);
  DMG_CUDA_OK(cudaSetDevice(m->device));
  DMG_CUDA_OK(cudaMemcpy(it->second.dst, data_host, (size_t)numel * 4, cudaMemcpyHostToDevice));
  m->committed = false;
  m->weights_set_externally = true;
  return 0;
}

int dmg_get_weight(dmg_model* m, const char* name, float* out_host, int64_t numel) {
  DMG_CHECK(m && name && out_host, "dmg_get_weight: null argument");
  auto it = m->reg.find(name);
  if (it == m->reg.end()) return 1;
  DMG_CHECK(it->second.numel == numel, "dmg_get_weight: %s has %lld elements, asked for %lld", name, it->second.numel,
            (long long)numel);
  DMG_CUDA_OK(cudaSetDevice(m->device));
  DMG_CUDA_OK(cudaMemcpy(out_host, it->second.dst, (size_t)numel * 4, cudaMemcpyDeviceToHost));
  return 0;
}

int dmg_commit_weights(dmg_model* m) {
  DMG_CHECK(m, "dmg_commit_weights: null model");
  DMG_CUDA_OK(cudaSetDevice(m->device));
  if (commit_weight(m, m->emb)) return -1;
  for (auto& L : m->layers) {
    if (commit_weight(m, L.wqkv) || commit_weight(m, L.wo) || commit_weight(m, L.w1) || commit_weight(m, L.w2)) return -1;
  }
  if (build_rd(m)) return -1;
  if (m->train && train_weights_reloaded(m, m->weights_set_externally)) return -1;
  m->weights_set_externally = false;
  DMG_CUDA_OK(cudaDeviceSynchronize());
  m->committed = true;
  return 0;
}

int dmg_reset(dmg_model* m, int batch) {
  DMG_CHECK(m, "dmg_reset: null model");
  DMG_CHECK(batch >= 0 && batch <= m->cfg.max_batch, "dmg_reset: batch %d outside [0, %d]", batch, m->cfg.max_batch);
  DMG_CUDA_OK(cudaSetDevice(m->device));
  m->pos_total = 0;
  m->mem_count = 0;
  m->batch = batch;
  m->logits_valid = false;
  DMG_CUDA_OK(cudaMemset(m->dev_state, 0, 16));
  return 0;
}

int dmg_select_hidden(dmg_model* m, const int32_t* idx_host, int n) {
  DMG_CHECK(m && idx_host, "dmg_select_hidden: null argument");
  const dmg_config& c = m->cfg;
  DMG_CHECK(n >= 1 && n <= c.max_batch, "dmg_select_hidden: %d streams outside [1, %d]", n, c.max_batch);
  if (c.mem_len == 0 || m->mem_count == 0) { m->batch = n; return 0; }
  for (int j = 0; j < n; j++)
    DMG_CHECK(idx_host[j] >= 0 && idx_host[j] < m->batch, "dmg_select_hidden: index %d out of range", idx_host[j]);
  DMG_CUDA_OK(cudaSetDevice(m->device));
  const size_t per_kv = (size_t)c.n_heads * c.mem_len * c.d_head * m->esz;
  const size_t per_h = (size_t)c.mem_len * c.d_model * 4;
  const size_t tmp_bytes = (size_t)m->batch * (per_kv > per_h ? per_kv : per_h);
  char* tmp = nullptr;
  DMG_CUDA_OK(cudaMalloc(&tmp, tmp_bytes));
  auto permute = [&](void* ring, size_t per) -> int {
    DMG_CUDA_OK(cudaMemcpy(tmp, ring, per * m->batch, cudaMemcpyDeviceToDevice));
    for (int j = 0; j < n; j++)
      DMG_CUDA_OK(cudaMemcpyAsync((char*)ring + per * j, tmp + per * idx_host[j], per, cudaMemcpyDeviceToDevice, 0));
    DMG_CUDA_OK(cudaDeviceSynchronize());
    return 0;
  };
  int rc = 0;
  for (auto& L : m->layers) {
    if (!rc) rc = permute(L.kring, per_kv);
    if (!rc) rc = permute(L.vring, per_kv);
  }
  for (float* h : m->hrings)
    if (!rc) rc = permute(h, per_h);
  cudaFree(tmp);
  if (rc) return rc;
  m->batch = n;
  m->logits_valid = false;
  return 0;
}

int dmg_forward(dmg_model* m, const int64_t* ids_dev, const int64_t* pos_dev, int bs, int x_len, int mask_win, int mask_k,
                int logits_mode, float* logits_dev, float* core_out_dev, void* stream) {
  DMG_CHECK(m && ids_dev, "dmg_forward: null argument");
  DMG_CHECK(mask_win >= 1, "dmg_forward: mask_win must be >= 1");
  DMG_CUDA_OK(cudaSetDevice(m->device));
  return forward_impl(m, (const long long*)ids_dev, (const long long*)pos_dev, bs, x_len, mask_win, mask_k, logits_mode,
                      logits_dev, core_out_dev, (cudaStream_t)stream);
}

int dmg_forward_varlen(dmg_model* m, const int64_t* ids_dev, const int64_t* pos_dev, const int32_t* lens_host, int bs, int T_max,
                       int logits_mode, float* logits_dev, float* core_out_dev, void* stream) {
  DMG_CHECK(m && ids_dev && pos_dev && lens_host, "dmg_forward_varlen: null argument");
  DMG_CHECK(logits_mode == DMG_LOGITS_NONE || logits_mode == DMG_LOGITS_ALL, "dmg_forward_varlen: logits_mode must be NONE or ALL");
  DMG_CUDA_OK(cudaSetDevice(m->device));
  cudaStream_t st = (cudaStream_t)stream;
  VarlenPlan p;
  if (varlen_setup(m, lens_host, bs, T_max, &p, st)) return -1;
  return forward_varlen(m, (const long long*)ids_dev, (const long long*)pos_dev, p, bs, T_max, logits_mode, logits_dev, core_out_dev, st);
}

int dmg_predict_mask_batch(dmg_model* m, int64_t* ids_dev, const int64_t* pos_dev, const int32_t* lens_host, const int32_t* mask_pos_host,
                           const int32_t* n_masks_host, const int32_t* stream_idx_host, int B, int T_max, int n_max,
                           const dmg_vocab_layout* vocab, const dmg_sampler_params* params, void* stream) {
  DMG_CHECK(m && ids_dev && pos_dev && lens_host && n_masks_host && stream_idx_host && vocab && params,
            "dmg_predict_mask_batch: null argument");
  DMG_CHECK(n_max >= 0 && n_max <= T_max && (n_max == 0 || mask_pos_host), "dmg_predict_mask_batch: n_max %d outside [0, T_max=%d]", n_max, T_max);
  DMG_CHECK(B >= 1 && B <= m->cfg.max_batch, "dmg_predict_mask_batch: %d items outside [1, max_batch=%d]", B, m->cfg.max_batch);
  for (int b = 0; b < B; b++) {
    const int L = lens_host[b], n = n_masks_host[b];
    DMG_CHECK(L >= 1 && L <= T_max, "dmg_predict_mask_batch: length %d of item %d outside [1, T_max=%d]", L, b, T_max);
    DMG_CHECK(n >= 0 && n <= n_max && n <= L, "dmg_predict_mask_batch: item %d has %d masks (n_max %d, length %d)", b, n, n_max, L);
    DMG_CHECK(stream_idx_host[b] >= 0, "dmg_predict_mask_batch: negative stream index of item %d", b);
    for (int s = 0; s < n; s++) {
      const int p = mask_pos_host[(size_t)b * n_max + s];
      DMG_CHECK(p >= 0 && p < L && (s == 0 || p > mask_pos_host[(size_t)b * n_max + s - 1]),
                "dmg_predict_mask_batch: mask position %d of item %d is outside [0, %d) or not ascending", p, b, L);
    }
  }
  DMG_CUDA_OK(cudaSetDevice(m->device));
  cudaStream_t st = (cudaStream_t)stream;
  VarlenPlan p;
  if (varlen_setup(m, lens_host, B, T_max, &p, st)) return -1;
  int steps = 0;
  for (int b = 0; b < B; b++) steps = n_masks_host[b] > steps ? n_masks_host[b] : steps;
  if (steps == 0) return 0;
  DMG_CUDA_OK(cudaMemcpyAsync(m->mk_pos, mask_pos_host, (size_t)B * n_max * 4, cudaMemcpyHostToDevice, st));
  DMG_CUDA_OK(cudaMemcpyAsync(m->mk_n, n_masks_host, (size_t)B * 4, cudaMemcpyHostToDevice, st));
  DMG_CUDA_OK(cudaMemcpyAsync(m->mk_streams, stream_idx_host, (size_t)B * 4, cudaMemcpyHostToDevice, st));
  DMG_CUDA_OK(cudaMemsetAsync(m->mk_rc, 0, (size_t)B * 4, st));
  DMG_CUDA_OK(cudaMemsetAsync(m->mk_step, 0, 4, st));
  const dmg_config& c = m->cfg;
  MaskStepArgs a;
  a.ids = (long long*)ids_dev; a.lens = m->vl_lens; a.mask_pos = m->mk_pos; a.n_masks = m->mk_n; a.step = m->mk_step;
  a.prev = m->mk_prev; a.repeat_count = m->mk_rc; a.logits = m->logits_buf; a.bias = m->head_b; a.tok = m->mk_tok;
  a.num_choices = m->mk_nc; a.B = B; a.T_max = T_max; a.n_max = n_max; a.d = c.d_model; a.V = c.vocab;
  SampleArgs sa;
  memset(&sa, 0, sizeof(sa));
  sa.logits = m->logits_buf; sa.V = c.vocab; sa.vocab = *vocab; sa.params = *params; sa.loop_mode = 0;
  sa.prev_idx = m->mk_prev; sa.repeat_count = m->mk_rc; sa.out_tokens = m->mk_tok; sa.num_choices = m->mk_nc;
  sa.stream_ids = m->mk_streams; sa.dev_offset = m->mk_step;
  const void* emb = m->is_bf16 ? (const void*)m->emb.b16 : (const void*)m->emb.f32;
  // one step: the encoder forward (no logits) over the current ids, then the mask step; its launches read the step counter on the
  // device, so from the second step on they are replayed as one CUDA graph (the first, eager step performs the one-time set-up)
  auto step = [&](cudaStream_t s) -> int {
    if (forward_varlen(m, (const long long*)ids_dev, (const long long*)pos_dev, p, B, T_max, DMG_LOGITS_NONE, nullptr, nullptr, s)) return -1;
    return mask_step_launch(a, m->xa, emb, m->is_bf16, sa, s);
  };
  const bool graphed = !(m->kflags & DMG_KF_NO_GRAPH) && steps > 1;
  cudaGraphExec_t exec = nullptr;
  int rc = step(st);
  for (int s = 1; s < steps && !rc; s++) {
    if (!graphed) { rc = step(st); continue; }
    if (exec == nullptr) {
      const long long before = g_launch_count;
      cudaGraph_t g = nullptr;
      DMG_CUDA_OK(cudaStreamBeginCapture(m->cap_stream, cudaStreamCaptureModeThreadLocal));
      rc = step(m->cap_stream);
      const cudaError_t e = cudaStreamEndCapture(m->cap_stream, &g);
      m->graph_launches = g_launch_count - before;
      g_launch_count = before;
      if (!rc && e != cudaSuccess) { set_error("dmg_predict_mask_batch: graph capture failed: %s", cudaGetErrorString(e)); rc = -1; }
      if (!rc && cudaGraphInstantiate(&exec, g, 0) != cudaSuccess) { set_error("dmg_predict_mask_batch: cudaGraphInstantiate failed"); rc = -1; }
      if (g) cudaGraphDestroy(g);
      if (rc) break;
    }
    if (cudaGraphLaunch(exec, st) != cudaSuccess) { set_error("dmg_predict_mask_batch: cudaGraphLaunch failed"); rc = -1; break; }
    g_launch_count += m->graph_launches;
  }
  if (exec) cudaGraphExecDestroy(exec);
  return rc;
}

int dmg_attn_bert_varlen(const void* qkv_dev, const void* rk_dev, int Dcap, const float* u, const float* v, void* out_dev,
                         const int32_t* lens_host, int B, int T_max, int H, int mma_sync_only, void* stream) {
  DMG_CHECK(qkv_dev && rk_dev && u && v && out_dev && lens_host, "dmg_attn_bert_varlen: null argument");
  DMG_CHECK(B >= 1 && T_max >= 1 && H >= 1 && H <= 256 && Dcap >= T_max, "dmg_attn_bert_varlen: B %d, T_max %d, H %d, Dcap %d", B, T_max, H, Dcap);
  for (int b = 0; b < B; b++)
    DMG_CHECK(lens_host[b] >= 1 && lens_host[b] <= T_max, "dmg_attn_bert_varlen: length %d of sequence %d outside [1, T_max=%d]", lens_host[b], b, T_max);
  cudaStream_t st = (cudaStream_t)stream;
  std::vector<int> items, seqs;
  int fl_max = 0;
  bert_varlen_plan(lens_host, B, H, !mma_sync_only && attn_bert_tc_supported(T_max, H, Dcap), items, seqs, &fl_max);
  int* buf = nullptr;
  DMG_CUDA_OK(cudaMalloc(&buf, (size_t)(B + items.size() + seqs.size() + 1) * 4));
  VarlenPlan p;
  p.lens = buf; p.tc_items = buf + B; p.n_tc_items = (int)items.size(); p.fl_seqs = buf + B + items.size();
  p.n_fl_seqs = (int)seqs.size(); p.fl_max_len = fl_max;
  int rc = 0;
  if (cudaMemcpyAsync(buf, lens_host, (size_t)B * 4, cudaMemcpyHostToDevice, st) != cudaSuccess ||
      (!items.empty() && cudaMemcpyAsync(buf + B, items.data(), items.size() * 4, cudaMemcpyHostToDevice, st) != cudaSuccess) ||
      (!seqs.empty() && cudaMemcpyAsync(buf + B + items.size(), seqs.data(), seqs.size() * 4, cudaMemcpyHostToDevice, st) != cudaSuccess)) {
    set_error("dmg_attn_bert_varlen: upload failed");
    rc = -1;
  }
  if (!rc) rc = attn_bert_varlen_bf16((const bf16*)qkv_dev, (const bf16*)rk_dev, Dcap, u, v, (bf16*)out_dev, p, B, T_max, H,
                                      0.125f, 0, st);
  const cudaError_t e = cudaStreamSynchronize(st);
  cudaFree(buf);
  if (rc) return rc;
  DMG_CUDA_OK(e);
  return 0;
}

int dmg_get_hidden(dmg_model* m, int level, float* out_dev, void* stream) {
  DMG_CHECK(m && out_dev, "dmg_get_hidden: null argument");
  DMG_CHECK(m->cfg.keep_hidden && !m->hrings.empty(), "dmg_get_hidden: model was created without keep_hidden");
  DMG_CHECK(level >= 0 && level <= m->cfg.n_layers, "dmg_get_hidden: level %d out of range", level);
  DMG_CUDA_OK(cudaSetDevice(m->device));
  return ring_export_hidden(m->hrings[level], out_dev, m->batch, m->cfg.d_model, m->cfg.mem_len, m->pos_total, m->mem_count,
                            (cudaStream_t)stream);
}

int dmg_sampler_init(dmg_model* m, const dmg_vocab_layout* vocab, const dmg_sampler_params* params,
                     const int32_t* prev_idx_host, const int64_t* last_pos_host, int bs) {
  DMG_CHECK(m && vocab && params && prev_idx_host, "dmg_sampler_init: null argument");
  DMG_CHECK(bs >= 1 && bs <= m->cfg.max_batch, "dmg_sampler_init: batch %d outside [1, %d]", bs, m->cfg.max_batch);
  DMG_CHECK(params->n_words > 0, "dmg_sampler_init: n_words must be positive");
  DMG_CUDA_OK(cudaSetDevice(m->device));
  SampleArgs& s = m->samp;
  s.V = m->cfg.vocab;
  s.vocab = *vocab;
  s.params = *params;
  s.loop_mode = 1;
  s.offset = 0;
  s.logits = m->logits_buf;
  s.next_ids = m->ids_buf;
  s.next_pos = m->pos_buf;
  s.num_choices = nullptr;
  std::vector<long long> lp(bs, 0);
  if (last_pos_host) for (int i = 0; i < bs; i++) lp[i] = last_pos_host[i];
  DMG_CUDA_OK(cudaMemcpy(s.prev_idx, prev_idx_host, (size_t)bs * 4, cudaMemcpyHostToDevice));
  DMG_CUDA_OK(cudaMemcpy(s.last_pos, lp.data(), (size_t)bs * 8, cudaMemcpyHostToDevice));
  DMG_CUDA_OK(cudaMemcpy(s.start_pos, lp.data(), (size_t)bs * 8, cudaMemcpyHostToDevice));
  DMG_CUDA_OK(cudaMemcpy(m->pos_buf, lp.data(), (size_t)bs * 8, cudaMemcpyHostToDevice));
  DMG_CUDA_OK(cudaMemset(s.repeat_count, 0, (size_t)bs * 4));
  DMG_CUDA_OK(cudaMemset(s.last_xxsep, 0, (size_t)bs * 4));
  DMG_CUDA_OK(cudaMemset(s.step, 0, (size_t)bs * 4));
  DMG_CUDA_OK(cudaMemset(s.status, 0, (size_t)bs * 4));
  m->samp_ready = true;
  return 0;
}

int dmg_generate(dmg_model* m, int n_steps, int32_t* tokens_dev, void* stream) {
  DMG_CHECK(m && tokens_dev, "dmg_generate: null argument");
  DMG_CHECK(m->samp_ready, "dmg_generate: call dmg_sampler_init first");
  DMG_CHECK(m->logits_valid, "dmg_generate: no logits to sample from (run dmg_forward with DMG_LOGITS_LAST first)");
  DMG_CHECK(m->cfg.arch == DMG_ARCH_TXL, "dmg_generate: only the Transformer-XL model generates");
  DMG_CUDA_OK(cudaSetDevice(m->device));
  cudaStream_t st = (cudaStream_t)stream;
  const int bs = m->batch;
  for (int s = 0; s < n_steps; s++) {
    SampleArgs a = m->samp;
    a.out_tokens = tokens_dev + (size_t)s * bs;
    if (sample_launch(a, bs, st)) return -1;
    if (decode_forward_graphed(m, bs, st)) return -1;
  }
  return 0;
}

int dmg_generate_step_host(dmg_model* m, const int64_t* ids_host, int32_t* tokens_host, void* stream) {
  DMG_CHECK(m && tokens_host, "dmg_generate_step_host: null argument");
  DMG_CHECK(m->samp_ready, "dmg_generate_step_host: call dmg_sampler_init first");
  DMG_CUDA_OK(cudaSetDevice(m->device));
  cudaStream_t st = (cudaStream_t)stream;
  const int bs = m->batch;
  if (ids_host) {
    DMG_CUDA_OK(cudaMemcpyAsync(m->ids_buf, ids_host, (size_t)bs * 8, cudaMemcpyHostToDevice, st));
    if (decode_forward_graphed(m, bs, st)) return -1;
  } else {
    DMG_CHECK(m->logits_valid, "dmg_generate_step_host: no logits to sample from");
  }
  SampleArgs a = m->samp;
  a.out_tokens = m->tok_buf;
  if (sample_launch(a, bs, st)) return -1;
  if (!ids_host && decode_forward_graphed(m, bs, st)) return -1;
  DMG_CUDA_OK(cudaMemcpyAsync(tokens_host, m->tok_buf, (size_t)bs * 4, cudaMemcpyDeviceToHost, st));
  DMG_CUDA_OK(cudaStreamSynchronize(st));
  return 0;
}

int dmg_sample_logits(dmg_model* m, const float* logits_dev, const int32_t* prev_idx_dev, const int32_t* repeat_count_dev,
                      int n, const dmg_vocab_layout* vocab, const dmg_sampler_params* params, uint64_t offset,
                      int32_t* out_dev, int32_t* num_choices_dev, void* stream) {
  DMG_CHECK(m && logits_dev && prev_idx_dev && repeat_count_dev && vocab && params && out_dev, "dmg_sample_logits: null argument");
  DMG_CUDA_OK(cudaSetDevice(m->device));
  SampleArgs a;
  memset(&a, 0, sizeof(a));
  a.logits = logits_dev;
  a.V = m->cfg.vocab;
  a.vocab = *vocab;
  a.params = *params;
  a.loop_mode = 0;
  a.offset = offset;
  a.prev_idx = const_cast<int*>(prev_idx_dev);
  a.repeat_count = const_cast<int*>(repeat_count_dev);
  a.out_tokens = out_dev;
  a.num_choices = num_choices_dev;
  return sample_launch(a, n, (cudaStream_t)stream);
}

int dmg_beam_step(dmg_model* m, const float* scores_dev, int n_scores, int nb, int top_k, int beam_sz, float* scores_out_dev,
                  int32_t* parents_out_dev, int32_t* tokens_out_dev, void* stream) {
  DMG_CHECK(m && scores_dev && scores_out_dev && parents_out_dev && tokens_out_dev, "dmg_beam_step: null argument");
  DMG_CHECK(m->logits_valid && nb == m->batch, "dmg_beam_step: needs the logits of a DMG_LOGITS_LAST forward over %d beams (have %d streams)",
            nb, m->batch);
  DMG_CHECK(n_scores == 1 || n_scores == nb, "dmg_beam_step: n_scores must be 1 or nb");
  DMG_CUDA_OK(cudaSetDevice(m->device));
  BeamArgs a;
  a.logits = m->logits_buf; a.V = m->cfg.vocab; a.nb = nb; a.top_k = top_k; a.beam_sz = beam_sz;
  a.scores_in = scores_dev; a.n_scores = n_scores; a.scores_out = scores_out_dev; a.parents = parents_out_dev; a.tokens = tokens_out_dev;
  return beam_step_launch(a, (cudaStream_t)stream);
}

int dmg_sample_probs(dmg_model* m, int predict_loop, const float* logits_dev, const int32_t* prev_idx_dev,
                     const int32_t* repeat_count_dev, const int32_t* last_xxsep_dev, const int64_t* pos_since_start_dev, int n,
                     const dmg_vocab_layout* vocab, const dmg_sampler_params* params, uint64_t offset, int32_t* out_dev,
                     int32_t* num_choices_dev, float* probs_dev, void* stream) {
  DMG_CHECK(m && logits_dev && prev_idx_dev && repeat_count_dev && vocab && params && out_dev, "dmg_sample_probs: null argument");
  DMG_CHECK(!predict_loop || (last_xxsep_dev && pos_since_start_dev), "dmg_sample_probs: the predict loop needs last_xxsep and positions");
  DMG_CUDA_OK(cudaSetDevice(m->device));
  SampleArgs a;
  memset(&a, 0, sizeof(a));
  a.logits = logits_dev;
  a.V = m->cfg.vocab;
  a.vocab = *vocab;
  a.params = *params;
  a.loop_mode = predict_loop ? 2 : 0;
  a.offset = offset;
  a.prev_idx = const_cast<int*>(prev_idx_dev);
  a.repeat_count = const_cast<int*>(repeat_count_dev);
  a.last_xxsep = const_cast<int*>(last_xxsep_dev);
  a.last_pos = (long long*)const_cast<int64_t*>(pos_since_start_dev);     // start_pos = 0: last_pos - start_pos = the given distance
  a.out_tokens = out_dev;
  a.num_choices = num_choices_dev;
  a.probs = probs_dev;
  return sample_launch(a, n, (cudaStream_t)stream);
}

int dmg_decode_timeline(dmg_model* m, uint64_t* out64_host) {
  DMG_CHECK(m && out64_host, "dmg_decode_timeline: null argument");
  DMG_CHECK(m->dl_dbg != nullptr, "dmg_decode_timeline: create the model with DMG_DECODE_TIMELINE=1 in the environment");
  DMG_CUDA_OK(cudaSetDevice(m->device));
  DMG_CUDA_OK(cudaDeviceSynchronize());
  DMG_CUDA_OK(cudaMemcpy(out64_host, m->dl_dbg, 64 * sizeof(uint64_t), cudaMemcpyDeviceToHost));
  return 0;
}

int dmg_attn_decode_layer(dmg_model* m, int layer, void* stream) {
  DMG_CHECK(m, "dmg_attn_decode_layer: null model");
  const dmg_config& c = m->cfg;
  DMG_CHECK(layer >= 0 && layer < c.n_layers, "dmg_attn_decode_layer: layer %d out of range", layer);
  DMG_CHECK(m->is_bf16 && c.arch == DMG_ARCH_TXL && attn_decode2_supported(c.d_head, c.mem_len) && m->layers[layer].has_ring_tm,
            "dmg_attn_decode_layer: the fused decode kernel needs bf16, d_head 64 and mem_len %% 64 == 0");
  DMG_CHECK(m->batch >= 1 && m->batch <= m->max_rows, "dmg_attn_decode_layer: no active streams");
  DMG_CUDA_OK(cudaSetDevice(m->device));
  LayerW& L = m->layers[layer];
  AttnDecodeArgs a;
  a.qkv = m->qkv; a.kring = (bf16*)L.kring; a.vring = (bf16*)L.vring; a.rd = (const bf16*)L.rd;
  a.u = m->u; a.v = m->v; a.out = (bf16*)m->attn; a.dev_state = m->dev_state;
  a.B = m->batch; a.H = c.n_heads; a.M = c.mem_len; a.Dcap = m->Dcap;
  a.scale = 1.f / sqrtf((float)c.d_head);
  return attn_decode2(&L.tmK, &L.tmV, &L.tmR, a, 0, m->num_sms, (cudaStream_t)stream);
}

int dmg_decode_dual_launch(dmg_model* m, int layer, void* stream) {
  DMG_CHECK(m, "dmg_decode_dual_launch: null model");
  const dmg_config& c = m->cfg;
  DMG_CHECK(layer >= 0 && layer + 1 < c.n_layers, "dmg_decode_dual_launch: layer %d out of range", layer);
  DMG_CHECK(m->batch >= 1 && m->batch <= m->dl_rows, "dmg_decode_dual_launch: no active streams");
  DMG_CUDA_OK(cudaSetDevice(m->device));
  const DecodeStep ds{m, 0, (cudaStream_t)stream};
  int hx = 0;
  DMG_CHECK(m->fused_decode && ds.pipelined(m->batch, &hx), "dmg_decode_dual_launch: the two-half pipeline is off for this model / batch");
  return ds.dual(layer + 1, 0, hx, layer, hx, m->batch);      // A_layer(second half) + F_{layer+1}(first half), as in the step
}

}  // extern "C"

// ---- unit-test entries of the one-token decode kernels: the checks and tensor maps of dmg_attn_decode / dmg_decode_layer_step /
// dmg_decode_dual, made before anything is launched
namespace dmg {

static_assert(sizeof(dmg_decode_attn_args) == 104 && sizeof(dmg_decode_layer_args) == 176, "tests/test_abi.py mirrors these layouts");

struct DecodeAttnPlan {
  AttnDecodeArgs a;
  TensorMap2D tmK, tmV, tmR;
  int b0 = 0, num_sms = 0;
  int state[2] = {0, 0};
};

static int plan_decode_attn(const dmg_decode_attn_args* p, DecodeAttnPlan& o, const char* who) {
  DMG_CHECK(p && p->qkv && p->kring && p->vring && p->rd && p->u && p->v && p->out && p->state, "%s: null argument", who);
  DMG_CHECK(p->Dh == 64, "%s: head size %d (only 64)", who, p->Dh);
  DMG_CHECK(p->kernel == 0 || p->kernel == 1, "%s: kernel %d (0 = the step's choice, 1 = the second-generation kernel)", who, p->kernel);
  // kernel 0 falls back to the second kernel where the third does not apply, so both choices need what the second one supports
  DMG_CHECK(attn_decode2_supported(64, p->M), "%s: mem_len %d not supported by the decode attention", who, p->M);
  DMG_CHECK(p->Dcap >= p->M + 1, "%s: rel-pos cache too small (Dcap %d < M + 1 = %d)", who, p->Dcap, p->M + 1);
  DMG_CHECK(p->B >= 1 && p->H >= 1 && p->H <= 64 && p->b0 >= 0 && (long long)p->b0 + p->B <= p->Bcap,
            "%s: B %d, H %d, streams [%d, %d) outside the ring's %d", who, p->B, p->H, p->b0, p->b0 + p->B, p->Bcap);
  DMG_CHECK(p->pos_total >= 0 && p->pos_total <= 0x7fffffffLL, "%s: pos_total %lld outside [0, 2^31)", who, (long long)p->pos_total);
  const long long ring_rows = (long long)p->Bcap * p->H * p->M;
  if (make_tmap_bf16(&o.tmK, p->kring, 64, ring_rows, 64, 64) || make_tmap_bf16(&o.tmV, p->vring, 64, ring_rows, 64, 64) ||
      make_tmap_bf16(&o.tmR, p->rd, 64, (long long)p->H * p->Dcap, 64, 64)) return -1;
  int dev = 0;
  DMG_CUDA_OK(cudaGetDevice(&dev));
  DMG_CUDA_OK(cudaDeviceGetAttribute(&o.num_sms, cudaDevAttrMultiProcessorCount, dev));
  AttnDecodeArgs& a = o.a;
  const size_t chunk = (size_t)p->b0 * p->H * p->M * 64;      // the kernels take ring pointers offset by b0 streams
  a.qkv = p->qkv; a.kring = (bf16*)p->kring + chunk; a.vring = (bf16*)p->vring + chunk; a.rd = (const bf16*)p->rd;
  a.u = p->u; a.v = p->v; a.out = (bf16*)p->out; a.dev_state = p->state;
  a.B = p->B; a.H = p->H; a.M = p->M; a.Dcap = p->Dcap;
  a.scale = 0.125f;
  a.force_v2 = p->kernel;
  o.b0 = p->b0;
  o.state[0] = (int)p->pos_total;
  o.state[1] = (int)(p->pos_total < p->M ? p->pos_total : p->M);   // mem_count, as state_advance keeps it
  return 0;
}

struct DecodeLayerPlan {
  DecodeLayerArgs a;
  TensorMap2D tmAttn, tmWo, tmW1, tmW2, tmWq;
};

static int plan_decode_layer(const dmg_decode_layer_args* p, DecodeLayerPlan& o, const char* who) {
  DMG_CHECK(p, "%s: null argument", who);
  const bool body = (p->mode & 1) != 0, next = (p->mode & 2) != 0;
  DMG_CHECK(p->mode >= 1 && p->mode <= 3, "%s: mode %d (bit 0 = layer body, bit 1 = next q|k|v)", who, p->mode);
  const int HD = p->n_heads * p->d_head;
  DMG_CHECK(p->d_head == 64 && decode_layer_supported(p->d_model, HD, p->d_inner, 3 * HD),
            "%s: geometry d_model %d, %d heads of %d, d_inner %d not supported", who, p->d_model, p->n_heads, p->d_head, p->d_inner);
  DMG_CHECK(p->x32 && p->pp, "%s: null argument", who);
  DMG_CHECK(!body || (p->attn && p->wo && p->w1 && p->w2 && p->ln1w && p->ln1b && p->ln2w && p->ln2b), "%s: null argument (layer body)", who);
  DMG_CHECK(!next || (p->wqkv && p->qkv), "%s: null argument (next q|k|v)", who);
  DMG_CHECK(p->row_base >= 0 && p->B > p->row_base, "%s: rows [%d, %d) empty", who, p->row_base, p->B);
  DMG_CHECK(!body || p->attn_rows >= p->B, "%s: attn_rows %d < B %d", who, p->attn_rows, p->B);
  const long long rows_pad = p->row_base + (long long)(p->B - p->row_base + DL_ROWS - 1) / DL_ROWS * DL_ROWS;
  DMG_CHECK(p->pp_stride >= rows_pad * p->d_model, "%s: pp_stride %lld < %lld rows x %d (whole %d-row clusters are written)", who,
            (long long)p->pp_stride, rows_pad, p->d_model, DL_ROWS);
  const int d = p->d_model, di = p->d_inner;
  // the kernel takes all five maps; a weight the mode does not read gets the map of one it does
  if (body) {
    if (make_tmap_bf16(&o.tmAttn, p->attn, HD, p->attn_rows, HD, DL_ROWS) || make_tmap_bf16(&o.tmWo, p->wo, HD, d, HD, 64) ||
        make_tmap_bf16(&o.tmW1, p->w1, d, di, d, 64) || make_tmap_bf16(&o.tmW2, p->w2, di, d, di, 64)) return -1;
  }
  if (next && make_tmap_bf16(&o.tmWq, p->wqkv, d, 3 * HD, d, 64)) return -1;
  if (!body) o.tmAttn = o.tmWo = o.tmW1 = o.tmW2 = o.tmWq;
  if (!next) o.tmWq = o.tmWo;
  DecodeLayerArgs& a = o.a;
  a.x32 = p->x32; a.xa_out = (bf16*)p->xa_out; a.qkv = p->qkv; a.PP = p->pp; a.pp_stride = p->pp_stride;
  a.bo = p->bo; a.b1 = p->b1; a.b2 = p->b2; a.bq = p->bqkv;
  a.ln1w = p->ln1w; a.ln1b = p->ln1b; a.ln2w = p->ln2w; a.ln2b = p->ln2b;
  a.row_base = p->row_base; a.B = p->B;
  a.d = d; a.HD = HD; a.di = di; a.n3 = 3 * HD;
  a.mode = p->mode;
  return 0;
}

}  // namespace dmg

extern "C" {

int dmg_attn_decode(const dmg_decode_attn_args* p, void* stream) {
  DecodeAttnPlan o;
  if (plan_decode_attn(p, o, "dmg_attn_decode")) return -1;
  cudaStream_t st = (cudaStream_t)stream;
  DMG_CUDA_OK(cudaMemcpyAsync(p->state, o.state, sizeof(o.state), cudaMemcpyHostToDevice, st));
  const int rc = attn_decode2(&o.tmK, &o.tmV, &o.tmR, o.a, o.b0, o.num_sms, st);
  const cudaError_t e = cudaStreamSynchronize(st);
  if (rc) return rc;
  DMG_CUDA_OK(e);
  return 0;
}

int dmg_decode_layer_step(const dmg_decode_layer_args* f, void* stream) {
  DecodeLayerPlan o;
  if (plan_decode_layer(f, o, "dmg_decode_layer_step")) return -1;
  cudaStream_t st = (cudaStream_t)stream;
  const int rc = decode_layer(&o.tmAttn, &o.tmWo, &o.tmW1, &o.tmW2, &o.tmWq, o.a, st);
  const cudaError_t e = cudaStreamSynchronize(st);
  if (rc) return rc;
  DMG_CUDA_OK(e);
  return 0;
}

int dmg_decode_dual(const dmg_decode_layer_args* f, const dmg_decode_attn_args* a, int attn_clusters, void* stream) {
  DecodeLayerPlan lo;
  DecodeAttnPlan ao;
  if (plan_decode_layer(f, lo, "dmg_decode_dual") || plan_decode_attn(a, ao, "dmg_decode_dual")) return -1;
  DMG_CHECK(a->kernel == 0 && decode_dual_supported(a->M), "dmg_decode_dual: the attention role runs the third-generation kernel only "
            "(kernel 0, M a multiple of 128 up to 512; got kernel %d, M %d)", a->kernel, a->M);
  DMG_CHECK(attn_clusters >= 0, "dmg_decode_dual: attn_clusters %d", attn_clusters);
  const long long items = (long long)a->B * a->H;
  if (attn_clusters == 0) {   // as DecodeStep::dual sizes the attention role
    const int n_fused = (f->B - f->row_base + DL_ROWS - 1) / DL_ROWS;
    attn_clusters = decode_dual_max_clusters() - n_fused;
    if ((long long)attn_clusters * DL_CLUSTER > items) attn_clusters = (int)((items + DL_CLUSTER - 1) / DL_CLUSTER);
    DMG_CHECK(attn_clusters >= 1, "dmg_decode_dual: no cluster left for the attention role");
  }
  DMG_CHECK(items <= decode_dual_max_items(attn_clusters), "dmg_decode_dual: %d x %d items do not fit %d attention clusters", a->B,
            a->H, attn_clusters);
  cudaStream_t st = (cudaStream_t)stream;
  DMG_CUDA_OK(cudaMemcpyAsync(a->state, ao.state, sizeof(ao.state), cudaMemcpyHostToDevice, st));
  const int rc = decode_dual(&lo.tmAttn, &lo.tmWo, &lo.tmW1, &lo.tmW2, &lo.tmWq, lo.a, &ao.tmK, &ao.tmV, &ao.tmR, ao.a, ao.b0,
                             attn_clusters, st);
  const cudaError_t e = cudaStreamSynchronize(st);
  if (rc) return rc;
  DMG_CUDA_OK(e);
  return 0;
}

int dmg_gemm_bf16(const void* a_dev, const void* w_dev, const float* bias_dev, void* c_dev, int M, int N, int K, int gelu,
                  int out_bf16, int backend, void* stream) {
  DMG_CHECK(a_dev && w_dev && c_dev, "dmg_gemm_bf16: null argument");
  cudaStream_t st = (cudaStream_t)stream;
  if (backend == DMG_GEMM_SIMT)
    return gemm_simt<bf16>((const bf16*)a_dev, K, (const bf16*)w_dev, K, bias_dev, c_dev, N, M, N, K, gelu, out_bf16, st);
  TensorMap2D ta, tw;
  const int BN = M <= 512 ? 32 : 128;
  if (make_tmap_bf16(&ta, a_dev, K, M, K, 128)) return -1;
  if (make_tmap_bf16(&tw, w_dev, K, N, K, BN)) return -1;
  if (backend == DMG_GEMM_AUTO && M <= 512 && gemm_tc_splitk_ways(K))
    return gemm_tc_splitk(&ta, &tw, bias_dev, c_dev, N, M, N, K, gelu, out_bf16, st);
  return gemm_tc(&ta, &tw, BN, bias_dev, c_dev, N, M, N, K, gelu, out_bf16, st);
}

}  // extern "C"
