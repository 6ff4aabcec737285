// Training step: forward with saved activations, loss, backward, Adam; C ABI (dmg_train_*).
// What fastai's Learner does for one batch around the reference models (SURVEY.md 3.3, App. A.3, A.7):
//   Transformer-XL: model(x) train-mode (deep_music_genre.py:1617-1647), CrossEntropyFlat + RNNTrainer AR/TAR, backward, Adam(true_wd).
//   Memory in training is the reference's own: hidden states of the previous segment per level (detached), re-projected
//   to K/V with the current weights every step (_update_mems, App. A.2).
//   Remix encoder (msk task): head(encoder(x_masked, pos)) train-mode (deep_music_remix.py:1874-1881, 1910-2104),
//   CrossEntropyFlat(ignore_index=pad_idx), backward, the same Adam(true_wd); no memory, no AR/TAR.
#include <cstring>
#include <string>
#include <vector>

#include "model.cuh"
#include "launch.cuh"
#include "train_kernels.cuh"

using namespace dmg;

namespace {

enum { SITE_EMBED = 0, SITE_ATTN = 1, SITE_RES1 = 2, SITE_FF = 3, SITE_RES2 = 4, SITE_OUT = 5 };

struct ParamRef {
  std::string name;
  float* p = nullptr;      // fp32 master
  bf16* p16 = nullptr;     // bf16 copy (matrices)
  long long n = 0;
  long long off = 0;       // offset in the flat gradient / Adam buffers
};

struct LayerAct {
  bf16 *xa_in = nullptr, *qkv_x = nullptr, *kv_m = nullptr, *attn = nullptr, *z1 = nullptr, *xa1 = nullptr, *hpre = nullptr,
       *hact = nullptr, *z2 = nullptr, *rk = nullptr;
  float* lse = nullptr;
  bf16* p_save = nullptr;    // [B*H, T, S] undropped attention probabilities saved by the tcgen05 forward (AttnTrainArgs::p_save)
  float* m_save = nullptr;   // [B*H, T, S/64] their reference maxima
  bf16 *qu_save = nullptr, *qv_save = nullptr;   // [rows, HD] q + u / q + v tiles stored by the tcgen05 forward
  float2 *st1 = nullptr, *st2 = nullptr;
};

struct LayerGrad {   // offsets into the flat buffer
  long long wqkv, wr, wo, w1, w2, bqkv, br, bo, b1, b2, ln1w, ln1b, ln2w, ln2b;
};

}  // namespace

struct dmg_train {
  dmg_train_config cfg;
  int B = 0, T = 0, rows = 0, S = 0, Vp = 0;
  std::vector<ParamRef> params;
  std::vector<LayerGrad> lg;
  long long g_head_b = 0, g_u = 0, g_v = 0, g_emb = 0, g_beat = 0, g_bar = 0;
  std::vector<long long> layer_lo_off, layer_hi_off;   // flat span of each layer
  long long tail_off = 0, total = 0;
  float *G = nullptr, *m1 = nullptr, *m2 = nullptr;
  bool own_G = false;
  std::vector<LayerAct> act;
  bf16* xa_last = nullptr;                   // output of the last layer (bf16) = hids[L]
  std::vector<bf16*> mem;                    // L+1 levels [B, M, d] bf16, right-aligned
  bf16* mem_scratch = nullptr;
  int mem_count = 0;
  bf16* pe = nullptr;                        // PositionalEncoding table [M + T, d] bf16
  // workspaces
  float *x32 = nullptr, *dx32 = nullptr, *logits = nullptr, *delta = nullptr, *drk32 = nullptr, *partial = nullptr, *acc = nullptr;
  bf16 *proj = nullptr, *dadd = nullptr, *dh = nullptr, *dattn = nullptr, *dqkv_x = nullptr, *dkv_m = nullptr, *ds_dist = nullptr,
       *qv = nullptr, *drk16 = nullptr, *dlogits = nullptr, *xdrop = nullptr, *dbr = nullptr, *p_buf = nullptr, *ds_buf = nullptr;
  bool dbr_valid = false;                    // dbr holds a branch gradient still to be added to dx32
  bool bert = false;                         // remix encoder (DMG_ARCH_BERT): the *_bert step functions
  long long emb_pad = -1;                    // token row of the embedding that lookups do not train (BERT: pad_idx)
  const long long *ids = nullptr, *pos = nullptr;     // of the latest forward (caller-owned, must stay alive until backward ends)
  int win = 1, k = 1, training = 1;
  long long step = 0;
  int opt_steps = 0;
  int next_layer = -1;                       // backward progress: next layer_hi expected (-1: no forward pending)
  bool mem_pending = false;
  // validation (dmg_train_eval_*): forward-only batches write (ce_sum, kept, correct) to row eval_n of eval_tab, never to acc
  bool eval_fwd = false;                     // the running forward is a validation batch: save nothing for a backward
  bool eval_last = false;                    // the latest forward was a validation batch: its activations are incomplete
  bool eval_open = false;                    // between dmg_train_eval_begin and dmg_train_eval_end
  int eval_cap = 0, eval_max = 0, eval_n = 0;   // allocated rows, rows of this validation, rows written
  double *eval_tab = nullptr, *eval_part = nullptr;   // [eval_cap][3], [EVAL_PART_SLOTS][3]
  const long long* eval_targets = nullptr;
  AdamTensor* adam_tensors = nullptr;
  AdamChunk* adam_chunks = nullptr;
  int n_adam_chunks = 0;
  std::vector<void*> allocs;
  long long bytes = 0;
};

namespace {

template <class T>
int talloc(dmg_train* t, T** p, size_t n) {
  void* q = nullptr;
  const size_t bytes = (n ? n : 1) * sizeof(T);
  DMG_CUDA_OK(cudaMalloc(&q, bytes));
  DMG_CUDA_OK(cudaMemset(q, 0, bytes));
  t->allocs.push_back(q);
  t->bytes += (long long)bytes;
  *p = (T*)q;
  return 0;
}

long long add_param(dmg_train* t, const std::string& name, float* p, bf16* p16, long long n) {
  ParamRef r;
  r.name = name; r.p = p; r.p16 = p16; r.n = n; r.off = t->total;
  t->total += (n + 3) & ~3ll;
  t->params.push_back(r);
  return r.off;
}

std::string reg_name(dmg_model* m, const float* p) {
  for (auto& kv : m->reg)
    if (kv.second.dst == p) return kv.first;
  return std::string();
}

// the parameter list in the order their gradients become final during backward:
// head bias | layer L-1 ... layer 0 | u, v, embedding (tied head weight), beat, bar
int build_params(dmg_model* m, dmg_train* t) {
  const dmg_config& c = m->cfg;
  const int d = c.d_model, HD = m->HD, L = c.n_layers;
  t->params.clear();
  t->total = 0;
  t->g_head_b = add_param(t, reg_name(m, m->head_b), m->head_b, nullptr, c.vocab);
  t->lg.assign(L, LayerGrad());
  t->layer_lo_off.assign(L, 0);
  t->layer_hi_off.assign(L, 0);
  for (int l = L - 1; l >= 0; l--) {
    LayerW& W = m->layers[l];
    LayerGrad& g = t->lg[l];
    t->layer_lo_off[l] = t->total;
    g.wqkv = add_param(t, reg_name(m, W.wqkv.f32), W.wqkv.f32, W.wqkv.b16, (long long)3 * HD * d);
    g.wr = add_param(t, reg_name(m, W.wr.f32), W.wr.f32, W.wr.b16, (long long)HD * d);
    g.wo = add_param(t, reg_name(m, W.wo.f32), W.wo.f32, W.wo.b16, (long long)d * HD);
    g.w1 = add_param(t, reg_name(m, W.w1.f32), W.w1.f32, W.w1.b16, (long long)c.d_inner * d);
    g.w2 = add_param(t, reg_name(m, W.w2.f32), W.w2.f32, W.w2.b16, (long long)d * c.d_inner);
    g.bqkv = g.br = g.bo = -1;
    if (c.attn_bias) {
      g.bqkv = add_param(t, reg_name(m, W.bqkv), W.bqkv, nullptr, 3 * HD);
      g.br = add_param(t, reg_name(m, W.br), W.br, nullptr, HD);
      g.bo = add_param(t, reg_name(m, W.bo), W.bo, nullptr, d);
    }
    g.b1 = add_param(t, reg_name(m, W.b1), W.b1, nullptr, c.d_inner);
    g.b2 = add_param(t, reg_name(m, W.b2), W.b2, nullptr, d);
    g.ln1w = add_param(t, reg_name(m, W.ln1w), W.ln1w, nullptr, d);
    g.ln1b = add_param(t, reg_name(m, W.ln1b), W.ln1b, nullptr, d);
    g.ln2w = add_param(t, reg_name(m, W.ln2w), W.ln2w, nullptr, d);
    g.ln2b = add_param(t, reg_name(m, W.ln2b), W.ln2b, nullptr, d);
    t->layer_hi_off[l] = t->total;
  }
  t->tail_off = t->total;
  t->g_u = add_param(t, reg_name(m, m->u), m->u, nullptr, HD);
  t->g_v = add_param(t, reg_name(m, m->v), m->v, nullptr, HD);
  t->g_emb = add_param(t, "0.encoder.weight", m->emb.f32, m->emb.b16, (long long)c.vocab * d);
  t->g_beat = t->g_bar = -1;
  if (c.encode_position) {
    t->g_beat = add_param(t, reg_name(m, m->beat), m->beat, nullptr, 32ll * d);
    t->g_bar = add_param(t, reg_name(m, m->bar), m->bar, nullptr, 1024ll * d);
  }
  return 0;
}

// remix encoder: same order, per layer q | k | v (one contiguous span: the model stores them as one [3*HD, d] matrix),
// r_attn, their biases, the LayerNorm; tail u, v, embedding (tied head weight), beat, bar
int build_params_bert(dmg_model* m, dmg_train* t) {
  const dmg_config& c = m->cfg;
  const int d = c.d_model, HD = m->HD, L = c.n_layers;
  const long long w = (long long)HD * d;
  t->params.clear();
  t->total = 0;
  t->g_head_b = add_param(t, "head.decoder.bias", m->head_b, nullptr, c.vocab);
  t->lg.assign(L, LayerGrad());
  t->layer_lo_off.assign(L, 0);
  t->layer_hi_off.assign(L, 0);
  for (int l = L - 1; l >= 0; l--) {
    LayerW& W = m->layers[l];
    LayerGrad& g = t->lg[l];
    const std::string p = "encoder.layers." + std::to_string(l) + ".mha1.";
    t->layer_lo_off[l] = t->total;
    g.wo = g.w1 = g.w2 = g.bo = g.b1 = g.b2 = g.ln2w = g.ln2b = g.bqkv = g.br = -1;
    g.wqkv = add_param(t, p + "q_wgt.weight", W.wqkv.f32, W.wqkv.b16, w);
    add_param(t, p + "k_wgt.weight", W.wqkv.f32 + w, W.wqkv.b16 + w, w);
    add_param(t, p + "v_wgt.weight", W.wqkv.f32 + 2 * w, W.wqkv.b16 + 2 * w, w);
    g.wr = add_param(t, p + "r_attn.weight", W.wr.f32, W.wr.b16, w);
    if (c.attn_bias) {
      g.bqkv = add_param(t, p + "q_wgt.bias", W.bqkv, nullptr, HD);
      add_param(t, p + "k_wgt.bias", W.bqkv + HD, nullptr, HD);
      add_param(t, p + "v_wgt.bias", W.bqkv + 2 * HD, nullptr, HD);
      g.br = add_param(t, p + "r_attn.bias", W.br, nullptr, HD);
    }
    g.ln1w = add_param(t, p + "ln.weight", W.ln1w, nullptr, d);
    g.ln1b = add_param(t, p + "ln.bias", W.ln1b, nullptr, d);
    t->layer_hi_off[l] = t->total;
  }
  t->tail_off = t->total;
  t->g_u = add_param(t, "encoder.u", m->u, nullptr, HD);
  t->g_v = add_param(t, "encoder.v", m->v, nullptr, HD);
  t->g_emb = add_param(t, "encoder.embed.embed.weight", m->emb.f32, m->emb.b16, (long long)c.vocab * d);
  t->g_beat = add_param(t, "encoder.embed.beat_enc.weight", m->beat, nullptr, 32ll * d);
  t->g_bar = add_param(t, "encoder.embed.bar_enc.weight", m->bar, nullptr, 1024ll * d);
  return 0;
}

// the r_attn weight has no bf16 copy in the inference model (the rel-pos cache is built in fp32): make one for training
int ensure_wr_b16(dmg_model* m, dmg_train* t) {
  for (auto& W : m->layers) {
    if (W.wr.b16 == nullptr) {
      if (talloc(t, &W.wr.b16, (size_t)W.wr.rows * W.wr.cols)) return -1;
    }
    if (train_cast_bf16(W.wr.f32, W.wr.b16, (long long)W.wr.rows * W.wr.cols, 0)) return -1;
  }
  return 0;
}

// split-K factor of a weight-gradient GEMM: as many K slices as fit in ONE wave of 256 x 256 CTA-pair tiles (the epilogue
// adds fp32 atomics per slice, so more slices than needed only add traffic), at least 8 k-blocks per slice
int pick_splitk(int M, int N, int K, int num_sms) {
  const long long tiles = (long long)((M + 255) / 256) * ((N + 255) / 256);
  const int num_kb = (K + 63) / 64;
  long long s = (num_sms / 2) / tiles;
  if (s > num_kb / 8) s = num_kb / 8;
  if (s < 1) s = 1;
  return (int)s;
}

// weight gradient: G[off] ([Nout, Nin]) += dY^T X  with dY [rows, Nout] (row stride ldy), X [rows, Nin] (row stride ldx)
int grad_w(dmg_model* m, dmg_train* t, const bf16* dY, long long ldy, const bf16* X, long long ldx, int Nout, int Nin, int rows,
           long long off, cudaStream_t st) {
  GemmEpi e;
  e.out = t->G + off; e.ldc = Nin; e.out_mode = GEMM_OUT_ATOMIC;
  return gemm_bf16_tc(dY, 1, ldy, X, 1, ldx, Nout, Nin, rows, pick_splitk(Nout, Nin, rows, m->num_sms), e, m->num_sms, st);
}

int apply_mem_update(dmg_model* m, dmg_train* t, cudaStream_t st, int level_lo, int level_hi) {
  const dmg_config& c = m->cfg;
  const int M = c.mem_len;
  if (M <= 0) return 0;
  for (int l = level_lo; l <= level_hi; l++) {
    if (t->T == M) {   // the whole memory is replaced: trade buffers instead of copying (the old memory becomes next step's scratch)
      std::swap(t->mem[l], l < c.n_layers ? t->act[l].xa_in : t->xa_last);
      continue;
    }
    const bf16* x = l < c.n_layers ? t->act[l].xa_in : t->xa_last;
    if (t->T >= M) {
      if (train_mem_update(t->mem[l], x, t->B, t->T, M, c.d_model, st)) return -1;
    } else {
      if (train_mem_update2(t->mem_scratch, t->mem[l], x, t->B, t->T, M, c.d_model, st)) return -1;
      std::swap(t->mem_scratch, t->mem[l]);
    }
  }
  return 0;
}

int finish_pending_mem(dmg_model* m, dmg_train* t, cudaStream_t st) {
  if (!t->mem_pending) return 0;
  if (apply_mem_update(m, t, st, 0, m->cfg.n_layers - 1)) return -1;
  const int nm = t->mem_count + t->T;
  t->mem_count = nm > m->cfg.mem_len ? m->cfg.mem_len : nm;
  t->mem_pending = false;
  return 0;
}

struct Drop {
  uint32_t thresh, seed;
  float scale;
};
Drop make_drop(dmg_train* t, float p, int site, int layer) {
  Drop d;
  d.thresh = (t->training && p > 0.f) ? drop_thresh16(p) : 0u;
  d.scale = d.thresh ? drop_scale(p) : 1.f;
  d.seed = drop_seed(t->cfg.seed, (uint64_t)t->step, site, layer);
  return d;
}

AttnTrainArgs attn_args(dmg_model* m, dmg_train* t, int l) {
  const dmg_config& c = m->cfg;
  LayerAct& A = t->act[l];
  AttnTrainArgs a;
  a.qkv_x = A.qkv_x; a.ldx = 3 * m->HD;
  a.kv_m = A.kv_m; a.ldm = 2 * m->HD;
  a.rk = A.rk; a.u = m->u; a.v = m->v;
  a.out = A.attn; a.lse = A.lse;
  a.B = t->B; a.T = t->T; a.H = c.n_heads; a.M = c.mem_len; a.mem_count = t->mem_count;
  a.win = t->win; a.k = t->k;
  a.scale = 1.f / sqrtf((float)c.d_head);
  const Drop dr = make_drop(t, t->cfg.attn_p, SITE_ATTN, l);
  a.drop_thresh = dr.thresh; a.drop_seed = dr.seed; a.drop_scale = dr.scale;
  if (A.p_save && !t->eval_fwd && attn_train_fwd_tc_supported(a)) {   // same predicate as the forward dispatch
    a.p_save = A.p_save; a.m_save = A.m_save; a.qu_save = A.qu_save; a.qv_save = A.qv_save;
  }
  return a;
}

// validation head: tied decoder on the last layer's output (the output dropout is the identity in eval mode) and the metrics of
// the batch into row eval_n of the validation table
int eval_head(dmg_model* m, dmg_train* t, long long ignore, cudaStream_t st) {
  const dmg_config& c = m->cfg;
  GemmEpi e; e.bias = m->head_b; e.out = t->logits; e.ldc = t->Vp; e.out_mode = GEMM_OUT_F32;
  if (gemm_bf16_tc(t->xa_last, 0, c.d_model, m->emb.b16, 0, c.d_model, t->rows, c.vocab, c.d_model, 1, e, m->num_sms, st)) return -1;
  return train_eval_metrics(t->logits, t->Vp, t->eval_targets, ignore, t->rows, c.vocab, t->eval_part, t->eval_tab + 3ll * t->eval_n, st);
}

int train_forward(dmg_model* m, dmg_train* t, const long long* ids, const long long* pos, const long long* targets,
                  cudaStream_t st) {
  const dmg_config& c = m->cfg;
  const int d = c.d_model, HD = m->HD, L = c.n_layers, M = c.mem_len, rows = t->rows, S = M + t->T, ns = m->num_sms;
  if (finish_pending_mem(m, t, st)) return -1;
  if (!t->eval_fwd) DMG_CUDA_OK(cudaMemsetAsync(t->acc, 0, 4 * sizeof(float), st));
  {
    const Drop dr = make_drop(t, t->cfg.embed_p, SITE_EMBED, 0);
    if (train_embed(ids, c.encode_position ? pos : nullptr, m->emb.f32, m->beat, m->bar, t->x32, t->act[0].xa_in, rows, d, c.vocab,
                    dr.thresh, dr.seed, dr.scale, st)) return -1;
  }
  for (int l = 0; l < L; l++) {
    LayerW& W = m->layers[l];
    LayerAct& A = t->act[l];
    bf16* xa_out = l + 1 < L ? t->act[l + 1].xa_in : t->xa_last;
    {   // relative-position keys of this step: Rk = PE[0..S) Wr^T (+br)
      GemmEpi e; e.bias = W.br; e.out = A.rk; e.ldc = HD; e.out_mode = GEMM_OUT_BF16;
      if (gemm_bf16_tc(t->pe, 0, d, W.wr.b16, 0, d, S, HD, d, 1, e, ns, st)) return -1;
    }
    {   // q | k | v of the segment
      GemmEpi e; e.bias = W.bqkv; e.out = A.qkv_x; e.ldc = 3 * HD; e.out_mode = GEMM_OUT_BF16;
      if (gemm_bf16_tc(A.xa_in, 0, d, W.wqkv.b16, 0, d, rows, 3 * HD, d, 1, e, ns, st)) return -1;
    }
    if (t->mem_count > 0) {   // k | v of the memory rows (hidden states of the previous segments, current weights)
      GemmEpi e; e.bias = W.bqkv ? W.bqkv + HD : nullptr; e.out = A.kv_m; e.ldc = 2 * HD; e.out_mode = GEMM_OUT_BF16;
      if (gemm_bf16_tc(t->mem[l], 0, d, W.wqkv.b16 + (size_t)HD * d, 0, d, t->B * M, 2 * HD, d, 1, e, ns, st)) return -1;
    }
    {
      const AttnTrainArgs a = attn_args(m, t, l);
      if (attn_train_fwd(a, st)) return -1;
    }
    {   // output projection, dropout, residual, LayerNorm
      GemmEpi e; e.bias = W.bo; e.out = t->proj; e.ldc = d; e.out_mode = GEMM_OUT_BF16;
      if (gemm_bf16_tc(A.attn, 0, HD, W.wo.b16, 0, HD, rows, d, HD, 1, e, ns, st)) return -1;
      const Drop dr = make_drop(t, t->cfg.resid_p, SITE_RES1, l);
      if (train_residual_ln_fwd(t->x32, t->proj, W.ln1w, W.ln1b, A.xa1, A.z1, A.st1, rows, d, dr.thresh, dr.seed, dr.scale, st)) return -1;
    }
    {   // FFN
      const Drop d3 = make_drop(t, t->cfg.ff_p, SITE_FF, l);
      // hpre receives the backward factor gelu'(pre) * dropout instead of the pre-activation (GEMM_ACT_GELU_GRADSAVE)
      GemmEpi e; e.bias = W.b1; e.act = GEMM_ACT_GELU_GRADSAVE; e.out = A.hact; e.ldc = c.d_inner; e.out_mode = GEMM_OUT_BF16;
      e.out2 = A.hpre; e.ld2 = c.d_inner; e.drop_thresh = d3.thresh; e.drop_seed = d3.seed; e.drop_scale = d3.scale;
      if (t->eval_fwd) { e.act = GEMM_ACT_GELU; e.out2 = nullptr; }   // validation: the activation only
      if (gemm_bf16_tc(A.xa1, 0, d, W.w1.b16, 0, d, rows, c.d_inner, d, 1, e, ns, st)) return -1;
      GemmEpi e2; e2.bias = W.b2; e2.out = t->proj; e2.ldc = d; e2.out_mode = GEMM_OUT_BF16;
      if (gemm_bf16_tc(A.hact, 0, c.d_inner, W.w2.b16, 0, c.d_inner, rows, d, c.d_inner, 1, e2, ns, st)) return -1;
      const Drop d4 = make_drop(t, t->cfg.ff_p, SITE_RES2, l);
      if (train_residual_ln_fwd(t->x32, t->proj, W.ln2w, W.ln2b, xa_out, A.z2, A.st2, rows, d, d4.thresh, d4.seed, d4.scale, st)) return -1;
    }
  }
  // head: RNN dropout, tied decoder, cross entropy (+ gradient of the logits), AR, TAR
  if (t->eval_fwd) {   // validation: no dropout, the metrics instead of the loss and dlogits; no AR / TAR (CrossEntropyFlat only)
    if (eval_head(m, t, -1, st)) return -1;
    if (M > 0 && apply_mem_update(m, t, st, L, L)) return -1;   // level L keeps what a training forward leaves there
  } else {
    const Drop dr = make_drop(t, t->cfg.output_p, SITE_OUT, 0);
    if (train_rnn_dropout(t->xa_last, t->xdrop, t->B, t->T, d, dr.thresh, dr.seed, dr.scale, st)) return -1;
    GemmEpi e; e.bias = m->head_b; e.out = t->logits; e.ldc = t->Vp; e.out_mode = GEMM_OUT_F32;
    if (gemm_bf16_tc(t->xdrop, 0, d, m->emb.b16, 0, d, rows, c.vocab, d, 1, e, ns, st)) return -1;
    if (targets) {
      if (train_ce_loss(t->logits, t->Vp, targets, t->dlogits, t->acc + 0, rows, c.vocab, 1.f / rows, st)) return -1;
    }
    if (train_sumsq(t->x32, (long long)rows * d, t->acc + 1, st)) return -1;
    if (M > 0) {
      if (apply_mem_update(m, t, st, L, L)) return -1;   // level L feeds nothing but the TAR value
      const int cnt = t->mem_count + t->T > M ? M : t->mem_count + t->T;
      if (train_tar(t->mem[L] + (size_t)(M - cnt) * d, (long long)M * d, t->B, cnt, d, t->acc + 2, st)) return -1;
    }
  }
  t->mem_pending = M > 0;
  return 0;
}

// dRk[h] = dS_dist[:, h]^T (q + v)[:, h]  ->  dWr = dRk^T PE, r_attn bias = column sums of dRk
int grad_rel_pos(dmg_model* m, dmg_train* t, const bf16* qv_op, const LayerGrad& g, cudaStream_t st) {
  const dmg_config& c = m->cfg;
  const int d = c.d_model, HD = m->HD, rows = t->rows, S = t->S, ns = m->num_sms;
  DMG_CUDA_OK(cudaMemsetAsync(t->drk32, 0, (size_t)S * HD * sizeof(float), st));
  {   // one grouped launch: group h reads dS_dist columns [h*S, (h+1)*S) and (q+v) columns [h*64, (h+1)*64)
    GemmEpi er; er.out = t->drk32; er.ldc = HD; er.out_mode = GEMM_OUT_ATOMIC;
    er.groups = c.n_heads; er.a_gs = S; er.b_gs = 64; er.c_gs = 64;
    int sk = (2 * ns) / (c.n_heads * ((S + 127) / 128));
    if (sk < 1) sk = 1;
    if (sk > rows / 512) sk = rows / 512 > 0 ? rows / 512 : 1;
    if (gemm_bf16_tc(t->ds_dist, 1, (long long)c.n_heads * S, qv_op, 1, HD, S, 64, rows, sk, er, ns, st)) return -1;
  }
  if (train_cast_bf16(t->drk32, t->drk16, (long long)S * HD, st)) return -1;
  if (grad_w(m, t, t->drk16, HD, t->pe, d, HD, d, S, g.wr, st)) return -1;
  if (g.br >= 0 && train_colsum_bf16(t->drk16, HD, S, HD, t->G + g.br, st)) return -1;
  return 0;
}

int backward_head(dmg_model* m, dmg_train* t, cudaStream_t st) {
  const dmg_config& c = m->cfg;
  const int d = c.d_model, rows = t->rows, ns = m->num_sms;
  DMG_CUDA_OK(cudaMemsetAsync(t->G, 0, (size_t)t->total * sizeof(float), st));
  // tied decoder weight: dE += dlogits^T xdrop ; bias ; input gradient
  if (grad_w(m, t, t->dlogits, t->Vp, t->xdrop, d, c.vocab, d, rows, t->g_emb, st)) return -1;
  if (train_colsum_bf16(t->dlogits, t->Vp, rows, c.vocab, t->G + t->g_head_b, st)) return -1;
  {
    GemmEpi e; e.out = t->dadd; e.ldc = d; e.out_mode = GEMM_OUT_BF16;
    if (gemm_bf16_tc(t->dlogits, 0, t->Vp, m->emb.b16, 1, d, rows, d, c.vocab, 1, e, ns, st)) return -1;
  }
  const Drop dr = make_drop(t, t->cfg.output_p, SITE_OUT, 0);
  const float ar_coef = 2.f * t->cfg.alpha / ((float)rows * d);
  t->dbr_valid = false;
  return train_head_bwd(t->dadd, t->x32, t->dx32, t->B, t->T, d, dr.thresh, dr.seed, dr.scale, ar_coef, st);
}

int backward_layer(dmg_model* m, dmg_train* t, int l, cudaStream_t st) {
  const dmg_config& c = m->cfg;
  const int d = c.d_model, HD = m->HD, M = c.mem_len, rows = t->rows, S = M + t->T, ns = m->num_sms, di = c.d_inner;
  LayerW& W = m->layers[l];
  LayerAct& A = t->act[l];
  const LayerGrad& g = t->lg[l];
  // ---- FFN block
  {
    const Drop d4 = make_drop(t, t->cfg.ff_p, SITE_RES2, l);
    if (train_ln_bwd(t->dx32, t->dbr_valid ? t->dbr : nullptr, A.z2, A.st2, W.ln2w, t->dadd, t->G + g.ln2w, t->G + g.ln2b, t->G + g.b2, rows, d,
                     d4.thresh, d4.seed, d4.scale, st)) return -1;   // also the FFN-down bias gradient
    if (grad_w(m, t, t->dadd, d, A.hact, di, d, di, rows, g.w2, st)) return -1;
    // hpre = gelu'(pre) * keep * scale, stored by the forward: one multiply
    GemmEpi e; e.aux = A.hpre; e.ld_aux = di; e.aux_mode = GEMM_AUX_MUL_BF16; e.out = t->dh; e.ldc = di; e.out_mode = GEMM_OUT_BF16;
    if (gemm_bf16_tc(t->dadd, 0, d, W.w2.b16, 1, di, rows, di, d, 1, e, ns, st)) return -1;
    if (grad_w(m, t, t->dh, di, A.xa1, d, di, d, rows, g.w1, st)) return -1;
    if (train_colsum_bf16(t->dh, di, rows, di, t->G + g.b1, st)) return -1;
    // input gradient of the FFN branch, bf16; the LayerNorm backward below adds it to the fp32 residual gradient
    GemmEpi e2; e2.out = t->dbr; e2.ldc = d; e2.out_mode = GEMM_OUT_BF16;
    if (gemm_bf16_tc(t->dh, 0, di, W.w1.b16, 1, d, rows, d, di, 1, e2, ns, st)) return -1;
  }
  // ---- attention block
  {
    const Drop d2 = make_drop(t, t->cfg.resid_p, SITE_RES1, l);
    if (train_ln_bwd(t->dx32, t->dbr, A.z1, A.st1, W.ln1w, t->dadd, t->G + g.ln1w, t->G + g.ln1b, g.bo >= 0 ? t->G + g.bo : nullptr, rows, d,
                     d2.thresh, d2.seed, d2.scale, st)) return -1;
    if (grad_w(m, t, t->dadd, d, A.attn, HD, d, HD, rows, g.wo, st)) return -1;
    GemmEpi e; e.out = t->dattn; e.ldc = HD; e.out_mode = GEMM_OUT_BF16;
    if (gemm_bf16_tc(t->dadd, 0, d, W.wo.b16, 1, HD, rows, HD, d, 1, e, ns, st)) return -1;

    AttnTrainBwdArgs ba;
    ba.f = attn_args(m, t, l);
    ba.dout = t->dattn; ba.delta = t->delta; ba.dqkv_x = t->dqkv_x; ba.dkv_m = t->dkv_m; ba.ds_dist = t->ds_dist; ba.qv = t->qv;
    ba.du = t->G + t->g_u; ba.dv = t->G + t->g_v;
    ba.p_buf = t->p_buf; ba.ds_buf = t->ds_buf;
    const bool q_saved = ba.f.qu_save != nullptr;    // the tcgen05 forward stored q + u and q + v
    if (q_saved) ba.qu = ba.f.qu_save;
    if (attn_train_bwd(ba, st)) return -1;
    const bf16* qv_op = q_saved ? ba.f.qv_save : t->qv;
    if (!q_saved && train_q_plus_bias(A.qkv_x, 3 * HD, m->v, t->qv, rows, HD, st)) return -1;
    if (grad_rel_pos(m, t, qv_op, g, st)) return -1;
    // dWqkv: segment rows, then the memory rows' k|v part
    if (grad_w(m, t, t->dqkv_x, 3 * HD, A.xa_in, d, 3 * HD, d, rows, g.wqkv, st)) return -1;
    if (g.bqkv >= 0 && train_colsum_bf16(t->dqkv_x, 3 * HD, rows, 3 * HD, t->G + g.bqkv, st)) return -1;
    if (t->mem_count > 0) {
      if (grad_w(m, t, t->dkv_m, 2 * HD, t->mem[l], d, 2 * HD, d, t->B * M, g.wqkv + (long long)HD * d, st)) return -1;
      if (g.bqkv >= 0 && train_colsum_bf16(t->dkv_m, 2 * HD, t->B * M, 2 * HD, t->G + g.bqkv + HD, st)) return -1;
    }
    // input gradient of the attention branch, bf16: consumed by the next LayerNorm backward (or the embedding backward)
    GemmEpi e2; e2.out = t->dbr; e2.ldc = d; e2.out_mode = GEMM_OUT_BF16;
    if (gemm_bf16_tc(t->dqkv_x, 0, 3 * HD, W.wqkv.b16, 1, d, rows, d, 3 * HD, 1, e2, ns, st)) return -1;
    t->dbr_valid = true;
  }
  return 0;
}

// remix encoder: per layer ln(x + drop_res(attn(x))) (no out-projection, no FFN), then the head and the masked cross entropy
int train_forward_bert(dmg_model* m, dmg_train* t, const long long* ids, const long long* pos, const long long* targets, cudaStream_t st) {
  const dmg_config& c = m->cfg;
  const int d = c.d_model, HD = m->HD, L = c.n_layers, rows = t->rows, T = t->T, ns = m->num_sms;
  if (!t->eval_fwd) DMG_CUDA_OK(cudaMemsetAsync(t->acc, 0, 8 * sizeof(float), st));
  {
    const Drop dr = make_drop(t, t->cfg.embed_p, SITE_EMBED, 0);
    if (train_embed(ids, pos, m->emb.f32, m->beat, m->bar, t->x32, t->act[0].xa_in, rows, d, c.vocab, dr.thresh, dr.seed, dr.scale, st))
      return -1;
  }
  for (int l = 0; l < L; l++) {
    LayerW& W = m->layers[l];
    LayerAct& A = t->act[l];
    bf16* xa_out = l + 1 < L ? t->act[l + 1].xa_in : t->xa_last;
    {   // relative-position keys Rk = PE[0..T) Wr^T (+br)
      GemmEpi e; e.bias = W.br; e.out = A.rk; e.ldc = HD; e.out_mode = GEMM_OUT_BF16;
      if (gemm_bf16_tc(t->pe, 0, d, W.wr.b16, 0, d, T, HD, d, 1, e, ns, st)) return -1;
    }
    {   // q | k | v
      GemmEpi e; e.bias = W.bqkv; e.out = A.qkv_x; e.ldc = 3 * HD; e.out_mode = GEMM_OUT_BF16;
      if (gemm_bf16_tc(A.xa_in, 0, d, W.wqkv.b16, 0, d, rows, 3 * HD, d, 1, e, ns, st)) return -1;
    }
    if (attn_bert_train_fwd(attn_args(m, t, l), st)) return -1;
    const Drop dr = make_drop(t, t->cfg.resid_p, SITE_RES1, l);   // attention output (HD == d) enters the residual directly
    if (train_residual_ln_fwd(t->x32, A.attn, W.ln1w, W.ln1b, xa_out, A.z1, A.st1, rows, d, dr.thresh, dr.seed, dr.scale, st)) return -1;
  }
  if (t->eval_fwd) return eval_head(m, t, t->cfg.pad_idx, st);
  const Drop dr = make_drop(t, t->cfg.output_p, SITE_OUT, 0);
  if (train_rnn_dropout(t->xa_last, t->xdrop, t->B, T, d, dr.thresh, dr.seed, dr.scale, st)) return -1;
  GemmEpi e; e.bias = m->head_b; e.out = t->logits; e.ldc = t->Vp; e.out_mode = GEMM_OUT_F32;
  if (gemm_bf16_tc(t->xdrop, 0, d, m->emb.b16, 0, d, rows, c.vocab, d, 1, e, ns, st)) return -1;
  if (targets && train_ce_loss_masked(t->logits, t->Vp, targets, t->cfg.pad_idx, t->dlogits, t->acc + 0, t->acc + 4, rows, c.vocab, st))
    return -1;
  return 0;
}

int backward_layer_bert(dmg_model* m, dmg_train* t, int l, cudaStream_t st) {
  const dmg_config& c = m->cfg;
  const int d = c.d_model, HD = m->HD, H = c.n_heads, rows = t->rows, T = t->T, ns = m->num_sms;
  LayerW& W = m->layers[l];
  LayerAct& A = t->act[l];
  const LayerGrad& g = t->lg[l];
  const Drop d2 = make_drop(t, t->cfg.resid_p, SITE_RES1, l);
  // dadd = gradient wrt the attention output
  if (train_ln_bwd(t->dx32, t->dbr_valid ? t->dbr : nullptr, A.z1, A.st1, W.ln1w, t->dadd, t->G + g.ln1w, t->G + g.ln1b, nullptr, rows, d,
                   d2.thresh, d2.seed, d2.scale, st)) return -1;
  AttnTrainBwdArgs ba;
  ba.f = attn_args(m, t, l);
  ba.dout = t->dadd; ba.delta = t->delta; ba.dqkv_x = t->dqkv_x; ba.dkv_m = nullptr; ba.ds_dist = t->ds_dist; ba.qv = t->qv;
  ba.du = t->G + t->g_u; ba.dv = t->G + t->g_v;
  ba.p_buf = t->p_buf; ba.ds_buf = t->ds_buf;
  if (attn_bert_train_bwd(ba, st)) return -1;
  // position part of dq: dq_pos[:, h] = dS_dist[:, h] Rk[:, h] (per head, into dattn); dv = its column sums; dq += dq_pos
  for (int h = 0; h < H; h++) {
    GemmEpi e; e.out = t->dattn + h * 64; e.ldc = HD; e.out_mode = GEMM_OUT_BF16;
    if (gemm_bf16_tc(t->ds_dist + (size_t)h * T, 0, (long long)H * T, A.rk + h * 64, 1, HD, rows, 64, T, 1, e, ns, st)) return -1;
  }
  if (train_colsum_bf16(t->dattn, HD, rows, HD, t->G + t->g_v, st)) return -1;
  if (train_add_bf16(t->dqkv_x, 3 * HD, t->dattn, HD, rows, HD, st)) return -1;
  if (train_q_plus_bias(A.qkv_x, 3 * HD, m->v, t->qv, rows, HD, st)) return -1;
  if (grad_rel_pos(m, t, t->qv, g, st)) return -1;
  if (grad_w(m, t, t->dqkv_x, 3 * HD, A.xa_in, d, 3 * HD, d, rows, g.wqkv, st)) return -1;
  if (g.bqkv >= 0 && train_colsum_bf16(t->dqkv_x, 3 * HD, rows, 3 * HD, t->G + g.bqkv, st)) return -1;
  // input gradient of the attention branch, consumed by the next LayerNorm backward (or the embedding backward)
  GemmEpi e2; e2.out = t->dbr; e2.ldc = d; e2.out_mode = GEMM_OUT_BF16;
  if (gemm_bf16_tc(t->dqkv_x, 0, 3 * HD, W.wqkv.b16, 1, d, rows, d, 3 * HD, 1, e2, ns, st)) return -1;
  t->dbr_valid = true;
  return 0;
}

int backward_embed(dmg_model* m, dmg_train* t, cudaStream_t st) {
  const dmg_config& c = m->cfg;
  const Drop dr = make_drop(t, t->cfg.embed_p, SITE_EMBED, 0);
  return train_embed_bwd(t->ids, c.encode_position ? t->pos : nullptr, t->dx32, t->dbr_valid ? t->dbr : nullptr, t->G + t->g_emb,
                         t->g_beat >= 0 ? t->G + t->g_beat : nullptr, t->g_bar >= 0 ? t->G + t->g_bar : nullptr, t->rows, c.d_model,
                         c.vocab, t->emb_pad, dr.thresh, dr.seed, dr.scale, st);
}

int check_train(dmg_model* m, const char* who) {
  DMG_CHECK(m && m->train, "%s: no training state (call dmg_train_create)", who);
  return 0;
}

}  // namespace

namespace dmg {
int train_weights_reloaded(dmg_model* m, bool reset_optimizer) {
  dmg_train* t = m->train;
  if (t == nullptr) return 0;
  if (ensure_wr_b16(m, t)) return -1;
  if (reset_optimizer) {   // a loaded checkpoint carries no optimizer state here: fastai's learn.create_opt on the new weights
    DMG_CUDA_OK(cudaMemset(t->m1, 0, (size_t)t->total * sizeof(float)));
    DMG_CUDA_OK(cudaMemset(t->m2, 0, (size_t)t->total * sizeof(float)));
    t->opt_steps = 0;
  }
  return 0;
}
}  // namespace dmg

extern "C" {

int64_t dmg_train_param_count(dmg_model* m) {
  if (!m) return -1;
  dmg_train tmp;
  if (m->cfg.arch == DMG_ARCH_BERT) build_params_bert(m, &tmp);
  else build_params(m, &tmp);
  return tmp.total;
}

void dmg_train_destroy(dmg_model* m) {
  if (!m || !m->train) return;
  cudaSetDevice(m->device);
  cudaDeviceSynchronize();
  for (void* p : m->train->allocs) cudaFree(p);
  cudaFree(m->train->eval_tab);
  cudaFree(m->train->eval_part);
  delete m->train;
  m->train = nullptr;
}

int dmg_train_create(dmg_model* m, const dmg_train_config* cfg, float* grad_flat_dev) {
  DMG_CHECK(m && cfg, "dmg_train_create: null argument");
  const dmg_config& c = m->cfg;
  const bool bert = c.arch == DMG_ARCH_BERT;
  DMG_CHECK(m->is_bf16 && m->use_tc, "dmg_train_create: training needs the bf16 tcgen05 model (DMG_BF16, DMG_GEMM_AUTO)");
  DMG_CHECK(m->committed, "dmg_train_create: weights not committed");
  DMG_CHECK(cfg->batch >= 1 && cfg->bptt >= 64 && cfg->bptt % 64 == 0, "dmg_train_create: batch %d / bptt %d (bptt must be a multiple of 64)",
            cfg->batch, cfg->bptt);
  DMG_CHECK(c.mem_len % 64 == 0, "dmg_train_create: mem_len %d must be a multiple of 64", c.mem_len);
  DMG_CHECK((bert || c.d_inner % 64 == 0) && c.d_model % 128 == 0, "dmg_train_create: d_inner %% 64 and d_model %% 128 required");
  DMG_CHECK(!bert || (cfg->pad_idx >= 0 && cfg->pad_idx < c.vocab), "dmg_train_create: pad_idx %d outside the vocabulary", cfg->pad_idx);
  const float ps[5] = {cfg->resid_p, cfg->attn_p, cfg->ff_p, cfg->embed_p, cfg->output_p};
  for (float p : ps) DMG_CHECK(p >= 0.f && p < 0.95f, "dmg_train_create: dropout probability %f outside [0, 0.95)", p);
  DMG_CUDA_OK(cudaSetDevice(m->device));
  if (m->train) dmg_train_destroy(m);
  dmg_train* t = new dmg_train();
  m->train = t;
  t->cfg = *cfg;
  t->B = cfg->batch; t->T = cfg->bptt; t->rows = t->B * t->T;
  const int d = c.d_model, HD = m->HD, L = c.n_layers, M = c.mem_len, rows = t->rows, S = M + t->T, di = c.d_inner;
  t->S = S;
  t->Vp = (c.vocab + 63) / 64 * 64;
  t->bert = bert;
  if (bert) {   // the encoder has no AR / TAR terms
    t->cfg.alpha = t->cfg.beta = 0.f;
    t->emb_pad = cfg->pad_idx;
    build_params_bert(m, t);
  } else {
    build_params(m, t);
  }
  int rc = 0;
#define TRY(x) do { if (!rc && (x)) rc = -1; } while (0)
  if (grad_flat_dev) { t->G = grad_flat_dev; t->own_G = false; }
  else { TRY(talloc(t, &t->G, (size_t)t->total)); t->own_G = true; }
  TRY(talloc(t, &t->m1, (size_t)t->total));
  TRY(talloc(t, &t->m2, (size_t)t->total));
  t->act.resize(L);
  const size_t BM = (size_t)t->B * (M > 0 ? M : 1);
  for (int l = 0; l < L && !rc && bert; l++) {
    LayerAct& A = t->act[l];
    TRY(talloc(t, &A.xa_in, (size_t)rows * d));
    TRY(talloc(t, &A.qkv_x, (size_t)(rows + 1) * 3 * HD));   // + the zero row the last query tile reads as "next row"
    TRY(talloc(t, &A.attn, (size_t)rows * HD));
    TRY(talloc(t, &A.z1, (size_t)rows * d));
    bf16* rk = nullptr;   // Rk rows -64 .. T+127: the zero rows the attention's rel-pos windows read past both ends
    TRY(talloc(t, &rk, (size_t)(S + 192) * HD));
    A.rk = rk + (size_t)64 * HD;
    TRY(talloc(t, &A.lse, (size_t)t->B * c.n_heads * t->T));
    TRY(talloc(t, &A.st1, (size_t)rows));
  }
  for (int l = 0; l < L && !rc && !bert; l++) {
    LayerAct& A = t->act[l];
    TRY(talloc(t, &A.xa_in, (size_t)rows * d));
    TRY(talloc(t, &A.qkv_x, (size_t)rows * 3 * HD));
    TRY(talloc(t, &A.kv_m, BM * 2 * HD));
    TRY(talloc(t, &A.attn, (size_t)rows * HD));
    TRY(talloc(t, &A.z1, (size_t)rows * d));
    TRY(talloc(t, &A.xa1, (size_t)rows * d));
    TRY(talloc(t, &A.hpre, (size_t)rows * di));
    TRY(talloc(t, &A.hact, (size_t)rows * di));
    TRY(talloc(t, &A.z2, (size_t)rows * d));
    TRY(talloc(t, &A.rk, (size_t)S * HD));
    TRY(talloc(t, &A.lse, (size_t)t->B * c.n_heads * t->T));
    if (t->T % 128 == 0 && c.mem_len % 128 == 0) {   // geometry the tcgen05 forward serves
      TRY(talloc(t, &A.p_save, (size_t)t->B * c.n_heads * t->T * S));
      TRY(talloc(t, &A.m_save, (size_t)t->B * c.n_heads * t->T * (S / 64)));
      TRY(talloc(t, &A.qu_save, (size_t)rows * HD));
      TRY(talloc(t, &A.qv_save, (size_t)rows * HD));
    }
    TRY(talloc(t, &A.st1, (size_t)rows));
    TRY(talloc(t, &A.st2, (size_t)rows));
  }
  TRY(talloc(t, &t->xa_last, (size_t)rows * d));
  if (M > 0) {
    t->mem.assign(L + 1, nullptr);
    for (int l = 0; l <= L; l++) TRY(talloc(t, &t->mem[l], BM * d));
    TRY(talloc(t, &t->mem_scratch, BM * d));
  }
  TRY(talloc(t, &t->pe, (size_t)S * d));
  TRY(talloc(t, &t->x32, (size_t)rows * d));
  TRY(talloc(t, &t->dx32, (size_t)rows * d));
  TRY(talloc(t, &t->logits, (size_t)rows * t->Vp));
  TRY(talloc(t, &t->dlogits, (size_t)rows * t->Vp));
  TRY(talloc(t, &t->xdrop, (size_t)rows * d));
  TRY(talloc(t, &t->delta, (size_t)t->B * c.n_heads * t->T));
  TRY(talloc(t, &t->drk32, (size_t)S * HD));
  TRY(talloc(t, &t->drk16, (size_t)S * HD));
  {
    size_t pn = (size_t)148 * 4 * 2 * (size_t)(di > 3 * HD ? di : 3 * HD);
    TRY(talloc(t, &t->partial, pn));
  }
  TRY(talloc(t, &t->acc, 8));
  TRY(talloc(t, &t->proj, (size_t)rows * d));
  TRY(talloc(t, &t->dadd, (size_t)rows * d));
  TRY(talloc(t, &t->dbr, (size_t)rows * d));
  if (!bert) TRY(talloc(t, &t->dh, (size_t)rows * di));
  TRY(talloc(t, &t->dattn, (size_t)rows * HD));
  TRY(talloc(t, &t->dqkv_x, (size_t)rows * 3 * HD));
  TRY(talloc(t, &t->dkv_m, BM * 2 * HD));
  TRY(talloc(t, &t->ds_dist, (size_t)rows * c.n_heads * S));
  TRY(talloc(t, &t->qv, (size_t)rows * HD));
  TRY(talloc(t, &t->p_buf, (size_t)rows * c.n_heads * S));    // P / dS spilled by the dQ kernel for dK / dV
  TRY(talloc(t, &t->ds_buf, (size_t)rows * c.n_heads * S));
  {   // multi-tensor Adam tables
    std::vector<AdamTensor> ht;
    std::vector<AdamChunk> hc;
    for (size_t i = 0; i < t->params.size(); i++) {
      const ParamRef& p = t->params[i];
      AdamTensor at; at.p = p.p; at.p16 = p.p16; at.off = p.off;
      ht.push_back(at);
      for (long long s0 = 0; s0 < p.n; s0 += 16384) {
        AdamChunk ch; ch.t = (int)i; ch.start = (int)s0; ch.len = (int)(p.n - s0 < 16384 ? p.n - s0 : 16384);
        hc.push_back(ch);
      }
    }
    t->n_adam_chunks = (int)hc.size();
    TRY(talloc(t, &t->adam_tensors, ht.size()));
    TRY(talloc(t, &t->adam_chunks, hc.size()));
    if (!rc && cudaMemcpy(t->adam_tensors, ht.data(), ht.size() * sizeof(AdamTensor), cudaMemcpyHostToDevice) != cudaSuccess) rc = -1;
    if (!rc && cudaMemcpy(t->adam_chunks, hc.data(), hc.size() * sizeof(AdamChunk), cudaMemcpyHostToDevice) != cudaSuccess) rc = -1;
  }
  TRY(train_posenc(t->pe, S, d, 0));
  TRY(ensure_wr_b16(m, t));
#undef TRY
  if (!rc && cudaDeviceSynchronize() != cudaSuccess) { set_error("dmg_train_create: device error after setup"); rc = -1; }
  if (rc) { dmg_train_destroy(m); return rc; }
  m->bytes += t->bytes;
  return 0;
}

int dmg_train_reset(dmg_model* m) {
  if (check_train(m, "dmg_train_reset")) return -2;
  m->train->mem_count = 0;
  m->train->mem_pending = false;
  m->train->next_layer = -1;
  return 0;
}

int dmg_train_forward(dmg_model* m, const int64_t* ids_dev, const int64_t* pos_dev, const int64_t* targets_dev, int mask_win,
                      int mask_k, int training, int64_t step, void* stream) {
  if (check_train(m, "dmg_train_forward")) return -2;
  DMG_CHECK(ids_dev, "dmg_train_forward: null ids");
  DMG_CHECK(!m->cfg.encode_position || pos_dev, "dmg_train_forward: model encodes position but pos is NULL");
  DMG_CHECK((mask_win == 1 && mask_k == 1) || (mask_win >= 1 && mask_k == 0), "dmg_train_forward: window mask (%d,%d) unsupported", mask_win, mask_k);
  DMG_CHECK(!m->train->bert || (mask_win == 1 && mask_k == 1), "dmg_train_forward: the remix encoder has no attention mask, (mask_win, mask_k) must be (1, 1), got (%d,%d)",
            mask_win, mask_k);
  DMG_CUDA_OK(cudaSetDevice(m->device));
  dmg_train* t = m->train;
  t->ids = (const long long*)ids_dev; t->pos = (const long long*)pos_dev;
  t->win = mask_win; t->k = mask_k; t->training = training ? 1 : 0; t->step = step;
  t->eval_last = false;
  if (t->bert ? train_forward_bert(m, t, t->ids, t->pos, (const long long*)targets_dev, (cudaStream_t)stream)
              : train_forward(m, t, t->ids, t->pos, (const long long*)targets_dev, (cudaStream_t)stream)) return -1;
  t->next_layer = targets_dev ? m->cfg.n_layers : -1;
  return 0;
}

int dmg_train_backward(dmg_model* m, int layer_hi, int layer_lo, void* stream) {
  if (check_train(m, "dmg_train_backward")) return -2;
  dmg_train* t = m->train;
  const int L = m->cfg.n_layers;
  DMG_CHECK(layer_hi >= layer_lo && layer_lo >= 0 && layer_hi <= L, "dmg_train_backward: bad slice [%d, %d)", layer_lo, layer_hi);
  DMG_CHECK(!t->eval_last, "dmg_train_backward: the latest forward was a validation batch (dmg_train_eval_batch), which saves nothing "
            "for a backward; run dmg_train_forward with targets first");
  DMG_CHECK(t->next_layer == layer_hi, "dmg_train_backward: slice starts at layer %d but %d is next (forward with targets first, slices in descending order)",
            layer_hi, t->next_layer);
  DMG_CUDA_OK(cudaSetDevice(m->device));
  cudaStream_t st = (cudaStream_t)stream;
  if (layer_hi == L && backward_head(m, t, st)) return -1;
  for (int l = layer_hi - 1; l >= layer_lo; l--)
    if (t->bert ? backward_layer_bert(m, t, l, st) : backward_layer(m, t, l, st)) return -1;
  t->next_layer = layer_lo;
  if (layer_lo == 0) {
    if (backward_embed(m, t, st)) return -1;
    if (finish_pending_mem(m, t, st)) return -1;
    t->next_layer = -1;
  }
  return 0;
}

int dmg_train_eval_begin(dmg_model* m, int max_batches) {
  if (check_train(m, "dmg_train_eval_begin")) return -2;
  DMG_CHECK(max_batches >= 1, "dmg_train_eval_begin: max_batches %d must be at least 1", max_batches);
  dmg_train* t = m->train;
  DMG_CUDA_OK(cudaSetDevice(m->device));
  DMG_CUDA_OK(cudaDeviceSynchronize());   // a previous table may still be read by queued work
  if (t->eval_part == nullptr) DMG_CUDA_OK(cudaMalloc(&t->eval_part, (size_t)EVAL_PART_SLOTS * 3 * sizeof(double)));
  if (t->eval_cap < max_batches) {
    cudaFree(t->eval_tab);
    t->eval_tab = nullptr;
    t->eval_cap = 0;
    DMG_CUDA_OK(cudaMalloc(&t->eval_tab, (size_t)max_batches * 3 * sizeof(double)));
    t->eval_cap = max_batches;
  }
  DMG_CUDA_OK(cudaMemset(t->eval_tab, 0, (size_t)t->eval_cap * 3 * sizeof(double)));
  DMG_CUDA_OK(cudaDeviceSynchronize());
  t->eval_max = max_batches;
  t->eval_n = 0;
  t->eval_open = true;
  return 0;
}

int dmg_train_eval_batch(dmg_model* m, const int64_t* ids_dev, const int64_t* pos_dev, const int64_t* targets_dev, void* stream) {
  if (check_train(m, "dmg_train_eval_batch")) return -2;
  dmg_train* t = m->train;
  DMG_CHECK(t->eval_open, "dmg_train_eval_batch: no validation table (call dmg_train_eval_begin first)");
  DMG_CHECK(t->eval_n < t->eval_max, "dmg_train_eval_batch: batch %d is past max_batches = %d of dmg_train_eval_begin", t->eval_n + 1,
            t->eval_max);
  DMG_CHECK(ids_dev && targets_dev, "dmg_train_eval_batch: null ids or targets");
  DMG_CHECK(!t->bert || pos_dev, "dmg_train_eval_batch: the remix encoder adds beat/bar embeddings, pos is required");
  DMG_CHECK(!m->cfg.encode_position || pos_dev, "dmg_train_eval_batch: model encodes position but pos is NULL");
  DMG_CUDA_OK(cudaSetDevice(m->device));
  // model.eval(): no dropout, the (1,1) mask; ids / pos / step of the latest training forward stay as they are
  t->win = 1; t->k = 1; t->training = 0;
  t->eval_fwd = true;
  t->eval_targets = (const long long*)targets_dev;
  const int rc = t->bert ? train_forward_bert(m, t, (const long long*)ids_dev, (const long long*)pos_dev, nullptr, (cudaStream_t)stream)
                         : train_forward(m, t, (const long long*)ids_dev, (const long long*)pos_dev, nullptr, (cudaStream_t)stream);
  t->eval_fwd = false;
  t->eval_targets = nullptr;
  t->eval_last = true;
  t->next_layer = -1;
  if (rc) return -1;
  t->eval_n++;
  return 0;
}

int dmg_train_eval_end(dmg_model* m, double* out_host, int n_batches, void* stream) {
  if (check_train(m, "dmg_train_eval_end")) return -2;
  dmg_train* t = m->train;
  DMG_CHECK(t->eval_open, "dmg_train_eval_end: no validation table (call dmg_train_eval_begin first)");
  DMG_CHECK(out_host, "dmg_train_eval_end: null output");
  DMG_CHECK(n_batches == t->eval_n, "dmg_train_eval_end: n_batches = %d but %d batches were validated", n_batches, t->eval_n);
  DMG_CUDA_OK(cudaSetDevice(m->device));
  t->eval_open = false;
  if (n_batches == 0) return 0;
  DMG_CUDA_OK(cudaMemcpyAsync(out_host, t->eval_tab, (size_t)n_batches * 3 * sizeof(double), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  DMG_CUDA_OK(cudaStreamSynchronize((cudaStream_t)stream));
  return 0;
}

int dmg_eval_metrics(const float* logits_dev, int64_t ldl, const int64_t* targets_dev, int64_t ignore, int rows, int V, double* out3_dev,
                     void* stream) {
  DMG_CHECK(logits_dev && targets_dev && out3_dev, "dmg_eval_metrics: null argument");
  DMG_CHECK(rows >= 0 && V >= 1 && ldl >= V, "dmg_eval_metrics: rows %d, V %d, ldl %lld (need rows >= 0, V >= 1, ldl >= V)", rows, V,
            (long long)ldl);
  return train_eval_metrics(logits_dev, ldl, (const long long*)targets_dev, ignore, rows, V, nullptr, out3_dev, (cudaStream_t)stream);
}

int dmg_train_grad_span(dmg_model* m, int layer_hi, int layer_lo, int64_t* offset, int64_t* count) {
  if (check_train(m, "dmg_train_grad_span")) return -2;
  dmg_train* t = m->train;
  const int L = m->cfg.n_layers;
  DMG_CHECK(offset && count && layer_hi >= layer_lo && layer_lo >= 0 && layer_hi <= L, "dmg_train_grad_span: bad arguments");
  // final after backward(layer_hi, layer_lo): the head bias (slice starting at L), the layers of the slice (stored in
  // descending order), and - only once layer 0 is done - u, v and the embeddings, which every layer accumulates into
  long long lo = 0, hi = 0;
  if (layer_hi > layer_lo) {
    lo = layer_hi == L ? 0 : t->layer_lo_off[layer_hi - 1];
    hi = layer_lo == 0 ? t->total : t->layer_hi_off[layer_lo];
  } else if (layer_hi == L) {
    lo = 0; hi = L > 0 ? t->layer_lo_off[L - 1] : t->total;
  } else if (layer_lo == 0) {
    lo = t->tail_off; hi = t->total;
  }
  *offset = lo;
  *count = hi - lo;
  return 0;
}

int dmg_train_grad_pack(dmg_model* m, int64_t offset, int64_t count, void* wire_bf16_dev, void* stream) {
  if (check_train(m, "dmg_train_grad_pack")) return -2;
  dmg_train* t = m->train;
  DMG_CHECK(wire_bf16_dev && offset >= 0 && count >= 0 && offset + count <= t->total, "dmg_train_grad_pack: bad span");
  DMG_CUDA_OK(cudaSetDevice(m->device));
  return train_grad_pack(t->G + offset, (bf16*)wire_bf16_dev, count, (cudaStream_t)stream);
}

int dmg_train_grad_unpack(dmg_model* m, int64_t offset, int64_t count, const void* wire_bf16_dev, void* stream) {
  if (check_train(m, "dmg_train_grad_unpack")) return -2;
  dmg_train* t = m->train;
  DMG_CHECK(wire_bf16_dev && offset >= 0 && count >= 0 && offset + count <= t->total, "dmg_train_grad_unpack: bad span");
  DMG_CUDA_OK(cudaSetDevice(m->device));
  return train_grad_unpack((const bf16*)wire_bf16_dev, t->G + offset, count, (cudaStream_t)stream);
}

int dmg_train_optimizer_step(dmg_model* m, float lr, float beta1, float beta2, float eps, float wd, float clip, float grad_scale,
                             void* stream) {
  if (check_train(m, "dmg_train_optimizer_step")) return -2;
  dmg_train* t = m->train;
  DMG_CUDA_OK(cudaSetDevice(m->device));
  cudaStream_t st = (cudaStream_t)stream;
  // the norm of the (all-reduced) gradient, summed in a fixed order: every rank must scale its update by the same bits
  if (train_sumsq_det(t->G, t->total, t->partial, 148 * 4, t->acc + 3, st)) return -1;
  t->opt_steps++;
  if (train_adam(t->adam_tensors, t->adam_chunks, t->n_adam_chunks, t->G, t->m1, t->m2, lr, beta1, beta2, eps, wd, t->opt_steps, clip,
                 t->acc + 3, grad_scale, st)) return -1;
  m->committed = false;   // the inference rel-pos key cache is stale now
  return 0;
}

int dmg_train_losses(dmg_model* m, float* out4_host, void* stream) {
  if (check_train(m, "dmg_train_losses")) return -2;
  DMG_CHECK(out4_host, "dmg_train_losses: null output");
  dmg_train* t = m->train;
  DMG_CUDA_OK(cudaSetDevice(m->device));
  float a[5];
  DMG_CUDA_OK(cudaMemcpyAsync(a, t->acc, sizeof(a), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  DMG_CUDA_OK(cudaStreamSynchronize((cudaStream_t)stream));
  const int d = m->cfg.d_model, M = m->cfg.mem_len;
  if (t->bert) {   // mean over the targets that are not pad_idx (NaN when there are none, as torch gives); no AR / TAR
    out4_host[0] = a[0] / a[4];
    out4_host[1] = out4_host[2] = 0.f;
    out4_host[3] = sqrtf(a[3]);
    return 0;
  }
  out4_host[0] = a[0] / t->rows;
  out4_host[1] = t->cfg.alpha * a[1] / ((float)t->rows * d);
  int cnt = t->mem_count + (t->mem_pending ? t->T : 0);
  if (cnt > M) cnt = M;
  out4_host[2] = (M > 0 && cnt > 1) ? t->cfg.beta * a[2] / ((float)t->B * (cnt - 1) * d) : 0.f;
  out4_host[3] = sqrtf(a[3]);
  return 0;
}

int dmg_train_get_grad(dmg_model* m, const char* name, float* out_host, int64_t numel) {
  if (check_train(m, "dmg_train_get_grad")) return -2;
  DMG_CHECK(name && out_host, "dmg_train_get_grad: null argument");
  dmg_train* t = m->train;
  std::string key = name;
  if (key == "1.decoder.weight") key = "0.encoder.weight";
  for (auto& p : t->params) {
    if (p.name != key) continue;
    DMG_CHECK(p.n == numel, "dmg_train_get_grad: %s has %lld elements, asked for %lld", name, p.n, (long long)numel);
    DMG_CUDA_OK(cudaSetDevice(m->device));
    DMG_CUDA_OK(cudaDeviceSynchronize());
    DMG_CUDA_OK(cudaMemcpy(out_host, t->G + p.off, (size_t)numel * 4, cudaMemcpyDeviceToHost));
    return 0;
  }
  return 1;
}

// Adam state of one parameter by its state-dict name: which = 1 (exp_avg) or 2 (exp_avg_sq); set = 0 reads into buf_host, 1 writes
int dmg_train_opt_state(dmg_model* m, const char* name, int which, int set, float* buf_host, int64_t numel) {
  if (check_train(m, "dmg_train_opt_state")) return -2;
  DMG_CHECK(name && buf_host && (which == 1 || which == 2), "dmg_train_opt_state: bad arguments");
  dmg_train* t = m->train;
  std::string key = name;
  if (key == "1.decoder.weight") key = "0.encoder.weight";
  for (auto& p : t->params) {
    if (p.name != key) continue;
    DMG_CHECK(p.n == numel, "dmg_train_opt_state: %s has %lld elements, got %lld", name, p.n, (long long)numel);
    DMG_CUDA_OK(cudaSetDevice(m->device));
    DMG_CUDA_OK(cudaDeviceSynchronize());
    float* dev = (which == 1 ? t->m1 : t->m2) + p.off;
    if (set) DMG_CUDA_OK(cudaMemcpy(dev, buf_host, (size_t)numel * 4, cudaMemcpyHostToDevice));
    else DMG_CUDA_OK(cudaMemcpy(buf_host, dev, (size_t)numel * 4, cudaMemcpyDeviceToHost));
    return 0;
  }
  return 1;
}

// optimizer step counter (Adam bias correction): value < 0 reads it, otherwise sets it; returns the (new) value
int64_t dmg_train_opt_steps(dmg_model* m, int64_t value) {
  if (!m || !m->train) return -1;
  if (value >= 0) m->train->opt_steps = (int)value;
  return m->train->opt_steps;
}

float* dmg_train_grad_buffer(dmg_model* m) { return (m && m->train) ? m->train->G : nullptr; }

int dmg_train_dropout_mask(dmg_model* m, int site, int layer, int64_t step, float* out_dev, int64_t numel, void* stream) {
  if (check_train(m, "dmg_train_dropout_mask")) return -2;
  dmg_train* t = m->train;
  DMG_CHECK(out_dev && site >= 0 && site <= 5, "dmg_train_dropout_mask: bad arguments");
  const float ps[6] = {t->cfg.embed_p, t->cfg.attn_p, t->cfg.resid_p, t->cfg.ff_p, t->cfg.ff_p, t->cfg.output_p};
  const float p = ps[site];
  const uint32_t th = p > 0.f ? drop_thresh16(p) : 0u;
  const uint32_t seed = drop_seed(t->cfg.seed, (uint64_t)step, site, (site == SITE_EMBED || site == SITE_OUT) ? 0 : layer);
  DMG_CUDA_OK(cudaSetDevice(m->device));
  return train_export_mask(out_dev, numel, th, seed, th ? drop_scale(p) : 1.f, (cudaStream_t)stream);
}

int dmg_gemm_train(const void* a_dev, int a_mn, int64_t lda, const void* b_dev, int b_mn, int64_t ldb, int M, int N, int K,
                   int splitk, const float* bias_dev, int gelu, const void* aux_dev, int64_t ld_aux, int aux_mode, void* out_dev,
                   int64_t ldc, int out_mode, void* out2_dev, int64_t ld2, float drop_p, uint32_t drop_seed_v, void* stream) {
  DMG_CHECK(a_dev && b_dev && out_dev, "dmg_gemm_train: null argument");
  int dev = 0, sms = 148;
  DMG_CUDA_OK(cudaGetDevice(&dev));
  DMG_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  GemmEpi e;
  e.bias = bias_dev; e.act = gelu; e.aux = aux_dev; e.ld_aux = ld_aux; e.aux_mode = aux_mode; e.out = out_dev; e.ldc = ldc;
  e.out_mode = out_mode; e.out2 = (bf16*)out2_dev; e.ld2 = ld2;
  if (drop_p > 0.f) { e.drop_thresh = drop_thresh16(drop_p); e.drop_scale = drop_scale(drop_p); e.drop_seed = drop_seed_v; }
  return gemm_bf16_tc((const bf16*)a_dev, a_mn, lda, (const bf16*)b_dev, b_mn, ldb, M, N, K, splitk, e, sms, (cudaStream_t)stream);
}

static AttnTrainArgs make_attn_args(const void* qkv_x, int64_t ldx, const void* kv_m, int64_t ldm, const void* rk, const float* u,
                                    const float* v, void* out, float* lse, int B, int T, int H, int M, int mem_count, int win, int k,
                                    float drop_p, uint32_t seed) {
  AttnTrainArgs a;
  a.qkv_x = (const bf16*)qkv_x; a.ldx = ldx; a.kv_m = (const bf16*)kv_m; a.ldm = ldm; a.rk = (const bf16*)rk; a.u = u; a.v = v;
  a.out = (bf16*)out; a.lse = lse; a.B = B; a.T = T; a.H = H; a.M = M; a.mem_count = mem_count; a.win = win; a.k = k;
  a.scale = 0.125f;
  a.drop_thresh = drop_p > 0.f ? drop_thresh16(drop_p) : 0u;
  a.drop_scale = drop_p > 0.f ? drop_scale(drop_p) : 1.f;
  a.drop_seed = seed;
  return a;
}

int dmg_attn_train_fwd(const void* qkv_x, int64_t ldx, const void* kv_m, int64_t ldm, const void* rk, const float* u, const float* v,
                       void* out, float* lse, int B, int T, int H, int M, int mem_count, int win, int k, float drop_p,
                       uint32_t drop_seed_v, void* p_save, float* m_save, void* stream) {
  DMG_CHECK(qkv_x && rk && u && v && out && lse, "dmg_attn_train_fwd: null argument");
  AttnTrainArgs a = make_attn_args(qkv_x, ldx, kv_m, ldm, rk, u, v, out, lse, B, T, H, M, mem_count, win, k, drop_p, drop_seed_v);
  if (p_save && m_save) {
    DMG_CHECK(attn_train_fwd_tc_supported(a), "dmg_attn_train_fwd: p_save needs the tcgen05 forward (T, M, mem_count multiples of 128)");
    a.p_save = (bf16*)p_save; a.m_save = m_save;
  }
  return attn_train_fwd(a, (cudaStream_t)stream);
}

int dmg_attn_train_bwd(const void* qkv_x, int64_t ldx, const void* kv_m, int64_t ldm, const void* rk, const float* u, const float* v,
                       const void* out, const float* lse, const void* dout, int B, int T, int H, int M, int mem_count, int win, int k,
                       float drop_p, uint32_t drop_seed_v, float* delta, void* dqkv_x, void* dkv_m, void* ds_dist, float* du,
                       float* dv, const void* p_save, const float* m_save, void* stream) {
  DMG_CHECK(qkv_x && rk && u && v && out && lse && dout && delta && dqkv_x && ds_dist && du && dv, "dmg_attn_train_bwd: null argument");
  AttnTrainBwdArgs ba;
  ba.f = make_attn_args(qkv_x, ldx, kv_m, ldm, rk, u, v, const_cast<void*>(out), const_cast<float*>(lse), B, T, H, M, mem_count, win,
                        k, drop_p, drop_seed_v);
  ba.dout = (const bf16*)dout; ba.delta = delta; ba.dqkv_x = (bf16*)dqkv_x; ba.dkv_m = (bf16*)dkv_m; ba.ds_dist = (bf16*)ds_dist;
  ba.qv = nullptr; ba.du = du; ba.dv = dv;
  if (p_save && m_save) { ba.f.p_save = (bf16*)const_cast<void*>(p_save); ba.f.m_save = const_cast<float*>(m_save); }
  static bf16* ws = nullptr;          // spill workspace of this test hook: kept between calls, regrown on demand
  static size_t ws_elems = 0;
  const size_t n = (size_t)B * H * T * (M + T);
  if (ws_elems < 2 * n) {
    if (ws) { DMG_CUDA_OK(cudaDeviceSynchronize()); cudaFree(ws); ws = nullptr; ws_elems = 0; }
    DMG_CUDA_OK(cudaMalloc(&ws, 2 * n * sizeof(bf16)));
    ws_elems = 2 * n;
  }
  ba.p_buf = ws; ba.ds_buf = ws + n;
  // (q + u) operand of the tcgen05 dK/dV kernel (in the trainer the tcgen05 forward stores it)
  static bf16* qu_ws = nullptr;
  static size_t qu_elems = 0;
  const size_t nq = (size_t)B * T * H * 64;
  if (qu_elems < nq) {
    if (qu_ws) { DMG_CUDA_OK(cudaDeviceSynchronize()); cudaFree(qu_ws); qu_ws = nullptr; qu_elems = 0; }
    DMG_CUDA_OK(cudaMalloc(&qu_ws, nq * sizeof(bf16)));
    qu_elems = nq;
  }
  if (train_q_plus_bias((const bf16*)qkv_x, ldx, u, qu_ws, B * T, H * 64, (cudaStream_t)stream)) return -1;
  ba.qu = qu_ws;
  return attn_train_bwd(ba, (cudaStream_t)stream);
}

int dmg_attn_bert_train_fwd(const void* qkv_x, int64_t ldx, const void* rk, const float* u, const float* v, void* out, float* lse,
                            int B, int T, int H, float drop_p, uint32_t drop_seed_v, void* stream) {
  DMG_CHECK(qkv_x && rk && u && v && out && lse, "dmg_attn_bert_train_fwd: null argument");
  return attn_bert_train_fwd(make_attn_args(qkv_x, ldx, nullptr, 0, rk, u, v, out, lse, B, T, H, 0, 0, 1, 1, drop_p, drop_seed_v),
                             (cudaStream_t)stream);
}

int dmg_attn_bert_train_bwd(const void* qkv_x, int64_t ldx, const void* rk, const float* u, const float* v, const void* out,
                            const float* lse, const void* dout, int B, int T, int H, float drop_p, uint32_t drop_seed_v, float* delta,
                            void* dqkv_x, void* ds_dist, float* du, void* p_buf, void* ds_buf, void* stream) {
  DMG_CHECK(qkv_x && rk && u && v && out && lse && dout && delta && dqkv_x && du, "dmg_attn_bert_train_bwd: null argument");
  DMG_CHECK(ds_dist, "dmg_attn_bert_train_bwd: ds_dist [B*T, H*T] is required");
  DMG_CHECK(p_buf && ds_buf, "dmg_attn_bert_train_bwd: p_buf and ds_buf [B*H, T, T] are required");
  AttnTrainBwdArgs ba;
  ba.f = make_attn_args(qkv_x, ldx, nullptr, 0, rk, u, v, const_cast<void*>(out), const_cast<float*>(lse), B, T, H, 0, 0, 1, 1, drop_p,
                        drop_seed_v);
  ba.dout = (const bf16*)dout; ba.delta = delta; ba.dqkv_x = (bf16*)dqkv_x; ba.dkv_m = nullptr; ba.ds_dist = (bf16*)ds_dist;
  ba.qv = nullptr; ba.du = du; ba.dv = nullptr;
  ba.p_buf = (bf16*)p_buf; ba.ds_buf = (bf16*)ds_buf;
  return attn_bert_train_bwd(ba, (cudaStream_t)stream);
}

}  // extern "C"
