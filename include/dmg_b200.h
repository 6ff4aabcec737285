/*
 * dmg_b200.h - C ABI of the B200-native DeepMusicGeneration hot path (libdmg_b200.so).
 *
 * The reference (AniketRajpoot/DeepMusicGeneration) is pure Python: it has no plugin / FFI layer, its
 * boundary is the Python call surface of the model and the learner.  Each entry point below names the
 * reference call it stands behind (paths relative to the reference checkout).  The Python host package
 * `deepmusicgeneration_b200` binds these with ctypes and re-creates that call surface on top.
 *
 * Conventions: plain pointers and sizes only; every function returns 0 on success, non-zero on error
 * (message via dmg_last_error()); no exceptions cross the ABI; no internal threads; all device work is
 * enqueued on the caller's stream (a cudaStream_t passed as void*, NULL = legacy default stream);
 * "_dev" pointers are device memory of the model's device, "_host" pointers are host memory;
 * the caller owns every buffer it passes; the model owns weights, the K/V memory rings, the
 * relative-position key cache and its workspaces.
 */
#ifndef DMG_B200_H
#define DMG_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct dmg_model dmg_model;

enum { DMG_ARCH_TXL = 0,   /* MusicTransformerXL + LinearDecoder   (deep_music_genre.py:1603-1647, fastai TransformerXL) */
       DMG_ARCH_BERT = 1   /* MultiTransformer 'msk' branch: MTEncoder + MTLinearDecoder (deep_music_remix.py:1864-2104) */ };
enum { DMG_F32 = 0, DMG_BF16 = 1 };
enum { DMG_GEMM_AUTO = 0,  /* bf16: tcgen05/TMEM/TMA kernels (cluster split-K for <= 512 rows); f32: SIMT fp32 kernel */
       DMG_GEMM_SIMT = 1,  /* debugging: SIMT kernel for every dtype */
       DMG_GEMM_TC_TILE = 2 /* dmg_gemm_bf16 only: the one-CTA-per-tile tcgen05 kernel even for skinny shapes */ };
enum { DMG_LOGITS_NONE = 0, DMG_LOGITS_ALL = 1, DMG_LOGITS_LAST = 2 };
/* dmg_config.kernel_flags: selectors of the non-default kernels, for the parity tests (every alternative kernel is compared with the
 * default one and with the oracle) and for reproducing the measurements in profiles/README.md.  0 = the product path.  The
 * environment variable DMG_<NAME> sets the same bit; the environment is read once, in dmg_create. */
enum { DMG_KF_NO_DECODE_KERNEL = 1,  /* one-token steps through the general attention kernel instead of attention_decode2.cu        */
       DMG_KF_NO_FLASH = 2,          /* memory-less bf16 segments (prefill, BERT) through the general FFMA attention kernel           */
       DMG_KF_NO_GRAPH = 4,          /* generation loop launched kernel by kernel instead of replaying the captured CUDA graph        */
       DMG_KF_BERT_MMA_SYNC = 8,     /* BERT attention on the mma.sync flash kernel for every length (env DMG_BERT_ATTN_MMA_SYNC)      */
       DMG_KF_BERT_FP32_STRIP = 16,  /* BERT tcgen05 attention with fp32 strip lines (env DMG_BERT_TC_FP32_STRIP)                      */
       DMG_KF_NO_SPLITK = 32,        /* one-token GEMMs without cluster split-K                                                       */
       DMG_KF_NO_BIG_GEMM = 64,      /* many-row GEMMs on gemm_tc_kernel instead of the persistent CTA-pair kernel                    */
       DMG_KF_GEMM_SIMT = 128,       /* every GEMM on the FFMA kernel                                                                 */
       DMG_KF_NO_FUSED_DECODE = 256, /* one-token step as separate GEMM / LayerNorm launches instead of the fused layer kernels       */
       DMG_KF_NO_DUAL_DECODE = 512,  /* fused layer kernels and attention as separate launches over all streams instead of the two-half
                                        software pipeline (fused step of one half + attention of the other half in ONE dual-role launch) */
       DMG_KF_ATTN_DECODE_V2 = 1024  /* one-token attention on the second-generation kernel (one consumer group, resident rel-pos keys)      */ };

/* Model hyper-parameters: the keys of the reference config dicts (app_utils.py:13-63, fastai tfmerXL_lm_config). */
typedef struct dmg_config {
  int32_t arch;             /* DMG_ARCH_*                                                                 */
  int32_t dtype;            /* DMG_F32 (parity mode) or DMG_BF16 (fast path)                              */
  int32_t vocab;            /* len(vocab.itos) = 324                                                      */
  int32_t d_model, n_layers, n_heads, d_head, d_inner;
  int32_t mem_len;          /* TXL segment-recurrence memory (config['mem_len']); 0 for the BERT encoder  */
  int32_t attn_bias;        /* config['bias']: bias on attention / r_attn (/ out) Linears                  */
  int32_t encode_position;  /* BeatPositionEncoder / TransformerEmbedding beat+bar embeddings             */
  int32_t max_batch;        /* streams whose K/V rings stay resident in HBM                               */
  int32_t max_seq;          /* longest x_len of one forward call                                          */
  int32_t max_rows;         /* activation workspace rows per chunk; 0 = max_batch*max_seq                 */
  int32_t keep_hidden;      /* also keep the reference's hidden-state mems (model[0].hidden) for export   */
  int32_t gemm_backend;     /* DMG_GEMM_*                                                                 */
  int32_t kernel_flags;     /* DMG_KF_* (0 = product path)                                                */
  int32_t reserved[3];
} dmg_config;

/* Index layout of MusicVocab (deep_music_genre.py:812-890); ranges are [lo, hi). */
typedef struct dmg_vocab_layout {
  int32_t bos, pad, eos, mask, ni, sep;
  int32_t special_lo, special_hi;    /* SPECIAL_TOKS */
  int32_t note_lo, note_hi, dur_lo, dur_hi, ins_lo, ins_hi;
} dmg_vocab_layout;

enum { DMG_SAMPLE_EARLY_STOP = 1,    /* the loop's break rules (deep_music_genre.py:1951-1963)                         */
       DMG_SAMPLE_MASK_UNUSED = 2,   /* also forbid ids >= ins_hi (mt*, dummy*), which the reference never filters      */
       DMG_SAMPLE_REMIX_FILTER = 4   /* filter_invalid_indexes of deep_music_remix.py:2394-2437 instead of the genre one */ };

/* Arguments of MusicLearner.predict (deep_music_genre.py:1853-1855). */
typedef struct dmg_sampler_params {
  double temperatures[3];    /* [0] after instrument/pad, [1] after note/xxsep, [2] after duration (:1913-1918);
                                Python floats in the reference, hence double                                   */
  int32_t min_bars;
  int32_t top_k;
  float top_p;
  int32_t n_words;
  uint32_t allowed_ins_mask; /* bit i set = instrument i allowed; 0 = allowed_ins is None                    */
  int32_t flags;             /* DMG_SAMPLE_*                                                                 */
  uint64_t seed;             /* Philox key of the device multinomial                                         */
} dmg_sampler_params;

const char* dmg_last_error(void);
int dmg_abi_version(void);

/* get_language_model / get_multitask_model (deep_music_genre.py:1793, deep_music_remix.py:1851-1862): allocate
 * the model on CUDA device `device`. */
int dmg_create(const dmg_config* cfg, int device, dmg_model** out);
void dmg_destroy(dmg_model* m);

/* load_state_dict(state['model'], strict=False) (deep_music_genre.py:1800): one call per tensor, fastai
 * state-dict key names (SURVEY.md App. A.8), fp32 host data in nn.Module layout.  Unknown names return 1
 * (ignored, like strict=False) without setting an error. */
int dmg_set_weight(dmg_model* m, const char* name, const float* data_host, int64_t numel);
int dmg_get_weight(dmg_model* m, const char* name, float* out_host, int64_t numel);
/* Must follow the last dmg_set_weight: makes bf16 copies, runs the rel-pos R-projection (r_attn over
 * PositionalEncoding) into the per-layer key cache, builds the TMA tensor maps. */
int dmg_commit_weights(dmg_model* m);

/* SequentialRNN.reset() -> TransformerXL.reset() (deep_music_genre.py:1857): drop all memory; `batch`
 * streams become active. */
int dmg_reset(dmg_model* m, int batch);
/* TransformerXL.select_hidden(idxs) (used by beam_search, deep_music_genre.py:1847): new stream j takes
 * the memory of old stream idx[j]. */
int dmg_select_hidden(dmg_model* m, const int32_t* idx_host, int n);
/* hidden[0].size(1) of the reference: number of memory positions currently held. */
int dmg_mem_count(dmg_model* m);

/* model(x) (deep_music_genre.py:1617-1647 + LinearDecoder; deep_music_remix.py:1874-1881 for DMG_ARCH_BERT).
 * ids_dev/pos_dev: int64 [bs, x_len] (pos_dev may be NULL unless encode_position).  mask_win/mask_k: the
 * (win_size, k) pair of window_mask (:1577-1584); eval mode is (1, 1).  logits_dev: fp32 [bs, x_len, V]
 * (DMG_LOGITS_ALL) or [bs, V] (DMG_LOGITS_LAST) or NULL.  core_out_dev: fp32 [bs, x_len, d_model] or NULL.
 * Appends the segment to the memory exactly like _update_mems. */
int dmg_forward(dmg_model* m, const int64_t* ids_dev, const int64_t* pos_dev, int bs, int x_len, int mask_win,
                int mask_k, int logits_mode, float* logits_dev, float* core_out_dev, void* stream);

/* raw_outputs[level] of the reference forward (= model[0].hidden[level]): fp32 [bs, mem_count, d_model].
 * Needs cfg.keep_hidden. */
int dmg_get_hidden(dmg_model* m, int level, float* out_dev, void* stream);

/* MusicLearner.predict state (deep_music_genre.py:1856-1881): per stream the previous token (item.data[-1]),
 * last_pos = pos[-1]; start_pos = last_pos. */
int dmg_sampler_init(dmg_model* m, const dmg_vocab_layout* vocab, const dmg_sampler_params* params,
                     const int32_t* prev_idx_host, const int64_t* last_pos_host, int bs);

/* The body of the `for i in range(n_words)` loop (deep_music_genre.py:1883-1967), n_steps times, entirely on
 * the device: sample from the logits of the latest forward (temperature, grammar filter, top-k/top-p,
 * multinomial), then run the one-token forward on the sampled ids.  dmg_forward(..., DMG_LOGITS_LAST, NULL)
 * (the prefill of the seed) must precede the first call.  tokens_dev: int32 [n_steps, bs]; -1 marks a stream
 * that has stopped (BOS predicted / bar rule); -2 marks a stream whose previous token has no temperature class
 * (the reference raises AssertionError there, :1920-1925). */
int dmg_generate(dmg_model* m, int n_steps, int32_t* tokens_dev, void* stream);
/* Same loop body, ONE step, through host buffers: copies ids_host (int64 [bs], may be NULL to keep the sampled
 * ids) in, runs sample+forward, copies the bs sampled tokens out to tokens_host and synchronises the stream. */
int dmg_generate_step_host(dmg_model* m, const int64_t* ids_host, int32_t* tokens_host, void* stream);

/* Sampling only (top_k_top_p + filter + multinomial over caller-provided logits), for predict_mask
 * (deep_music_remix.py:2586-2609; temperatures[0] after duration/pad else [1], the ten special ids forbidden,
 * the remix filter): logits_dev fp32 [n, V]; prev_idx_dev, repeat_count_dev int32 [n]; out_dev (sampled ids) and
 * num_choices_dev (non-zero probabilities, drives repeat_count) int32 [n]. */
int dmg_sample_logits(dmg_model* m, const float* logits_dev, const int32_t* prev_idx_dev,
                      const int32_t* repeat_count_dev, int n, const dmg_vocab_layout* vocab,
                      const dmg_sampler_params* params, uint64_t offset, int32_t* out_dev, int32_t* num_choices_dev,
                      void* stream);

/* One step of MusicLearner.beam_search (deep_music_genre.py:1834-1847) on the logits of the latest DMG_LOGITS_LAST forward over `nb`
 * beams: log_softmax, top_k per beam, scores = -logp + previous score (scores_dev: fp32 [n_scores], n_scores = 1 broadcasts like the
 * reference's zeros(1)), the beam_sz lowest scores survive.  Outputs (device): scores [beam_sz], the parent beam of each survivor
 * (feed it to dmg_select_hidden) and the token it appends.  Exact ties go to the lower candidate index. */
int dmg_beam_step(dmg_model* m, const float* scores_dev, int n_scores, int nb, int top_k, int beam_sz, float* scores_out_dev,
                  int32_t* parents_out_dev, int32_t* tokens_out_dev, void* stream);

/* Test hook: ONE sampling step for n independent rows that also returns the final probabilities probs_dev fp32 [n, V] (may be
 * NULL) - their support is the set kept by the grammar filter, top-k and top-p.  predict_loop = 0: predict_mask's step (as
 * dmg_sample_logits; last_xxsep_dev / pos_since_start_dev ignored).  predict_loop = 1: the step of MusicLearner.predict
 * (deep_music_genre.py:1895-1944) on caller-provided loop state: prev_idx, repeat_count, last_xxsep as they are BEFORE the update
 * of :1897-1901, and last_pos - start_pos (for the min_bars rule :1937); nothing is written back. */
int dmg_sample_probs(dmg_model* m, int predict_loop, const float* logits_dev, const int32_t* prev_idx_dev,
                     const int32_t* repeat_count_dev, const int32_t* last_xxsep_dev, const int64_t* pos_since_start_dev, int n,
                     const dmg_vocab_layout* vocab, const dmg_sampler_params* params, uint64_t offset, int32_t* out_dev,
                     int32_t* num_choices_dev, float* probs_dev, void* stream);

/* Introspection for tests / bench. */
int64_t dmg_device_bytes(dmg_model* m);          /* bytes of HBM owned by the model */
int64_t dmg_launch_count(void);                  /* kernels launched by this library so far (process-wide) */
int dmg_uses_tcgen05(dmg_model* m);              /* 1 when GEMMs run on the tcgen05 kernel */

/* Measurement hook: %globaltimer marks (ns) of CTA 0 of one mid-stack launch of the fused one-token layer kernel (decode_layer.cu):
 * 3 roles (TMA producer, MMA issuer, epilogue thread) x 16 marks, then - when that launch is a dual-role launch - 4 marks of the attention
 * role ([48] first attention CTA starts, [49] its rel-pos table is built, [50] it ends, [51] the last attention CTA ends): 64 values.
 * Needs DMG_DECODE_TIMELINE=1 in the environment at dmg_create. */
int dmg_decode_timeline(dmg_model* m, uint64_t* out64_host);

/* Measurement hook for bench.py's roofline: re-launch ONLY the fused decode-attention kernel of `layer` on the
 * current ring state and the q/k/v of the latest one-token forward (idempotent: the ring position is not advanced). */
int dmg_attn_decode_layer(dmg_model* m, int layer, void* stream);

/* The same for the dominant launch of the pipelined one-token step (decode_dual_kernel): the attention of `layer` over the second
 * half of the streams together with the fused layer step (body of `layer`, q|k|v of `layer + 1`) of the first half, exactly as the
 * step issues it.  Advances nothing on the host side, but rewrites the residual stream of the first half: call it after the run. */
int dmg_decode_dual_launch(dmg_model* m, int layer, void* stream);

/* Stand-alone GEMM entry (unit tests / micro-benchmarks): C[M,N] = A[M,K] * W[N,K]^T (+bias) (gelu),
 * bf16 inputs on the device, fp32 or bf16 output.  backend: DMG_GEMM_AUTO = tcgen05, DMG_GEMM_SIMT. */
int dmg_gemm_bf16(const void* a_dev, const void* w_dev, const float* bias_dev, void* c_dev, int M, int N, int K,
                  int gelu, int out_bf16, int backend, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Training step (SURVEY.md 3.3, App. A.7): what fastai's Learner.fit does around the reference model for one batch -
 * model(x) in train mode (deep_music_genre.py:1617-1647 with dropout and rand_window_mask :1586-1590), CrossEntropyFlat
 * + RNNTrainer's AR/TAR terms, loss.backward(), Adam with decoupled weight decay.  bf16 compute (tcgen05 GEMMs, mma.sync
 * flash attention with the rel-pos term), fp32 master weights / residual stream / gradients.  Needs a DMG_BF16 model:
 * DMG_ARCH_TXL, or DMG_ARCH_BERT for masked-LM training of the remix encoder (the msk task of MultiTransformer,
 * deep_music_remix.py:1874-1881: CrossEntropyFlat(ignore_index=pad_idx), no memory, no AR/TAR, no attention mask).
 * Data-parallel training: every rank runs forward/backward on its own sequences and all-reduces the flat gradient buffer
 * (dmg_train_grad_span tells which slice is final after which backward call) before the step.
 * ------------------------------------------------------------------------------------------------------------------ */
typedef struct dmg_train_config {
  int32_t batch;            /* sequences per step on this GPU (each keeps its own memory, like bs rows of the reference batch) */
  int32_t bptt;             /* tokens per sequence and step (x_len), a multiple of 64                                          */
  float resid_p, attn_p, ff_p, embed_p, output_p;   /* dropout probabilities, already multiplied by drop_mult (App. A.1/A.2)    */
  float alpha, beta;        /* RNNTrainer activation regularisation (AR) and temporal AR (TAR, value only), App. A.7           */
  uint64_t seed;            /* base seed of the counter-based dropout masks                                                    */
  int32_t pad_idx;          /* DMG_ARCH_BERT: the loss's ignore index and the embedding's padding_idx (ignored for DMG_ARCH_TXL) */
  int32_t reserved[3];
} dmg_train_config;

/* Allocates activations / gradient / Adam state.  grad_flat_dev: caller-owned fp32 device buffer of
 * dmg_train_param_count() elements that receives the gradients (e.g. a torch tensor handed to NCCL), or NULL to let the
 * model own one.  Call dmg_train_param_count first (it works before dmg_train_create). */
int64_t dmg_train_param_count(dmg_model* m);
int dmg_train_create(dmg_model* m, const dmg_train_config* cfg, float* grad_flat_dev);
void dmg_train_destroy(dmg_model* m);
/* RNNTrainer.on_epoch_begin -> model.reset(): forget the training memory (hidden states of the previous segments); a no-op
 * for DMG_ARCH_BERT, which has no memory. */
int dmg_train_reset(dmg_model* m);
/* model(x) in train mode + loss.  ids/targets (and pos when encode_position): int64 [batch, bptt] on the device.
 * (mask_win, mask_k): what rand_window_mask drew on the host, (1,1) or (w,0); always (1,1) for DMG_ARCH_BERT, whose
 * targets are the masked copy of x (mask_tfm) with pad_idx at every position not to be predicted.  training = 0 disables every dropout
 * (model.eval() semantics with the training memory).  `step` keys the dropout masks. */
int dmg_train_forward(dmg_model* m, const int64_t* ids_dev, const int64_t* pos_dev, const int64_t* targets_dev, int mask_win,
                      int mask_k, int training, int64_t step, void* stream);
/* loss.backward() in slices so that the gradient all-reduce can overlap: runs the head (when layer_hi == n_layers) and
 * the layers layer_hi-1 ... layer_lo; layer_lo == 0 also runs the embedding and finishes the step (memory update).
 * Slices must be issued in descending order and cover n_layers..0 exactly once per forward. */
int dmg_train_backward(dmg_model* m, int layer_hi, int layer_lo, void* stream);
/* Flat-gradient slice that is final once dmg_train_backward(m, layer_hi, layer_lo) has run. */
int dmg_train_grad_span(dmg_model* m, int layer_hi, int layer_lo, int64_t* offset, int64_t* count);
/* Wire format of the data-parallel gradient exchange: the slice [offset, offset+count) of the flat fp32 gradient packed to bf16
 * (round to nearest even) into a caller-owned device buffer of `count` bf16 elements, and back (overwrites the fp32 slice) after
 * the all-reduce.  Halves the bytes on NVLink (SURVEY.md 8e: 109.5 MB instead of 219 MB per step for the 16-layer model). */
int dmg_train_grad_pack(dmg_model* m, int64_t offset, int64_t count, void* wire_bf16_dev, void* stream);
int dmg_train_grad_unpack(dmg_model* m, int64_t offset, int64_t count, const void* wire_bf16_dev, void* stream);
/* Adam(betas, eps) with fastai's true_wd (p *= 1 - lr*wd first), gradients scaled by grad_scale (1/world_size after a
 * SUM all-reduce) and clipped to global norm `clip` (<= 0: no clipping); refreshes the bf16 weight copies.
 * Inference entry points need dmg_commit_weights() again afterwards (the rel-pos key cache follows r_attn). */
int dmg_train_optimizer_step(dmg_model* m, float lr, float beta1, float beta2, float eps, float wd, float clip,
                             float grad_scale, void* stream);
/* MusicLearner.save(with_opt=True) / the optimizer half of music_model_learner(pretrained_path=...) (deep_music_genre.py:1801-1803,
 * 1812-1821): Adam's exp_avg (which = 1) / exp_avg_sq (which = 2) of one parameter by its state-dict name, fp32 host buffer;
 * set = 0 reads, 1 writes.  Unknown names return 1.  dmg_train_opt_steps: the step counter of the bias correction (value < 0 reads). */
int dmg_train_opt_state(dmg_model* m, const char* name, int which, int set, float* buf_host, int64_t numel);
int64_t dmg_train_opt_steps(dmg_model* m, int64_t value);
/* Synchronises the stream and returns {cross-entropy (mean), alpha*AR, beta*TAR, gradient norm (after grad_scale; 0 before
 * the first optimizer step)} of the latest step.  DMG_ARCH_BERT: {mean CE over the targets != pad_idx (NaN if there are
 * none; the gradients are then zero), 0, 0, gradient norm}. */
int dmg_train_losses(dmg_model* m, float* out4_host, void* stream);
/* Tests: gradient of one parameter by its state-dict name; the dropout mask (keep ? 1/(1-p) : 0) of a site as the kernels
 * generate it (site 0 embedding [rows,d], 1 attention [B,H,T,S], 2 attention-residual [rows,d], 3 FFN inner [rows,d_inner],
 * 4 FFN residual [rows,d], 5 output RNN dropout [B,d]; DMG_ARCH_BERT uses 0, 1 [B,H,T,T], 2 and 5); the device pointer of the
 * owned gradient buffer. */
int dmg_train_get_grad(dmg_model* m, const char* name, float* out_host, int64_t numel);
int dmg_train_dropout_mask(dmg_model* m, int site, int layer, int64_t step, float* out_dev, int64_t numel, void* stream);
float* dmg_train_grad_buffer(dmg_model* m);
/* Unit-test entry of the training GEMM (persistent tcgen05 kernel): C[M,N] = op(A) op(B); a_mn / b_mn = 1 when the
 * reduction index is the slow one in memory; out_mode 0 fp32, 1 bf16, 2 fp32 atomic accumulate (split-K allowed);
 * aux_mode 0 none, 1 multiply by gelu'(aux bf16), 2 add aux bf16, 3 add aux fp32. */
int dmg_gemm_train(const void* a_dev, int a_mn, int64_t lda, const void* b_dev, int b_mn, int64_t ldb, int M, int N, int K,
                   int splitk, const float* bias_dev, int gelu, const void* aux_dev, int64_t ld_aux, int aux_mode, void* out_dev,
                   int64_t ldc, int out_mode, void* out2_dev, int64_t ld2, float drop_p, uint32_t drop_seed, void* stream);
/* Unit-test entries of the training attention kernels (attention_train.cu, attention_train_tc.cu): see AttnTrainArgs for
 * the layouts.  p_save [B*H, T, M+T] bf16 and m_save [B*H, T, (M+T)/64] fp32 are optional (both or neither, tcgen05
 * forward only = T, M, mem_count multiples of 128): the forward saves the undropped probabilities there and the backward,
 * given the same pair, rebuilds P from them instead of recomputing the scores. */
int dmg_attn_train_fwd(const void* qkv_x, int64_t ldx, const void* kv_m, int64_t ldm, const void* rk, const float* u,
                       const float* v, void* out, float* lse, int B, int T, int H, int M, int mem_count, int win, int k,
                       float drop_p, uint32_t drop_seed, void* p_save, float* m_save, void* stream);
int dmg_attn_train_bwd(const void* qkv_x, int64_t ldx, const void* kv_m, int64_t ldm, const void* rk, const float* u,
                       const float* v, const void* out, const float* lse, const void* dout, int B, int T, int H, int M,
                       int mem_count, int win, int k, float drop_p, uint32_t drop_seed, float* delta, void* dqkv_x, void* dkv_m,
                       void* ds_dist, float* du, float* dv, const void* p_save, const float* m_save, void* stream);

/* ---- training data feed (SURVEY.md section 8 f4) ------------------------------------------------------------------------
 * dmg_preload_fill = MusicPreloader.__getitem__ / fill_row (deep_music_genre.py:1088-1125) for all `bs` rows of one batch.
 * Everything is device memory: `tokens` / `positions` the flat ragged corpus (int32), `offsets` [n_items+1] (int64), `perm` the
 * CircularIndex permutation (:1005-1014, int64), `transpose` the per-item semitone shift or NULL (MusicItem.transpose :1247,
 * applied to ids in [note_lo, note_hi)), `ro` / `ri` [bs] the row cursors (in/out), `x` / `y` [bs, bptt] int64 (y = the stream
 * shifted by y_offset), `xpos` [bs, bptt] the positions of x or NULL (batch_position_tfm :1129-1136).  forward = !backwards. */
int dmg_preload_fill(const int32_t* tokens, const int32_t* positions, const int64_t* offsets, const int64_t* perm, int n_items,
                     int forward, const int32_t* transpose, int note_lo, int note_hi, int64_t* ro, int64_t* ri, int bs, int bptt,
                     int y_offset, int64_t* x, int64_t* y, int64_t* xpos, void* stream);
/* mask_tfm (deep_music_remix.py:1208-1223) in place on device tensors of n elements: tokens inside [mask_lo, mask_hi) are
 * masked with probability 0.8 p, replaced by a random token of the range with 0.1 p, left with 0.1 p; y becomes pad_idx where
 * nothing was selected.  rand_out / wrong_out (nullable, n elements) export the uniform draw and the replacement candidate of
 * every element (test hooks: the oracle replays them). */
int dmg_mask_tfm(int64_t* x, int64_t* y, int64_t n, int mask_lo, int mask_hi, int mask_idx, int pad_idx, double p, uint32_t seed,
                 float* rand_out, int64_t* wrong_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DMG_B200_H */
