// Model object of libdmg_b200.so, shared by model.cu (inference) and train.cu (training).
#pragma once
#include <map>
#include <string>
#include <vector>

#include "../../include/dmg_b200.h"
#include "kernels.cuh"
#include "sampling.cuh"

struct dmg_train;

namespace dmg {

struct Weight {
  float* f32 = nullptr;   // master copy, nn.Linear layout [rows(out), cols(in)]
  bf16* b16 = nullptr;
  int rows = 0, cols = 0;
  TensorMap2D tm32, tm128;   // TMA maps with 32- and 128-row boxes
  TensorMap2D tm64;          // 64-row boxes (fused decode layer kernel)
  bool has_tm = false;
};

struct LayerW {
  Weight wqkv, wr, wo, w1, w2;
  float *bqkv = nullptr, *br = nullptr, *bo = nullptr, *b1 = nullptr, *b2 = nullptr;
  float *ln1w = nullptr, *ln1b = nullptr, *ln2w = nullptr, *ln2b = nullptr;
  void* rd = nullptr;      // [H][Dcap][Dh] compute dtype: r_attn(PositionalEncoding(dist))
  void* kring = nullptr;   // [max_batch][H][M][Dh] compute dtype
  void* vring = nullptr;
  TensorMap2D tmK, tmV, tmR;   // 64-row boxes over the rings / the rel-pos cache (decode attention v2)
  bool has_ring_tm = false;
};

struct RegEntry {
  float* dst;
  long long numel;
};

enum ABuf { A_XA = 0, A_ATTN = 1, A_H = 2, A_XLAST = 3, A_COUNT = 4 };


}  // namespace dmg

using dmg::Weight; using dmg::LayerW; using dmg::RegEntry; using dmg::TensorMap2D; using dmg::SampleArgs; using dmg::A_COUNT;

struct dmg_model {
  dmg_config cfg;
  int kflags = 0;   // DMG_KF_* kernel selectors: cfg.kernel_flags | the DMG_* environment variables, read ONCE at dmg_create
  int device = 0;
  bool is_bf16 = false, use_tc = false, committed = false;
  bool weights_set_externally = false;   // dmg_set_weight since the last commit (a checkpoint was loaded over a live trainer)
  int HD = 0, Dcap = 0, max_rows = 0, esz = 4, num_sms = 148;
  Weight emb;   // [V, d] (tied head)
  float *beat = nullptr, *bar = nullptr, *u = nullptr, *v = nullptr, *head_b = nullptr;
  std::vector<LayerW> layers;
  std::vector<float*> hrings;   // (L+1) x [max_batch][M][d] fp32 when keep_hidden
  std::map<std::string, RegEntry> reg;
  std::vector<void*> allocs;
  long long bytes = 0;
  // memory state: per stream {pos_total (tokens appended since reset), mem_count (valid memory positions, <= mem_len)}, on the device
  // ([max_batch][2], read by the kernels, also under graph replay) and its host mirror.  Rows >= batch are zero.
  std::vector<long long> pos_total;
  std::vector<int> mem_count;
  int batch = 0;
  int* dev_state = nullptr;
  // workspaces
  float *x32 = nullptr, *qkv = nullptr, *proj = nullptr, *logits_buf = nullptr;
  bf16* qkv16 = nullptr;        // bf16 q|k|v of a segment for the flash-attention path
  void *xa = nullptr, *attn = nullptr, *hbuf = nullptr, *xlast = nullptr;
  TensorMap2D tmA[A_COUNT];
  // fused one-token layer step (decode_layer.cu)
  bool fused_decode = false;
  float* dl_PP = nullptr;
  long long dl_pp_stride = 0;
  int dl_rows = 0, dl_max_clusters = 0;
  bool dl_dual = false;                    // the two-half software pipeline with dual-role launches
  TensorMap2D tmAttn16;
  unsigned long long* dl_dbg = nullptr;   // DMG_DECODE_TIMELINE=1: timeline of the fused kernel's CTA 0 (the LAST launch wins)
  int a_rows[A_COUNT], a_cols[A_COUNT];
  // generation loop
  bool samp_ready = false, logits_valid = false;
  SampleArgs samp;
  long long *ids_buf = nullptr, *pos_buf = nullptr;
  int* tok_buf = nullptr;
  cudaStream_t cap_stream = nullptr;
  cudaGraphExec_t step_graph = nullptr;
  int graph_bs = -1;
  long long graph_launches = 0;
  dmg_train* train = nullptr;   // training state (train.cu), created by dmg_train_create
  // batched remix (remix_batch.cu), BERT models: per-sequence lengths with their attention routing, and the mask loop's device state
  int *vl_lens = nullptr, *vl_items = nullptr, *vl_seqs = nullptr;
  int *mk_pos = nullptr, *mk_n = nullptr, *mk_streams = nullptr, *mk_prev = nullptr, *mk_rc = nullptr, *mk_tok = nullptr, *mk_nc = nullptr,
      *mk_step = nullptr;
};

namespace dmg {

// train.cu: called by dmg_commit_weights when a trainer exists - refreshes the bf16 r_attn copies the training forward multiplies
// with and, when the weights were replaced from outside (load_state_dict over a live trainer), restarts Adam (zero moments, step 0)
int train_weights_reloaded(dmg_model* m, bool reset_optimizer);

template <class T>
inline int dalloc(dmg_model* m, T** p, size_t n, bool zero = true) {
  void* q = nullptr;
  const size_t bytes = (n ? n : 1) * sizeof(T);
  DMG_CUDA_OK(cudaMalloc(&q, bytes));
  if (zero) DMG_CUDA_OK(cudaMemset(q, 0, bytes));
  m->allocs.push_back(q);
  m->bytes += (long long)bytes;
  *p = (T*)q;
  return 0;
}

}  // namespace dmg
