#pragma once
#include "../../include/dmg_b200.h"
#include "common.cuh"

namespace dmg {

struct SampleArgs {
  const float* logits;        // [n, V] fp32
  int V;
  dmg_vocab_layout vocab;
  dmg_sampler_params params;
  int loop_mode;              // 1: MusicLearner.predict loop state below; 0: stateless (predict_mask);
                              // 2: one stateless step of the predict loop (test hook: state is read, never written)
  unsigned long long offset;  // Philox counter base
  // loop state, one entry per stream
  int* prev_idx;
  int* repeat_count;
  int* last_xxsep;
  long long* last_pos;
  long long* start_pos;
  int* step;
  int* status;                // 0 running, 1 stopped (break), 2 no temperature class (reference AssertionError)
  // outputs
  int* out_tokens;            // [n] sampled id, -1 stopped, -2 error (may be NULL in loop mode)
  long long* next_ids;        // [n] input ids of the next one-token forward (loop mode)
  long long* next_pos;        // [n] beat position of the next token (loop mode, may be NULL)
  int* num_choices;           // [n] optional
  float* probs;               // [n, V] optional: the final probabilities (after filter / top-k / top-p / softmax)
  // optional (the batched remix): Philox stream of row i = stream_ids[i] instead of i; *dev_offset is added to the counter
  const int* stream_ids;
  const int* dev_offset;
};

int sample_launch(const SampleArgs& a, int n, cudaStream_t st);

// The mask step of the batched remix (remix_batch.cu): device state of B items of a padded batch (row b*T_max + t)
struct MaskStepArgs {
  long long* ids;             // [B*T_max] in / out: the sampled tokens replace the masks
  const int* lens;            // [B]
  const int* mask_pos;        // [B, n_max] ascending mask positions of each item
  const int* n_masks;         // [B]
  int* step;                  // [1] the loop step s (advanced by the step itself: the launches can be replayed as a graph)
  int* prev;                  // [B] the token before the masked position (the sampler's prev_idx)
  int* repeat_count;          // [B]
  float* logits;              // [B, V] the masked positions' logits
  const float* bias;          // [V] head bias
  int* tok;                   // [B] sampled ids
  int* num_choices;           // [B]
  int B, T_max, n_max, d, V;
};
// head row -> sampler (samp: the remix sampler over a.logits, prev, repeat_count, tok, num_choices) -> write-back
int mask_step_launch(const MaskStepArgs& a, const void* h, const void* emb, bool bf16_operands, const SampleArgs& samp, cudaStream_t st);

struct BeamArgs {
  const float* logits;      // [nb, V] fp32: last-position logits of the live beams
  int V, nb, top_k, beam_sz;
  const float* scores_in;   // [n_scores]: accumulated negative log-probabilities (n_scores == 1: broadcast, the first step)
  int n_scores;
  float* scores_out;        // [beam_sz]
  int* parents;             // [beam_sz] beam each survivor extends
  int* tokens;              // [beam_sz] appended token
};
int beam_step_launch(const BeamArgs& a, cudaStream_t st);

}  // namespace dmg
