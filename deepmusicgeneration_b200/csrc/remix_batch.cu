// The batched remix (MultitaskLearner.predict_mask_batch): per-sequence lengths in the encoder attention and the mask step.
//
// Items of different lengths share one padded batch, row b*T_max + t.  Each sequence is computed as if it were alone at its own
// length L_b: the attention kernels take the lengths (attention_bert_tc.cu, attention_flash.cu, attention.cu), the attention-output
// rows >= L_b are zeroed here so that the padding rows stay finite through LayerNorm and the next layer, and the row-wise launches
// (embedding, GEMMs, residual + LayerNorm) need nothing.
//
// The mask step replaces the B*T*V logits GEMM and the host round trips of predict_mask (deep_music_remix.py:2563-2613): for every item
// with masks left at step s it computes ONE row of logits (the masked position's), samples it with the remix sampler of sampling.cu and
// writes the token back into the ids of the next forward.
#include <vector>

#include "kernels.cuh"
#include "launch.cuh"
#include "sampling.cuh"

namespace dmg {

namespace {

// rows [b*T_max + lens[b], (b+1)*T_max) of out [B*T_max, HD] (16-byte chunks; HD * sizeof(T) is a multiple of 16)
template <class T>
__global__ void varlen_zero_rows_kernel(T* out, const int* lens, int B, int T_max, int HD) {
  pdl_launch_dependents();
  pdl_wait();
  const int chunks = HD * (int)sizeof(T) / 16;
  const long long n = (long long)B * T_max * chunks;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const long long row = i / chunks;
    const int b = (int)(row / T_max), t = (int)(row % T_max);
    if (t >= lens[b]) ((uint4*)out)[i] = make_uint4(0u, 0u, 0u, 0u);
  }
}

// one CTA per item: logits[b] = h[b*T_max + p] . Emb^T + bias, p = mask_pos[b][step]; prev[b] = ids[p - 1], or the item's own last
// token when p == 0.  Operands as the head GEMM's (bf16 x bf16 or fp32 x fp32), fp32 accumulation.
constexpr int MH_THREADS = 256;
template <class T>
__global__ void __launch_bounds__(MH_THREADS) mask_head_kernel(MaskStepArgs a, const T* h, const T* emb) {
  extern __shared__ float mh_row[];
  pdl_launch_dependents();
  pdl_wait();
  const int b = blockIdx.x, s = *a.step;
  if (s >= a.n_masks[b]) return;
  const int p = a.mask_pos[(size_t)b * a.n_max + s];
  const size_t row = (size_t)b * a.T_max + p;
  for (int k = threadIdx.x; k < a.d; k += MH_THREADS) mh_row[k] = to_f32(h[row * a.d + k]);
  if (threadIdx.x == 0) a.prev[b] = (int)a.ids[p > 0 ? row - 1 : (size_t)b * a.T_max + a.lens[b] - 1];
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int v = warp; v < a.V; v += MH_THREADS / 32) {
    const T* e = emb + (size_t)v * a.d;
    float acc = 0.f;
    for (int k = lane; k < a.d; k += 32) acc = fmaf(mh_row[k], to_f32(e[k]), acc);
    acc = warp_sum(acc);
    if (lane == 0) a.logits[(size_t)b * a.V + v] = acc + a.bias[v];
  }
}

// one CTA: the sampled token of every item that had a mask at this step goes into ids; repeat_count follows the reference rule
// (+1 if num_choices <= 2, else halved); the step counter advances
__global__ void mask_scatter_kernel(MaskStepArgs a) {
  pdl_launch_dependents();
  pdl_wait();
  const int s = *a.step;
  for (int b = threadIdx.x; b < a.B; b += blockDim.x) {
    if (s >= a.n_masks[b]) continue;
    a.ids[(size_t)b * a.T_max + a.mask_pos[(size_t)b * a.n_max + s]] = a.tok[b];
    a.repeat_count[b] = a.num_choices[b] <= 2 ? a.repeat_count[b] + 1 : a.repeat_count[b] / 2;
  }
  __syncthreads();
  if (threadIdx.x == 0) *a.step = s + 1;
}

}  // namespace

template <class T>
int varlen_zero_rows(T* out, const int* lens_dev, int B, int T_max, int HD, cudaStream_t st) {
  DMG_CHECK(HD * (int)sizeof(T) % 16 == 0, "varlen_zero_rows: row of %d elements is not a multiple of 16 bytes", HD);
  const long long n = (long long)B * T_max * (HD * (int)sizeof(T) / 16);
  const int blocks = (int)((n + 255) / 256 < 4096 ? (n + 255) / 256 : 4096);
  return launch_k(varlen_zero_rows_kernel<T>, dim3(blocks), dim3(256), 0, st, 1, out, lens_dev, B, T_max, HD);
}
template int varlen_zero_rows<float>(float*, const int*, int, int, int, cudaStream_t);
template int varlen_zero_rows<bf16>(bf16*, const int*, int, int, int, cudaStream_t);

void bert_varlen_plan(const int* lens_host, int B, int H, bool use_tc, std::vector<int>& tc_items, std::vector<int>& fl_seqs,
                      int* fl_max_len) {
  tc_items.clear();
  fl_seqs.clear();
  *fl_max_len = 0;
  for (int b = 0; b < B; b++) {
    const int L = lens_host[b];
    if (use_tc && L >= 128) {
      for (int h = 0; h < H; h++)
        for (int it = 0; it < (L + 127) / 128; it++) tc_items.push_back((b << 16) | (h << 8) | it);
    } else {
      fl_seqs.push_back(b);
      if (L > *fl_max_len) *fl_max_len = L;
    }
  }
}

int attn_bert_varlen_bf16(const bf16* qkv, const bf16* rd, int Dcap, const float* u, const float* v, bf16* out, const VarlenPlan& p,
                          int B, int T_max, int H, float scale, int fp32_strip, cudaStream_t st) {
  if (p.n_tc_items > 0 &&
      attn_bert_tc_varlen(qkv, rd, Dcap, u, v, out, p.lens, p.tc_items, p.n_tc_items, B, T_max, H, scale, fp32_strip, st)) return -1;
  if (p.n_fl_seqs > 0 && attn_flash_varlen(qkv, rd, Dcap, u, v, out, p.lens, p.fl_seqs, p.n_fl_seqs, p.fl_max_len, T_max, H, scale, st))
    return -1;
  return varlen_zero_rows<bf16>(out, p.lens, B, T_max, H * 64, st);
}

int mask_step_launch(const MaskStepArgs& a, const void* h, const void* emb, bool bf16_operands, const SampleArgs& samp, cudaStream_t st) {
  DMG_CHECK(a.d <= 1024, "mask step: d_model %d too large", a.d);
  const size_t smem = (size_t)a.d * 4;
  const int rc = bf16_operands ? launch_k(mask_head_kernel<bf16>, dim3(a.B), dim3(MH_THREADS), smem, st, 1, a, (const bf16*)h, (const bf16*)emb)
                               : launch_k(mask_head_kernel<float>, dim3(a.B), dim3(MH_THREADS), smem, st, 1, a, (const float*)h, (const float*)emb);
  if (rc) return rc;
  if (sample_launch(samp, a.B, st)) return -1;
  return launch_k(mask_scatter_kernel, dim3(1), dim3(256), 0, st, 1, a);
}

}  // namespace dmg
