#pragma once
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "engine_common.h"

namespace ls {

// Token -> mu front half of CausalMaskedDiffWithXvec.inference (speech/cosyvoice/flow/flow.py:461-489; SURVEY section 8
// f-1) on the tensor cores: input embedding, UpsampleConformerEncoder (transformer/upsample_encoder.py:266-318: 6 rel-pos
// conformer layers at 25 Hz, nearest x2 + conv5, 4 layers at 50 Hz), encoder_proj, speaker-embedding affine.
// Time-major activations [B][T][512]: fp32 residual stream, bf16 GEMM operands.  Every linear / convolution is a
// conv_gemm launch; self-attention is the estimator's flash-attention kernel with the relative-position term
// bd[i, j] = (q_i + v) . p[T-1-i+j] (attention.py:225-247's rel_shift in closed form) added to the scores from a
// [B][H][T][2T-1] matrix that one conv_gemm launch per head writes.  Right-padded batches through per-utterance key bounds.
class FrontEngine {
 public:
  FrontEngine(const Weights& w, int device);
  ~FrontEngine();
  // tokens [B,T_all] int64 (device), embedding [B,spk_dim] -> mu [B,80,2(T_all - n_context)], spks [B,80]
  // token_len (device, nullable): per-utterance token counts of a right-padded batch (mu is zero past 2 * token_len)
  void encode(const long long* tokens, const float* embedding, float* mu, float* spks, int B, int T_all, int n_context,
              bool streaming, const int* token_len, cudaStream_t s);
  // Session mode: row b holds token_len[b] tokens of which the last n_context[b] (0 or 3) are look-ahead context, and
  // comes out equal to an encode of that row alone: mu [B,80,2T], zero past 2 * (token_len[b] - n_context[b]).  Rows
  // with invalid entries (n_context not 0 or 3, fewer than 1 output token, token_len > T_all or more than T output
  // tokens) get an all-zero mu.  token_len and n_context are device int32 [B].
  void encode_sessions(const long long* tokens, const float* embedding, float* mu, float* spks, int B, int T_all, int T,
                       const int* token_len, const int* n_context, bool streaming, cudaStream_t s);
  int out_dim() const { return out_; }
  int spk_dim() const { return spk_; }
  int device() const { return device_; }

 private:
  void run(const long long* tokens, const float* embedding, float* mu, float* spks, int B, int T_all, int T, bool streaming,
           const int* token_len, const int* n_context, cudaStream_t s);
  struct LayerW {
    PackedLinear qkv, pos, out, ff1, ff2;
    size_t g_mha, b_mha, g_ff, b_ff, bias_u, bias_v;
  };
  struct EmbedW {
    PackedLinear lin;
    size_t g, b;
  };
  struct Plan;
  void ensure_workspace(int B, int T_all, int T, cudaStream_t s);
  const Plan& plan_for(int B, int T_all, int T);
  template <typename T>
  T* ws(size_t off) const { return reinterpret_cast<T*>(ws_base_ + off); }

  int device_ = 0, num_sms_ = 148, d_ = 512, ff_ = 2048, vocab_ = 6561, out_ = 80, spk_ = 192, heads_ = 8, chunk_ = 25;
  Arena arena_;
  size_t emb_table_ = 0;  // bf16 [vocab][d]
  size_t spk_w_ = 0, spk_b_ = 0;
  EmbedW embed_, up_embed_;
  PackedLinear pre1_, pre2_, up_conv_, proj_;
  size_t g_after_ = 0, b_after_ = 0;
  std::vector<LayerW> layers_, up_layers_;
  uint8_t* ws_base_ = nullptr;
  long long cap_rows_ = 0, cap_bd_ = 0;
  size_t o_x_ = 0, o_y_ = 0, o_nb_ = 0, o_qkv_ = 0, o_qv_ = 0, o_att_ = 0, o_h_ = 0, o_pe_ = 0, o_pp_ = 0, o_pph_ = 0, o_bd_ = 0,
         o_spk_ = 0;
  std::map<std::vector<int>, std::unique_ptr<Plan>> plans_;
};

// LearnableSpeakerEncoder (speech/cosyvoice/llm/llm.py:34-96; SURVEY section 8 f-4) on the tensor cores: the 1x1 convolutions
// (init, qkv, proj_out) are conv_gemm launches, QKVAttentionLegacy is the estimator's flash-attention kernel (the head-major
// [q|k|v] rows of the qkv weight are permuted to Q | K | V column blocks at load; its scale 64^-1/4 on q and k is the
// kernel's 1/8 on the product), GroupNorm32 is a small kernel over the fp32 residual stream.  Equal-length clips.
class SpeakerEngine {
 public:
  SpeakerEngine(const Weights& w, int device);
  ~SpeakerEngine();
  // mel [n_refs][B,mel,T] -> emb [B,out]; n_refs > 1 averages the per-clip embeddings (flow.py:336-366)
  void encode(const float* mel, float* emb, int B, int T, int n_refs, cudaStream_t s);
  int device() const { return device_; }

 private:
  struct BlockW {
    PackedLinear qkv, proj;
    size_t g, b;
  };
  struct Plan;
  const Plan& plan_for(int R, int T, cudaStream_t s);
  template <typename T>
  T* ws(size_t off) const { return reinterpret_cast<T*>(ws_base_ + off); }

  int device_ = 0, num_sms_ = 148, mel_ = 80, out_ = 192, heads_ = 8, groups_ = 32;
  Arena arena_;
  PackedLinear init_;
  size_t out_w_ = 0, out_b_ = 0;
  std::vector<BlockW> blocks_;
  uint8_t* ws_base_ = nullptr;
  long long cap_rows_ = 0;
  size_t o_h_ = 0, o_nb_ = 0, o_qkv_ = 0, o_att_ = 0, o_mel_ = 0, o_emb_ = 0;
  std::map<std::pair<int, int>, std::unique_ptr<Plan>> plans_;
};

}  // namespace ls
