// fp32 mode of the hot path ("<= 1e-4 in fp32 mode", north_star): the same call surface as FlowEngine / DacEngine,
// computed end to end in fp32 on the CUDA cores with plain (unfused) kernels in the reference's own NCT layout.
// It exists to show that the data flow -- masks, padding, causal convolutions, weight-norm folding, CFG, the Euler
// update -- is the reference's, free of bf16 rounding; it is a validation mode, not the fast path.
#pragma once
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "engine_common.h"

namespace ls {

// every state_dict tensor as a device fp32 array, by name
class F32Weights {
 public:
  F32Weights() = default;
  ~F32Weights();
  void add(const std::string& name, const float* host, size_t n, std::vector<long long> shape);
  const float* ptr(const std::string& name) const;
  const std::vector<long long>& shape(const std::string& name) const;
  bool has(const std::string& name) const { return items_.count(name) != 0; }

 private:
  struct Item {
    float* dev = nullptr;
    std::vector<long long> shape;
  };
  std::map<std::string, Item> items_;
};

// grow-only scratch memory, bump-allocated per call (no allocation once every shape has been seen)
class F32Scratch {
 public:
  ~F32Scratch();
  void reset() { used_ = 0; }
  float* get(size_t n_floats, cudaStream_t s);

 private:
  float* base_ = nullptr;
  size_t cap_ = 0, used_ = 0;
  std::vector<float*> retired_;  // outgrown blocks stay alive until destruction (in-flight kernels may use them)
};

class FlowEngineF32 {
 public:
  FlowEngineF32(const Weights& w, int device);
  void estimator_forward(const float* x, const float* mask, const float* mu, const float* t, const float* spks,
                         const float* cond, float* out, int rows, int T, bool streaming, cudaStream_t s);
  void solve(const float* mu, const float* mask, const float* spks, const float* cond, const float* noise,
             long long noise_stride, const float* t_span, int n_steps, float temperature, float cfg_rate,
             bool streaming, float* out, int B, int T, cudaStream_t s);
  int feat() const { return feat_; }
  int device() const { return device_; }

 private:
  void run(const float* x, const float* mask, const float* mu, const float* t, const float* spks, const float* cond,
           float* out, int R, int T, bool streaming, cudaStream_t s);
  float* group(const std::string& prefix, const float* h, int cin, const float* mask, const float* temb,
               const int* lens, int R, int T, bool streaming, cudaStream_t s);
  float* resnet(const std::string& p, const float* x, int cin, const float* mask, const float* temb, int R, int T,
                cudaStream_t s);
  float* causal_block(const std::string& p, const float* x, int cin, const float* mask, const float* addvec, int R,
                      int T, cudaStream_t s);
  int device_ = 0, feat_ = 80, C_ = 256, heads_ = 8, n_blocks_ = 0, n_mid_ = 0, chunk_ = 50;
  bool causal_ = true;   // false: the non-causal ConditionalDecoder (Conv1d pad 1 + GroupNorm(8) blocks)
  int conv_pad_ = 2;
  const int* lens_ = nullptr;  // device lengths of the call in flight (GroupNorm statistics run over the valid frames)
  F32Weights w_;
  F32Scratch scratch_;
};

class DacEngineF32 {
 public:
  DacEngineF32(const Weights& w, int device);
  void decode(const float* z, const int* lengths, float* wav, int B, int L, cudaStream_t s);
  // DACVAE.encode (SURVEY section 8 f-3): audio [B,1,S] -> z, m, logs [B,latent,S/hop]; noise (nullable) [B,latent,S/hop];
  // lengths (device int32 [B], nullable): latent frames per clip, each clip encoded alone, outputs zero past it
  void encode(const float* audio, const int* lengths, const float* noise, float* z, float* m, float* logs, int B, int S,
              cudaStream_t s);
  bool has_encoder() const { return !enc_rates_.empty(); }
  bool has_decoder() const { return !rates_.empty(); }
  int hop() const { return hop_; }
  int latent_dim() const { return latent_; }
  int device() const { return device_; }

 private:
  float* residual_unit(const std::string& u, const float* x, int B, int C, int len, int dil, cudaStream_t s);
  void encode_dense(const float* audio, const float* noise, float* z, float* m, float* logs, int B, int S, cudaStream_t s);
  void decode_dense(const float* z, long long z_bstride, float* wav, long long wav_bstride, int B, int L, int L_alloc,
                    cudaStream_t s);
  int device_ = 0, latent_ = 80, hop_ = 1;
  std::vector<int> rates_, enc_rates_;
  F32Weights w_;  // weight-norm folded: "<prefix>.weight", "<prefix>.bias", "<prefix>.alpha"
  F32Scratch scratch_;
};

// token -> mu front half of CausalMaskedDiffWithXvec.inference (flow/flow.py:437-511; SURVEY section 8 f-1): input
// embedding, UpsampleConformerEncoder (rel-pos conformer layers at 25 Hz, x2 upsample, conformer layers at 50 Hz),
// encoder_proj, speaker-embedding affine.  fp32 mode; right-padded batches; finalize = True or a non-final chunk
// (3 look-ahead context tokens), optional block-causal streaming attention.
class FrontEngineF32 {
 public:
  FrontEngineF32(const Weights& w, int device);
  // tokens [B,T_all] int64 (device), embedding [B,spk_dim] -> mu [B,80,2(T_all - n_context)], spks [B,80]
  // token_len (device, nullable): per-utterance token counts of a right-padded batch
  void encode(const long long* tokens, const float* embedding, float* mu, float* spks, int B, int T_all, int n_context,
              bool streaming, const int* token_len, cudaStream_t s);
  // session mode: see FrontEngine::encode_sessions
  void encode_sessions(const long long* tokens, const float* embedding, float* mu, float* spks, int B, int T_all, int T,
                       const int* token_len, const int* n_context, bool streaming, cudaStream_t s);
  int out_dim() const { return out_; }
  int spk_dim() const { return spk_; }
  int device() const { return device_; }

 private:
  void run(const long long* tokens, const float* embedding, float* mu, float* spks, int B, int T_all, int T, bool streaming,
           const int* token_len, const int* n_context, cudaStream_t s);
  float* layer(const std::string& p, float* x, const float* pe, int B, int T, int chunk, const int* lens, cudaStream_t s);
  float* embed(const std::string& p, const float* x, int B, int T, float** pe, cudaStream_t s);
  int device_ = 0, d_ = 512, vocab_ = 6561, out_ = 80, spk_ = 192, heads_ = 8, n_blocks_ = 0, n_up_ = 0, chunk_ = 25;
  F32Weights w_;
  F32Scratch scratch_;
};

// LearnableSpeakerEncoder (speech/cosyvoice/llm/llm.py:34-96; SURVEY section 8 f-4): reference mel [B,80,T] -> L2-normalised
// speaker embedding [B,192] (the `embedding` input of the front half).  fp32 mode; equal-length clips.
class SpeakerEngineF32 {
 public:
  SpeakerEngineF32(const Weights& w, int device);
  // mel [n_refs][B,mel,T] -> emb [B,out]; n_refs > 1 averages the per-clip embeddings (flow.py:336-366)
  void encode(const float* mel, float* emb, int B, int T, int n_refs, cudaStream_t s);
  int mel_dim() const { return mel_; }
  int out_dim() const { return out_; }
  int device() const { return device_; }

 private:
  int device_ = 0, mel_ = 80, d_ = 512, out_ = 192, heads_ = 8, groups_ = 32, n_blocks_ = 0;
  F32Weights w_;
  F32Scratch scratch_;
};

// S3TokenizerV2 (speech/tools/S3Tokenizer/s3tokenizer/model_v2.py:290-415; SURVEY section 8 f-4): 100 Hz log-mel
// [B,n_mels,T] + lengths -> 25 Hz FSQ token ids (vocabulary 3^8) + token counts.  fp32 mode only: a token is a rounding
// decision, and the tensor-core operand types move activations near a rounding boundary across it.
class S3EngineF32 {
 public:
  S3EngineF32(const Weights& w, int device);
  // mel [B,n_mels,T], mel_len [B] (device) -> codes [B,T2] int32, code_len [B] int32; hidden_out (nullable): [B,T2,n_state]
  void quantize(const float* mel, const int* mel_len, int* codes, int* code_len, float* hidden_out, int B, int T, cudaStream_t s);
  static void code_frames(int T, int* T1, int* T2);  // frames after each of the two stride-2 convs
  int n_mels() const { return mels_; }
  int n_state() const { return d_; }
  int device() const { return device_; }

 private:
  int device_ = 0, mels_ = 128, d_ = 1280, heads_ = 20, ksize_ = 31, n_blocks_ = 0, table_len_ = 0;
  F32Weights w_;
  F32Scratch scratch_;
};

}  // namespace ls
