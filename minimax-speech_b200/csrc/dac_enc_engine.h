#pragma once
#include <map>
#include <memory>
#include <vector>

#include "dac_engine.h"

namespace ls {

// DAC-VAE encoder (dac-vae/model.py:146-234 Encoder / EncoderBlock, 469-483 encode) on time-major activations,
// tensor-core path: every ResidualUnit convolution and every downsampling convolution is a conv_gemm launch.
class DacEncEngine {
 public:
  // fp16: fp16 instead of bf16 GEMM operands (weights and the Snake outputs the convolutions consume); accumulation,
  // the residual stream and z / m / logs stay fp32
  DacEncEngine(const Weights& w, int device, bool fp16 = false);
  ~DacEncEngine();
  // audio [B,1,S] fp32 (S a multiple of the hop) -> z, m, logs [B,latent,S/hop] fp32; noise nullable ([B,latent,S/hop]).
  // lengths (device int32 [B], nullable): latent frames per clip; clip b is encoded as if alone at lengths[b] * hop
  // samples (the rest of its row is never read) and its outputs are zero from frame lengths[b] on.
  void encode(const float* audio, const int* lengths, const float* noise, float* z, float* m, float* logs, int B, int S,
              cudaStream_t s);
  int hop() const { return hop_; }
  int latent_dim() const { return latent_; }
  int device() const { return device_; }

 private:
  struct UnitW {
    PackedLinear conv7, conv1;
    size_t a0, ia0, a2, ia2;
  };
  struct StageW {
    int stride, cin;       // cin channels in, 2*cin out
    UnitW unit[3];
    size_t a_dn, ia_dn;    // Snake before the downsampling conv
    PackedLinear down;     // 3-tap polyphase form over the [L/s][s*cin] view of the input
  };
  struct Plan;
  void ensure_workspace(int B, int S, cudaStream_t s);
  const Plan& plan_for(int B, int S);
  template <typename T>
  T* ws(size_t off) const { return reinterpret_cast<T*>(ws_base_ + off); }

  int device_ = 0, num_sms_ = 148, latent_ = 80, hop_ = 1, dim0_ = 64, fp16_ = 0;
  Arena arena_;
  size_t in_w_ = 0, in_b_ = 0;       // first conv (1 -> dim0, k = 7), fp32 [dim0][7] + bias
  size_t post_w_ = 0, post_b_ = 0;   // en_conv_post folded, fp32 [2*latent][latent] + bias
  size_t final_alpha_ = 0, final_ialpha_ = 0;
  PackedLinear final_;               // conv3 (C_last -> latent)
  std::vector<StageW> stages_;
  uint8_t* ws_base_ = nullptr;
  long long cap_samples_ = 0;
  size_t o_x_ = 0, o_sA_ = 0, o_sB_ = 0, o_y_ = 0;
  std::map<std::pair<int, int>, std::unique_ptr<Plan>> plans_;
};

}  // namespace ls
