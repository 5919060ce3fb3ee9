#pragma once
#include <cmath>
#include <map>
#include <memory>
#include <vector>

#include <cuda_fp16.h>

#include "engine_common.h"

namespace ls {

// One folded weight as a 16-bit GEMM operand of the handle's format: bf16, or fp16 (ls_dac_create_fp16: the same
// kernels compiled for fp16 operands).  A checkpoint is outside input: a weight past fp16's range (|w| > 65504) would
// become inf, so the layer p is refused instead.
inline __nv_bfloat16 dac_w16(float x, bool fp16, const std::string& p) {
  if (!fp16) return __float2bfloat16(x);
  if (!(std::fabs(x) <= 65504.f))  // (the message is built on failure only: this runs once per weight element)
    throw EngineError(LS_ERR_UNSUPPORTED, "folded weight of " + p + " is not finite in fp16 (|w| > 65504)");
  const __half h = __float2half_rn(x);
  __nv_bfloat16 out;
  std::memcpy(&out, &h, 2);
  return out;
}

// shared with the encoder engine (dac_enc_engine.cu): weight-norm folding + 16-bit [taps][N][K] packing (fp16: fp16
// operands instead of bf16)
PackedLinear pack_wn_conv(Arena& a, const Weights& w, const std::string& p, bool fp16, int n_pad_to = 0);
void finalize_linear(const Arena& a, PackedLinear& pl);

// DAC-VAE decoder (dac-vae/model.py:326-379, 485-488) on time-major activations.
class DacEngine {
 public:
  // fp16: fp16 instead of bf16 GEMM operands (weights, z and every Snake / LeakyReLU output a convolution consumes);
  // accumulation stays fp32, the residual stream fp16, the waveform fp32
  DacEngine(const Weights& w, int device, bool fp16 = false);
  ~DacEngine();
  void decode(const float* z, const int* lengths, float* wav, int B, int L, cudaStream_t s);
  int hop() const { return hop_; }
  int latent_dim() const { return latent_; }
  int device() const { return device_; }
  unsigned long long ws_generation() const { return ws_generation_; }

 private:
  struct UnitW;
  struct StageW;
  struct Plan;
  void ensure_workspace(int B, int L, cudaStream_t s);
  const Plan& plan_for(int B, int L);
  template <typename T>
  T* ws(size_t off) const { return reinterpret_cast<T*>(ws_base_ + off); }

  int device_ = 0, num_sms_ = 148, fp16_ = 0;
  int latent_ = 80, dim_ = 1536, hop_ = 1, out_ch_ = 1;
  std::vector<int> rates_;
  Arena arena_;
  PackedLinear pre_, in_, final_;
  std::vector<StageW> stages_;
  size_t final_alpha_ = 0, final_ialpha_ = 0;

  uint8_t* ws_base_ = nullptr;
  long long cap_frames_ = 0;  // B*L capacity
  int cap_b_ = 0;
  unsigned long long ws_generation_ = 0;
  size_t o_zt_ = 0, o_a0_ = 0, o_x_ = 0, o_sA_[2] = {0, 0}, o_sB_ = 0, o_len_ = 0;
  std::map<std::pair<int, int>, std::unique_ptr<Plan>> plans_;
};

}  // namespace ls
