#pragma once
#include <map>
#include <memory>
#include <vector>

#include "dac_engine.h"

namespace ls {

// S3TokenizerV2 (speech/tools/S3Tokenizer/s3tokenizer/model_v2.py:290-415) on the tensor cores with bf16x3 operands:
// every dense linear / convolution computes A_hi W_hi + A_lo W_hi + A_hi W_lo (hi = bf16(x), lo = bf16(x - hi)) with
// fp32 accumulation, which keeps the encoder output at fp32-level error (a token is a rounding decision).  The split is a
// longer K: activations that feed a GEMM are stored as [hi | lo | hi] rows of 3K bf16, weights once as [N][3K] =
// [W_hi | W_hi | W_lo], and one ordinary conv_gemm launch with K' = 3K does the rest.  Residual stream, LayerNorm
// statistics, rotary, FSMN and attention stay fp32.  Time-major activations; right-padded batches, each clip computed as
// if alone (bitwise).
class S3Engine {
 public:
  S3Engine(const Weights& w, int device);
  ~S3Engine();
  // mel [B,n_mels,T], mel_len [B] (device) -> codes [B,T2] int32, code_len [B] int32; hidden_out (nullable): [B,T2,n_state]
  // (rows past code_len[b] are zero)
  void quantize(const float* mel, const int* mel_len, int* codes, int* code_len, float* hidden_out, int B, int T, cudaStream_t s);
  int n_mels() const { return mels_; }
  int n_state() const { return d_; }
  int device() const { return device_; }

 private:
  struct BlockW {
    PackedLinear qkv, out, ff1, ff2;  // split weights [N][3K]
    size_t ln1_g, ln1_b, ln2_g, ln2_b, fsmn;
  };
  struct Layout {
    size_t l1, mel_s, x, a_s, qkv, xm, x1, h, h_s, total;
  };
  struct Plan;
  static Layout layout(int B, int T, int mels, int d);
  const Plan& plan_for(int B, int T, const Layout& L);
  template <typename T>
  T* ws(size_t off) const { return reinterpret_cast<T*>(ws_base_ + off); }

  int device_ = 0, num_sms_ = 148, mels_ = 128, d_ = 1280, heads_ = 20, ksize_ = 31, table_len_ = 0;
  Arena arena_;
  PackedLinear conv1_, conv2_;  // 2-tap forms over the [T/2][2 * 3C] view of the split input
  std::vector<BlockW> blocks_;
  size_t cos_ = 0, sin_ = 0, fsq_w_ = 0, fsq_b_ = 0;
  uint8_t* ws_base_ = nullptr;
  size_t ws_bytes_ = 0;
  std::map<std::pair<int, int>, std::unique_ptr<Plan>> plans_;
};

}  // namespace ls
