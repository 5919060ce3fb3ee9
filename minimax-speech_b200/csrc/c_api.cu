// extern "C" surface declared in include/ls_b200.h.
#include <algorithm>
#include <atomic>
#include <cstdarg>
#include <mutex>
#include <vector>

#include "dac_enc_engine.h"
#include "dac_engine.h"
#include "engine_common.h"
#include "f32_path.h"
#include "flow_engine.h"
#include "front_engine.h"
#include "profiler.h"
#include "s3_engine.h"

namespace ls {

std::atomic<long long> g_launch_count{0};
long long* g_debug_buffer = nullptr;
bool pdl_enabled() {
  static const bool on = [] {
    const char* e = getenv("LS_NO_PDL");
    return !(e && e[0] == '1');
  }();
  return on;
}
long long g_debug_bytes = 0;
int conv_halo_mode() {  // 0: per-tap boxes; 1: halo box, descriptor base offset set; 2: halo box, base offset 0
  static const int mode = [] {
    const char* e = getenv("LS_CONV_HALO");
    return e && e[0] >= '0' && e[0] <= '2' ? e[0] - '0' : 2;
  }();
  return mode;
}
bool conv_halo_enabled() { return conv_halo_mode() != 0; }
bool conv_fuse_res_enabled() {
  static const bool on = [] {
    const char* e = getenv("LS_CONV_FUSE_RES");
    return !(e && e[0] == '0');
  }();
  return on;
}
bool conv_dual_enabled() {
  static const bool on = [] {
    const char* e = getenv("LS_CONV_DUAL");
    return !(e && e[0] == '0');
  }();
  return on;
}
bool conv_tma_out_enabled() {
  static const bool on = [] {
    const char* e = getenv("LS_CONV_TMA_OUT");
    return !(e && e[0] == '0');
  }();
  return on;
}
bool conv_resident_enabled() {
  static const bool on = [] {
    const char* e = getenv("LS_CONV_RESIDENT");
    return !(e && e[0] == '0');
  }();
  return on;
}

static thread_local std::string t_error;
void set_error(const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  t_error = buf;
}
const char* get_error() { return t_error.c_str(); }

template <typename F>
static int32_t guarded(F&& f) {
  try {
    f();
    return LS_OK;
  } catch (const EngineError& e) {
    set_error("%s", e.what());
    return e.code;
  } catch (const std::exception& e) {
    set_error("%s", e.what());
    return LS_ERR_INVALID;
  } catch (...) {
    set_error("unknown failure");
    return LS_ERR_INVALID;
  }
}

// Calls that reach one handle are serialised: a per-handle mutex orders the host threads, and when the handle is used on
// a different stream than its previous call the new stream first waits for an event recorded at the end of that call
// (the handle's workspace, plans and staging buffers are shared state).  Different handles stay independent.  While a
// stream is being captured into a CUDA graph nothing is recorded or waited for (the capture owns the ordering).
struct StreamSerial {
  std::mutex mu;
  cudaEvent_t ev = nullptr;
  cudaStream_t last = nullptr;
  bool used = false;
  ~StreamSerial() {
    if (ev) cudaEventDestroy(ev);
  }
};
class SerialScope {
 public:
  SerialScope(StreamSerial& ss, int device, cudaStream_t s) : ss_(ss), s_(s) {
    ss_.mu.lock();
    try {
      LS_CUDA(cudaSetDevice(device));
      cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
      LS_CUDA(cudaStreamIsCapturing(s, &st));
      capturing_ = st != cudaStreamCaptureStatusNone;
      if (!capturing_) {
        if (!ss_.ev) LS_CUDA(cudaEventCreateWithFlags(&ss_.ev, cudaEventDisableTiming));
        if (ss_.used && ss_.last != s) LS_CUDA(cudaStreamWaitEvent(s, ss_.ev, 0));
      }
    } catch (...) {
      ss_.mu.unlock();
      throw;
    }
  }
  ~SerialScope() {
    if (!capturing_ && ss_.ev && cudaEventRecord(ss_.ev, s_) == cudaSuccess) ss_.last = s_, ss_.used = true;
    ss_.mu.unlock();
  }
  SerialScope(const SerialScope&) = delete;
  SerialScope& operator=(const SerialScope&) = delete;

 private:
  StreamSerial& ss_;
  cudaStream_t s_;
  bool capturing_ = false;
};

}  // namespace ls

struct ls_flow {
  ls::StreamSerial serial;
  std::unique_ptr<ls::FlowEngine> eng;        // bf16 tensor-core path (default)
  std::unique_ptr<ls::FlowEngineF32> eng32;   // fp32 mode (ls_flow_create_fp32)
  int feat() const { return eng ? eng->feat() : eng32->feat(); }
  int device() const { return eng ? eng->device() : eng32->device(); }
  template <typename... A>
  void solve(A&&... a) {
    if (eng) eng->solve(std::forward<A>(a)...);
    else eng32->solve(std::forward<A>(a)...);
  }
  template <typename... A>
  void estimator_forward(A&&... a) {
    if (eng) eng->estimator_forward(std::forward<A>(a)...);
    else eng32->estimator_forward(std::forward<A>(a)...);
  }
  // staging for ls_synthesize_host
  float* stage = nullptr;
  size_t stage_bytes = 0;
};
struct ls_dac {
  ls::StreamSerial serial;
  int device() const { return eng ? eng->device() : enc ? enc->device() : eng32->device(); }
  std::unique_ptr<ls::DacEngine> eng;       // tensor-core decoder (state dict holds decoder.* / de_conv_pre.*)
  std::unique_ptr<ls::DacEncEngine> enc;    // tensor-core encoder (state dict holds encoder.* / en_conv_post.*)
  std::unique_ptr<ls::DacEngineF32> eng32;  // fp32 mode: both directions
  int hop() const { return eng ? eng->hop() : enc ? enc->hop() : eng32->hop(); }
  void decode(const float* z, const int* lengths, float* wav, int B, int L, cudaStream_t s) {
    if (eng) eng->decode(z, lengths, wav, B, L, s);
    else if (eng32) eng32->decode(z, lengths, wav, B, L, s);
    else throw ls::EngineError(LS_ERR_WEIGHTS, "this handle holds no decoder weights");
  }
};

struct ls_front {
  ls::StreamSerial serial;
  int device() const { return eng ? eng->device() : eng32->device(); }
  std::unique_ptr<ls::FrontEngine> eng;       // tensor-core path
  std::unique_ptr<ls::FrontEngineF32> eng32;  // fp32 mode
};

struct ls_speaker {
  ls::StreamSerial serial;
  int device() const { return eng ? eng->device() : eng32->device(); }
  std::unique_ptr<ls::SpeakerEngine> eng;        // tensor-core path
  std::unique_ptr<ls::SpeakerEngineF32> eng32;   // fp32 mode
};

struct ls_s3 {
  ls::StreamSerial serial;
  int device() const { return eng ? eng->device() : eng32->device(); }
  std::unique_ptr<ls::S3Engine> eng;       // bf16x3 tensor-core mode (fp32-level error: tokens are rounding decisions)
  std::unique_ptr<ls::S3EngineF32> eng32;  // fp32 mode
};

struct ls_resampler {
  int device = 0;
  ls::ResamplePlan plan;
  float* taps = nullptr;
  int2* fc = nullptr;
  ~ls_resampler() {
    if (taps) cudaFree(taps);
    if (fc) cudaFree(fc);
  }
};

extern "C" {

int32_t ls_s3_create_fp32(const ls_tensor* weights, int32_t n_weights, int32_t device, ls_s3** out) {
  return ls::guarded([&] {
    ls::require(weights && out && n_weights > 0, "ls_s3_create_fp32: null argument");
    ls::Weights w(weights, n_weights);
    auto h = std::make_unique<ls_s3>();
    h->eng32 = std::make_unique<ls::S3EngineF32>(w, device);
    *out = h.release();
  });
}
int32_t ls_s3_create(const ls_tensor* weights, int32_t n_weights, int32_t device, ls_s3** out) {
  return ls::guarded([&] {
    ls::require(weights && out && n_weights > 0, "ls_s3_create: null argument");
    ls::Weights w(weights, n_weights);
    auto h = std::make_unique<ls_s3>();
    h->eng = std::make_unique<ls::S3Engine>(w, device);
    *out = h.release();
  });
}
void ls_s3_destroy(ls_s3* h) { delete h; }
int32_t ls_s3_code_frames(int32_t T) {
  int t1 = 0, t2 = 0;
  if (T > 0) ls::S3EngineF32::code_frames(T, &t1, &t2);
  return t2;
}
int32_t ls_s3_quantize(ls_s3* h, const float* mel, const int32_t* mel_len, int32_t* codes, int32_t* code_len, float* hidden,
                       int32_t B, int32_t T, void* stream) {
  return ls::guarded([&] {
    ls::require(h && mel && mel_len && codes && code_len, "ls_s3_quantize: null argument");
    ls::SerialScope scope(h->serial, h->device(), (cudaStream_t)stream);
    if (h->eng) h->eng->quantize(mel, mel_len, codes, code_len, hidden, B, T, (cudaStream_t)stream);
    else h->eng32->quantize(mel, mel_len, codes, code_len, hidden, B, T, (cudaStream_t)stream);
  });
}

int32_t ls_front_create_fp32(const ls_tensor* weights, int32_t n_weights, int32_t device, ls_front** out) {
  return ls::guarded([&] {
    ls::require(weights && out && n_weights > 0, "ls_front_create_fp32: null argument");
    ls::Weights w(weights, n_weights);
    auto h = std::make_unique<ls_front>();
    h->eng32 = std::make_unique<ls::FrontEngineF32>(w, device);
    *out = h.release();
  });
}
int32_t ls_front_create(const ls_tensor* weights, int32_t n_weights, int32_t device, ls_front** out) {
  return ls::guarded([&] {
    ls::require(weights && out && n_weights > 0, "ls_front_create: null argument");
    ls::Weights w(weights, n_weights);
    auto h = std::make_unique<ls_front>();
    h->eng = std::make_unique<ls::FrontEngine>(w, device);
    *out = h.release();
  });
}
void ls_front_destroy(ls_front* h) { delete h; }
int32_t ls_front_encode(ls_front* h, const int64_t* tokens, const float* embedding, float* mu, float* spks, int32_t B,
                        int32_t T, int32_t n_context, int32_t streaming, const int32_t* token_len, void* stream) {
  return ls::guarded([&] {
    ls::require(h && tokens && embedding && mu && spks, "ls_front_encode: null argument");
    ls::SerialScope scope(h->serial, h->device(), (cudaStream_t)stream);
    if (h->eng) h->eng->encode(reinterpret_cast<const long long*>(tokens), embedding, mu, spks, B, T, n_context, streaming != 0,
                               token_len, (cudaStream_t)stream);
    else h->eng32->encode(reinterpret_cast<const long long*>(tokens), embedding, mu, spks, B, T, n_context, streaming != 0,
                          token_len, (cudaStream_t)stream);
  });
}
int32_t ls_front_encode_sessions(ls_front* h, const int64_t* tokens, const float* embedding, float* mu, float* spks, int32_t B,
                                 int32_t T_all, int32_t T, const int32_t* token_len, const int32_t* n_context, int32_t streaming,
                                 void* stream) {
  return ls::guarded([&] {
    ls::require(h && tokens && embedding && mu && spks && token_len && n_context, "ls_front_encode_sessions: null argument");
    ls::SerialScope scope(h->serial, h->device(), (cudaStream_t)stream);
    const auto* tok = reinterpret_cast<const long long*>(tokens);
    if (h->eng) h->eng->encode_sessions(tok, embedding, mu, spks, B, T_all, T, token_len, n_context, streaming != 0, (cudaStream_t)stream);
    else h->eng32->encode_sessions(tok, embedding, mu, spks, B, T_all, T, token_len, n_context, streaming != 0, (cudaStream_t)stream);
  });
}

int32_t ls_speaker_create_fp32(const ls_tensor* weights, int32_t n_weights, int32_t device, ls_speaker** out) {
  return ls::guarded([&] {
    ls::require(weights && out && n_weights > 0, "ls_speaker_create_fp32: null argument");
    ls::Weights w(weights, n_weights);
    auto h = std::make_unique<ls_speaker>();
    h->eng32 = std::make_unique<ls::SpeakerEngineF32>(w, device);
    *out = h.release();
  });
}
int32_t ls_speaker_create(const ls_tensor* weights, int32_t n_weights, int32_t device, ls_speaker** out) {
  return ls::guarded([&] {
    ls::require(weights && out && n_weights > 0, "ls_speaker_create: null argument");
    ls::Weights w(weights, n_weights);
    auto h = std::make_unique<ls_speaker>();
    h->eng = std::make_unique<ls::SpeakerEngine>(w, device);
    *out = h.release();
  });
}
void ls_speaker_destroy(ls_speaker* h) { delete h; }
int32_t ls_speaker_encode(ls_speaker* h, const float* mel, float* embedding, int32_t B, int32_t T, int32_t n_refs, void* stream) {
  return ls::guarded([&] {
    ls::require(h && mel && embedding, "ls_speaker_encode: null argument");
    ls::SerialScope scope(h->serial, h->device(), (cudaStream_t)stream);
    if (h->eng) h->eng->encode(mel, embedding, B, T, n_refs, (cudaStream_t)stream);
    else h->eng32->encode(mel, embedding, B, T, n_refs, (cudaStream_t)stream);
  });
}

int32_t ls_abi_version(void) { return LS_ABI_VERSION; }
const char* ls_last_error(void) { return ls::get_error(); }
int64_t ls_launch_count(void) { return ls::g_launch_count.load(); }

int32_t ls_device_check(int32_t device, int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor) {
  return ls::guarded([&] {
    cudaDeviceProp prop;
    LS_CUDA(cudaGetDeviceProperties(&prop, device));
    if (sm_count) *sm_count = prop.multiProcessorCount;
    if (cc_major) *cc_major = prop.major;
    if (cc_minor) *cc_minor = prop.minor;
    ls::require(prop.major == 10, "device is not sm_100 (B200)", LS_ERR_UNSUPPORTED);
  });
}

int32_t ls_flow_create(const ls_tensor* weights, int32_t n_weights, int32_t device, ls_flow** out) {
  return ls::guarded([&] {
    ls::require(weights && out && n_weights > 0, "ls_flow_create: null argument");
    ls::Weights w(weights, n_weights);
    auto h = std::make_unique<ls_flow>();
    h->eng = std::make_unique<ls::FlowEngine>(w, device);
    *out = h.release();
  });
}
int32_t ls_flow_create_fp16(const ls_tensor* weights, int32_t n_weights, int32_t device, ls_flow** out) {
  return ls::guarded([&] {
    ls::require(weights && out && n_weights > 0, "ls_flow_create_fp16: null argument");
    ls::Weights w(weights, n_weights);
    auto h = std::make_unique<ls_flow>();
    h->eng = std::make_unique<ls::FlowEngine>(w, device, true);
    *out = h.release();
  });
}
int32_t ls_flow_create_fp32(const ls_tensor* weights, int32_t n_weights, int32_t device, ls_flow** out) {
  return ls::guarded([&] {
    ls::require(weights && out && n_weights > 0, "ls_flow_create_fp32: null argument");
    ls::Weights w(weights, n_weights);
    auto h = std::make_unique<ls_flow>();
    h->eng32 = std::make_unique<ls::FlowEngineF32>(w, device);
    *out = h.release();
  });
}
void ls_flow_destroy(ls_flow* h) {
  if (!h) return;
  if (h->stage) cudaFree(h->stage);
  delete h;
}

int32_t ls_flow_estimator_forward(ls_flow* h, const float* x, const float* mask, const float* mu, const float* t,
                                  const float* spks, const float* cond, float* out, int32_t rows, int32_t T,
                                  int32_t streaming, void* stream) {
  return ls::guarded([&] {
    ls::require(h && x && mask && mu && t && spks && cond && out, "ls_flow_estimator_forward: null argument");
    ls::SerialScope scope(h->serial, h->device(), (cudaStream_t)stream);
    h->estimator_forward(x, mask, mu, t, spks, cond, out, rows, T, streaming != 0, (cudaStream_t)stream);
  });
}

int32_t ls_flow_solve(ls_flow* h, const float* mu, const float* mask, const float* spks, const float* cond,
                      const float* noise, int64_t noise_stride, const float* t_span_host, int32_t n_timesteps,
                      float temperature, float cfg_rate, int32_t streaming, float* out, int32_t B, int32_t T,
                      void* stream) {
  return ls::guarded([&] {
    ls::require(h && mu && mask && spks && cond && noise && t_span_host && out, "ls_flow_solve: null argument");
    ls::SerialScope scope(h->serial, h->device(), (cudaStream_t)stream);
    h->solve(mu, mask, spks, cond, noise, noise_stride, t_span_host, n_timesteps, temperature, cfg_rate, streaming != 0,
             out, B, T, (cudaStream_t)stream);
  });
}

namespace {
// ls_dac_create / ls_dac_create_fp16: the decoder, the encoder, or both, from whatever the state dict holds
int32_t dac_create(const ls_tensor* weights, int32_t n_weights, int32_t device, ls_dac** out, bool fp16, const char* fn) {
  return ls::guarded([&] {
    ls::require(weights && out && n_weights > 0, std::string(fn) + ": null argument");
    ls::Weights w(weights, n_weights);
    auto h = std::make_unique<ls_dac>();
    const bool has_dec = w.has("decoder.model.0.0.weight_v"), has_enc = w.has("encoder.block.0.0.weight_v");
    ls::require(has_dec || has_enc, std::string(fn) + ": neither decoder.* nor encoder.* weights found", LS_ERR_WEIGHTS);
    if (has_dec) h->eng = std::make_unique<ls::DacEngine>(w, device, fp16);
    if (has_enc) h->enc = std::make_unique<ls::DacEncEngine>(w, device, fp16);
    *out = h.release();
  });
}
}  // namespace

int32_t ls_dac_create(const ls_tensor* weights, int32_t n_weights, int32_t device, ls_dac** out) {
  return dac_create(weights, n_weights, device, out, false, "ls_dac_create");
}
int32_t ls_dac_create_fp16(const ls_tensor* weights, int32_t n_weights, int32_t device, ls_dac** out) {
  return dac_create(weights, n_weights, device, out, true, "ls_dac_create_fp16");
}
int32_t ls_dac_create_fp32(const ls_tensor* weights, int32_t n_weights, int32_t device, ls_dac** out) {
  return ls::guarded([&] {
    ls::require(weights && out && n_weights > 0, "ls_dac_create_fp32: null argument");
    ls::Weights w(weights, n_weights);
    auto h = std::make_unique<ls_dac>();
    h->eng32 = std::make_unique<ls::DacEngineF32>(w, device);
    *out = h.release();
  });
}
void ls_dac_destroy(ls_dac* h) { delete h; }
int32_t ls_dac_hop_length(const ls_dac* h) { return h ? h->hop() : 0; }

int32_t ls_dac_decode(ls_dac* h, const float* z, const int32_t* lengths, float* wav, int32_t B, int32_t L,
                      void* stream) {
  return ls::guarded([&] {
    ls::require(h && z && wav, "ls_dac_decode: null argument");
    ls::SerialScope scope(h->serial, h->device(), (cudaStream_t)stream);
    h->decode(z, lengths, wav, B, L, (cudaStream_t)stream);
  });
}

int32_t ls_dac_encode_lengths(ls_dac* h, const float* audio, const int32_t* lengths, const float* noise, float* z, float* m,
                              float* logs, int32_t B, int32_t S, void* stream) {
  return ls::guarded([&] {
    ls::require(h && audio && z && m && logs, "ls_dac_encode: null argument");
    ls::require(h->enc != nullptr || h->eng32 != nullptr, "ls_dac_encode: this handle holds no encoder weights",
                LS_ERR_WEIGHTS);
    ls::SerialScope scope(h->serial, h->device(), (cudaStream_t)stream);
    if (h->enc) h->enc->encode(audio, lengths, noise, z, m, logs, B, S, (cudaStream_t)stream);
    else h->eng32->encode(audio, lengths, noise, z, m, logs, B, S, (cudaStream_t)stream);
  });
}

int32_t ls_dac_encode(ls_dac* h, const float* audio, const float* noise, float* z, float* m, float* logs, int32_t B,
                      int32_t S, void* stream) {
  return ls_dac_encode_lengths(h, audio, nullptr, noise, z, m, logs, B, S, stream);
}

int32_t ls_synthesize_host(ls_flow* flow, ls_dac* dac, const float* mu_host, const float* mask_host,
                           const float* spks_host, const float* cond_host, const float* noise_dev,
                           int64_t noise_stride, const float* t_span_host, int32_t n_timesteps, float temperature,
                           float cfg_rate, float* wav_host, int32_t B, int32_t T, void* stream) {
  return ls::guarded([&] {
    ls::require(flow && dac && mu_host && mask_host && spks_host && cond_host && noise_dev && wav_host,
                "ls_synthesize_host: null argument");
    ls::require(B > 0 && T > 0, "B and T must be positive");
    cudaStream_t s = (cudaStream_t)stream;
    const int F = flow->feat();
    const int hop = dac->hop();
    const size_t n_mu = (size_t)B * F * T, n_mask = (size_t)B * T, n_spk = (size_t)B * F;
    const size_t n_wav = (size_t)B * T * hop;
    // staging layout: mu | cond | latent | mask | spks | lengths(int) | wav
    const size_t need = (3 * n_mu + n_mask + n_spk + (size_t)B + n_wav) * sizeof(float) + 7 * 256;
    ls::SerialScope scope_f(flow->serial, flow->device(), s);
    ls::SerialScope scope_d(dac->serial, dac->device(), s);
    if (need > flow->stage_bytes) {  // stream-ordered growth: no synchronisation
      uint8_t* st = reinterpret_cast<uint8_t*>(flow->stage);
      ls::ws_release(st, s);
      flow->stage = nullptr, flow->stage_bytes = 0;
      ls::ws_alloc(st, need, s);
      flow->stage = reinterpret_cast<float*>(st);
      flow->stage_bytes = need;
    }
    auto al = [](size_t n) { return (n + 63) & ~size_t(63); };
    float* d_mu = flow->stage;
    float* d_cond = d_mu + al(n_mu);
    float* d_lat = d_cond + al(n_mu);
    float* d_mask = d_lat + al(n_mu);
    float* d_spk = d_mask + al(n_mask);
    int32_t* d_len = reinterpret_cast<int32_t*>(d_spk + al(n_spk));
    float* d_wav = reinterpret_cast<float*>(d_len) + al((size_t)B);
    LS_CUDA(cudaMemcpyAsync(d_mu, mu_host, n_mu * 4, cudaMemcpyHostToDevice, s));
    LS_CUDA(cudaMemcpyAsync(d_cond, cond_host, n_mu * 4, cudaMemcpyHostToDevice, s));
    LS_CUDA(cudaMemcpyAsync(d_mask, mask_host, n_mask * 4, cudaMemcpyHostToDevice, s));
    LS_CUDA(cudaMemcpyAsync(d_spk, spks_host, n_spk * 4, cudaMemcpyHostToDevice, s));
    flow->solve(d_mu, d_mask, d_spk, d_cond, noise_dev, noise_stride, t_span_host, n_timesteps, temperature, cfg_rate, false,
                d_lat, B, T, s);
    LS_CUDA(ls::launch_mask_to_lengths(d_mask, d_len, B, T, 1, s));
    dac->decode(d_lat, d_len, d_wav, B, T, s);
    LS_CUDA(cudaMemcpyAsync(wav_host, d_wav, n_wav * 4, cudaMemcpyDeviceToHost, s));
    LS_CUDA(cudaStreamSynchronize(s));
  });
}

int32_t ls_fsq_encode(const float* hidden, const float* project_down_weight, const float* project_down_bias, int32_t* tokens,
                      int64_t rows, int32_t dim, void* stream) {
  return ls::guarded([&] {
    ls::require(hidden && project_down_weight && project_down_bias && tokens && rows >= 0 && dim > 0, "ls_fsq_encode: bad argument");
    LS_CUDA(ls::launch_fsq_encode(hidden, project_down_weight, project_down_bias, tokens, rows, dim, (cudaStream_t)stream));
  });
}

int32_t ls_s3_log_mel(const float* audio, const int32_t* audio_len, const float* filters, int32_t n_mels, float* mel,
                      int32_t* mel_len, int32_t B, int64_t S, void* stream) {
  return ls::guarded([&] {
    ls::require(audio && audio_len && filters && mel && mel_len, "ls_s3_log_mel: null argument");
    ls::require(B > 0 && B <= 65535 && S >= 0, "ls_s3_log_mel: B must be in [1, 65535] and S >= 0");
    ls::require(n_mels >= 1 && n_mels <= 128, "ls_s3_log_mel: n_mels must be in [1, 128]");
    LS_CUDA(ls::launch_s3_log_mel(audio, audio_len, filters, n_mels, mel, mel_len, B, S, (cudaStream_t)stream));
  });
}

int32_t ls_resample_taps(int32_t orig_freq, int32_t new_freq, int32_t* orig_red, int32_t* new_red, int32_t* width,
                         int32_t* max_taps, int32_t* first, int32_t* count, float* taps) {
  return ls::guarded([&] {
    ls::ResampleTable t;
    const bool fill = first || count || taps;
    const int code = ls::resample_table(orig_freq, new_freq, &t, fill);
    if (orig_red) *orig_red = t.O;
    if (new_red) *new_red = t.N;
    if (width) *width = t.width;
    if (max_taps) *max_taps = code == LS_OK ? t.max_taps : 0;
    ls::require(code != LS_ERR_INVALID, "ls_resample_taps: rates must be positive");
    ls::require(code == LS_OK, "ls_resample_taps: the tap table exceeds 96 KiB", LS_ERR_UNSUPPORTED);
    if (first) std::copy(t.first.begin(), t.first.end(), first);
    if (count) std::copy(t.count.begin(), t.count.end(), count);
    if (taps) std::copy(t.taps.begin(), t.taps.end(), taps);
  });
}

int32_t ls_resampler_create(int32_t orig_freq, int32_t new_freq, int32_t device, ls_resampler** out) {
  return ls::guarded([&] {
    ls::require(out != nullptr, "ls_resampler_create: null argument");
    ls::ResampleTable t;
    const int code = ls::resample_table(orig_freq, new_freq, &t);
    ls::require(code != LS_ERR_INVALID, "ls_resampler_create: rates must be positive");
    ls::require(code == LS_OK, "ls_resampler_create: the tap table exceeds 96 KiB", LS_ERR_UNSUPPORTED);
    auto h = std::make_unique<ls_resampler>();
    ls::require(ls::resample_plan(t, &h->plan) == LS_OK, "ls_resampler_create: the tile does not fit shared memory",
                LS_ERR_UNSUPPORTED);
    // device layout: rows padded to the plan's odd stride
    const int N = t.N, stride = h->plan.stride;
    std::vector<float> taps((size_t)N * stride, 0.0f);
    std::vector<int2> fc(N);
    for (int p = 0; p < N; ++p) {
      std::copy_n(t.taps.begin() + (size_t)p * t.max_taps, t.max_taps, taps.begin() + (size_t)p * stride);
      fc[p] = make_int2(t.first[p], t.count[p]);
    }
    h->device = device;
    LS_CUDA(cudaSetDevice(device));
    LS_CUDA(cudaMalloc(&h->taps, taps.size() * sizeof(float)));
    LS_CUDA(cudaMalloc(&h->fc, fc.size() * sizeof(int2)));
    LS_CUDA(cudaMemcpy(h->taps, taps.data(), taps.size() * sizeof(float), cudaMemcpyHostToDevice));
    LS_CUDA(cudaMemcpy(h->fc, fc.data(), fc.size() * sizeof(int2), cudaMemcpyHostToDevice));
    h->plan.taps = h->taps, h->plan.fc = h->fc;
    *out = h.release();
  });
}
void ls_resampler_destroy(ls_resampler* h) { delete h; }
int32_t ls_resample(ls_resampler* h, const float* audio, const int32_t* audio_len, float* out, int32_t* out_len, int32_t B,
                    int64_t S_in, int64_t S_out, void* stream) {
  return ls::guarded([&] {
    ls::require(h && audio && audio_len && out && out_len, "ls_resample: null argument");
    ls::require(B > 0 && B <= 65535 && S_in >= 1 && S_in <= INT32_MAX && S_out <= INT32_MAX,
                "ls_resample: B must be in [1, 65535] and 1 <= S_in, S_out < 2^31");
    const long long need = ((long long)h->plan.N * S_in + h->plan.O - 1) / h->plan.O;
    ls::require(S_out >= need, "ls_resample: S_out must be at least ceil(new * S_in / orig) = " + std::to_string(need));
    LS_CUDA(cudaSetDevice(h->device));
    LS_CUDA(ls::launch_resample(h->plan, audio, audio_len, out, out_len, B, S_in, S_out, (cudaStream_t)stream));
  });
}

int32_t ls_latent_resize_linear(const float* z, const int32_t* len_in, const int32_t* len_out, float* out, int32_t B, int32_t C,
                                int32_t L_in, int32_t L_out, void* stream) {
  return ls::guarded([&] {
    ls::require(z && len_in && len_out && out, "ls_latent_resize_linear: null argument");
    ls::require(B > 0 && C > 0 && L_in > 0 && L_out > 0 && (long long)B * C <= INT32_MAX,
                "ls_latent_resize_linear: B, C, L_in, L_out must be positive");
    LS_CUDA(ls::launch_latent_resize_linear(z, len_in, len_out, out, B, C, L_in, L_out, (cudaStream_t)stream));
  });
}

int32_t ls_mask_to_lengths(const float* mask, int32_t* lengths, int32_t B, int32_t T, void* stream) {
  return ls::guarded([&] {
    ls::require(mask && lengths && B > 0 && T > 0, "ls_mask_to_lengths: bad argument");
    LS_CUDA(ls::launch_mask_to_lengths(mask, lengths, B, T, 1, (cudaStream_t)stream));
  });
}

}  // extern "C"

// ---- CUDA-graph replay of one fixed-shape solve (+ decode) --------------------------------------------------------
// The n-step solve is ~1800 PDL-chained launches (flow_matching.py:103 is the loop); for small batches the step is
// launch-bound, so the whole sequence is captured once per shape over buffers owned by this object and replayed with
// one cudaGraphLaunch.  The graph bakes the engines' workspace addresses: if a larger call on the same handles made a
// workspace grow in between (ws_generation changed) the sequence is captured again at the next launch.
struct ls_graph {
  ls_flow* flow = nullptr;
  ls_dac* dac = nullptr;  // may be null: solve only
  int B = 0, T = 0, n_steps = 0, streaming = 0;
  float temperature = 1.f, cfg_rate = 0.f;
  const float* noise = nullptr;
  long long noise_stride = 0;
  std::vector<float> t_span;
  uint8_t* buf = nullptr;
  float *mu = nullptr, *mask = nullptr, *spks = nullptr, *cond = nullptr, *lat = nullptr, *wav = nullptr;
  int32_t* len = nullptr;
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  cudaStream_t cap = nullptr;  // private capture stream
  unsigned long long gen_flow = 0, gen_dac = 0;
  long long launches = 0;  // kernels per replay

  void run(cudaStream_t s) {
    flow->solve(mu, mask, spks, cond, noise, noise_stride, t_span.data(), n_steps, temperature, cfg_rate, streaming != 0, lat, B,
                T, s);
    if (dac) {
      LS_CUDA(ls::launch_mask_to_lengths(mask, len, B, T, 1, s));
      dac->decode(lat, len, wav, B, T, s);
    }
  }
  void drop() {
    if (exec) cudaGraphExecDestroy(exec);
    if (graph) cudaGraphDestroy(graph);
    exec = nullptr, graph = nullptr;
  }
  void capture(cudaStream_t s) {
    drop();
    run(s);  // eager pass: workspace growth, plans, per-device attribute opt-ins all happen outside the capture
    // the capture runs on a private stream: the caller's stream may be the legacy default stream, which cannot be captured
    if (!cap) LS_CUDA(cudaStreamCreateWithFlags(&cap, cudaStreamNonBlocking));
    const long long before = ls::g_launch_count.load();
    LS_CUDA(cudaStreamBeginCapture(cap, cudaStreamCaptureModeThreadLocal));
    try {
      run(cap);
    } catch (...) {
      cudaGraph_t g = nullptr;
      cudaStreamEndCapture(cap, &g);
      if (g) cudaGraphDestroy(g);
      throw;
    }
    LS_CUDA(cudaStreamEndCapture(cap, &graph));
    launches = ls::g_launch_count.load() - before;
    LS_CUDA(cudaGraphInstantiate(&exec, graph, 0));
    gen_flow = flow->eng ? flow->eng->ws_generation() : 0;
    gen_dac = dac && dac->eng ? dac->eng->ws_generation() : 0;
  }
  bool current() const {
    return exec && gen_flow == (flow->eng ? flow->eng->ws_generation() : 0) &&
           gen_dac == (dac && dac->eng ? dac->eng->ws_generation() : 0);
  }
  ~ls_graph() {
    drop();
    if (cap) cudaStreamDestroy(cap);
    if (buf) cudaFree(buf);
  }
};

namespace {
// the SM count a test hook launches for: 0 = the device's own; anything outside [0, device SMs] is refused
int test_hook_sms(int32_t num_sms, const char* what) {
  int dev = 0, sms = 0;
  LS_CUDA(cudaGetDevice(&dev));
  LS_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  ls::require(num_sms >= 0 && num_sms <= sms, std::string(what) + ": num_sms outside [0, device SMs]");
  return num_sms == 0 ? sms : num_sms;
}
}  // namespace

extern "C" {

int32_t ls_graph_create(ls_flow* flow, ls_dac* dac, const float* noise_dev, int64_t noise_stride, const float* t_span_host,
                        int32_t n_timesteps, float temperature, float cfg_rate, int32_t streaming, int32_t B, int32_t T,
                        void* stream, ls_graph** out) {
  return ls::guarded([&] {
    ls::require(flow && noise_dev && t_span_host && out, "ls_graph_create: null argument");
    ls::require(flow->eng != nullptr && (!dac || dac->eng != nullptr), "ls_graph_create: tensor-core handles only (fp32 mode is not graphed)",
                LS_ERR_UNSUPPORTED);
    ls::require(B > 0 && T > 0 && n_timesteps > 0 && n_timesteps <= 64, "ls_graph_create: need B, T > 0 and 1 <= n_timesteps <= 64");
    cudaStream_t s = (cudaStream_t)stream;
    auto g = std::make_unique<ls_graph>();
    g->flow = flow, g->dac = dac, g->B = B, g->T = T, g->n_steps = n_timesteps, g->streaming = streaming;
    g->temperature = temperature, g->cfg_rate = cfg_rate, g->noise = noise_dev, g->noise_stride = noise_stride;
    g->t_span.assign(t_span_host, t_span_host + n_timesteps + 1);
    const int F = flow->feat();
    const size_t n_mu = (size_t)B * F * T, n_mask = (size_t)B * T, n_spk = (size_t)B * F;
    const size_t n_wav = dac ? (size_t)B * T * dac->hop() : 0;
    auto al = [](size_t n) { return (n + 63) & ~size_t(63); };
    const size_t floats = 3 * al(n_mu) + al(n_mask) + al(n_spk) + al((size_t)B) + al(n_wav);
    ls::SerialScope scope_f(flow->serial, flow->device(), s);
    std::unique_ptr<ls::SerialScope> scope_d;
    if (dac) scope_d = std::make_unique<ls::SerialScope>(dac->serial, dac->device(), s);
    LS_CUDA(cudaMalloc(&g->buf, floats * sizeof(float)));
    LS_CUDA(cudaMemsetAsync(g->buf, 0, floats * sizeof(float), s));
    float* f = reinterpret_cast<float*>(g->buf);
    g->mu = f, f += al(n_mu);
    g->cond = f, f += al(n_mu);
    g->lat = f, f += al(n_mu);
    g->mask = f, f += al(n_mask);
    g->spks = f, f += al(n_spk);
    g->len = reinterpret_cast<int32_t*>(f), f += al((size_t)B);
    g->wav = dac ? f : nullptr;
    // the capture pass needs a valid mask: all frames valid until the caller writes the real one
    std::vector<float> ones(n_mask, 1.0f);
    LS_CUDA(cudaMemcpyAsync(g->mask, ones.data(), n_mask * 4, cudaMemcpyHostToDevice, s));
    LS_CUDA(cudaStreamSynchronize(s));  // (`ones` leaves scope; creation is not a hot call)
    g->capture(s);
    *out = g.release();
  });
}

void* ls_graph_buffer(ls_graph* g, int32_t which) {
  if (!g) return nullptr;
  switch (which) {
    case 0: return g->mu;
    case 1: return g->mask;
    case 2: return g->spks;
    case 3: return g->cond;
    case 4: return g->lat;
    case 5: return g->wav;
    default: return nullptr;
  }
}

int32_t ls_graph_launch(ls_graph* g, void* stream) {
  return ls::guarded([&] {
    ls::require(g != nullptr, "ls_graph_launch: null argument");
    cudaStream_t s = (cudaStream_t)stream;
    ls::SerialScope scope_f(g->flow->serial, g->flow->device(), s);
    std::unique_ptr<ls::SerialScope> scope_d;
    if (g->dac) scope_d = std::make_unique<ls::SerialScope>(g->dac->serial, g->dac->device(), s);
    g->flow->eng->check_sticky();
    if (!g->current()) g->capture(s);
    LS_CUDA(cudaGraphLaunch(g->exec, s));
    ls::g_launch_count.fetch_add(g->launches, std::memory_order_relaxed);
  });
}

int64_t ls_graph_kernel_count(const ls_graph* g) { return g ? g->launches : 0; }

void ls_graph_destroy(ls_graph* g) { delete g; }

int32_t ls_debug_set_buffer(void* dev_ptr, int64_t bytes) {
  ls::g_debug_buffer = reinterpret_cast<long long*>(dev_ptr);
  ls::g_debug_bytes = dev_ptr ? bytes : 0;
  return LS_OK;
}

int32_t ls_profile_begin(void) {
  ls::prof_begin();
  return LS_OK;
}
int32_t ls_profile_end(ls_profile_entry* out4, int32_t n_entries) {
  return ls::guarded([&] {
    ls::require(out4 != nullptr && n_entries == ls::PK_COUNT, "ls_profile_end: need LS_PROFILE_KINDS entries");
    long long n[ls::PK_COUNT];
    double ms[ls::PK_COUNT], fl[ls::PK_COUNT], by[ls::PK_COUNT];
    ls::prof_end(n, ms, fl, by);
    for (int k = 0; k < ls::PK_COUNT; ++k) out4[k] = ls_profile_entry{n[k], ms[k], fl[k], by[k]};
  });
}

int32_t ls_test_conv_gemm(const ls_conv_gemm_desc* d, int32_t num_sms, int32_t* plan_out, void* stream) {
  return ls::guarded([&] {
    ls::require(d && d->a0 && d->w, "ls_test_conv_gemm: null argument");
    const int sms = test_hook_sms(num_sms, "ls_test_conv_gemm");
    CUtensorMap a0, a1, w;
    const bool halo = ls::conv_halo_enabled();
    const int box = halo ? ls::conv_halo_box_rows(d->taps, d->dil) : 128;
    ls::require(ls::make_act_map(&a0, d->a0, d->a0_C, d->T_in, d->B, d->a0_C, (long long)d->T_in * d->a0_C, box),
                "tensor map a0", LS_ERR_CUDA);
    if (d->a1)
      ls::require(ls::make_act_map(&a1, d->a1, d->a1_C, d->T_in, d->B, d->a1_C, (long long)d->T_in * d->a1_C, box),
                  "tensor map a1", LS_ERR_CUDA);
    else
      a1 = a0;
    ls::require(ls::make_weight_map(&w, d->w, d->K, d->taps * d->N, d->block_n), "tensor map w", LS_ERR_CUDA);
    ls::ConvGemmParams p{};
    p.B = d->B, p.M = d->M, p.N = d->N, p.block_n = d->block_n, p.taps = d->taps, p.dil = d->dil, p.pad = d->pad;
    p.kb_per_tap = (d->K + 63) / 64;
    p.kb_split = d->a1 ? d->a0_C / 64 : p.kb_per_tap;
    p.lengths = d->lengths, p.m_len_mul = d->m_len_mul, p.m_len_add = d->m_len_add, p.skip_halo = d->skip_halo;
    p.chan_mod = d->chan_mod, p.bias = d->bias, p.act = d->act, p.ln_g = d->ln_g, p.ln_b = d->ln_b;
    p.temb = d->temb, p.temb_bstride = d->temb_bstride, p.addend = d->addend, p.addend_dtype = d->addend_dtype;
    p.out0 = d->out0, p.out0_dtype = d->out0_dtype, p.out1 = d->out1, p.out1_mode = d->out1_mode;
    p.p1_a = d->p1_a, p.p1_b = d->p1_b, p.n_store = d->n_store;
    p.out_ld = d->out_ld, p.out_shift = d->out_shift, p.out_bstride = d->out_bstride, p.out_alloc = d->out_alloc;
    p.out_valid_mul = d->out_valid_mul;
    ls::require(d->fp16 == 0 || d->fp16 == 1, "ls_test_conv_gemm: fp16 must be 0 or 1");
    p.k_true = d->K, p.tag = 0, p.halo_mode = ls::conv_halo_mode(), p.fp16 = d->fp16;
    p.zero_skipped = d->zero_skipped;
    if (d->res_w) {  // the fused residual GEMM, set up as flow_engine.cu does (128-row activation boxes whatever the halo mode)
      ls::require(d->res_a0 != nullptr && !d->addend && d->res_K == d->res_a0_C + d->res_a1_C &&
                      (d->res_a1 == nullptr || d->res_a0_C % 64 == 0),
                  "ls_test_conv_gemm: the residual GEMM needs res_a0, no addend, res_K = res_a0_C + res_a1_C and "
                  "res_a0_C % 64 == 0 with two sources");
      ls::require(ls::make_act_map(&p.res_a0, d->res_a0, d->res_a0_C, d->T_in, d->B, d->res_a0_C,
                                   (long long)d->T_in * d->res_a0_C, 128),
                  "tensor map res_a0", LS_ERR_CUDA);
      if (d->res_a1)
        ls::require(ls::make_act_map(&p.res_a1, d->res_a1, d->res_a1_C, d->T_in, d->B, d->res_a1_C,
                                     (long long)d->T_in * d->res_a1_C, 128),
                    "tensor map res_a1", LS_ERR_CUDA);
      else
        p.res_a1 = p.res_a0;
      ls::require(ls::make_weight_map(&p.res_w, d->res_w, d->res_K, d->N, d->block_n), "tensor map res_w", LS_ERR_CUDA);
      p.addend = nullptr, p.addend_dtype = ls::ADD_GEMM;
      p.res_kb = (d->res_K + 63) / 64, p.res_split = d->res_a1 ? d->res_a0_C / 64 : p.res_kb, p.res_k_true = d->res_K;
      p.res_bias = d->res_bias;
    }
    LS_CUDA(ls::launch_conv_gemm(a0, a1, w, p, sms, (cudaStream_t)stream, plan_out));
  });
}

int32_t ls_test_attention(const void* qkv, void* out, const int32_t* lengths, int32_t B, int32_t T, int32_t H,
                          int32_t chunk, int32_t fp16, const float* bias, int64_t bias_ld, int64_t bias_bh,
                          void* stream) {
  return ls::guarded([&] {
    ls::require(qkv && out, "ls_test_attention: null argument");
    ls::require(B >= 1 && B <= 65535 && T >= 1 && H >= 1 && H <= 65535 && chunk >= 0,
                "ls_test_attention: B, T, H or chunk out of range");
    ls::require(fp16 == 0 || fp16 == 1, "ls_test_attention: fp16 must be 0 or 1");
    if (bias)
      ls::require(bias_ld >= 2LL * T - 1 && bias_bh >= (long long)T * bias_ld,
                  "ls_test_attention: bias needs bias_ld >= 2T-1 and bias_bh >= T*bias_ld");
    CUtensorMap m;
    ls::require(ls::make_act_map(&m, qkv, 3 * H * 64, T, B, 3 * H * 64, (long long)T * 3 * H * 64, ATTN_KV),
                "tensor map qkv", LS_ERR_CUDA);
    ls::AttnParams ap{};
    ap.B = B, ap.T = T, ap.H = H, ap.lengths = lengths, ap.chunk = chunk;
    ap.scale_log2e = 0.125f * 1.4426950408889634f;
    ap.out = reinterpret_cast<__nv_bfloat16*>(out);
    ap.bias = bias, ap.bias_ld = bias_ld, ap.bias_bh = bias_bh;
    ap.fp16 = fp16;
    LS_CUDA(ls::launch_attention(m, ap, (cudaStream_t)stream));
  });
}

int32_t ls_test_tblock(const void* att, float* u, const void* wo, const void* w1, const void* w2, const void* wqkv,
                       const float* vec, void* qkv_out, void* tail_out, const int32_t* lengths, int32_t R, int32_t T,
                       int32_t tail_mode, int32_t fp16, int32_t no_skip, int32_t num_sms, int32_t* plan_out,
                       void* stream) {
  return ls::guarded([&] {
    ls::require(att && u && wo && w1 && w2 && wqkv && vec, "ls_test_tblock: null argument");
    ls::require(fp16 == 0 || fp16 == 1, "ls_test_tblock: fp16 must be 0 or 1");
    const int sms = test_hook_sms(num_sms, "ls_test_tblock");
    ls::require(tail_mode != 1 ? qkv_out != nullptr : tail_out != nullptr, "ls_test_tblock: missing output");
    ls::TBlockMaps m;
    ls::require(ls::make_tile_map(&m.att, att, 2, 512, R, 128) && ls::make_tile_map(&m.u, u, 4, 256, R, 128),
                "tensor map att / u", LS_ERR_CUDA);
    ls::require(ls::make_weight_map(&m.wo, wo, 512, 256, TBLOCK_WIDE_BOX_ROWS) &&
                    ls::make_weight_map(&m.w2, w2, 1024, 256, TBLOCK_WIDE_BOX_ROWS) &&
                    (TBLOCK_PAIR ? ls::make_weight_map_kb(&m.w1, w1, 256, 1024, 64, 2) &&
                                       ls::make_weight_map_kb(&m.wqkv, wqkv, 256, 1536, 64, 2)
                                 : ls::make_weight_map(&m.w1, w1, 256, 1024, TBLOCK_WBOX_ROWS) &&
                                       ls::make_weight_map(&m.wqkv, wqkv, 256, 1536, TBLOCK_WBOX_ROWS)),
                "tensor map weights", LS_ERR_CUDA);
    m.qkv_out = m.att, m.tail_out = m.att;
    if (tail_mode != 1)
      ls::require(ls::make_tile_map(&m.qkv_out, qkv_out, 2, 1536, R, 128), "tensor map qkv", LS_ERR_CUDA);
    else
      ls::require(ls::make_tile_map(&m.tail_out, tail_out, 2, 256, R, 128), "tensor map tail", LS_ERR_CUDA);
    ls::TBlockParams p{};
    p.R = R, p.T = T, p.lengths = lengths, p.vec = vec, p.tail_mode = tail_mode, p.fp16 = fp16, p.no_skip = no_skip;
    LS_CUDA(ls::launch_tblock(m, p, sms, (cudaStream_t)stream, plan_out));
  });
}

int32_t ls_test_groupnorm_mish(const float* x, void* stats, const float* gamma, const float* beta, const float* temb,
                               int64_t temb_bstride, const float* addend, float* out_f32, void* out_h, int32_t B,
                               int32_t C, int32_t T, int32_t G, const int32_t* lengths, int32_t fp16, void* stream) {
  return ls::guarded([&] {
    ls::require(x && stats && gamma && beta, "ls_test_groupnorm_mish: null argument");
    LS_CUDA(ls::launch_groupnorm_mish(x, reinterpret_cast<float2*>(stats), gamma, beta, temb, temb_bstride, addend, out_f32,
                                      reinterpret_cast<__nv_bfloat16*>(out_h), B, C, T, G, lengths, fp16,
                                      (cudaStream_t)stream));
  });
}

}  // extern "C"
