// DAC-VAE decoder engine: z [B,80,L] -> 24 kHz waveform [B,1,L*hop].
//
// Layer order follows dac-vae/model.py:485-488 (de_conv_pre -> Decoder), :326-379 (Decoder), :237-323
// (DecoderBlock), :107-143 (ResidualUnit), with every generator Conv1d followed by LeakyReLU(0.1)
// (the shadowing WNConv1d at model.py:509-514).  weight_norm (layers.py:9-14) is folded once here.
// All convolutions run as conv_gemm launches; Snake1d (layers.py:18-33) is never a pass of its own: each
// epilogue emits snake(x) for the *next* convolution as its 16-bit secondary output (bf16, or fp16 for a handle
// built with fp16 operands).
#include <cmath>

#include "dac_engine.h"

namespace ls {

// Conv1d weight_v [N][K][taps] with weight_g [N] -> folded 16-bit [taps][Npad][K]
PackedLinear pack_wn_conv(Arena& a, const Weights& w, const std::string& p, bool fp16, int n_pad_to) {
  const ls_tensor& v = w.get(p + ".weight_v");
  const ls_tensor& g = w.get(p + ".weight_g");
  const ls_tensor& b = w.get(p + ".bias");
  require(v.ndim == 3 && g.shape[0] == v.shape[0], "unexpected weight_norm tensors at " + p, LS_ERR_WEIGHTS);
  PackedLinear pl;
  const int N = (int)v.shape[0];
  pl.K = (int)v.shape[1];
  pl.taps = (int)v.shape[2];
  pl.N = n_pad_to > N ? n_pad_to : N;
  pl.block_n = pick_block_n(pl.N);
  pl.w_off = a.reserve((size_t)pl.taps * pl.N * pl.K * 2);
  __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(a.host(pl.w_off));
  for (size_t i = 0; i < (size_t)pl.taps * pl.N * pl.K; ++i) dst[i] = __float2bfloat16(0.f);  // 0 has the same bits in fp16
  const size_t per = (size_t)pl.K * pl.taps;
  for (int n = 0; n < N; ++n) {
    double ss = 0;
    for (size_t i = 0; i < per; ++i) ss += (double)v.data[n * per + i] * v.data[n * per + i];
    const float scale = g.data[n] / (float)std::sqrt(ss);
    for (int k = 0; k < pl.K; ++k)
      for (int t = 0; t < pl.taps; ++t)
        dst[((size_t)t * pl.N + n) * pl.K + k] = dac_w16(v.data[(n * (size_t)pl.K + k) * pl.taps + t] * scale, fp16, p);
  }
  std::vector<float> bias(pl.N, 0.f);
  for (int n = 0; n < N; ++n) bias[n] = b.data[n];
  pl.bias_off = a.put_f32(bias.data(), pl.N);
  pl.has_bias = true;
  return pl;
}

void finalize_linear(const Arena& a, PackedLinear& pl) {
  require(make_weight_map(&pl.map, a.ptr<uint8_t>(pl.w_off), pl.K, pl.taps * pl.N, pl.block_n),
          "cuTensorMapEncodeTiled failed for a weight matrix", LS_ERR_CUDA);
  pl.bias = a.ptr<float>(pl.bias_off);
}

namespace {

// ConvTranspose1d weight_v [Cin][Cout][2s], weight_g [Cin] -> two-tap polyphase GEMM, 16-bit [2][s*Cout][Cin]:
//   out[q*s + phi - pad] = in[q] . W[:, :, phi] + in[q-1] . W[:, :, phi + s]        (model.py:255-262)
// tap 0 multiplies in[q-1], tap 1 multiplies in[q]  (A row = q + tap - 1).
PackedLinear pack_wn_convT(Arena& a, const Weights& w, const std::string& p, int stride, bool fp16) {
  const ls_tensor& v = w.get(p + ".weight_v");
  const ls_tensor& g = w.get(p + ".weight_g");
  const ls_tensor& b = w.get(p + ".bias");
  require(v.ndim == 3 && v.shape[2] == 2 * stride && g.shape[0] == v.shape[0], "unexpected ConvTranspose1d at " + p,
          LS_ERR_WEIGHTS);
  const int cin = (int)v.shape[0], cout = (int)v.shape[1], k2 = 2 * stride;
  PackedLinear pl;
  pl.K = cin, pl.taps = 2, pl.N = stride * cout, pl.block_n = pick_block_n(pl.N);
  pl.w_off = a.reserve((size_t)2 * pl.N * cin * 2);
  __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(a.host(pl.w_off));
  const size_t per = (size_t)cout * k2;
  for (int c = 0; c < cin; ++c) {
    double ss = 0;
    for (size_t i = 0; i < per; ++i) ss += (double)v.data[c * per + i] * v.data[c * per + i];
    const float scale = g.data[c] / (float)std::sqrt(ss);  // weight_norm dim 0 = Cin for ConvTranspose
    for (int n = 0; n < cout; ++n)
      for (int phi = 0; phi < stride; ++phi) {
        const float w_q = v.data[(c * (size_t)cout + n) * k2 + phi] * scale;            // multiplies in[q]
        const float w_qm1 = v.data[(c * (size_t)cout + n) * k2 + phi + stride] * scale;  // multiplies in[q-1]
        dst[((size_t)0 * pl.N + phi * cout + n) * cin + c] = dac_w16(w_qm1, fp16, p);
        dst[((size_t)1 * pl.N + phi * cout + n) * cin + c] = dac_w16(w_q, fp16, p);
      }
  }
  pl.bias_off = a.put_f32(b.data, cout);
  pl.has_bias = true;
  return pl;
}

}  // namespace

struct DacEngine::UnitW {
  PackedLinear conv7, conv1;
  size_t a0, ia0, a2, ia2;  // Snake alpha / 1/(alpha+1e-9) before conv7 and before conv1
};
struct DacEngine::StageW {
  int stride, cin, cout;
  size_t a_in, ia_in;  // Snake before the transposed conv
  PackedLinear up;
  UnitW unit[3];
};
// sA[i]/sB[i]: stage-i views (i = 0: output of the input conv).  Every consumer of a buffer gets a view whose box
// carries the halo of its convolution: up = 2-tap transposed conv, d[j] = conv7 with dilation 1 / 3 / 9.
struct DacEngine::Plan {
  CUtensorMap zt, a0;
  struct {
    CUtensorMap up, d[3];
  } sA[6];
  CUtensorMap sB[6];
};

DacEngine::~DacEngine() {
  if (ws_base_) cudaFree(ws_base_);
}

DacEngine::DacEngine(const Weights& w, int device, bool fp16) : device_(device), fp16_(fp16 ? 1 : 0) {
  LS_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  LS_CUDA(cudaGetDeviceProperties(&prop, device));
  require(prop.major == 10, "this library only runs on sm_100 (B200) devices", LS_ERR_UNSUPPORTED);
  num_sms_ = prop.multiProcessorCount;

  auto snake = [&](const std::string& name, int c, size_t* a_off, size_t* ia_off) {
    const ls_tensor& al = w.get(name, {1, c, 1});
    std::vector<float> ia(c);
    for (int i = 0; i < c; ++i) ia[i] = 1.0f / (al.data[i] + 1e-9f);  // layers.py:22
    *a_off = arena_.put_f32(al.data, c);
    *ia_off = arena_.put_f32(ia.data(), c);
  };

  pre_ = pack_wn_conv(arena_, w, "de_conv_pre.0", fp16);
  in_ = pack_wn_conv(arena_, w, "decoder.model.0.0", fp16);
  latent_ = pre_.K;
  dim_ = in_.N;
  require(pre_.taps == 1 && in_.taps == 7 && latent_ % 16 == 0 && dim_ % 16 == 0, "unexpected DAC decoder stem",
          LS_ERR_UNSUPPORTED);
  int c = dim_;
  hop_ = 1;
  for (int i = 1; w.has("decoder.model." + std::to_string(i) + ".block.1.weight_v"); ++i) {
    const std::string p = "decoder.model." + std::to_string(i) + ".block";
    StageW st;
    st.stride = (int)w.get(p + ".1.weight_v").shape[2] / 2;
    st.cin = c, st.cout = c / 2;
    require(st.cout % 16 == 0, "decoder channel count must stay a multiple of 16", LS_ERR_UNSUPPORTED);
    snake(p + ".0.alpha", c, &st.a_in, &st.ia_in);
    st.up = pack_wn_convT(arena_, w, p + ".1", st.stride, fp16);
    for (int j = 0; j < 3; ++j) {
      const std::string q = p + "." + std::to_string(j + 2) + ".block";
      snake(q + ".0.alpha", st.cout, &st.unit[j].a0, &st.unit[j].ia0);
      st.unit[j].conv7 = pack_wn_conv(arena_, w, q + ".1.0", fp16);
      snake(q + ".2.alpha", st.cout, &st.unit[j].a2, &st.unit[j].ia2);
      st.unit[j].conv1 = pack_wn_conv(arena_, w, q + ".3.0", fp16);
      require(st.unit[j].conv7.taps == 7 && st.unit[j].conv1.taps == 1, "unexpected ResidualUnit at " + q,
              LS_ERR_UNSUPPORTED);
    }
    rates_.push_back(st.stride);
    hop_ *= st.stride;
    c = st.cout;
    stages_.push_back(st);
  }
  const int n = (int)stages_.size();
  require(n >= 1 && n <= 5, "DAC decoder must have 1..5 upsampling stages", LS_ERR_UNSUPPORTED);
  snake("decoder.model." + std::to_string(n + 1) + ".alpha", c, &final_alpha_, &final_ialpha_);
  final_ = pack_wn_conv(arena_, w, "decoder.model." + std::to_string(n + 2) + ".0", fp16, 16);
  out_ch_ = (int)w.get("decoder.model." + std::to_string(n + 2) + ".0.bias").shape[0];
  require(out_ch_ == 1 && final_.taps == 7, "only mono output (d_out=1) is covered", LS_ERR_UNSUPPORTED);

  arena_.upload();
  finalize_linear(arena_, pre_);
  finalize_linear(arena_, in_);
  finalize_linear(arena_, final_);
  for (auto& st : stages_) {
    finalize_linear(arena_, st.up);
    for (auto& u : st.unit) {
      finalize_linear(arena_, u.conv7);
      finalize_linear(arena_, u.conv1);
    }
  }
}

void DacEngine::ensure_workspace(int B, int L, cudaStream_t s) {
  const long long frames = (long long)B * L;
  if (frames <= cap_frames_ && B <= cap_b_) return;
  ws_release(ws_base_, s);
  plans_.clear();
  cap_frames_ = std::max(frames, cap_frames_);
  cap_b_ = std::max(B, cap_b_);
  long long per_frame = dim_;  // elements per latent frame of the widest activation
  long long r = 1;
  for (auto& st : stages_) {
    r *= st.stride;
    per_frame = std::max(per_frame, r * st.cout);
  }
  size_t off = 0;
  auto take = [&](size_t bytes) {
    size_t o = off;
    off = (off + bytes + 1023) & ~size_t(1023);
    return o;
  };
  const size_t F = (size_t)cap_frames_;
  o_zt_ = take(F * latent_ * 2);
  o_a0_ = take(F * latent_ * 2);
  o_x_ = take(F * per_frame * 4);
  o_sA_[0] = take(F * per_frame * 2);
  o_sA_[1] = take(F * per_frame * 2);
  o_sB_ = take(F * per_frame * 2);
  o_len_ = take((size_t)cap_b_ * 4);
  ws_alloc(ws_base_, off, s);
  ++ws_generation_;
}

const DacEngine::Plan& DacEngine::plan_for(int B, int L) {
  auto key = std::make_pair(B, L);
  auto it = plans_.find(key);
  if (it != plans_.end()) return *it->second;
  auto pl = std::make_unique<Plan>();
  const bool halo = conv_halo_enabled();
  auto mk = [&](CUtensorMap* m, size_t off, int C, long long rows, int taps, int dil) {
    require(make_act_map(m, ws_base_ + off, C, (int)rows, B, C, rows * C, halo ? conv_halo_box_rows(taps, dil) : 128),
            "cuTensorMapEncodeTiled failed for an activation buffer", LS_ERR_CUDA);
  };
  static const int dils[3] = {1, 3, 9};
  mk(&pl->zt, o_zt_, latent_, L, 1, 1);
  mk(&pl->a0, o_a0_, latent_, L, 7, 1);
  mk(&pl->sA[0].up, o_sA_[0], dim_, L, 2, 1);
  long long rows = L;
  for (size_t i = 0; i < stages_.size(); ++i) {
    rows *= stages_[i].stride;
    mk(&pl->sA[i + 1].up, o_sA_[(i + 1) & 1], stages_[i].cout, rows, 2, 1);
    for (int j = 0; j < 3; ++j) mk(&pl->sA[i + 1].d[j], o_sA_[(i + 1) & 1], stages_[i].cout, rows, 7, dils[j]);
    mk(&pl->sB[i + 1], o_sB_, stages_[i].cout, rows, 1, 1);
  }
  const Plan& ref = *pl;
  plans_[key] = std::move(pl);
  return ref;
}

void DacEngine::decode(const float* z, const int* lengths, float* wav, int B, int L, cudaStream_t s) {
  require(B > 0 && L > 0, "B and L must be positive");
  require((long long)L * hop_ < (1ll << 31), "utterance too long");
  LS_CUDA(cudaSetDevice(device_));
  ensure_workspace(B, L, s);
  const Plan& pl = plan_for(B, L);
  auto f32 = [&](size_t off) { return arena_.ptr<float>(off); };
  const bool halo = conv_halo_enabled();

  // generic launcher: rows = output rows per item of this layer, C_out = channel count of the output layout
  auto conv = [&](const CUtensorMap& a, const PackedLinear& w, long long rows, int rate, int dil, ConvGemmParams p) {
    p.B = B, p.M = (int)rows, p.N = w.N, p.block_n = w.block_n;
    p.taps = w.taps, p.dil = dil, p.pad = (w.taps - 1) / 2 * dil;
    p.kb_per_tap = (w.K + 63) / 64, p.kb_split = p.kb_per_tap;
    p.lengths = lengths, p.m_len_mul = rate, p.m_len_add = 0, p.skip_halo = 64;
    p.bias = w.bias;
    if (p.chan_mod == 0) p.chan_mod = w.N;
    if (p.n_store == 0) p.n_store = w.N;
    if (p.out_ld == 0) {
      p.out_ld = w.N, p.out_shift = 0, p.out_bstride = rows * w.N, p.out_alloc = rows * w.N;
      p.out_valid_mul = (long long)rate * w.N;
    }
    p.k_true = w.K, p.tag = 1, p.halo_mode = halo ? conv_halo_mode() : 0, p.fp16 = fp16_;
    LS_CUDA(launch_conv_gemm(a, a, w.map, p, num_sms_, s));
  };

  LS_CUDA(launch_pack_nct(z, ws<__nv_bfloat16>(o_zt_), B, latent_, L, (long long)latent_ * L, latent_, 0, lengths, s, fp16_));
  {  // de_conv_pre: 1x1 + LeakyReLU
    ConvGemmParams p{};
    p.act = ACT_LRELU, p.out1 = ws<void>(o_a0_), p.out1_mode = OUT1_COPY;
    conv(pl.zt, pre_, L, 1, 1, p);
  }
  {  // input conv k=7 + LeakyReLU, then the first block's Snake
    ConvGemmParams p{};
    p.act = ACT_LRELU, p.out1 = ws<void>(o_sA_[0]), p.out1_mode = OUT1_SNAKE;
    p.p1_a = f32(stages_[0].a_in), p.p1_b = f32(stages_[0].ia_in);
    conv(pl.a0, in_, L, 1, 1, p);
  }
  long long rows = L;
  int rate = 1;
  // residual stream x of the five stages: written by the transposed conv, read + rewritten by each unit's conv1.
  // Kept as fp16 (11 significand bits, no fewer than the 16-bit operands the convolutions consume): the thin stages
  // are bound by the bytes their epilogues move, and x was half of them as fp32.  -DLS_DAC_X_F32=1 keeps it fp32.
#ifndef LS_DAC_X_F32
#define LS_DAC_X_F32 0
#endif
  constexpr int kXDtype = LS_DAC_X_F32 ? OUT_F32 : OUT_F16;
  void* x = ws<void>(o_x_);
  for (size_t i = 0; i < stages_.size(); ++i) {
    const StageW& st = stages_[i];
    const long long rows_in = rows;
    const int rate_in = rate;
    rows *= st.stride, rate *= st.stride;
    void* sA = ws<void>(o_sA_[(i + 1) & 1]);
    void* sB = ws<void>(o_sB_);
    {  // transposed conv as a two-tap GEMM over q in [0, rows_in]; output row = q*stride + phi - pad
      const int padT = (st.stride + 1) / 2;  // math.ceil(stride / 2)
      ConvGemmParams p{};
      p.B = B, p.M = (int)rows_in + 1, p.N = st.up.N, p.block_n = st.up.block_n;
      p.taps = 2, p.dil = 1, p.pad = 1;
      p.kb_per_tap = (st.cin + 63) / 64, p.kb_split = p.kb_per_tap;
      p.lengths = lengths, p.m_len_mul = rate_in, p.m_len_add = 1, p.skip_halo = 64;
      p.chan_mod = st.cout, p.bias = st.up.bias, p.act = ACT_NONE;
      p.out0 = x, p.out0_dtype = kXDtype;
      p.out1 = sA, p.out1_mode = OUT1_SNAKE, p.p1_a = f32(st.unit[0].a0), p.p1_b = f32(st.unit[0].ia0);
      p.n_store = st.up.N;
      p.out_ld = st.up.N, p.out_shift = -(long long)padT * st.cout;
      p.out_bstride = rows * st.cout, p.out_alloc = rows * st.cout, p.out_valid_mul = (long long)rate * st.cout;
      p.k_true = st.cin, p.tag = 1, p.halo_mode = halo ? conv_halo_mode() : 0, p.fp16 = fp16_;
      LS_CUDA(launch_conv_gemm(pl.sA[i].up, pl.sA[i].up, st.up.map, p, num_sms_, s));
    }
    static const int dils[3] = {1, 3, 9};
    for (int j = 0; j < 3; ++j) {
      const UnitW& u = st.unit[j];
      {  // Snake (already applied) -> conv7 dilated -> LeakyReLU -> Snake
        ConvGemmParams p{};
        p.act = ACT_LRELU, p.out1 = sB, p.out1_mode = OUT1_SNAKE, p.p1_a = f32(u.a2), p.p1_b = f32(u.ia2);
        conv(pl.sA[i + 1].d[j], u.conv7, rows, rate, dils[j], p);
      }
      {  // conv1 -> LeakyReLU -> + x ; secondary output = Snake of whatever consumes x next
        ConvGemmParams p{};
        p.act = ACT_LRELU, p.addend = x, p.addend_dtype = kXDtype;
        const bool last_unit = j == 2;
        if (!last_unit) p.out0 = x, p.out0_dtype = kXDtype;
        size_t na, nia;
        if (!last_unit) na = st.unit[j + 1].a0, nia = st.unit[j + 1].ia0;
        else if (i + 1 < stages_.size()) na = stages_[i + 1].a_in, nia = stages_[i + 1].ia_in;
        else na = final_alpha_, nia = final_ialpha_;
        p.out1 = sA, p.out1_mode = OUT1_SNAKE, p.p1_a = f32(na), p.p1_b = f32(nia);
        conv(pl.sB[i + 1], u.conv1, rows, rate, 1, p);
      }
    }
  }
  {  // final Snake (applied) -> conv7 -> LeakyReLU -> tanh, mono fp32 waveform
    ConvGemmParams p{};
    p.act = ACT_LRELU_TANH, p.out0 = wav, p.out0_dtype = OUT_F32;
    p.chan_mod = 16, p.n_store = 1, p.zero_skipped = 1;
    p.out_ld = 1, p.out_shift = 0, p.out_bstride = rows, p.out_alloc = rows, p.out_valid_mul = rate;
    conv(pl.sA[stages_.size()].d[0], final_, rows, rate, 1, p);
  }
}

}  // namespace ls
