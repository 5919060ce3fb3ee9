// DAC-VAE encoder engine: 24 kHz audio [B,1,S] -> latents (z, m, logs) [B,latent,S/hop].
//
// Layer order follows dac-vae/model.py:195-234 (Encoder), :146-192 (EncoderBlock: ResidualUnit x3 (dil 1,3,9) ->
// Snake -> WNConv1d(k = 2s, stride s, pad ceil(s/2))), :107-143 (ResidualUnit), :469-483 (encode: leaky_relu ->
// en_conv_post -> split -> clamp -> m + noise * exp(logs)); every WNConv1d carries the shadow's LeakyReLU(0.1)
// (model.py:509-514).  Like in the decoder engine Snake is never a pass of its own.
//
// A stride-s convolution over time-major activations [L][C] is a plain 3-tap convolution over the SAME memory viewed
// as [L/s][s*C]:  out[t] = sum_k W[k] x[t*s + k - pad];  with k - pad = q*s + r (0 <= r < s) the sample is row t+q,
// channel block r of the view, q in {-1, 0, 1} -- so conv_gemm needs no strided mode, only re-packed weights
// W'[q+1][n][r*C + c] = W[n][c][q*s + r + pad] (zero where that k falls outside [0, 2s)).
#include <cmath>

#include "dac_enc_engine.h"
#include "ptx.cuh"

namespace ls {
namespace {

// first convolution (1 -> C0, k = 7, pad 3) + LeakyReLU(0.1): x fp32 [B][S][C0] and snake(x) for the first unit, in the
// handle's 16-bit operand format (fp16 = 1: IEEE half, else bf16).
// lengths (nullable, latent frames): item b is the samples [0, lengths[b] * hop) of its row; later samples are never
// read (they count as the convolution's zero padding) and rows from there to S are written as zeros.
__global__ void __launch_bounds__(128) enc_in_conv_kernel(const float* __restrict__ audio, const int* __restrict__ lengths,
                                                          int hop, const float* __restrict__ w,
                                                          const float* __restrict__ bias, const float* __restrict__ alpha,
                                                          const float* __restrict__ ialpha, float* __restrict__ x,
                                                          __nv_bfloat16* __restrict__ sn, int S, int C0, int fp16) {
  const int t = blockIdx.x * 128 + threadIdx.x;
  const int b = blockIdx.y;
  if (t >= S) return;
  const int n_valid = lengths ? min(max(lengths[b], 0), S / hop) * hop : S;
  float* xo = x + ((size_t)b * S + t) * C0;
  __nv_bfloat16* so = sn + ((size_t)b * S + t) * C0;
  if (t >= n_valid) {
    for (int n = 0; n < C0; n += 4) {
      *reinterpret_cast<float4*>(xo + n) = make_float4(0.f, 0.f, 0.f, 0.f);
      *reinterpret_cast<uint2*>(so + n) = make_uint2(0u, 0u);
    }
    return;
  }
  float a[7];
#pragma unroll
  for (int k = 0; k < 7; ++k) {
    const int tt = t + k - 3;
    a[k] = (tt >= 0 && tt < n_valid) ? audio[(size_t)b * S + tt] : 0.f;
  }
  for (int n = 0; n < C0; n += 4) {
    float4 v;
    float* vv = &v.x;
    uint32_t pk[2];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float acc = bias[n + j];
#pragma unroll
      for (int k = 0; k < 7; ++k) acc = fmaf(a[k], w[(n + j) * 7 + k], acc);
      acc = acc > 0.f ? acc : 0.1f * acc;
      vv[j] = acc;
    }
    *reinterpret_cast<float4*>(xo + n) = v;
    float s4[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) s4[j] = snake_f(vv[j], alpha[n + j], ialpha[n + j]);
    if (fp16) pk[0] = pack_f16x2(s4[0], s4[1]), pk[1] = pack_f16x2(s4[2], s4[3]);
    else pk[0] = pack_bf16x2(s4[0], s4[1]), pk[1] = pack_bf16x2(s4[2], s4[3]);
    *reinterpret_cast<uint2*>(so + n) = make_uint2(pk[0], pk[1]);
  }
}

// y fp32 [B][L][latent] (conv3 + LeakyReLU(0.1) done) -> leaky_relu(0.01) -> en_conv_post (1x1, + LeakyReLU(0.1)) ->
// split, clamp, reparameterise; outputs NCT [B][latent][L], zero at frames t >= lengths[b] (lengths nullable)
__global__ void enc_post_kernel(const float* __restrict__ y, const int* __restrict__ lengths, const float* __restrict__ w,
                                const float* __restrict__ bias, const float* __restrict__ noise, float* __restrict__ z,
                                float* __restrict__ m, float* __restrict__ logs, int L, int latent) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;  // latent channel
  const int t = blockIdx.y, b = blockIdx.z;
  if (c >= latent) return;
  if (lengths && t >= lengths[b]) {
    const size_t o = ((size_t)b * latent + c) * L + t;
    m[o] = 0.f, logs[o] = 0.f, z[o] = 0.f;
    return;
  }
  const float* yr = y + ((size_t)b * L + t) * latent;
  float am = bias[c], al = bias[latent + c];
  for (int k = 0; k < latent; ++k) {
    float v = yr[k];
    v = v > 0.f ? v : 0.01f * v;
    am = fmaf(v, w[(size_t)c * latent + k], am);
    al = fmaf(v, w[(size_t)(latent + c) * latent + k], al);
  }
  am = am > 0.f ? am : 0.1f * am;
  al = al > 0.f ? al : 0.1f * al;
  al = fminf(fmaxf(al, -14.0f), 14.0f);
  const size_t o = ((size_t)b * latent + c) * L + t;
  m[o] = am, logs[o] = al;
  z[o] = noise ? am + noise[o] * expf(al) : am;
}

// stride-s WNConv1d weight_v [N][C][2s] -> 3-tap polyphase 16-bit [3][N][s*C] (see the header comment)
PackedLinear pack_wn_down(Arena& a, const Weights& w, const std::string& p, int stride, bool fp16) {
  const ls_tensor& v = w.get(p + ".weight_v");
  const ls_tensor& g = w.get(p + ".weight_g");
  const ls_tensor& b = w.get(p + ".bias");
  require(v.ndim == 3 && v.shape[2] == 2 * stride && g.shape[0] == v.shape[0], "unexpected downsampling conv at " + p,
          LS_ERR_WEIGHTS);
  const int N = (int)v.shape[0], C = (int)v.shape[1], k2 = 2 * stride, pad = (stride + 1) / 2;
  PackedLinear pl;
  pl.N = N, pl.K = stride * C, pl.taps = 3, pl.block_n = pick_block_n(N);
  pl.w_off = a.reserve((size_t)3 * N * pl.K * 2);
  __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(a.host(pl.w_off));
  for (size_t i = 0; i < (size_t)3 * N * pl.K; ++i) dst[i] = __float2bfloat16(0.f);  // 0 has the same bits in fp16
  const size_t per = (size_t)C * k2;
  for (int n = 0; n < N; ++n) {
    double ss = 0;
    for (size_t i = 0; i < per; ++i) ss += (double)v.data[n * per + i] * v.data[n * per + i];
    const float scale = g.data[n] / (float)std::sqrt(ss);
    for (int q = -1; q <= 1; ++q)
      for (int r = 0; r < stride; ++r) {
        const int k = q * stride + r + pad;
        if (k < 0 || k >= k2) continue;
        for (int c = 0; c < C; ++c)
          dst[((size_t)(q + 1) * N + n) * pl.K + (size_t)r * C + c] = dac_w16(v.data[(n * (size_t)C + c) * k2 + k] * scale, fp16, p);
      }
  }
  pl.bias_off = a.put_f32(b.data, N);
  pl.has_bias = true;
  return pl;
}

}  // namespace

struct DacEncEngine::Plan {
  struct {
    CUtensorMap d[3];   // sA viewed for conv7 with dilation 1 / 3 / 9
    CUtensorMap b;      // sB for conv1
    CUtensorMap down;   // sA viewed [L/s][s*C] for the downsampling conv
  } st[5];
  CUtensorMap fin;      // sA of the last stage for conv3
};

DacEncEngine::~DacEncEngine() {
  if (ws_base_) cudaFree(ws_base_);
}

DacEncEngine::DacEncEngine(const Weights& w, int device, bool fp16) : device_(device), fp16_(fp16 ? 1 : 0) {
  LS_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  LS_CUDA(cudaGetDeviceProperties(&prop, device));
  require(prop.major == 10, "this library only runs on sm_100 (B200) devices", LS_ERR_UNSUPPORTED);
  num_sms_ = prop.multiProcessorCount;
  auto snake = [&](const std::string& name, int c, size_t* a_off, size_t* ia_off) {
    const ls_tensor& al = w.get(name, {1, c, 1});
    std::vector<float> ia(c);
    for (int i = 0; i < c; ++i) ia[i] = 1.0f / (al.data[i] + 1e-9f);
    *a_off = arena_.put_f32(al.data, c);
    *ia_off = arena_.put_f32(ia.data(), c);
  };
  auto fold_f32 = [&](const std::string& p, size_t* w_off, size_t* b_off) {  // small convs kept in fp32 [N][C*k]
    const ls_tensor& v = w.get(p + ".weight_v");
    const ls_tensor& g = w.get(p + ".weight_g");
    const ls_tensor& b = w.get(p + ".bias");
    const size_t N = (size_t)v.shape[0], per = (size_t)v.shape[1] * v.shape[2];
    std::vector<float> f(N * per);
    for (size_t n = 0; n < N; ++n) {
      double ss = 0;
      for (size_t i = 0; i < per; ++i) ss += (double)v.data[n * per + i] * v.data[n * per + i];
      const float scale = g.data[n] / (float)std::sqrt(ss);
      for (size_t i = 0; i < per; ++i) f[n * per + i] = v.data[n * per + i] * scale;
    }
    *w_off = arena_.put_f32(f.data(), f.size());
    *b_off = arena_.put_f32(b.data, N);
  };
  const ls_tensor& v0 = w.get("encoder.block.0.0.weight_v");
  require(v0.ndim == 3 && v0.shape[1] == 1 && v0.shape[2] == 7 && v0.shape[0] % 16 == 0, "unexpected encoder stem (mono, k = 7)",
          LS_ERR_UNSUPPORTED);
  dim0_ = (int)v0.shape[0];
  fold_f32("encoder.block.0.0", &in_w_, &in_b_);
  int c = dim0_;
  hop_ = 1;
  for (int i = 1; w.has("encoder.block." + std::to_string(i) + ".block.4.0.weight_v"); ++i) {
    const std::string p = "encoder.block." + std::to_string(i) + ".block";
    StageW st;
    st.stride = (int)w.get(p + ".4.0.weight_v").shape[2] / 2;
    st.cin = c;
    for (int j = 0; j < 3; ++j) {
      const std::string q = p + "." + std::to_string(j) + ".block";
      snake(q + ".0.alpha", c, &st.unit[j].a0, &st.unit[j].ia0);
      st.unit[j].conv7 = pack_wn_conv(arena_, w, q + ".1.0", fp16);
      snake(q + ".2.alpha", c, &st.unit[j].a2, &st.unit[j].ia2);
      st.unit[j].conv1 = pack_wn_conv(arena_, w, q + ".3.0", fp16);
      require(st.unit[j].conv7.taps == 7 && st.unit[j].conv1.taps == 1, "unexpected ResidualUnit at " + q, LS_ERR_UNSUPPORTED);
    }
    snake(p + ".3.alpha", c, &st.a_dn, &st.ia_dn);
    st.down = pack_wn_down(arena_, w, p + ".4.0", st.stride, fp16);
    hop_ *= st.stride;
    c *= 2;
    stages_.push_back(st);
  }
  const int n = (int)stages_.size();
  require(n >= 1 && n <= 5, "DAC encoder must have 1..5 downsampling stages", LS_ERR_UNSUPPORTED);
  snake("encoder.block." + std::to_string(n + 1) + ".alpha", c, &final_alpha_, &final_ialpha_);
  final_ = pack_wn_conv(arena_, w, "encoder.block." + std::to_string(n + 2) + ".0", fp16);
  latent_ = final_.N;
  require(final_.taps == 3 && latent_ % 16 == 0, "unexpected encoder head", LS_ERR_UNSUPPORTED);
  const ls_tensor& vp = w.get("en_conv_post.0.weight_v");
  require(vp.shape[0] == 2 * latent_ && vp.shape[1] == latent_ && vp.shape[2] == 1, "unexpected en_conv_post", LS_ERR_WEIGHTS);
  fold_f32("en_conv_post.0", &post_w_, &post_b_);
  arena_.upload();
  finalize_linear(arena_, final_);
  for (auto& st : stages_) {
    finalize_linear(arena_, st.down);
    for (auto& u : st.unit) finalize_linear(arena_, u.conv7), finalize_linear(arena_, u.conv1);
  }
}

void DacEncEngine::ensure_workspace(int B, int S, cudaStream_t s) {
  const long long samples = (long long)B * S;
  if (samples <= cap_samples_) return;
  ws_release(ws_base_, s);
  plans_.clear();
  cap_samples_ = samples;
  // widest activation in elements per input sample: stage i holds (S / prod strides) x (dim0 * 2^i)
  double per = dim0_, rate = 1.0, chan = dim0_;
  for (auto& st : stages_) rate /= st.stride, chan *= 2, per = std::max(per, rate * chan);
  const size_t elems = (size_t)std::ceil(per * (double)samples) + 4096;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    size_t o = off;
    off = (off + bytes + 1023) & ~size_t(1023);
    return o;
  };
  o_x_ = take(elems * 4);
  o_sA_ = take(elems * 2);
  o_sB_ = take(elems * 2);
  o_y_ = take((size_t)(samples / hop_ + 1) * latent_ * 4);
  ws_alloc(ws_base_, off, s);
}

const DacEncEngine::Plan& DacEncEngine::plan_for(int B, int S) {
  auto key = std::make_pair(B, S);
  auto it = plans_.find(key);
  if (it != plans_.end()) return *it->second;
  auto pl = std::make_unique<Plan>();
  const bool halo = conv_halo_enabled();
  auto mk = [&](CUtensorMap* m, size_t off, int C, long long rows, int taps, int dil) {
    require(make_act_map(m, ws_base_ + off, C, (int)rows, B, C, rows * C, halo ? conv_halo_box_rows(taps, dil) : 128),
            "cuTensorMapEncodeTiled failed for an activation buffer", LS_ERR_CUDA);
  };
  static const int dils[3] = {1, 3, 9};
  long long rows = S;
  int c = dim0_;
  for (size_t i = 0; i < stages_.size(); ++i) {
    for (int j = 0; j < 3; ++j) mk(&pl->st[i].d[j], o_sA_, c, rows, 7, dils[j]);
    mk(&pl->st[i].b, o_sB_, c, rows, 1, 1);
    const int s = stages_[i].stride;
    mk(&pl->st[i].down, o_sA_, s * c, rows / s, 3, 1);
    rows /= s, c *= 2;
  }
  mk(&pl->fin, o_sA_, c, rows, 3, 1);
  const Plan& ref = *pl;
  plans_[key] = std::move(pl);
  return ref;
}

void DacEncEngine::encode(const float* audio, const int* lengths, const float* noise, float* z, float* m, float* logs,
                          int B, int S, cudaStream_t s) {
  require(B > 0 && S > 0 && S % hop_ == 0, "audio length must be a positive multiple of the hop (pad first, model.py:455-462)");
  LS_CUDA(cudaSetDevice(device_));
  ensure_workspace(B, S, s);
  const Plan& pl = plan_for(B, S);
  auto f32 = [&](size_t off) { return arena_.ptr<float>(off); };
  const bool halo = conv_halo_enabled();
  float* x = ws<float>(o_x_);
  void* sA = ws<void>(o_sA_);
  void* sB = ws<void>(o_sB_);

  // Mixed lengths (lengths != nullptr, latent frames; clip b is the samples [0, n_b = lengths[b] * hop)): each clip is
  // encoded as if alone at its own length.  A layer at rate r (rows per latent frame: hop / prod(strides[:i]) inside
  // stage i, hop / prod(strides[:i+1]) for its downsampling conv, 1 for conv3) has L_b * r valid rows; every launch
  // writes zeros to the rows of a computed tile past them and skips (leaves stale) the tiles starting at or past
  // L_b * r + 64.  So the rows [L_b * r, L_b * r + 64) of every activation are zero (enc_in_conv_kernel zeroes the
  // whole tail of stage 0), and no valid output reaches further: the conv7 at dilation 9 reads 27 rows past its own,
  // the downsampling conv's pad of 1 view row is the input rows [L_b * r, L_b * r + s) with s < 64 -- the view stays
  // aligned because n_b is a multiple of the hop -- and conv3 reads 1 row past.  Those zeros are exactly the zero
  // padding the clip alone would see, so a valid output reads the same values either way; rows that are computed
  // from stale data are past the valid length and written as zeros.
  auto conv = [&](const CUtensorMap& a, const PackedLinear& w, long long rows, int rate, int dil, int pad, ConvGemmParams p) {
    p.B = B, p.M = (int)rows, p.N = w.N, p.block_n = w.block_n;
    p.taps = w.taps, p.dil = dil, p.pad = pad;
    p.kb_per_tap = (w.K + 63) / 64, p.kb_split = p.kb_per_tap;
    if (lengths) p.lengths = lengths, p.m_len_mul = rate, p.m_len_add = 0, p.skip_halo = 64;
    else p.lengths = nullptr, p.m_len_mul = 1, p.m_len_add = 0, p.skip_halo = 0;
    p.bias = w.bias, p.chan_mod = w.N, p.n_store = w.N;
    p.out_ld = w.N, p.out_shift = 0, p.out_bstride = rows * w.N, p.out_alloc = rows * w.N;
    p.out_valid_mul = lengths ? (long long)rate * w.N : w.N;
    p.k_true = w.K, p.tag = 1, p.halo_mode = halo ? conv_halo_mode() : 0, p.fp16 = fp16_;
    LS_CUDA(launch_conv_gemm(a, a, w.map, p, num_sms_, s));
  };

  count_launch();
  enc_in_conv_kernel<<<dim3((S + 127) / 128, B), 128, 0, s>>>(audio, lengths, hop_, f32(in_w_), f32(in_b_),
                                                            f32(stages_[0].unit[0].a0), f32(stages_[0].unit[0].ia0), x,
                                                            ws<__nv_bfloat16>(o_sA_), S, dim0_, fp16_);
  LS_CUDA(cudaGetLastError());
  long long rows = S;
  int rate = hop_;
  static const int dils[3] = {1, 3, 9};
  for (size_t i = 0; i < stages_.size(); ++i) {
    const StageW& st = stages_[i];
    for (int j = 0; j < 3; ++j) {
      const UnitW& u = st.unit[j];
      {  // Snake (already applied) -> conv7 dilated -> LeakyReLU -> Snake
        ConvGemmParams p{};
        p.act = ACT_LRELU, p.out1 = sB, p.out1_mode = OUT1_SNAKE, p.p1_a = f32(u.a2), p.p1_b = f32(u.ia2);
        conv(pl.st[i].d[j], u.conv7, rows, rate, dils[j], 3 * dils[j], p);
      }
      {  // conv1 -> LeakyReLU -> + x; secondary output = Snake of whatever consumes x next
        ConvGemmParams p{};
        p.act = ACT_LRELU, p.addend = x, p.addend_dtype = OUT_F32;
        const bool last_unit = j == 2;
        if (!last_unit) p.out0 = x, p.out0_dtype = OUT_F32;
        p.out1 = sA, p.out1_mode = OUT1_SNAKE;
        p.p1_a = f32(last_unit ? st.a_dn : st.unit[j + 1].a0), p.p1_b = f32(last_unit ? st.ia_dn : st.unit[j + 1].ia0);
        conv(pl.st[i].b, u.conv1, rows, rate, 1, 0, p);
      }
    }
    {  // downsampling conv on the [rows/s][s*C] view: 3 taps, pad 1 -> LeakyReLU -> x of the next stage + its Snake
      rows /= st.stride, rate /= st.stride;
      const bool last = i + 1 == stages_.size();
      ConvGemmParams p{};
      p.act = ACT_LRELU;
      if (!last) p.out0 = x, p.out0_dtype = OUT_F32;
      p.out1 = sB, p.out1_mode = OUT1_SNAKE;  // (sA is this launch's input: the Snake output goes to sB, then swaps)
      p.p1_a = f32(last ? final_alpha_ : stages_[i + 1].unit[0].a0), p.p1_b = f32(last ? final_ialpha_ : stages_[i + 1].unit[0].ia0);
      conv(pl.st[i].down, st.down, rows, rate, 1, 1, p);
      // the next stage reads its Snake input from sA: copy (the tensors shrink by >= 2x per stage; this is a small
      // fraction of the stage's traffic)
      LS_CUDA(cudaMemcpyAsync(sA, sB, (size_t)B * rows * st.down.N * 2, cudaMemcpyDeviceToDevice, s));
    }
  }
  {  // final Snake (applied) -> conv3 -> LeakyReLU(0.1): fp32 [B][L][latent]
    ConvGemmParams p{};
    p.act = ACT_LRELU, p.out0 = ws<float>(o_y_), p.out0_dtype = OUT_F32;
    conv(pl.fin, final_, rows, rate, 1, 1, p);
  }
  count_launch();
  enc_post_kernel<<<dim3((latent_ + 127) / 128, (unsigned)rows, B), 128, 0, s>>>(ws<float>(o_y_), lengths, f32(post_w_),
                                                                             f32(post_b_), noise, z, m, logs, (int)rows, latent_);
  LS_CUDA(cudaGetLastError());
}

}  // namespace ls
