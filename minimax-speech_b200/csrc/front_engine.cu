// Token -> mu front half on the tensor cores: see front_engine.h.  Reference lines next to each step.
#include <cmath>

#include "front_engine.h"
#include "ptx.cuh"

namespace ls {
namespace {

constexpr int kD = 512;  // encoder width (config.yaml:73-88); the small kernels below are written for it

// e[r][:] = table[clamp(tok[r], 0, vocab-1)][:]   (flow.py:476: input_embedding(torch.clamp(token, min=0)))
// rows past the utterance's token count are zero (flow.py:475-476: input_embedding(token) * mask)
__global__ void __launch_bounds__(64) front_gather_kernel(const long long* __restrict__ tok, const __nv_bfloat16* __restrict__ table,
                                                          __nv_bfloat16* __restrict__ e, int vocab, int T_all,
                                                          const int* __restrict__ lens) {
  const size_t r = blockIdx.x;
  long long id = tok[r];
  id = id < 0 ? 0 : (id >= vocab ? vocab - 1 : id);
  uint4 v = reinterpret_cast<const uint4*>(table + (size_t)id * kD)[threadIdx.x];
  if (lens && (int)(r % T_all) >= lens[r / T_all]) v = make_uint4(0u, 0u, 0u, 0u);
  reinterpret_cast<uint4*>(e + r * kD)[threadIdx.x] = v;
}
// lens0[b] = min(token_len[b], T) (keys at 25 Hz), lens1[b] = 2 * lens0[b] (keys and valid frames at 50 Hz).
// Session mode (n_ctx != nullptr): lens0[b] = token_len[b] - n_ctx[b], the row's own output tokens, or 0 for a row
// with invalid entries (its mu comes out all zero).
__global__ void front_lens_kernel(const int* __restrict__ token_len, const int* __restrict__ n_ctx, int* __restrict__ lens0,
                                  int* __restrict__ lens1, int B, int T_all, int T) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  int l = max(0, min(token_len[b], T));
  if (n_ctx) {
    const int n = token_len[b], c = n_ctx[b];
    l = ((c == 0 || c == 3) && n - c >= 1 && n <= T_all && n - c <= T) ? n - c : 0;
  }
  lens0[b] = l, lens1[b] = 2 * l;
}

// LayerNorm over the 512 channels of a row (eps 1e-5), times `scale` (the rel-pos encoding's sqrt(d) input scale,
// embedding.py:268): fp32 (optional) and bf16 outputs.  One warp per row, the row held in registers.  lens (nullable):
// rows r with r % T >= lens[r / T] are written as zeros (right padding of a batch of sessions: what F.pad gives the
// pre-lookahead convolution of a call alone).
__global__ void __launch_bounds__(128) front_ln_rows_kernel(const float* __restrict__ x, const float* __restrict__ g,
                                                            const float* __restrict__ be, float scale, float* __restrict__ yf,
                                                            __nv_bfloat16* __restrict__ yb, long long R,
                                                            const int* __restrict__ lens, int T) {
  const long long r = (long long)blockIdx.x * 4 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (r >= R) return;
  if (lens && (int)(r % T) >= lens[r / T]) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if (yf) reinterpret_cast<float4*>(yf + r * kD)[i * 32 + lane] = make_float4(0.f, 0.f, 0.f, 0.f);
      reinterpret_cast<uint2*>(yb + r * kD)[i * 32 + lane] = make_uint2(0u, 0u);
    }
    return;
  }
  const float4* xr = reinterpret_cast<const float4*>(x + r * kD);
  float4 v[4];
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    v[i] = xr[i * 32 + lane];
    sum += v[i].x + v[i].y + v[i].z + v[i].w;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  const float mean = sum * (1.0f / kD);
  float sq = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float a = v[i].x - mean, b = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
    sq += a * a + b * b + c * c + d * d;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
  const float rstd = rsqrtf(sq * (1.0f / kD) + 1e-5f);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float4 gm = reinterpret_cast<const float4*>(g)[i * 32 + lane];
    const float4 bt = reinterpret_cast<const float4*>(be)[i * 32 + lane];
    float4 o;
    o.x = ((v[i].x - mean) * rstd * gm.x + bt.x) * scale;
    o.y = ((v[i].y - mean) * rstd * gm.y + bt.y) * scale;
    o.z = ((v[i].z - mean) * rstd * gm.z + bt.z) * scale;
    o.w = ((v[i].w - mean) * rstd * gm.w + bt.w) * scale;
    if (yf) reinterpret_cast<float4*>(yf + r * kD)[i * 32 + lane] = o;
    reinterpret_cast<uint2*>(yb + r * kD)[i * 32 + lane] = make_uint2(pack_bf16x2(o.x, o.y), pack_bf16x2(o.z, o.w));
  }
}

// q + pos_bias_u (in place, the Q columns of the packed QKV rows) and q + pos_bias_v (attention.py:283-291)
__global__ void front_q_prep_kernel(__nv_bfloat16* __restrict__ qkv, const float* __restrict__ bu, const float* __restrict__ bv,
                                    __nv_bfloat16* __restrict__ qv, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const size_t r = i / kD;
  const int c = (int)(i % kD);
  const float q = __bfloat162float(qkv[r * 3 * kD + c]);
  qkv[r * 3 * kD + c] = __float2bfloat16(q + bu[c]);
  qv[i] = __float2bfloat16(q + bv[c]);
}

// EspnetRelPositionalEncoding (transformer/embedding.py:224-300): pe[n][:] for relative position T-1-n, n in [0, 2T-1)
__global__ void front_rel_pos_kernel(__nv_bfloat16* __restrict__ pe, int T) {
  const int c2 = blockIdx.x * blockDim.x + threadIdx.x;
  const int n = blockIdx.y;
  if (c2 >= kD / 2) return;
  const float pos = (float)(T - 1 - n);
  const float div = expf((float)(2 * c2) * -(logf(10000.0f) / (float)kD));
  pe[(size_t)n * kD + 2 * c2] = __float2bfloat16(sinf(pos * div));
  pe[(size_t)n * kD + 2 * c2 + 1] = __float2bfloat16(cosf(pos * div));
}

// projected positions [P][512] -> head-major [H][Ppad][64] (rows >= P stay zero): the "weights" of the per-head bd GEMMs
__global__ void front_split_heads_kernel(const __nv_bfloat16* __restrict__ pp, __nv_bfloat16* __restrict__ pph, int P, int Ppad) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)P * kD) return;
  const size_t n = i / kD;
  const int c = (int)(i % kD);
  pph[((size_t)(c >> 6) * Ppad + n) * 64 + (c & 63)] = pp[i];
}

// nearest-neighbour x2 along time (transformer/upsample_encoder.py:60): fp32 [B][T][512] -> bf16 [B][2T][512]
__global__ void front_upsample2_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ y, int T, size_t n_out) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_out) return;
  const int c = (int)(i % kD);
  const size_t row = i / kD;  // b*2T + t2
  const size_t b = row / (2 * (size_t)T);
  const int t2 = (int)(row % (2 * (size_t)T));
  y[i] = __float2bfloat16(x[(b * T + t2 / 2) * kD + c]);
}

// spks[b][:] = W (e / max(|e|, 1e-12)) + bias   (flow.py:463, 469)
__global__ void __launch_bounds__(128) front_spk_kernel(const float* __restrict__ e, const float* __restrict__ w,
                                                        const float* __restrict__ bias, float* __restrict__ spks, int K, int N) {
  const int b = blockIdx.x;
  __shared__ float red[4];
  __shared__ float inv;
  float ss = 0.f;
  for (int k = threadIdx.x; k < K; k += 128) ss = fmaf(e[(size_t)b * K + k], e[(size_t)b * K + k], ss);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ss;
  __syncthreads();
  if (threadIdx.x == 0) inv = 1.0f / fmaxf(sqrtf(red[0] + red[1] + red[2] + red[3]), 1e-12f);
  __syncthreads();
  for (int n = threadIdx.x; n < N; n += 128) {
    float acc = 0.f;
    for (int k = 0; k < K; ++k) acc = fmaf(e[(size_t)b * K + k], w[(size_t)n * K + k], acc);
    spks[(size_t)b * N + n] = acc * inv + bias[n];
  }
}

inline unsigned blocks(size_t n) { return (unsigned)((n + 255) / 256); }

// weight [N][K] (linear) or [N][K][taps] (conv1d) -> bf16 [taps][N][K]
PackedLinear pack_dense(Arena& a, const ls_tensor& w, const ls_tensor* bias) {
  PackedLinear pl;
  pl.N = (int)w.shape[0];
  pl.K = (int)w.shape[1];
  pl.taps = w.ndim == 3 ? (int)w.shape[2] : 1;
  pl.block_n = pick_block_n(pl.N);
  pl.w_off = a.reserve((size_t)pl.taps * pl.N * pl.K * 2);
  __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(a.host(pl.w_off));
  for (int t = 0; t < pl.taps; ++t)
    for (int n = 0; n < pl.N; ++n)
      for (int k = 0; k < pl.K; ++k)
        dst[((size_t)t * pl.N + n) * pl.K + k] = __float2bfloat16(w.data[((size_t)n * pl.K + k) * pl.taps + t]);
  if (bias) {
    require(bias->shape[0] == pl.N, std::string("bias shape mismatch for ") + w.name, LS_ERR_WEIGHTS);
    pl.bias_off = a.put_f32(bias->data, pl.N);
    pl.has_bias = true;
  }
  return pl;
}

void finalize_dense(const Arena& a, PackedLinear& pl) {
  require(make_weight_map(&pl.map, a.ptr<uint8_t>(pl.w_off), pl.K, pl.taps * pl.N, pl.block_n),
          "cuTensorMapEncodeTiled failed for a weight matrix", LS_ERR_CUDA);
  pl.bias = pl.has_bias ? a.ptr<float>(pl.bias_off) : nullptr;
}

inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

}  // namespace

struct FrontEngine::Plan {
  struct Level {          // one per frame rate: T rows per utterance
    int T = 0, P = 0, Ppad = 0, bd_block_n = 0;
    CUtensorMap nb, att, h, qkv_attn, pe;
    CUtensorMap qv[8], pph[8];
  } lv[2];
  CUtensorMap tok, pre1, pre2, up;
};

FrontEngine::~FrontEngine() {
  if (ws_base_) cudaFree(ws_base_);
}

FrontEngine::FrontEngine(const Weights& w, int device) : device_(device) {
  LS_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  LS_CUDA(cudaGetDeviceProperties(&prop, device));
  require(prop.major == 10, "this library only runs on sm_100 (B200) devices", LS_ERR_UNSUPPORTED);
  num_sms_ = prop.multiProcessorCount;
  const ls_tensor& emb = w.get("input_embedding.weight");
  vocab_ = (int)emb.shape[0];
  require(emb.ndim == 2 && emb.shape[1] == kD, "token encoder: expected width 512 (config.yaml:73-88)", LS_ERR_UNSUPPORTED);
  emb_table_ = arena_.reserve((size_t)vocab_ * kD * 2);
  {
    __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(arena_.host(emb_table_));
    for (size_t i = 0; i < (size_t)vocab_ * kD; ++i) dst[i] = __float2bfloat16(emb.data[i]);
  }
  auto vec = [&](const std::string& name, long long n) { return arena_.put_f32(w.get(name, {n}).data, (size_t)n); };
  const ls_tensor& sw = w.get("spk_embed_affine_layer.weight");
  out_ = (int)sw.shape[0], spk_ = (int)sw.shape[1];
  spk_w_ = arena_.put_f32(sw.data, (size_t)out_ * spk_);
  spk_b_ = vec("spk_embed_affine_layer.bias", out_);
  auto embed = [&](const std::string& p) {
    EmbedW e;
    e.lin = pack_dense(arena_, w.get(p + ".out.0.weight", {kD, kD}), &w.get(p + ".out.0.bias"));
    e.g = vec(p + ".out.1.weight", kD), e.b = vec(p + ".out.1.bias", kD);
    return e;
  };
  embed_ = embed("encoder.embed");
  up_embed_ = embed("encoder.up_embed");
  pre1_ = pack_dense(arena_, w.get("encoder.pre_lookahead_layer.conv1.weight", {kD, kD, 4}), &w.get("encoder.pre_lookahead_layer.conv1.bias"));
  pre2_ = pack_dense(arena_, w.get("encoder.pre_lookahead_layer.conv2.weight", {kD, kD, 3}), &w.get("encoder.pre_lookahead_layer.conv2.bias"));
  up_conv_ = pack_dense(arena_, w.get("encoder.up_layer.conv.weight", {kD, kD, 5}), &w.get("encoder.up_layer.conv.bias"));
  proj_ = pack_dense(arena_, w.get("encoder_proj.weight", {out_, kD}), &w.get("encoder_proj.bias"));
  require(out_ % 16 == 0 && out_ <= 256, "encoder_proj width must be a multiple of 16", LS_ERR_UNSUPPORTED);
  g_after_ = vec("encoder.after_norm.weight", kD), b_after_ = vec("encoder.after_norm.bias", kD);
  heads_ = (int)w.get("encoder.encoders.0.self_attn.pos_bias_u").shape[0];
  require(heads_ == 8 && kD == heads_ * 64, "token encoder: expected 8 heads of 64 channels", LS_ERR_UNSUPPORTED);
  auto layer = [&](const std::string& p) {
    LayerW L;
    const std::string a = p + ".self_attn";
    {  // Q | K | V as one [1536][512] projection
      const ls_tensor& wq = w.get(a + ".linear_q.weight", {kD, kD});
      const ls_tensor& wk = w.get(a + ".linear_k.weight", {kD, kD});
      const ls_tensor& wv = w.get(a + ".linear_v.weight", {kD, kD});
      std::vector<float> cat((size_t)3 * kD * kD), bias((size_t)3 * kD);
      std::memcpy(cat.data(), wq.data, (size_t)kD * kD * 4);
      std::memcpy(cat.data() + (size_t)kD * kD, wk.data, (size_t)kD * kD * 4);
      std::memcpy(cat.data() + (size_t)2 * kD * kD, wv.data, (size_t)kD * kD * 4);
      std::memcpy(bias.data(), w.get(a + ".linear_q.bias", {kD}).data, kD * 4);
      std::memcpy(bias.data() + kD, w.get(a + ".linear_k.bias", {kD}).data, kD * 4);
      std::memcpy(bias.data() + 2 * kD, w.get(a + ".linear_v.bias", {kD}).data, kD * 4);
      ls_tensor tw{}, tb{};
      tw.name = wq.name, tw.data = cat.data(), tw.ndim = 2, tw.shape[0] = 3 * kD, tw.shape[1] = kD;
      tb.name = wq.name, tb.data = bias.data(), tb.ndim = 1, tb.shape[0] = 3 * kD;
      L.qkv = pack_dense(arena_, tw, &tb);
    }
    L.pos = pack_dense(arena_, w.get(a + ".linear_pos.weight", {kD, kD}), nullptr);
    L.out = pack_dense(arena_, w.get(a + ".linear_out.weight", {kD, kD}), &w.get(a + ".linear_out.bias"));
    const ls_tensor& w1 = w.get(p + ".feed_forward.w_1.weight");
    ff_ = (int)w1.shape[0];
    require(w1.ndim == 2 && w1.shape[1] == kD && ff_ % 64 == 0, "unexpected feed-forward shape at " + p, LS_ERR_WEIGHTS);
    L.ff1 = pack_dense(arena_, w1, &w.get(p + ".feed_forward.w_1.bias"));
    L.ff2 = pack_dense(arena_, w.get(p + ".feed_forward.w_2.weight", {kD, ff_}), &w.get(p + ".feed_forward.w_2.bias"));
    L.g_mha = vec(p + ".norm_mha.weight", kD), L.b_mha = vec(p + ".norm_mha.bias", kD);
    L.g_ff = vec(p + ".norm_ff.weight", kD), L.b_ff = vec(p + ".norm_ff.bias", kD);
    L.bias_u = arena_.put_f32(w.get(a + ".pos_bias_u", {heads_, 64}).data, kD);
    L.bias_v = arena_.put_f32(w.get(a + ".pos_bias_v", {heads_, 64}).data, kD);
    return L;
  };
  for (int i = 0; w.has("encoder.encoders." + std::to_string(i) + ".norm_mha.weight"); ++i)
    layers_.push_back(layer("encoder.encoders." + std::to_string(i)));
  for (int i = 0; w.has("encoder.up_encoders." + std::to_string(i) + ".norm_mha.weight"); ++i)
    up_layers_.push_back(layer("encoder.up_encoders." + std::to_string(i)));
  arena_.upload();
  for (PackedLinear* pl : {&embed_.lin, &up_embed_.lin, &pre1_, &pre2_, &up_conv_, &proj_}) finalize_dense(arena_, *pl);
  for (auto* v : {&layers_, &up_layers_})
    for (LayerW& L : *v)
      for (PackedLinear* pl : {&L.qkv, &L.pos, &L.out, &L.ff1, &L.ff2}) finalize_dense(arena_, *pl);
}

void FrontEngine::ensure_workspace(int B, int T_all, int T, cudaStream_t s) {
  const int T2 = 2 * T;
  const long long rows = (long long)B * std::max(T2, T_all);
  const int Ppad = round_up(2 * T2 - 1, 128);
  const long long bd = (long long)B * heads_ * T2 * Ppad;
  if (rows <= cap_rows_ && bd <= cap_bd_) return;
  ws_release(ws_base_, s);
  plans_.clear();
  cap_rows_ = std::max(rows, cap_rows_), cap_bd_ = std::max(bd, cap_bd_);
  size_t off = 0;
  auto take = [&](size_t bytes) {
    size_t o = off;
    off = (off + bytes + 1023) & ~size_t(1023);
    return o;
  };
  const size_t R = (size_t)cap_rows_ + 256;  // slack rows: tiles overhang the last utterance
  // positions: P <= 2*max(T2) - 1; bound it by the bd capacity of a single-utterance call (B = 1 gives the longest T)
  const size_t Pcap = (size_t)round_up((int)std::min<long long>(4 * cap_rows_ + 128, 1 << 20), 128);
  o_x_ = take(R * kD * 4);
  o_y_ = take(R * kD * 4);
  o_nb_ = take(R * kD * 2);
  o_qkv_ = take(R * 3 * kD * 2);
  o_qv_ = take(R * kD * 2);
  o_att_ = take(R * kD * 2);
  o_h_ = take(R * (size_t)std::max(ff_, kD) * 2);
  o_pe_ = take(Pcap * kD * 2);
  o_pp_ = take(Pcap * kD * 2);
  o_pph_ = take(Pcap * kD * 2);
  o_bd_ = take(((size_t)cap_bd_ + 4096) * 4);
  o_spk_ = take(4096);  // int lens0[512] | lens1[512]
  ws_alloc(ws_base_, off, s);
}

const FrontEngine::Plan& FrontEngine::plan_for(int B, int T_all, int T) {
  std::vector<int> key{B, T_all, T};
  auto it = plans_.find(key);
  if (it != plans_.end()) return *it->second;
  auto pl = std::make_unique<Plan>();
  const bool halo = conv_halo_enabled();
  auto mk = [&](CUtensorMap* m, size_t off, int C, int rows, int nb, int taps) {
    require(make_act_map(m, ws_base_ + off, C, rows, nb, C, (long long)rows * C, halo ? conv_halo_box_rows(taps, 1) : 128),
            "cuTensorMapEncodeTiled failed for an activation buffer", LS_ERR_CUDA);
  };
  mk(&pl->tok, o_h_, kD, T_all, B, 1);
  mk(&pl->pre1, o_nb_, kD, T_all, B, 4);
  mk(&pl->pre2, o_att_, kD, T, B, 3);
  mk(&pl->up, o_nb_, kD, 2 * T, B, 5);
  for (int l = 0; l < 2; ++l) {
    Plan::Level& lv = pl->lv[l];
    lv.T = l == 0 ? T : 2 * T;
    lv.P = 2 * lv.T - 1;
    lv.Ppad = round_up(lv.P, 128);
    lv.bd_block_n = pick_block_n(lv.Ppad);
    mk(&lv.nb, o_nb_, kD, lv.T, B, 1);
    mk(&lv.att, o_att_, kD, lv.T, B, 1);
    mk(&lv.h, o_h_, ff_, lv.T, B, 1);
    mk(&lv.pe, o_pe_, kD, lv.P, 1, 1);
    require(make_act_map(&lv.qkv_attn, ws_base_ + o_qkv_, 3 * kD, lv.T, B, 3 * kD, (long long)lv.T * 3 * kD, ATTN_KV),
            "cuTensorMapEncodeTiled failed for the QKV buffer", LS_ERR_CUDA);
    for (int h = 0; h < heads_; ++h) {
      require(make_act_map(&lv.qv[h], ws_base_ + o_qv_ + (size_t)h * 64 * 2, 64, lv.T, B, kD, (long long)lv.T * kD, 128) &&
                  make_weight_map(&lv.pph[h], ws_base_ + o_pph_ + (size_t)h * lv.Ppad * 64 * 2, 64, lv.Ppad, lv.bd_block_n),
              "cuTensorMapEncodeTiled failed for the relative-position operands", LS_ERR_CUDA);
    }
  }
  const Plan& ref = *pl;
  plans_[key] = std::move(pl);
  return ref;
}

void FrontEngine::encode(const long long* tokens, const float* embedding, float* mu, float* spks, int B, int T_all,
                         int n_context, bool streaming, const int* token_len, cudaStream_t s) {
  require(B > 0 && T_all - n_context > 0 && (n_context == 0 || n_context == 3), "B, T must be positive; context is 0 or 3 tokens");
  run(tokens, embedding, mu, spks, B, T_all, T_all - n_context, streaming, token_len, nullptr, s);
}

void FrontEngine::encode_sessions(const long long* tokens, const float* embedding, float* mu, float* spks, int B, int T_all,
                                  int T, const int* token_len, const int* n_context, bool streaming, cudaStream_t s) {
  require(B > 0 && T > 0 && T <= T_all && token_len && n_context, "B, T must be positive, T <= T_all, lengths given");
  run(tokens, embedding, mu, spks, B, T_all, T, streaming, token_len, n_context, s);
}

// T_all token rows per utterance in, T output tokens (2T frames) out; T_all > T: the rows past T are look-ahead context.
// n_context (session mode, with token_len): per-utterance context, see front_lens_kernel.
void FrontEngine::run(const long long* tokens, const float* embedding, float* mu, float* spks, int B, int T_all, int T,
                      bool streaming, const int* token_len, const int* n_context, cudaStream_t s) {
  const int T2 = 2 * T;
  LS_CUDA(cudaSetDevice(device_));
  ensure_workspace(B, T_all, T, s);
  const Plan& pl = plan_for(B, T_all, T);
  auto f32 = [&](size_t off) { return arena_.ptr<float>(off); };
  const bool halo = conv_halo_enabled();
  float* x = ws<float>(o_x_);
  float* y = ws<float>(o_y_);
  __nv_bfloat16* nb = ws<__nv_bfloat16>(o_nb_);
  __nv_bfloat16* qkv = ws<__nv_bfloat16>(o_qkv_);
  __nv_bfloat16* qv = ws<__nv_bfloat16>(o_qv_);
  __nv_bfloat16* att = ws<__nv_bfloat16>(o_att_);
  __nv_bfloat16* hb = ws<__nv_bfloat16>(o_h_);
  __nv_bfloat16* pe = ws<__nv_bfloat16>(o_pe_);
  __nv_bfloat16* pp = ws<__nv_bfloat16>(o_pp_);
  __nv_bfloat16* pph = ws<__nv_bfloat16>(o_pph_);
  float* bd = ws<float>(o_bd_);

  // D[b][t][:] = epilogue(sum_tap A[b][t + tap - pad][:] W[tap]^T): dense [nb][rows][N] outputs
  auto conv = [&](const CUtensorMap& a, const PackedLinear& w, int nbatch, int rows, int pad, ConvGemmParams p) {
    p.B = nbatch, p.M = rows, p.N = w.N, p.block_n = w.block_n;
    p.taps = w.taps, p.dil = 1, p.pad = pad;
    p.kb_per_tap = (w.K + 63) / 64, p.kb_split = p.kb_per_tap;
    p.lengths = nullptr, p.m_len_mul = 1, p.m_len_add = 0, p.skip_halo = 0;
    p.bias = w.bias, p.chan_mod = w.N, p.n_store = w.N;
    p.out_ld = w.N, p.out_shift = 0, p.out_bstride = (long long)rows * w.N, p.out_alloc = (long long)rows * w.N, p.out_valid_mul = w.N;
    p.k_true = w.K, p.tag = 0, p.halo_mode = (halo && w.taps > 1) ? conv_halo_mode() : 0;
    LS_CUDA(launch_conv_gemm(a, a, w.map, p, num_sms_, s));
  };
  auto ln = [&](const float* in, size_t g, size_t b, float scale, float* of, __nv_bfloat16* ob, long long R,
                const int* zero_past = nullptr) {
    count_launch();
    front_ln_rows_kernel<<<(unsigned)((R + 3) / 4), 128, 0, s>>>(in, f32(g), f32(b), scale, of, ob, R, zero_past, T_all);
    LS_CUDA(cudaGetLastError());
  };
  auto rel_pos = [&](int Tl) {
    count_launch();
    front_rel_pos_kernel<<<dim3((kD / 2 + 127) / 128, 2 * Tl - 1), 128, 0, s>>>(pe, Tl);
    LS_CUDA(cudaGetLastError());
  };
  // ConformerEncoderLayer (encoder_layer.py:109-, normalize_before, no macaron, no conv module) on the residual stream xr
  auto layer = [&](const LayerW& L, const Plan::Level& lv, float* xr, int chunk, const int* lens) {
    const int Tl = lv.T;
    const long long R = (long long)B * Tl;
    ln(xr, L.g_mha, L.b_mha, 1.0f, nullptr, nb, R);
    {
      ConvGemmParams p{};
      p.out1 = qkv, p.out1_mode = OUT1_COPY;
      conv(lv.nb, L.qkv, B, Tl, 0, p);
    }
    count_launch();
    front_q_prep_kernel<<<blocks((size_t)R * kD), 256, 0, s>>>(qkv, f32(L.bias_u), f32(L.bias_v), qv, (size_t)R * kD);
    LS_CUDA(cudaGetLastError());
    {  // linear_pos (no bias) on the relative-position table, then head-major for the bd GEMMs
      ConvGemmParams p{};
      p.out1 = pp, p.out1_mode = OUT1_COPY;
      conv(lv.pe, L.pos, 1, lv.P, 0, p);
      count_launch();
      front_split_heads_kernel<<<blocks((size_t)lv.P * kD), 256, 0, s>>>(pp, pph, lv.P, lv.Ppad);
      LS_CUDA(cudaGetLastError());
    }
    for (int h = 0; h < heads_; ++h) {  // bd_full[b][h][i][n] = (q_i + v)_h . p_h[n]
      PackedLinear w;
      w.N = lv.Ppad, w.K = 64, w.taps = 1, w.block_n = lv.bd_block_n, w.map = lv.pph[h], w.bias = nullptr;
      ConvGemmParams p{};
      p.B = B, p.M = Tl, p.N = w.N, p.block_n = w.block_n;
      p.taps = 1, p.dil = 1, p.pad = 0, p.kb_per_tap = 1, p.kb_split = 1;
      p.m_len_mul = 1, p.chan_mod = w.N, p.n_store = w.N;
      p.out0 = bd + (size_t)h * Tl * lv.Ppad, p.out0_dtype = OUT_F32;
      p.out_ld = lv.Ppad, p.out_shift = 0, p.out_bstride = (long long)heads_ * Tl * lv.Ppad, p.out_alloc = (long long)Tl * lv.Ppad;
      p.out_valid_mul = lv.Ppad, p.k_true = 64, p.tag = 0, p.halo_mode = 0;
      LS_CUDA(launch_conv_gemm(lv.qv[h], lv.qv[h], w.map, p, num_sms_, s));
    }
    {
      AttnParams ap{};
      ap.B = B, ap.T = Tl, ap.H = heads_, ap.lengths = lens, ap.chunk = chunk;
      ap.scale_log2e = 0.125f * 1.4426950408889634f;
      ap.out = att;
      ap.bias = bd, ap.bias_ld = lv.Ppad, ap.bias_bh = (long long)Tl * lv.Ppad;
      LS_CUDA(launch_attention(lv.qkv_attn, ap, s));
    }
    {
      ConvGemmParams p{};
      p.addend = xr, p.addend_dtype = OUT_F32, p.out0 = xr, p.out0_dtype = OUT_F32;
      conv(lv.att, L.out, B, Tl, 0, p);
    }
    ln(xr, L.g_ff, L.b_ff, 1.0f, nullptr, nb, R);
    {
      ConvGemmParams p{};
      p.act = ACT_SILU, p.out1 = hb, p.out1_mode = OUT1_COPY;
      conv(lv.nb, L.ff1, B, Tl, 0, p);
    }
    {
      ConvGemmParams p{};
      p.addend = xr, p.addend_dtype = OUT_F32, p.out0 = xr, p.out0_dtype = OUT_F32;
      conv(lv.h, L.ff2, B, Tl, 0, p);
    }
  };

  count_launch();
  front_spk_kernel<<<B, 128, 0, s>>>(embedding, f32(spk_w_), f32(spk_b_), spks, spk_, out_);
  LS_CUDA(cudaGetLastError());
  count_launch();
  int *lens0 = nullptr, *lens1 = nullptr;
  if (token_len) {  // right-padded batch: key bounds of the two frame rates
    require(B <= 512, "at most 512 utterances per call with token lengths");
    lens0 = ws<int>(o_spk_), lens1 = lens0 + 512;
    count_launch();
    front_lens_kernel<<<(B + 127) / 128, 128, 0, s>>>(token_len, n_context, lens0, lens1, B, T_all, T);
    LS_CUDA(cudaGetLastError());
  }
  front_gather_kernel<<<(unsigned)((size_t)B * T_all), 64, 0, s>>>(tokens, arena_.ptr<__nv_bfloat16>(emb_table_), hb, vocab_, T_all,
                                                                   token_len);
  LS_CUDA(cudaGetLastError());
  const float sqrt_d = sqrtf((float)kD);
  {  // LinearNoSubsampling (subsampling.py:69-113) on tokens and context alike: Linear, LayerNorm, x sqrt(d)
    ConvGemmParams p{};
    p.out0 = y, p.out0_dtype = OUT_F32;
    conv(pl.tok, embed_.lin, B, T_all, 0, p);
    // session mode: the rows past a session's tokens are the zeros F.pad feeds the pre-lookahead layer of a call alone
    // (the reference's padded batch embeds them instead: bias and LayerNorm make them non-zero)
    ln(y, embed_.g, embed_.b, sqrt_d, x, nb, (long long)B * T_all, n_context ? token_len : nullptr);
  }
  float* xr = x;
  {  // PreLookaheadLayer (upsample_encoder.py:66-107): [x | context or zeros] -> conv k=4 -> leaky_relu -> causal conv k=3, + x
    ConvGemmParams p{};
    p.act = ACT_LRELU001, p.out1 = att, p.out1_mode = OUT1_COPY;
    conv(pl.pre1, pre1_, B, T, 0, p);  // reads rows t .. t+3 of the T_all-row input (rows past it are zero)
    if (T_all > T) {  // the residual stream keeps the first T rows of every utterance
      LS_CUDA(cudaMemcpy2DAsync(y, (size_t)T * kD * 4, x, (size_t)T_all * kD * 4, (size_t)T * kD * 4, B, cudaMemcpyDeviceToDevice, s));
      xr = y;
    }
    ConvGemmParams q{};
    q.addend = xr, q.addend_dtype = OUT_F32, q.out0 = xr, q.out0_dtype = OUT_F32;
    conv(pl.pre2, pre2_, B, T, 2, q);
  }
  const int chunk = streaming ? chunk_ : 0;
  rel_pos(T);
  for (const LayerW& L : layers_) layer(L, pl.lv[0], xr, chunk, lens0);
  {  // Upsample1D (upsample_encoder.py:37-63): nearest x2, left-pad 4, conv k=5; then up_embed
    count_launch();
    front_upsample2_kernel<<<blocks((size_t)B * T2 * kD), 256, 0, s>>>(xr, nb, T, (size_t)B * T2 * kD);
    LS_CUDA(cudaGetLastError());
    ConvGemmParams p{};
    p.out1 = att, p.out1_mode = OUT1_COPY;
    conv(pl.up, up_conv_, B, T2, 4, p);
    ConvGemmParams q{};
    q.out0 = y, q.out0_dtype = OUT_F32;
    conv(pl.lv[1].att, up_embed_.lin, B, T2, 0, q);
    ln(y, up_embed_.g, up_embed_.b, sqrt_d, x, nb, (long long)B * T2);
  }
  rel_pos(T2);
  for (const LayerW& L : up_layers_) layer(L, pl.lv[1], x, 2 * chunk, lens1);
  ln(x, g_after_, b_after_, 1.0f, nullptr, nb, (long long)B * T2);
  {
    ConvGemmParams p{};
    p.out0 = y, p.out0_dtype = OUT_F32;
    conv(pl.lv[1].nb, proj_, B, T2, 0, p);
  }
  LS_CUDA(launch_unpack_nct(y, mu, B, out_, T2, lens1, s));  // frames past 2 * token_len are zero
}

// ------------------------------------------------------------------------------------------------ speaker encoder (f-4)
namespace {

// GroupNorm32 (arch_util.py:21-41) on the time-major fp32 residual stream [R][T][512]: statistics over (16 channels x T
// frames) of one (clip, group), eps 1e-5, per-channel affine; bf16 output (the operand of the qkv GEMM).
// One block per (group, clip); thread = (row phase, float4 of the group's 16 channels).
__global__ void __launch_bounds__(256) spk_group_norm_kernel(const float* __restrict__ x, const float* __restrict__ g,
                                                             const float* __restrict__ be, __nv_bfloat16* __restrict__ y, int T) {
  const int grp = blockIdx.x, r = blockIdx.y;
  const int q4 = threadIdx.x & 3, ph = threadIdx.x >> 2;  // 64 row phases
  const float* xb = x + (size_t)r * T * kD + grp * 16 + q4 * 4;
  __shared__ float red[8];
  __shared__ float stat;
  auto block_sum = [&](float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
      float t = 0.f;
      for (int i = 0; i < 8; ++i) t += red[i];
      stat = t;
    }
    __syncthreads();
    return stat;
  };
  const float n = 16.0f * (float)T;
  float a = 0.f;
  for (int t = ph; t < T; t += 64) {
    const float4 v = *reinterpret_cast<const float4*>(xb + (size_t)t * kD);
    a += v.x + v.y + v.z + v.w;
  }
  const float mean = block_sum(a) / n;
  float q = 0.f;
  for (int t = ph; t < T; t += 64) {
    const float4 v = *reinterpret_cast<const float4*>(xb + (size_t)t * kD);
    const float d0 = v.x - mean, d1 = v.y - mean, d2 = v.z - mean, d3 = v.w - mean;
    q += d0 * d0 + d1 * d1 + d2 * d2 + d3 * d3;
  }
  const float rstd = rsqrtf(block_sum(q) / n + 1e-5f);
  const float4 gm = *reinterpret_cast<const float4*>(g + grp * 16 + q4 * 4);
  const float4 bt = *reinterpret_cast<const float4*>(be + grp * 16 + q4 * 4);
  __nv_bfloat16* yb = y + (size_t)r * T * kD + grp * 16 + q4 * 4;
  for (int t = ph; t < T; t += 64) {
    const float4 v = *reinterpret_cast<const float4*>(xb + (size_t)t * kD);
    const uint2 o = make_uint2(pack_bf16x2((v.x - mean) * rstd * gm.x + bt.x, (v.y - mean) * rstd * gm.y + bt.y),
                               pack_bf16x2((v.z - mean) * rstd * gm.z + bt.z, (v.w - mean) * rstd * gm.w + bt.w));
    *reinterpret_cast<uint2*>(yb + (size_t)t * kD) = o;
  }
}

// first-frame pooling (llm.py:88), output_proj, L2 normalise; n_refs > 1: mean of the per-clip unit vectors, normalised
// again (flow.py:336-366).  h is [n_refs][B][T][512]; one block per utterance b.
__global__ void __launch_bounds__(256) spk_head_kernel(const float* __restrict__ h, const float* __restrict__ w,
                                                       const float* __restrict__ bias, float* __restrict__ emb, int B, int T,
                                                       int n_refs, int N) {
  const int b = blockIdx.x;
  __shared__ float v[256];    // this clip's projection (N <= 256)
  __shared__ float acc[256];  // sum of the unit vectors
  __shared__ float red[8];
  __shared__ float nrm;
  auto block_norm = [&](float x2) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x2 += __shfl_xor_sync(0xffffffffu, x2, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = x2;
    __syncthreads();
    if (threadIdx.x == 0) {
      float t = 0.f;
      for (int i = 0; i < 8; ++i) t += red[i];
      nrm = fmaxf(sqrtf(t), 1e-12f);
    }
    __syncthreads();
    return nrm;
  };
  acc[threadIdx.x] = 0.f;
  for (int i = 0; i < n_refs; ++i) {
    const float* row = h + ((size_t)i * B + b) * T * kD;  // frame 0 of clip (i, b)
    float y = 0.f;
    if (threadIdx.x < N) {
      y = bias[threadIdx.x];
      for (int k = 0; k < kD; ++k) y = fmaf(row[k], w[(size_t)threadIdx.x * kD + k], y);
    }
    v[threadIdx.x] = y;
    const float nn = block_norm(threadIdx.x < N ? y * y : 0.f);
    acc[threadIdx.x] += v[threadIdx.x] / nn;
    __syncthreads();
  }
  if (n_refs == 1) {
    if (threadIdx.x < N) emb[(size_t)b * N + threadIdx.x] = acc[threadIdx.x];
    return;
  }
  const float m = acc[threadIdx.x] / (float)n_refs;
  const float nn = block_norm(threadIdx.x < N ? m * m : 0.f);
  if (threadIdx.x < N) emb[(size_t)b * N + threadIdx.x] = m / nn;
}

}  // namespace

struct SpeakerEngine::Plan {
  CUtensorMap mel, nb, att, qkv_attn;
};

SpeakerEngine::~SpeakerEngine() {
  if (ws_base_) cudaFree(ws_base_);
}

SpeakerEngine::SpeakerEngine(const Weights& w, int device) : device_(device) {
  LS_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  LS_CUDA(cudaGetDeviceProperties(&prop, device));
  require(prop.major == 10, "this library only runs on sm_100 (B200) devices", LS_ERR_UNSUPPORTED);
  num_sms_ = prop.multiProcessorCount;
  const ls_tensor& wi = w.get("init.weight");
  require(wi.ndim == 3 && wi.shape[0] == kD && wi.shape[2] == 1 && wi.shape[1] % 8 == 0, "speaker encoder: expected Conv1d(mel, 512, 1)",
          LS_ERR_UNSUPPORTED);
  mel_ = (int)wi.shape[1];
  init_ = pack_dense(arena_, wi, &w.get("init.bias"));
  const ls_tensor& wo = w.get("output_proj.weight");
  out_ = (int)wo.shape[0];
  require(wo.ndim == 2 && wo.shape[1] == kD && out_ <= 256, "speaker encoder: unexpected output_proj", LS_ERR_UNSUPPORTED);
  out_w_ = arena_.put_f32(wo.data, (size_t)out_ * kD);
  out_b_ = arena_.put_f32(w.get("output_proj.bias", {out_}).data, out_);
  for (int i = 0; w.has("attn." + std::to_string(i) + ".norm.weight"); ++i) {
    const std::string p = "attn." + std::to_string(i);
    BlockW bw;
    {  // qkv conv rows are head-major [q_h | k_h | v_h] (QKVAttentionLegacy, arch_util.py:57-60) -> Q | K | V column blocks
      const ls_tensor& wq = w.get(p + ".qkv.weight", {3 * kD, kD, 1});
      const ls_tensor& bq = w.get(p + ".qkv.bias", {3 * kD});
      std::vector<float> cat((size_t)3 * kD * kD), bias((size_t)3 * kD);
      for (int part = 0; part < 3; ++part)
        for (int hh = 0; hh < heads_; ++hh)
          for (int d = 0; d < 64; ++d) {
            const size_t src = (size_t)hh * 192 + part * 64 + d, dst = (size_t)part * kD + hh * 64 + d;
            std::memcpy(cat.data() + dst * kD, wq.data + src * kD, (size_t)kD * 4);
            bias[dst] = bq.data[src];
          }
      ls_tensor tw{}, tb{};
      tw.name = wq.name, tw.data = cat.data(), tw.ndim = 2, tw.shape[0] = 3 * kD, tw.shape[1] = kD;
      tb.name = wq.name, tb.data = bias.data(), tb.ndim = 1, tb.shape[0] = 3 * kD;
      bw.qkv = pack_dense(arena_, tw, &tb);
    }
    bw.proj = pack_dense(arena_, w.get(p + ".proj_out.weight", {kD, kD, 1}), &w.get(p + ".proj_out.bias"));
    bw.g = arena_.put_f32(w.get(p + ".norm.weight", {kD}).data, kD);
    bw.b = arena_.put_f32(w.get(p + ".norm.bias", {kD}).data, kD);
    blocks_.push_back(bw);
  }
  arena_.upload();
  finalize_dense(arena_, init_);
  for (BlockW& bw : blocks_) finalize_dense(arena_, bw.qkv), finalize_dense(arena_, bw.proj);
}

const SpeakerEngine::Plan& SpeakerEngine::plan_for(int R, int T, cudaStream_t s) {
  const long long rows = (long long)R * T;
  if (rows > cap_rows_) {
    ws_release(ws_base_, s);
    plans_.clear();
    cap_rows_ = rows;
    size_t off = 0;
    auto take = [&](size_t bytes) {
      size_t o = off;
      off = (off + bytes + 1023) & ~size_t(1023);
      return o;
    };
    const size_t n = (size_t)rows + 256;
    o_h_ = take(n * kD * 4), o_nb_ = take(n * kD * 2), o_qkv_ = take(n * 3 * kD * 2), o_att_ = take(n * kD * 2);
    o_mel_ = take(n * (size_t)mel_ * 2), o_emb_ = take(4096);
    ws_alloc(ws_base_, off, s);
  }
  auto key = std::make_pair(R, T);
  auto it = plans_.find(key);
  if (it != plans_.end()) return *it->second;
  auto pl = std::make_unique<Plan>();
  require(make_act_map(&pl->mel, ws_base_ + o_mel_, mel_, T, R, mel_, (long long)T * mel_, 128) &&
              make_act_map(&pl->nb, ws_base_ + o_nb_, kD, T, R, kD, (long long)T * kD, 128) &&
              make_act_map(&pl->att, ws_base_ + o_att_, kD, T, R, kD, (long long)T * kD, 128) &&
              make_act_map(&pl->qkv_attn, ws_base_ + o_qkv_, 3 * kD, T, R, 3 * kD, (long long)T * 3 * kD, ATTN_KV),
          "cuTensorMapEncodeTiled failed for a speaker-encoder buffer", LS_ERR_CUDA);
  const Plan& ref = *pl;
  plans_[key] = std::move(pl);
  return ref;
}

// LearnableSpeakerEncoder.forward (llm.py:70-96): init conv -> AttentionBlocks (x + proj_out(attn(qkv(GroupNorm(x))))) ->
// first frame -> output_proj -> L2 normalise (-> mean over reference clips -> normalise)
void SpeakerEngine::encode(const float* mel, float* emb, int B, int T, int n_refs, cudaStream_t s) {
  require(B > 0 && T > 0 && n_refs > 0, "B, T, n_refs must be positive");
  LS_CUDA(cudaSetDevice(device_));
  const int R = B * n_refs;  // every clip is an independent batch row
  const Plan& pl = plan_for(R, T, s);
  auto f32 = [&](size_t off) { return arena_.ptr<float>(off); };
  float* h = ws<float>(o_h_);
  __nv_bfloat16* nb = ws<__nv_bfloat16>(o_nb_);
  __nv_bfloat16* qkv = ws<__nv_bfloat16>(o_qkv_);
  __nv_bfloat16* att = ws<__nv_bfloat16>(o_att_);
  auto conv = [&](const CUtensorMap& a, const PackedLinear& w, ConvGemmParams p) {
    p.B = R, p.M = T, p.N = w.N, p.block_n = w.block_n;
    p.taps = 1, p.dil = 1, p.pad = 0;
    p.kb_per_tap = (w.K + 63) / 64, p.kb_split = p.kb_per_tap;
    p.lengths = nullptr, p.m_len_mul = 1, p.m_len_add = 0, p.skip_halo = 0;
    p.bias = w.bias, p.chan_mod = w.N, p.n_store = w.N;
    p.out_ld = w.N, p.out_shift = 0, p.out_bstride = (long long)T * w.N, p.out_alloc = (long long)T * w.N, p.out_valid_mul = w.N;
    p.k_true = w.K, p.tag = 0, p.halo_mode = 0;
    LS_CUDA(launch_conv_gemm(a, a, w.map, p, num_sms_, s));
  };
  LS_CUDA(launch_pack_nct(mel, ws<__nv_bfloat16>(o_mel_), R, mel_, T, (long long)mel_ * T, mel_, 0, nullptr, s));
  {
    ConvGemmParams p{};
    p.out0 = h, p.out0_dtype = OUT_F32;
    conv(pl.mel, init_, p);
  }
  for (const BlockW& bw : blocks_) {
    count_launch();
    spk_group_norm_kernel<<<dim3(groups_, R), 256, 0, s>>>(h, f32(bw.g), f32(bw.b), nb, T);
    LS_CUDA(cudaGetLastError());
    {
      ConvGemmParams p{};
      p.out1 = qkv, p.out1_mode = OUT1_COPY;
      conv(pl.nb, bw.qkv, p);
    }
    {
      AttnParams ap{};
      ap.B = R, ap.T = T, ap.H = heads_, ap.lengths = nullptr, ap.chunk = 0;
      ap.scale_log2e = 0.125f * 1.4426950408889634f;  // (q 64^-1/4) . (k 64^-1/4)
      ap.out = att;
      LS_CUDA(launch_attention(pl.qkv_attn, ap, s));
    }
    {
      ConvGemmParams p{};
      p.addend = h, p.addend_dtype = OUT_F32, p.out0 = h, p.out0_dtype = OUT_F32;
      conv(pl.att, bw.proj, p);
    }
  }
  count_launch();
  spk_head_kernel<<<B, 256, 0, s>>>(h, f32(out_w_), f32(out_b_), emb, B, T, n_refs, out_);
  LS_CUDA(cudaGetLastError());
}

}  // namespace ls
