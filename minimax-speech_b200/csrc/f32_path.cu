// fp32 mode of the hot path: see f32_path.h.  Plain CUDA-core kernels in the reference's NCT layout, one per
// reference op, no fusion, accurate libm (no fast-math intrinsics).  Reference lines next to each kernel.
#include <cmath>
#include <utility>

#include "f32_path.h"

namespace ls {
namespace {

constexpr int kTB = 128;  // threads per block: one thread per time step
constexpr int kNB = 4;    // output channels per thread

inline dim3 grid_t(int T, int n, int B) { return dim3((unsigned)((T + kTB - 1) / kTB), (unsigned)n, (unsigned)B); }
#define F32_LAUNCH(kernel, grid, block, stream, ...)   \
  do {                                                 \
    count_launch();                                    \
    kernel<<<grid, block, 0, stream>>>(__VA_ARGS__);   \
    LS_CUDA(cudaGetLastError());                       \
  } while (0)

// out[b,n,t] = act(bias[n] + sum_c sum_k in[b,c,t + k*dil - pad] * m_in[b,t'] * w[n,c,k]) * m_out[b,t]
// Conv1d / CausalConv1d (pad = K-1, flow/decoder.py:36-62) / 1x1 / Linear over channels; x*mask fused on the input
// (decoder.py:68, matcha decoder.py:60) and on the output (decoder.py:496).  lrelu < 0: no activation.
__global__ void __launch_bounds__(kTB) conv1d_nct_kernel(const float* __restrict__ in, const float* __restrict__ m_in,
                                                         const float* __restrict__ w, const float* __restrict__ bias,
                                                         float* __restrict__ out, const float* __restrict__ m_out, int Cin,
                                                         int Tin, int T, int N, int K, int dil, int pad, int stride,
                                                         float lrelu) {
  // Tin: input length, T: output length; stride > 1 = the encoder's downsampling convs (dac-vae/model.py:183-189)
  const int t = blockIdx.x * kTB + threadIdx.x;
  const int n0 = blockIdx.y * kNB;
  const int b = blockIdx.z;
  if (t >= T) return;
  float acc[kNB];
#pragma unroll
  for (int j = 0; j < kNB; ++j) acc[j] = (bias && n0 + j < N) ? bias[n0 + j] : 0.f;
  const float* inb = in + (size_t)b * Cin * Tin;
  const float* mb = m_in ? m_in + (size_t)b * Tin : nullptr;
  for (int k = 0; k < K; ++k) {
    const int tt = t * stride + k * dil - pad;
    if (tt < 0 || tt >= Tin) continue;
    const float mv = mb ? mb[tt] : 1.f;
    for (int c = 0; c < Cin; ++c) {
      const float v = inb[(size_t)c * Tin + tt] * mv;
#pragma unroll
      for (int j = 0; j < kNB; ++j)
        if (n0 + j < N) acc[j] = fmaf(v, w[((size_t)(n0 + j) * Cin + c) * K + k], acc[j]);
    }
  }
  const float mo = m_out ? m_out[(size_t)b * T + t] : 1.f;
#pragma unroll
  for (int j = 0; j < kNB; ++j)
    if (n0 + j < N) {
      float y = acc[j];
      if (lrelu >= 0.f) y = y > 0.f ? y : lrelu * y;
      out[((size_t)b * N + n0 + j) * T + t] = y * mo;
    }
}

// ConvTranspose1d (dac-vae/model.py:255-262): out[b,n,t] = bias[n] + sum_c sum_{k: (t+pad-k) % s == 0} in[b,c,(t+pad-k)/s] w[c,n,k]
__global__ void __launch_bounds__(kTB) convt1d_nct_kernel(const float* __restrict__ in, const float* __restrict__ w,
                                                          const float* __restrict__ bias, float* __restrict__ out, int Cin,
                                                          int Lin, int N, int K, int stride, int pad, int Lout) {
  const int t = blockIdx.x * kTB + threadIdx.x;
  const int n0 = blockIdx.y * kNB;
  const int b = blockIdx.z;
  if (t >= Lout) return;
  float acc[kNB];
#pragma unroll
  for (int j = 0; j < kNB; ++j) acc[j] = n0 + j < N ? bias[n0 + j] : 0.f;
  const float* inb = in + (size_t)b * Cin * Lin;
  for (int k = (t + pad) % stride; k < K; k += stride) {
    const int i = (t + pad - k) / stride;
    if (t + pad - k < 0 || i >= Lin) continue;
    for (int c = 0; c < Cin; ++c) {
      const float v = inb[(size_t)c * Lin + i];
#pragma unroll
      for (int j = 0; j < kNB; ++j)
        if (n0 + j < N) acc[j] = fmaf(v, w[((size_t)c * N + n0 + j) * K + k], acc[j]);
    }
  }
#pragma unroll
  for (int j = 0; j < kNB; ++j)
    if (n0 + j < N) out[((size_t)b * N + n0 + j) * Lout + t] = acc[j];
}

__device__ __forceinline__ float mish_exact(float x) {  // F.mish: x * tanh(softplus(x)), softplus threshold 20
  const float sp = x > 20.f ? x : log1pf(expf(x));
  return x * tanhf(sp);
}

// LayerNorm over the channel dim of [B,C,T] per (b,t), eps 1e-5 (decoder.py:70-76 via two transposes;
// transformer.py:243,303), then optionally Mish, * mask, + vec[b,c] (the time-embedding add, matcha decoder.py:58)
__global__ void __launch_bounds__(kTB) layernorm_nct_kernel(const float* __restrict__ x, const float* __restrict__ g,
                                                            const float* __restrict__ be, float* __restrict__ y, int C,
                                                            int T, int do_mish, const float* __restrict__ mask,
                                                            const float* __restrict__ vec, float eps = 1e-5f) {
  const int t = blockIdx.x * kTB + threadIdx.x;
  const int b = blockIdx.z;
  if (t >= T) return;
  const float* xb = x + (size_t)b * C * T + t;
  float mean = 0.f;
  for (int c = 0; c < C; ++c) mean += xb[(size_t)c * T];
  mean /= (float)C;
  float var = 0.f;
  for (int c = 0; c < C; ++c) {
    const float d = xb[(size_t)c * T] - mean;
    var = fmaf(d, d, var);
  }
  const float rstd = 1.0f / sqrtf(var / (float)C + eps);
  const float mv = mask ? mask[(size_t)b * T + t] : 1.f;
  float* yb = y + (size_t)b * C * T + t;
  for (int c = 0; c < C; ++c) {
    float v = (xb[(size_t)c * T] - mean) * rstd * g[c] + be[c];
    if (do_mish) v = mish_exact(v);
    v *= mv;
    if (vec) v += vec[(size_t)b * C + c];
    yb[(size_t)c * T] = v;
  }
}

// GroupNorm(G) -> Mish -> * mask (-> + vec[b,c]) on [B,C,T]: matcha Block1D (decoder.py:32-43), the block of the NON-causal
// ConditionalDecoder (flow/decoder.py:88-291).  Statistics over the (C/G channels x valid frames) of one (b, group) -- the
// frames of utterance b alone, as in one reference call per utterance -- two passes (mean, centred variance), eps 1e-5.
__global__ void __launch_bounds__(256) group_norm_mish_nct_kernel(const float* __restrict__ x, const float* __restrict__ g,
                                                                  const float* __restrict__ be, float* __restrict__ y, int C,
                                                                  int T, int G, const int* __restrict__ lens,
                                                                  const float* __restrict__ vec) {
  const int grp = blockIdx.x, b = blockIdx.y;
  const int cpg = C / G;
  const int len = min(lens[b], T);
  const float* xb = x + ((size_t)b * C + (size_t)grp * cpg) * T;
  float* yb = y + ((size_t)b * C + (size_t)grp * cpg) * T;
  __shared__ float red[8];
  __shared__ float stat;
  auto block_sum = [&](float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();  // red / stat of the previous reduction have been consumed
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
  const int n = cpg * len;
  float a = 0.f;
  for (int i = threadIdx.x; i < n; i += 256) a += xb[(size_t)(i / len) * T + i % len];
  const float mean = n ? block_sum(a) / (float)n : block_sum(0.f);
  float q = 0.f;
  for (int i = threadIdx.x; i < n; i += 256) {
    const float d = xb[(size_t)(i / len) * T + i % len] - mean;
    q = fmaf(d, d, q);
  }
  const float rstd = 1.0f / sqrtf((n ? block_sum(q) / (float)n : block_sum(0.f)) + 1e-5f);
  for (int i = threadIdx.x; i < cpg * T; i += 256) {
    const int cl = i / T, t = i - cl * T, c = grp * cpg + cl;
    float v = 0.f;
    if (t < len) v = mish_exact((xb[i] - mean) * rstd * g[c] + be[c]);
    if (vec) v += vec[(size_t)b * C + c];
    yb[i] = v;
  }
}

// diffusers Attention / AttnProcessor2_0 on q,k,v [R,H*64,T] with the additive mask of mask.py:161-236 +
// common.py:160-168: key j visible iff j < len[r] (and, streaming, j < (i/chunk+1)*chunk); a query row with no
// visible key sees every key (mask.py:233-235).  One thread per (r, h, query).
__global__ void __launch_bounds__(kTB) attention_nct_kernel(const float* __restrict__ q, const float* __restrict__ k,
                                                            const float* __restrict__ v, float* __restrict__ o,
                                                            const int* __restrict__ lens, int H, int T, int chunk,
                                                            float scale) {
  const int i = blockIdx.x * kTB + threadIdx.x;
  const int h = blockIdx.y, r = blockIdx.z;
  if (i >= T) return;
  const size_t base = ((size_t)r * H + h) * 64 * T;
  int limit = lens[r];
  if (chunk > 0) limit = min(limit, (i / chunk + 1) * chunk);
  if (limit <= 0) limit = T;
  float qr[64], acc[64];
#pragma unroll
  for (int d = 0; d < 64; ++d) qr[d] = q[base + (size_t)d * T + i], acc[d] = 0.f;
  float m = -INFINITY, l = 0.f;
  for (int j = 0; j < limit; ++j) {
    float s = 0.f;
#pragma unroll
    for (int d = 0; d < 64; ++d) s = fmaf(qr[d], k[base + (size_t)d * T + j], s);
    s *= scale;
    const float m_new = fmaxf(m, s);
    const float corr = expf(m - m_new);  // exp(-inf) = 0 on the first key
    const float p = expf(s - m_new);
    l = l * corr + p;
#pragma unroll
    for (int d = 0; d < 64; ++d) acc[d] = fmaf(p, v[base + (size_t)d * T + j], acc[d] * corr);
    m = m_new;
  }
  const float inv = 1.0f / l;
#pragma unroll
  for (int d = 0; d < 64; ++d) o[base + (size_t)d * T + i] = acc[d] * inv;
}

enum { EW_ADD = 0, EW_GELU = 1, EW_TANH = 2, EW_LRELU001 = 3, EW_SILU = 4 };
__global__ void ew_kernel(const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ y, size_t n, int op) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float x = a[i];
  float r;
  if (op == EW_ADD) r = x + b[i];
  else if (op == EW_GELU) r = 0.5f * x * (1.0f + erff(x * 0.70710678118654752f));  // F.gelu(approximate="none")
  else if (op == EW_TANH) r = tanhf(x);
  else if (op == EW_SILU) r = x / (1.0f + expf(-x));  // swish (transformer/positionwise_feed_forward.py:55)
  else r = x > 0.f ? x : 0.01f * x;  // F.leaky_relu default slope (dac-vae/model.py:475)
  y[i] = r;
}
// snake(x) = x + (alpha + 1e-9)^-1 sin^2(alpha x), alpha per channel (dac-vae/layers.py:18-24)
__global__ void snake_nct_kernel(const float* __restrict__ x, const float* __restrict__ alpha, float* __restrict__ y, int C,
                                 int T, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float a = alpha[(i / T) % C];
  const float sn = sinf(a * x[i]);
  y[i] = x[i] + (1.0f / (a + 1e-9f)) * sn * sn;
}
// y[r,n] = act_out(bias[n] + sum_k act_in(x[r,k]) w[n,k]); act_in: 0 none, 1 Mish; act_out: 0 none, 1 SiLU
__global__ void linear_rows_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ bias,
                                   float* __restrict__ y, int R, int K, int N, int act_in, int act_out) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  const int r = blockIdx.y;
  if (n >= N) return;
  float acc = bias ? bias[n] : 0.f;
  for (int k = 0; k < K; ++k) {
    float v = x[(size_t)r * K + k];
    if (act_in == 1) v = mish_exact(v);
    acc = fmaf(v, w[(size_t)n * K + k], acc);
  }
  if (act_out == 1) acc = acc / (1.0f + expf(-acc));
  y[(size_t)r * N + n] = acc;
}
// SinusoidalPosEmb (matcha decoder.py:14-29): [sin(1000 t f_i) | cos(1000 t f_i)], f_i = exp(-i ln(1e4)/(half-1))
__global__ void sinusoid_kernel(const float* __restrict__ t, float* __restrict__ y, int R, int dim) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int r = blockIdx.y;
  const int half = dim / 2;
  if (i >= half) return;
  const float f = expf((float)i * -(logf(10000.0f) / (float)(half - 1)));
  const float e = 1000.0f * t[r] * f;
  y[(size_t)r * dim + i] = sinf(e);
  y[(size_t)r * dim + half + i] = cosf(e);
}
// h0 = cat[x | mu | spks (broadcast over T) | cond] (flow/decoder.py:427-433)
__global__ void build_input_kernel(const float* __restrict__ x, const float* __restrict__ mu, const float* __restrict__ spks,
                                   const float* __restrict__ cond, float* __restrict__ h, int F, int T, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int t = (int)(i % T);
  const int c = (int)((i / T) % (4 * F));
  const size_t r = i / ((size_t)T * 4 * F);
  const int part = c / F, cc = c % F;
  const size_t src = (r * F + cc) * T + t;
  h[i] = part == 0 ? x[src] : part == 1 ? mu[src] : part == 2 ? spks[r * F + cc] : cond[src];
}
__global__ void cat_channels_kernel(const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ y, int Ca,
                                    int Cb, int T, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int t = (int)(i % T);
  const int c = (int)((i / T) % (Ca + Cb));
  const size_t r = i / ((size_t)T * (Ca + Cb));
  y[i] = c < Ca ? a[(r * Ca + c) * T + t] : b[(r * Cb + c - Ca) * T + t];
}
__global__ void mask_lengths_kernel(const float* __restrict__ mask, int* __restrict__ lens, int T) {
  const int r = blockIdx.x;
  int n = 0;
  for (int t = threadIdx.x; t < T; t += blockDim.x) n += mask[(size_t)r * T + t] != 0.f;
  __shared__ int sh[32];
  for (int o = 16; o; o >>= 1) n += __shfl_down_sync(0xffffffffu, n, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = n;
  __syncthreads();
  if (threadIdx.x == 0) {
    int tot = 0;
    for (int i = 0; i < (int)(blockDim.x + 31) / 32; ++i) tot += sh[i];
    lens[r] = tot;
  }
}
// CFG batch of flow_matching.py:105-110 for B >= 1: rows [0,B) conditional, [B,2B) with mu = spks = cond = 0
__global__ void cfg_pack_kernel(const float* __restrict__ x, const float* __restrict__ mu, const float* __restrict__ cond,
                                const float* __restrict__ mask, float* __restrict__ x2, float* __restrict__ mu2,
                                float* __restrict__ cond2, float* __restrict__ mask2, int F, int T, int B) {
  const size_t n = (size_t)B * F * T;
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    x2[i] = x[i], x2[n + i] = x[i];
    mu2[i] = mu[i], mu2[n + i] = 0.f;
    cond2[i] = cond[i], cond2[n + i] = 0.f;
  }
  const size_t nm = (size_t)B * T;
  if (i < nm) mask2[i] = mask[i], mask2[nm + i] = mask[i];
}
__global__ void cfg_small_kernel(const float* __restrict__ spks, float* __restrict__ spks2, float* __restrict__ t2, float t,
                                 int F, int B) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < B * F) spks2[i] = spks[i], spks2[B * F + i] = 0.f;
  if (i < 2 * B) t2[i] = t;
}
// x += dt * ((1 + w) v_c - w v_u)   (flow_matching.py:118-121)
__global__ void euler_kernel(float* __restrict__ x, const float* __restrict__ v, float dt, float w, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float vv = (1.0f + w) * v[i] - w * v[n + i];
  x[i] = x[i] + dt * vv;
}
__global__ void init_noise_kernel(const float* __restrict__ noise, long long stride, float temperature, float* __restrict__ x,
                                  int F, int T, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int t = (int)(i % T);
  const int c = (int)((i / T) % F);
  x[i] = noise[(size_t)c * stride + t] * temperature;
}
__global__ void mul_mask_kernel(const float* __restrict__ x, const float* __restrict__ mask, float* __restrict__ y, int C, int T,
                                size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  y[i] = x[i] * mask[(i / ((size_t)C * T)) * T + i % T];
}

// m, logs = split(x); logs = clamp(logs, -14, 14); z = m + noise * exp(logs)   (dac-vae/model.py:477-481)
__global__ void reparam_kernel(const float* __restrict__ x, const float* __restrict__ noise, float* __restrict__ z,
                               float* __restrict__ m, float* __restrict__ logs, int latent, int L, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int t = (int)(i % L);
  const int c = (int)((i / L) % latent);
  const size_t b = i / ((size_t)L * latent);
  const float mv = x[(b * 2 * latent + c) * L + t];
  const float lv = fminf(fmaxf(x[(b * 2 * latent + latent + c) * L + t], -14.0f), 14.0f);
  m[i] = mv, logs[i] = lv;
  z[i] = noise ? mv + noise[i] * expf(lv) : mv;
}

// ---- token -> mu front half (SURVEY section 8 f-1) -------------------------------------------------------------
// x[b,c,t] = E[clamp(tok[b,t], 0)][c]   (flow/flow.py:476: input_embedding(torch.clamp(token, min=0)))
// rows past the utterance's token count are zero (flow.py:475-476: input_embedding(token) * mask)
__global__ void embed_tokens_kernel(const long long* __restrict__ tok, const float* __restrict__ E, float* __restrict__ x, int d,
                                    int T, int vocab, size_t n, const int* __restrict__ lens) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int t = (int)(i % T);
  const int c = (int)((i / T) % d);
  const size_t b = i / ((size_t)T * d);
  long long id = tok[b * T + t];
  id = id < 0 ? 0 : (id >= vocab ? vocab - 1 : id);
  x[i] = (lens && t >= lens[b]) ? 0.f : E[(size_t)id * d + c];
}
// y[b,c,t] = 0 for t >= lens[b]
__global__ void zero_tail_nct_kernel(float* __restrict__ y, const int* __restrict__ lens, int C, int T, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if ((int)(i % T) >= lens[i / ((size_t)C * T)]) y[i] = 0.f;
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
__global__ void scale_kernel(float* __restrict__ x, float sc, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) x[i] *= sc;
}
// EspnetRelPositionalEncoding (transformer/embedding.py:224-300): pe[n][:] for relative position T-1-n, n in [0, 2T-1)
__global__ void rel_pos_emb_kernel(float* __restrict__ pe, int T, int d) {
  const int c2 = blockIdx.x * blockDim.x + threadIdx.x;  // pair index
  const int n = blockIdx.y;
  if (c2 >= d / 2) return;
  const float pos = (float)(T - 1 - n);
  const float div = expf((float)(2 * c2) * -(logf(10000.0f) / (float)d));
  pe[(size_t)n * d + 2 * c2] = sinf(pos * div);
  pe[(size_t)n * d + 2 * c2 + 1] = cosf(pos * div);
}
// RelPositionMultiHeadedAttention (transformer/attention.py:249-330) on q,k,v [B,H*64,T] (NCT) and the projected
// positions pp [2T-1][H*64]: score(i,j) = ((q_i + u) . k_j + (q_i + v) . pp[T-1-i+j]) / sqrt(64) for j < len[b]
// (rel_shift of :225-247 in closed form); softmax; . v.  One thread per (b, h, query).
__global__ void __launch_bounds__(kTB) rel_attention_nct_kernel(const float* __restrict__ q, const float* __restrict__ k,
                                                                const float* __restrict__ v, const float* __restrict__ pp,
                                                                const float* __restrict__ bu, const float* __restrict__ bv,
                                                                float* __restrict__ o, int H, int T, int len, int chunk,
                                                                const int* __restrict__ lens) {
  const int i = blockIdx.x * kTB + threadIdx.x;
  const int h = blockIdx.y, b = blockIdx.z;
  if (i >= T) return;
  if (lens) len = min(len, lens[b]);  // key-padding mask of a mixed-length batch (attention.py:84-127)
  if (chunk > 0) len = min(len, (i / chunk + 1) * chunk);  // block-causal (utils/mask.py:127-158)
  const size_t base = ((size_t)b * H + h) * 64 * T;
  const int inner = H * 64;
  float qu[64], qv[64], acc[64];
#pragma unroll
  for (int d = 0; d < 64; ++d) {
    const float qq = q[base + (size_t)d * T + i];
    qu[d] = qq + bu[h * 64 + d], qv[d] = qq + bv[h * 64 + d], acc[d] = 0.f;
  }
  float m = -INFINITY, l = 0.f;
  for (int j = 0; j < len; ++j) {
    const float* pr = pp + (size_t)(T - 1 - i + j) * inner + h * 64;
    float s = 0.f;
#pragma unroll
    for (int d = 0; d < 64; ++d) s = fmaf(qu[d], k[base + (size_t)d * T + j], fmaf(qv[d], pr[d], s));
    s *= 0.125f;
    const float m_new = fmaxf(m, s);
    const float corr = expf(m - m_new);
    const float p = expf(s - m_new);
    l = l * corr + p;
#pragma unroll
    for (int d = 0; d < 64; ++d) acc[d] = fmaf(p, v[base + (size_t)d * T + j], acc[d] * corr);
    m = m_new;
  }
  const float inv = l > 0.f ? 1.0f / l : 0.f;
#pragma unroll
  for (int d = 0; d < 64; ++d) o[base + (size_t)d * T + i] = acc[d] * inv;
}
// y[b,c,t] = x[b,c,t] for t < T of rows that are Tin long
__global__ void slice_time_kernel(const float* __restrict__ x, float* __restrict__ y, int Tin, int T, size_t n_out) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_out) return;
  y[i] = x[(i / T) * Tin + i % T];
}
// nearest-neighbour x2 along time (transformer/upsample_encoder.py:60)
__global__ void upsample2_nct_kernel(const float* __restrict__ x, float* __restrict__ y, int T, size_t n_out) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_out) return;
  const size_t row = i / (2 * (size_t)T);
  const int t = (int)(i % (2 * (size_t)T));
  y[i] = x[row * T + t / 2];
}
// F.normalize(x, dim=1) over rows [R][K] (flow.py:463)
__global__ void normalize_rows_kernel(const float* __restrict__ x, float* __restrict__ y, int K) {
  const int r = blockIdx.x;
  __shared__ float sh;
  if (threadIdx.x == 0) {
    float ss = 0.f;
    for (int k = 0; k < K; ++k) ss = fmaf(x[(size_t)r * K + k], x[(size_t)r * K + k], ss);
    sh = fmaxf(sqrtf(ss), 1e-12f);
  }
  __syncthreads();
  for (int k = threadIdx.x; k < K; k += blockDim.x) y[(size_t)r * K + k] = x[(size_t)r * K + k] / sh;
}

// ---- speaker encoder (SURVEY section 8 f-4): llm/llm.py:34-96, transformer/arch_util.py:21-123 --------------------
// GroupNorm32 (arch_util.py:21-41): statistics over (C/G channels x T) of one (b, group) -- contiguous in NCT --
// eps 1e-5, per-channel affine.  One block per (group, b); two passes (mean, then centred variance).
__global__ void __launch_bounds__(256) group_norm_nct_kernel(const float* __restrict__ x, const float* __restrict__ g,
                                                             const float* __restrict__ be, float* __restrict__ y, int C,
                                                             int T, int G) {
  const int grp = blockIdx.x, b = blockIdx.y;
  const int cpg = C / G;
  const size_t n = (size_t)cpg * T;
  const float* xb = x + ((size_t)b * C + (size_t)grp * cpg) * T;
  float* yb = y + ((size_t)b * C + (size_t)grp * cpg) * T;
  __shared__ float red[8];
  __shared__ float stat;
  auto block_sum = [&](float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();  // red / stat of the previous reduction have been consumed
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
  float a = 0.f;
  for (size_t i = threadIdx.x; i < n; i += 256) a += xb[i];
  const float mean = block_sum(a) / (float)n;
  float q = 0.f;
  for (size_t i = threadIdx.x; i < n; i += 256) {
    const float d = xb[i] - mean;
    q = fmaf(d, d, q);
  }
  const float rstd = 1.0f / sqrtf(block_sum(q) / (float)n + 1e-5f);
  for (size_t i = threadIdx.x; i < n; i += 256) {
    const int c = grp * cpg + (int)(i / T);
    yb[i] = (xb[i] - mean) * rstd * g[c] + be[c];
  }
}
// QKVAttentionLegacy (arch_util.py:44-77) on qkv [B, H*3*64, T]: heads are split BEFORE q/k/v (head h owns channels
// [192h, 192h+192) = [q | k | v]); weight = softmax((q*s) . (k*s)), s = 64^-1/4, over all T keys (no mask); a = weight . v
// -> [B, H*64, T].  One thread per (b, h, query).
__global__ void __launch_bounds__(kTB) qkv_legacy_attention_kernel(const float* __restrict__ qkv, float* __restrict__ o, int H,
                                                                   int T) {
  const int i = blockIdx.x * kTB + threadIdx.x;
  const int h = blockIdx.y, b = blockIdx.z;
  if (i >= T) return;
  const float* q = qkv + ((size_t)b * H + h) * 192 * T;
  const float* k = q + (size_t)64 * T;
  const float* v = q + (size_t)128 * T;
  const float sc = 1.0f / sqrtf(sqrtf(64.0f));
  float qr[64], acc[64];
#pragma unroll
  for (int d = 0; d < 64; ++d) qr[d] = q[(size_t)d * T + i] * sc, acc[d] = 0.f;
  float m = -INFINITY, l = 0.f;
  for (int j = 0; j < T; ++j) {
    float s = 0.f;
#pragma unroll
    for (int d = 0; d < 64; ++d) s = fmaf(qr[d], k[(size_t)d * T + j] * sc, s);
    const float m_new = fmaxf(m, s);
    const float corr = expf(m - m_new);
    const float p = expf(s - m_new);
    l = l * corr + p;
#pragma unroll
    for (int d = 0; d < 64; ++d) acc[d] = fmaf(p, v[(size_t)d * T + j], acc[d] * corr);
    m = m_new;
  }
  const float inv = 1.0f / l;
  float* ob = o + ((size_t)b * H + h) * 64 * T;
#pragma unroll
  for (int d = 0; d < 64; ++d) ob[(size_t)d * T + i] = acc[d] * inv;
}
// y[b,c] = x[b,c,0]   (first-position pooling, llm.py:88)
__global__ void first_frame_kernel(const float* __restrict__ x, float* __restrict__ y, int T, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) y[i] = x[i * T];
}
// y = mean over N stacked embeddings [N][B*K] (flow.py:355, several reference clips)
__global__ void mean_stack_kernel(const float* __restrict__ x, float* __restrict__ y, int N, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float a = 0.f;
  for (int k = 0; k < N; ++k) a += x[(size_t)k * n + i];
  y[i] = a / (float)N;
}

// ---- S3 tokenizer trunk (tools/S3Tokenizer/s3tokenizer/model_v2.py) -------------------------------------------------
// lengths after the two stride-2 convs (model_v2.py:330-334: (len + 2 - 2 - 1) / 2 + 1) and the float masks of
// make_non_pad_mask (utils.py) for the input and the two conv outputs
__global__ void s3_lens_kernel(const int* __restrict__ mel_len, int* __restrict__ l1, int* __restrict__ l2, float* __restrict__ m0,
                               float* __restrict__ m1, float* __restrict__ m2, int T, int T1, int T2) {
  const int b = blockIdx.x;
  const int n0 = mel_len[b];
  const int n1 = (n0 - 1) / 2 + 1, n2 = (n1 - 1) / 2 + 1;
  if (threadIdx.x == 0) l1[b] = n1, l2[b] = n2;
  for (int t = threadIdx.x; t < T; t += blockDim.x) m0[(size_t)b * T + t] = t < n0 ? 1.f : 0.f;
  for (int t = threadIdx.x; t < T1; t += blockDim.x) m1[(size_t)b * T1 + t] = t < n1 ? 1.f : 0.f;
  for (int t = threadIdx.x; t < T2; t += blockDim.x) m2[(size_t)b * T2 + t] = t < n2 ? 1.f : 0.f;
}
// apply_rotary_emb (model_v2.py:51-70) in place on x [B, H*64, T]: per head, x * cos + cat(-x[32:], x[:32]) * sin with the
// table of precompute_freqs_cis(64, .) concatenated with itself (angle index d mod 32); cs / sn: [table_len][32]
__global__ void rotary_nct_kernel(float* __restrict__ x, const float* __restrict__ cs, const float* __restrict__ sn, int H, int T,
                                  size_t n_pairs) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_pairs) return;
  const int t = (int)(i % T);
  const int d = (int)((i / T) % 32);
  const size_t bh = i / ((size_t)T * 32);
  float* lo = x + (bh * 64 + d) * T + t;
  float* hi = lo + (size_t)32 * T;
  const float c = cs[(size_t)t * 32 + d], s = sn[(size_t)t * 32 + d];
  const float a = *lo, b = *hi;
  *lo = a * c + (-b) * s;
  *hi = b * c + a * s;
}
// FSMNMultiHeadAttention.forward_fsmn (model_v2.py:177-189): vm = v * mask; (depthwise conv over time, kernel K with
// (K-1)/2 zeros on the left and the rest on the right, + vm) * mask.  v, y: [B, C, T]; w: [C][K]
__global__ void __launch_bounds__(kTB) fsmn_nct_kernel(const float* __restrict__ v, const float* __restrict__ mask,
                                                       const float* __restrict__ w, float* __restrict__ y, int C, int T, int K) {
  const int t = blockIdx.x * kTB + threadIdx.x;
  const int c = blockIdx.y, b = blockIdx.z;
  if (t >= T) return;
  const float* vb = v + ((size_t)b * C + c) * T;
  const float* mb = mask + (size_t)b * T;
  const int left = (K - 1) / 2;
  float acc = 0.f;
  for (int k = 0; k < K; ++k) {
    const int tt = t + k - left;
    if (tt >= 0 && tt < T) acc = fmaf(vb[tt] * mb[tt], w[(size_t)c * K + k], acc);
  }
  y[((size_t)b * C + c) * T + t] = (acc + vb[t] * mb[t]) * mb[t];
}
// [B, C, T] -> [B, T, C] (the row layout the FSQ head reads)
__global__ void nct_to_rows_kernel(const float* __restrict__ x, float* __restrict__ y, int C, int T, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int c = (int)(i % C);
  const int t = (int)((i / C) % T);
  const size_t b = i / ((size_t)C * T);
  y[i] = x[(b * C + c) * T + t];
}

inline unsigned blocks(size_t n) { return (unsigned)((n + 255) / 256); }

void conv1d(const float* in, const float* m_in, const float* w, const float* bias, float* out, const float* m_out, int B,
            int Cin, int T, int N, int K, int dil, int pad, float lrelu, cudaStream_t s, int stride = 1, int t_out = 0) {
  const int Tout = t_out > 0 ? t_out : (stride == 1 ? T : (T + 2 * pad - K) / stride + 1);
  F32_LAUNCH(conv1d_nct_kernel, grid_t(Tout, (N + kNB - 1) / kNB, B), kTB, s, in, m_in, w, bias, out, m_out, Cin, T, Tout, N,
             K, dil, pad, stride, lrelu);
}
void ew(const float* a, const float* b, float* y, size_t n, int op, cudaStream_t s) {
  F32_LAUNCH(ew_kernel, blocks(n), 256, s, a, b, y, n, op);
}

}  // namespace

// ---------------------------------------------------------------------------------------------- infrastructure
F32Weights::~F32Weights() {
  for (auto& kv : items_)
    if (kv.second.dev) cudaFree(kv.second.dev);
}
void F32Weights::add(const std::string& name, const float* host, size_t n, std::vector<long long> shape) {
  Item it;
  LS_CUDA(cudaMalloc(&it.dev, (n ? n : 1) * sizeof(float)));
  LS_CUDA(cudaMemcpy(it.dev, host, n * sizeof(float), cudaMemcpyHostToDevice));
  it.shape = std::move(shape);
  items_[name] = it;
}
const float* F32Weights::ptr(const std::string& name) const {
  auto it = items_.find(name);
  if (it == items_.end()) throw EngineError(LS_ERR_WEIGHTS, "missing weight '" + name + "'");
  return it->second.dev;
}
const std::vector<long long>& F32Weights::shape(const std::string& name) const {
  auto it = items_.find(name);
  if (it == items_.end()) throw EngineError(LS_ERR_WEIGHTS, "missing weight '" + name + "'");
  return it->second.shape;
}
F32Scratch::~F32Scratch() {
  if (base_) cudaFree(base_);
  for (float* p : retired_) cudaFree(p);
}
float* F32Scratch::get(size_t n, cudaStream_t) {
  n = (n + 63) & ~size_t(63);
  if (used_ + n > cap_) {
    // grow: the old block stays alive (kernels already queued may still use pointers into it)
    const size_t want = (used_ + n) * 2 + (size_t(1) << 20);
    if (base_) retired_.push_back(base_);
    LS_CUDA(cudaMalloc(&base_, want * sizeof(float)));
    cap_ = want, used_ = 0;
  }
  float* p = base_ + used_;
  used_ += n;
  return p;
}

static void upload_all(const Weights& w, F32Weights* dst) {
  for (const auto& kv : w.all()) {
    const ls_tensor& t = *kv.second;
    size_t n = 1;
    std::vector<long long> shape;
    for (int i = 0; i < t.ndim; ++i) n *= (size_t)t.shape[i], shape.push_back(t.shape[i]);
    dst->add(kv.first, t.data, n, shape);
  }
}

// ---------------------------------------------------------------------------------------------- flow (estimator + solve)
FlowEngineF32::FlowEngineF32(const Weights& w, int device) : device_(device) {
  LS_CUDA(cudaSetDevice(device));
  upload_all(w, &w_);
  while (w_.has("down_blocks.0.1." + std::to_string(n_blocks_) + ".norm1.weight")) ++n_blocks_;
  while (w_.has("mid_blocks." + std::to_string(n_mid_) + ".0.mlp.1.weight")) ++n_mid_;
  C_ = (int)w_.shape("final_proj.weight")[1];
  feat_ = (int)w_.shape("final_proj.weight")[0];
  require(n_blocks_ > 0 && (int)w_.shape("down_blocks.0.1.0.attn1.to_q.weight")[0] == heads_ * 64,
          "fp32 estimator: expected 8 heads x 64", LS_ERR_UNSUPPORTED);
  // CausalConditionalDecoder: LayerNorm at block.2 (after a Transpose); ConditionalDecoder: GroupNorm at block.1
  causal_ = w_.has("final_block.block.2.weight");
  conv_pad_ = causal_ ? 2 : 1;
  require(causal_ || w_.has("final_block.block.1.weight"), "estimator state dict: neither block.2 (causal) nor block.1 norms",
          LS_ERR_WEIGHTS);
}

// CausalBlock1D (decoder.py:65-78): conv3 causal on x*mask -> LayerNorm(C) -> Mish -> *mask (-> + addvec); for the
// non-causal ConditionalDecoder, matcha's Block1D: conv3 pad 1 -> GroupNorm(8) over the utterance's frames -> Mish -> *mask
float* FlowEngineF32::causal_block(const std::string& p, const float* x, int cin, const float* mask, const float* addvec,
                                   int R, int T, cudaStream_t s) {
  float* c = scratch_.get((size_t)R * C_ * T, s);
  conv1d(x, mask, w_.ptr(p + ".block.0.weight"), w_.ptr(p + ".block.0.bias"), c, nullptr, R, cin, T, C_, 3, 1, conv_pad_, -1.f,
         s);
  float* y = scratch_.get((size_t)R * C_ * T, s);
  if (!causal_) {
    F32_LAUNCH(group_norm_mish_nct_kernel, dim3(8, R), 256, s, c, w_.ptr(p + ".block.1.weight"), w_.ptr(p + ".block.1.bias"), y,
               C_, T, 8, lens_, addvec);
    return y;
  }
  F32_LAUNCH(layernorm_nct_kernel, grid_t(T, 1, R), kTB, s, c, w_.ptr(p + ".block.2.weight"), w_.ptr(p + ".block.2.bias"), y,
             C_, T, 1, mask, addvec);
  return y;
}

// ResnetBlock1D.forward (matcha decoder.py:56-61) with causal blocks (flow/decoder.py:81-85)
float* FlowEngineF32::resnet(const std::string& p, const float* x, int cin, const float* mask, const float* temb, int R,
                             int T, cudaStream_t s) {
  float* tvec = scratch_.get((size_t)R * C_, s);
  F32_LAUNCH(linear_rows_kernel, dim3((C_ + 127) / 128, R), 128, s, temb, w_.ptr(p + ".mlp.1.weight"),
             w_.ptr(p + ".mlp.1.bias"), tvec, R, (int)w_.shape(p + ".mlp.1.weight")[1], C_, 1, 0);
  float* h = causal_block(p + ".block1", x, cin, mask, tvec, R, T, s);
  float* h2 = causal_block(p + ".block2", h, C_, mask, nullptr, R, T, s);
  float* rc = scratch_.get((size_t)R * C_ * T, s);
  conv1d(x, mask, w_.ptr(p + ".res_conv.weight"), w_.ptr(p + ".res_conv.bias"), rc, nullptr, R, cin, T, C_, 1, 1, 0, -1.f, s);
  ew(h2, rc, h2, (size_t)R * C_ * T, EW_ADD, s);
  return h2;
}

// one resnet + n_blocks BasicTransformerBlocks (transformer.py:243-316), all in NCT (a Linear is a 1x1 conv)
float* FlowEngineF32::group(const std::string& prefix, const float* h, int cin, const float* mask, const float* temb,
                            const int* lens, int R, int T, bool streaming, cudaStream_t s) {
  float* u = resnet(prefix + ".0", h, cin, mask, temb, R, T, s);
  const size_t n = (size_t)R * C_ * T;
  const int inner = heads_ * 64;
  for (int j = 0; j < n_blocks_; ++j) {
    const std::string p = prefix + ".1." + std::to_string(j);
    float* nrm = scratch_.get(n, s);
    F32_LAUNCH(layernorm_nct_kernel, grid_t(T, 1, R), kTB, s, u, w_.ptr(p + ".norm1.weight"), w_.ptr(p + ".norm1.bias"), nrm,
               C_, T, 0, (const float*)nullptr, (const float*)nullptr);
    float* q = scratch_.get((size_t)R * inner * T, s);
    float* k = scratch_.get((size_t)R * inner * T, s);
    float* v = scratch_.get((size_t)R * inner * T, s);
    conv1d(nrm, nullptr, w_.ptr(p + ".attn1.to_q.weight"), nullptr, q, nullptr, R, C_, T, inner, 1, 1, 0, -1.f, s);
    conv1d(nrm, nullptr, w_.ptr(p + ".attn1.to_k.weight"), nullptr, k, nullptr, R, C_, T, inner, 1, 1, 0, -1.f, s);
    conv1d(nrm, nullptr, w_.ptr(p + ".attn1.to_v.weight"), nullptr, v, nullptr, R, C_, T, inner, 1, 1, 0, -1.f, s);
    float* att = scratch_.get((size_t)R * inner * T, s);
    F32_LAUNCH(attention_nct_kernel, grid_t(T, heads_, R), kTB, s, q, k, v, att, lens, heads_, T, streaming ? chunk_ : 0,
               0.125f);
    float* o = scratch_.get(n, s);
    conv1d(att, nullptr, w_.ptr(p + ".attn1.to_out.0.weight"), w_.ptr(p + ".attn1.to_out.0.bias"), o, nullptr, R, inner, T,
           C_, 1, 1, 0, -1.f, s);
    float* u1 = scratch_.get(n, s);
    ew(u, o, u1, n, EW_ADD, s);
    F32_LAUNCH(layernorm_nct_kernel, grid_t(T, 1, R), kTB, s, u1, w_.ptr(p + ".norm3.weight"), w_.ptr(p + ".norm3.bias"), nrm,
               C_, T, 0, (const float*)nullptr, (const float*)nullptr);
    const int ff = (int)w_.shape(p + ".ff.net.0.proj.weight")[0];
    float* hh = scratch_.get((size_t)R * ff * T, s);
    conv1d(nrm, nullptr, w_.ptr(p + ".ff.net.0.proj.weight"), w_.ptr(p + ".ff.net.0.proj.bias"), hh, nullptr, R, C_, T, ff, 1,
           1, 0, -1.f, s);
    ew(hh, nullptr, hh, (size_t)R * ff * T, EW_GELU, s);
    conv1d(hh, nullptr, w_.ptr(p + ".ff.net.2.weight"), w_.ptr(p + ".ff.net.2.bias"), o, nullptr, R, ff, T, C_, 1, 1, 0, -1.f,
           s);
    float* u2 = scratch_.get(n, s);
    ew(u1, o, u2, n, EW_ADD, s);
    u = u2;
  }
  return u;
}

// CausalConditionalDecoder.forward (flow/decoder.py:405-496), channels = [C]
void FlowEngineF32::run(const float* x, const float* mask, const float* mu, const float* t, const float* spks,
                        const float* cond, float* out, int R, int T, bool streaming, cudaStream_t s) {
  const int F = feat_;
  int* lens = reinterpret_cast<int*>(scratch_.get((size_t)R, s));
  F32_LAUNCH(mask_lengths_kernel, R, 256, s, mask, lens, T);
  lens_ = lens;
  if (!causal_) streaming = false;  // ConditionalDecoder.forward ignores the flag: full attention (decoder.py:241)
  // time embedding: sinusoid -> Linear -> SiLU -> Linear (matcha decoder.py:14-29, 73-117)
  const int tdim = (int)w_.shape("time_mlp.linear_1.weight")[1], thid = (int)w_.shape("time_mlp.linear_1.weight")[0];
  float* e0 = scratch_.get((size_t)R * tdim, s);
  F32_LAUNCH(sinusoid_kernel, dim3((tdim / 2 + 127) / 128, R), 128, s, t, e0, R, tdim);
  float* e1 = scratch_.get((size_t)R * thid, s);
  F32_LAUNCH(linear_rows_kernel, dim3((thid + 127) / 128, R), 128, s, e0, w_.ptr("time_mlp.linear_1.weight"),
             w_.ptr("time_mlp.linear_1.bias"), e1, R, tdim, thid, 0, 1);
  float* temb = scratch_.get((size_t)R * thid, s);
  F32_LAUNCH(linear_rows_kernel, dim3((thid + 127) / 128, R), 128, s, e1, w_.ptr("time_mlp.linear_2.weight"),
             w_.ptr("time_mlp.linear_2.bias"), temb, R, thid, thid, 0, 0);
  const size_t n_in = (size_t)R * 4 * F * T;
  float* h0 = scratch_.get(n_in, s);
  F32_LAUNCH(build_input_kernel, blocks(n_in), 256, s, x, mu, spks, cond, h0, F, T, n_in);

  float* h = group("down_blocks.0", h0, 4 * F, mask, temb, lens, R, T, streaming, s);
  float* skip = h;
  float* d = scratch_.get((size_t)R * C_ * T, s);
  conv1d(h, mask, w_.ptr("down_blocks.0.2.weight"), w_.ptr("down_blocks.0.2.bias"), d, nullptr, R, C_, T, C_, 3, 1, conv_pad_, -1.f,
         s);
  h = d;
  for (int i = 0; i < n_mid_; ++i) h = group("mid_blocks." + std::to_string(i), h, C_, mask, temb, lens, R, T, streaming, s);
  const size_t n_cat = (size_t)R * 2 * C_ * T;
  float* cat = scratch_.get(n_cat, s);
  F32_LAUNCH(cat_channels_kernel, blocks(n_cat), 256, s, h, skip, cat, C_, C_, T, n_cat);
  h = group("up_blocks.0", cat, 2 * C_, mask, temb, lens, R, T, streaming, s);
  float* uo = scratch_.get((size_t)R * C_ * T, s);
  conv1d(h, mask, w_.ptr("up_blocks.0.2.weight"), w_.ptr("up_blocks.0.2.bias"), uo, nullptr, R, C_, T, C_, 3, 1, conv_pad_, -1.f,
         s);
  float* fb = causal_block("final_block", uo, C_, mask, nullptr, R, T, s);
  conv1d(fb, mask, w_.ptr("final_proj.weight"), w_.ptr("final_proj.bias"), out, mask, R, C_, T, F, 1, 1, 0, -1.f, s);
}

void FlowEngineF32::estimator_forward(const float* x, const float* mask, const float* mu, const float* t, const float* spks,
                                      const float* cond, float* out, int rows, int T, bool streaming, cudaStream_t s) {
  require(rows > 0 && T > 0, "rows and T must be positive");
  LS_CUDA(cudaSetDevice(device_));
  scratch_.reset();
  // out may alias x: compute into scratch, then copy
  float* tmp = scratch_.get((size_t)rows * feat_ * T, s);
  run(x, mask, mu, t, spks, cond, tmp, rows, T, streaming, s);
  LS_CUDA(cudaMemcpyAsync(out, tmp, (size_t)rows * feat_ * T * sizeof(float), cudaMemcpyDeviceToDevice, s));
}

// CausalConditionalCFM.forward + ConditionalCFM.solve_euler (flow_matching.py:323-348, 74-126), B >= 1
void FlowEngineF32::solve(const float* mu, const float* mask, const float* spks, const float* cond, const float* noise,
                          long long noise_stride, const float* t_span, int n_steps, float temperature, float cfg_rate,
                          bool streaming, float* out, int B, int T, cudaStream_t s) {
  require(B > 0 && T > 0 && n_steps > 0, "B, T and n_timesteps must be positive");
  require(noise_stride >= T, "noise buffer shorter than T");
  LS_CUDA(cudaSetDevice(device_));
  const int F = feat_;
  const size_t n = (size_t)B * F * T;
  float t = t_span[0], dt = t_span[1] - t_span[0];
  // persistent state across steps lives at the bottom of the scratch block of the first step; to keep it simple the
  // state is kept in `out` (fp32 [B,80,T]) itself
  scratch_.reset();
  F32_LAUNCH(init_noise_kernel, blocks(n), 256, s, noise, noise_stride, temperature, out, F, T, n);
  for (int step = 1; step <= n_steps; ++step) {
    scratch_.reset();
    float* x2 = scratch_.get(2 * n, s);
    float* mu2 = scratch_.get(2 * n, s);
    float* cond2 = scratch_.get(2 * n, s);
    float* mask2 = scratch_.get((size_t)2 * B * T, s);
    float* spks2 = scratch_.get((size_t)2 * B * F, s);
    float* t2 = scratch_.get((size_t)2 * B, s);
    float* v = scratch_.get(2 * n, s);
    F32_LAUNCH(cfg_pack_kernel, blocks(n > (size_t)B * T ? n : (size_t)B * T), 256, s, out, mu, cond, mask, x2, mu2, cond2, mask2,
               F, T, B);
    F32_LAUNCH(cfg_small_kernel, blocks((size_t)B * F + 2 * B), 256, s, spks, spks2, t2, t, F, B);
    run(x2, mask2, mu2, t2, spks2, cond2, v, 2 * B, T, streaming, s);
    F32_LAUNCH(euler_kernel, blocks(n), 256, s, out, v, dt, cfg_rate, n);
    t = t + dt;
    if (step < n_steps) dt = t_span[step + 1] - t;
  }
  F32_LAUNCH(mul_mask_kernel, blocks(n), 256, s, out, mask, out, F, T, n);  // API: zero where mask == 0
}

// ---------------------------------------------------------------------------------------------- DAC-VAE decoder
DacEngineF32::DacEngineF32(const Weights& w, int device) : device_(device) {
  LS_CUDA(cudaSetDevice(device));
  // fold weight-norm (layers.py:9-14): w = g * v / ||v||, norm over all dims but 0 (dim 0 = Cin for ConvTranspose1d)
  for (const auto& kv : w.all()) {
    const std::string& name = kv.first;
    const ls_tensor& t = *kv.second;
    size_t n = 1;
    std::vector<long long> shape;
    for (int i = 0; i < t.ndim; ++i) n *= (size_t)t.shape[i], shape.push_back(t.shape[i]);
    const std::string suf_v = ".weight_v";
    if (name.size() > suf_v.size() && name.compare(name.size() - suf_v.size(), suf_v.size(), suf_v) == 0) {
      const std::string base = name.substr(0, name.size() - suf_v.size());
      const ls_tensor& g = w.get(base + ".weight_g");
      const size_t d0 = (size_t)t.shape[0], inner = n / d0;
      std::vector<float> folded(n);
      for (size_t i = 0; i < d0; ++i) {
        double ss = 0.0;
        for (size_t j = 0; j < inner; ++j) ss += (double)t.data[i * inner + j] * t.data[i * inner + j];
        const float scale = g.data[i] / (float)std::sqrt(ss);
        for (size_t j = 0; j < inner; ++j) folded[i * inner + j] = t.data[i * inner + j] * scale;
      }
      w_.add(base + ".weight", folded.data(), n, shape);
    } else if (name.find(".weight_g") == std::string::npos) {
      w_.add(name, t.data, n, shape);
    }
  }
  if (w_.has("de_conv_pre.0.weight")) {
    latent_ = (int)w_.shape("de_conv_pre.0.weight")[1];
    while (w_.has("decoder.model." + std::to_string(rates_.size() + 1) + ".block.1.weight")) {
      const auto& sh = w_.shape("decoder.model." + std::to_string(rates_.size() + 1) + ".block.1.weight");
      rates_.push_back((int)sh[2] / 2);
    }
  }
  if (w_.has("en_conv_post.0.weight")) {
    latent_ = (int)w_.shape("en_conv_post.0.weight")[1];
    while (w_.has("encoder.block." + std::to_string(enc_rates_.size() + 1) + ".block.4.0.weight")) {
      const auto& sh = w_.shape("encoder.block." + std::to_string(enc_rates_.size() + 1) + ".block.4.0.weight");
      enc_rates_.push_back((int)sh[2] / 2);
    }
  }
  require(!rates_.empty() || !enc_rates_.empty(), "fp32 DAC-VAE: neither decoder nor encoder weights found", LS_ERR_WEIGHTS);
  hop_ = 1;
  for (int r : (rates_.empty() ? enc_rates_ : rates_)) hop_ *= r;
}

// ResidualUnit (dac-vae/model.py:107-143): x + LReLU(conv1(snake(LReLU(conv7_dil(snake(x))))))
float* DacEngineF32::residual_unit(const std::string& u, const float* x, int B, int C, int len, int dil, cudaStream_t s) {
  const size_t n = (size_t)B * C * len;
  float* a = scratch_.get(n, s);
  F32_LAUNCH(snake_nct_kernel, blocks(n), 256, s, x, w_.ptr(u + ".0.alpha"), a, C, len, n);
  float* c7 = scratch_.get(n, s);
  conv1d(a, nullptr, w_.ptr(u + ".1.0.weight"), w_.ptr(u + ".1.0.bias"), c7, nullptr, B, C, len, C, 7, dil, 3 * dil, 0.1f, s);
  F32_LAUNCH(snake_nct_kernel, blocks(n), 256, s, c7, w_.ptr(u + ".2.alpha"), a, C, len, n);
  conv1d(a, nullptr, w_.ptr(u + ".3.0.weight"), w_.ptr(u + ".3.0.bias"), c7, nullptr, B, C, len, C, 1, 1, 0, 0.1f, s);
  float* xn = scratch_.get(n, s);
  ew(x, c7, xn, n, EW_ADD, s);
  return xn;
}

// DACVAE.encode (dac-vae/model.py:469-483) after Encoder (model.py:146-234); audio [B,1,S], S a multiple of the hop
void DacEngineF32::encode(const float* audio, const int* lengths, const float* noise, float* z, float* m, float* logs,
                          int B, int S, cudaStream_t s) {
  require(!enc_rates_.empty(), "this handle holds no encoder weights", LS_ERR_WEIGHTS);
  int hop = 1;
  for (int r : enc_rates_) hop *= r;
  require(B > 0 && S > 0 && S % hop == 0, "audio length must be a positive multiple of the hop (pad first, model.py:455-462)");
  LS_CUDA(cudaSetDevice(device_));
  scratch_.reset();
  if (!lengths) {
    encode_dense(audio, noise, z, m, logs, B, S, s);
    return;
  }
  // per-clip semantics: each clip is encoded alone at its own length (what a loop over the reference gives); the
  // noise rows and the outputs have row stride L, so the clip's noise is gathered and its outputs scattered
  const int L = S / hop;
  const size_t row = (size_t)latent_ * L;
  std::vector<int> h(B);
  LS_CUDA(cudaMemcpyAsync(h.data(), lengths, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, s));
  LS_CUDA(cudaStreamSynchronize(s));
  for (float* o : {z, m, logs}) LS_CUDA(cudaMemsetAsync(o, 0, (size_t)B * row * sizeof(float), s));
  for (int b = 0; b < B; ++b) {
    const int n = h[b] < L ? h[b] : L;
    if (n <= 0) continue;
    scratch_.reset();
    const size_t nd = (size_t)latent_ * n;
    float* nz = noise ? scratch_.get(nd, s) : nullptr;
    if (noise)
      LS_CUDA(cudaMemcpy2DAsync(nz, (size_t)n * 4, noise + b * row, (size_t)L * 4, (size_t)n * 4, latent_,
                                cudaMemcpyDeviceToDevice, s));
    float* zd = scratch_.get(nd, s);
    float* md = scratch_.get(nd, s);
    float* ld = scratch_.get(nd, s);
    encode_dense(audio + (size_t)b * S, nz, zd, md, ld, 1, n * hop, s);
    const float* src[3] = {zd, md, ld};
    float* dst[3] = {z, m, logs};
    for (int k = 0; k < 3; ++k)
      LS_CUDA(cudaMemcpy2DAsync(dst[k] + b * row, (size_t)L * 4, src[k], (size_t)n * 4, (size_t)n * 4, latent_,
                                cudaMemcpyDeviceToDevice, s));
  }
}

// audio [B,1,S] -> z, m, logs [B,latent,S/hop], all dense (the scratch memory is taken, not reset)
void DacEngineF32::encode_dense(const float* audio, const float* noise, float* z, float* m, float* logs, int B, int S,
                                cudaStream_t s) {
  int C = (int)w_.shape("encoder.block.0.0.weight")[0], len = S;
  float* x = scratch_.get((size_t)B * C * len, s);
  conv1d(audio, nullptr, w_.ptr("encoder.block.0.0.weight"), w_.ptr("encoder.block.0.0.bias"), x, nullptr, B, 1, len, C, 7, 1, 3,
         0.1f, s);
  const int dils[3] = {1, 3, 9};
  for (size_t i = 0; i < enc_rates_.size(); ++i) {
    const std::string p = "encoder.block." + std::to_string(i + 1) + ".block";
    for (int j = 0; j < 3; ++j) x = residual_unit(p + "." + std::to_string(j) + ".block", x, B, C, len, dils[j], s);
    const size_t n = (size_t)B * C * len;
    float* sn = scratch_.get(n, s);
    F32_LAUNCH(snake_nct_kernel, blocks(n), 256, s, x, w_.ptr(p + ".3.alpha"), sn, C, len, n);
    const int st = enc_rates_[i];
    float* d = scratch_.get((size_t)B * 2 * C * (len / st), s);
    conv1d(sn, nullptr, w_.ptr(p + ".4.0.weight"), w_.ptr(p + ".4.0.bias"), d, nullptr, B, C, len, 2 * C, 2 * st, 1, (st + 1) / 2,
           0.1f, s, st);
    x = d, C *= 2, len /= st;
  }
  const int nst = (int)enc_rates_.size();
  const size_t n = (size_t)B * C * len;
  float* sn = scratch_.get(n, s);
  F32_LAUNCH(snake_nct_kernel, blocks(n), 256, s, x, w_.ptr("encoder.block." + std::to_string(nst + 1) + ".alpha"), sn, C, len, n);
  const std::string fin = "encoder.block." + std::to_string(nst + 2) + ".0";
  float* y = scratch_.get((size_t)B * latent_ * len, s);
  conv1d(sn, nullptr, w_.ptr(fin + ".weight"), w_.ptr(fin + ".bias"), y, nullptr, B, C, len, latent_, 3, 1, 1, 0.1f, s);
  ew(y, nullptr, y, (size_t)B * latent_ * len, EW_LRELU001, s);
  float* post = scratch_.get((size_t)B * 2 * latent_ * len, s);
  conv1d(y, nullptr, w_.ptr("en_conv_post.0.weight"), w_.ptr("en_conv_post.0.bias"), post, nullptr, B, latent_, len, 2 * latent_,
         1, 1, 0, 0.1f, s);
  const size_t nz = (size_t)B * latent_ * len;
  F32_LAUNCH(reparam_kernel, blocks(nz), 256, s, post, noise, z, m, logs, latent_, len, nz);
}

// Decoder (dac-vae/model.py:326-379) after de_conv_pre (model.py:485-488); every Conv1d is followed by LeakyReLU(0.1)
// (the shadowing WNConv1d, model.py:509-514)
void DacEngineF32::decode_dense(const float* z, long long z_bstride, float* wav, long long wav_bstride, int B, int L,
                                int L_alloc, cudaStream_t s) {
  (void)L_alloc;
  auto W = [&](const std::string& p) { return w_.ptr(p + ".weight"); };
  auto Bv = [&](const std::string& p) { return w_.ptr(p + ".bias"); };
  // gather the batch into a dense [B,latent,L] buffer (rows of z may be longer than L)
  float* zin = scratch_.get((size_t)B * latent_ * L, s);
  for (int b = 0; b < B; ++b)
    LS_CUDA(cudaMemcpy2DAsync(zin + (size_t)b * latent_ * L, (size_t)L * 4, z + (size_t)b * z_bstride, (size_t)(z_bstride / latent_) * 4,
                              (size_t)L * 4, latent_, cudaMemcpyDeviceToDevice, s));
  int C = latent_;
  float* x = scratch_.get((size_t)B * C * L, s);
  conv1d(zin, nullptr, W("de_conv_pre.0"), Bv("de_conv_pre.0"), x, nullptr, B, C, L, C, 1, 1, 0, 0.1f, s);
  const int dim = (int)w_.shape("decoder.model.0.0.weight")[0];
  float* y = scratch_.get((size_t)B * dim * L, s);
  conv1d(x, nullptr, W("decoder.model.0.0"), Bv("decoder.model.0.0"), y, nullptr, B, C, L, dim, 7, 1, 3, 0.1f, s);
  x = y, C = dim;
  int len = L;
  for (size_t i = 0; i < rates_.size(); ++i) {
    const std::string p = "decoder.model." + std::to_string(i + 1) + ".block";
    const int st = rates_[i], Cout = C / 2, Lout = len * st;
    const size_t n_in = (size_t)B * C * len, n_out = (size_t)B * Cout * Lout;
    float* sn = scratch_.get(n_in, s);
    F32_LAUNCH(snake_nct_kernel, blocks(n_in), 256, s, x, w_.ptr(p + ".0.alpha"), sn, C, len, n_in);
    float* up = scratch_.get(n_out, s);
    F32_LAUNCH(convt1d_nct_kernel, grid_t(Lout, (Cout + kNB - 1) / kNB, B), kTB, s, sn, W(p + ".1"), Bv(p + ".1"), up, C, len, Cout,
               2 * st, st, (st + 1) / 2, Lout);
    x = up, C = Cout, len = Lout;
    const int dils[3] = {1, 3, 9};
    for (int j = 0; j < 3; ++j) x = residual_unit(p + "." + std::to_string(j + 2) + ".block", x, B, C, len, dils[j], s);
  }
  const int nst = (int)rates_.size();
  const size_t n_last = (size_t)B * C * len;
  float* sn = scratch_.get(n_last, s);
  F32_LAUNCH(snake_nct_kernel, blocks(n_last), 256, s, x, w_.ptr("decoder.model." + std::to_string(nst + 1) + ".alpha"), sn, C, len,
             n_last);
  const std::string fin = "decoder.model." + std::to_string(nst + 2) + ".0";
  float* fo = scratch_.get((size_t)B * len, s);
  conv1d(sn, nullptr, W(fin), Bv(fin), fo, nullptr, B, C, len, 1, 7, 1, 3, 0.1f, s);
  ew(fo, nullptr, fo, (size_t)B * len, EW_TANH, s);
  for (int b = 0; b < B; ++b)
    LS_CUDA(cudaMemcpyAsync(wav + (size_t)b * wav_bstride, fo + (size_t)b * len, (size_t)len * 4, cudaMemcpyDeviceToDevice, s));
}

void DacEngineF32::decode(const float* z, const int* lengths, float* wav, int B, int L, cudaStream_t s) {
  require(B > 0 && L > 0, "B and L must be positive");
  require(!rates_.empty(), "this handle holds no decoder weights", LS_ERR_WEIGHTS);
  LS_CUDA(cudaSetDevice(device_));
  scratch_.reset();
  if (!lengths) {
    decode_dense(z, (long long)latent_ * L, wav, (long long)L * hop_, B, L, L, s);
    return;
  }
  // per-utterance semantics: each item is decoded alone at its own length (what a loop over the reference gives)
  std::vector<int> h(B);
  LS_CUDA(cudaMemcpyAsync(h.data(), lengths, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, s));
  LS_CUDA(cudaStreamSynchronize(s));
  LS_CUDA(cudaMemsetAsync(wav, 0, (size_t)B * L * hop_ * sizeof(float), s));
  for (int b = 0; b < B; ++b) {
    const int n = h[b] < L ? h[b] : L;
    if (n <= 0) continue;
    scratch_.reset();
    decode_dense(z + (size_t)b * latent_ * L, (long long)latent_ * L, wav + (size_t)b * L * hop_, (long long)L * hop_, 1, n, L, s);
  }
}

// ---------------------------------------------------------------------------------------------- token -> mu (f-1)
FrontEngineF32::FrontEngineF32(const Weights& w, int device) : device_(device) {
  LS_CUDA(cudaSetDevice(device));
  upload_all(w, &w_);
  d_ = (int)w_.shape("input_embedding.weight")[1];
  vocab_ = (int)w_.shape("input_embedding.weight")[0];
  out_ = (int)w_.shape("encoder_proj.weight")[0];
  spk_ = (int)w_.shape("spk_embed_affine_layer.weight")[1];
  heads_ = (int)w_.shape("encoder.encoders.0.self_attn.pos_bias_u")[0];
  require(d_ == heads_ * 64, "fp32 token encoder: expected head dim 64", LS_ERR_UNSUPPORTED);
  while (w_.has("encoder.encoders." + std::to_string(n_blocks_) + ".norm_mha.weight")) ++n_blocks_;
  while (w_.has("encoder.up_encoders." + std::to_string(n_up_) + ".norm_mha.weight")) ++n_up_;
}

// ConformerEncoderLayer (normalize_before, no macaron, no conv module): x += attn(LN(x)); x += w_2(swish(w_1(LN(x))))
float* FrontEngineF32::layer(const std::string& p, float* x, const float* pe, int B, int T, int chunk, const int* lens,
                             cudaStream_t s) {
  const size_t n = (size_t)B * d_ * T;
  const int P = 2 * T - 1;
  float* nrm = scratch_.get(n, s);
  F32_LAUNCH(layernorm_nct_kernel, grid_t(T, 1, B), kTB, s, x, w_.ptr(p + ".norm_mha.weight"), w_.ptr(p + ".norm_mha.bias"), nrm, d_,
             T, 0, (const float*)nullptr, (const float*)nullptr);
  float* q = scratch_.get(n, s);
  float* k = scratch_.get(n, s);
  float* v = scratch_.get(n, s);
  const std::string a = p + ".self_attn";
  conv1d(nrm, nullptr, w_.ptr(a + ".linear_q.weight"), w_.ptr(a + ".linear_q.bias"), q, nullptr, B, d_, T, d_, 1, 1, 0, -1.f, s);
  conv1d(nrm, nullptr, w_.ptr(a + ".linear_k.weight"), w_.ptr(a + ".linear_k.bias"), k, nullptr, B, d_, T, d_, 1, 1, 0, -1.f, s);
  conv1d(nrm, nullptr, w_.ptr(a + ".linear_v.weight"), w_.ptr(a + ".linear_v.bias"), v, nullptr, B, d_, T, d_, 1, 1, 0, -1.f, s);
  float* pp = scratch_.get((size_t)P * d_, s);
  F32_LAUNCH(linear_rows_kernel, dim3((d_ + 127) / 128, P), 128, s, pe, w_.ptr(a + ".linear_pos.weight"), (const float*)nullptr, pp, P,
             d_, d_, 0, 0);
  float* att = scratch_.get(n, s);
  F32_LAUNCH(rel_attention_nct_kernel, grid_t(T, heads_, B), kTB, s, q, k, v, pp, w_.ptr(a + ".pos_bias_u"), w_.ptr(a + ".pos_bias_v"),
             att, heads_, T, T, chunk, lens);
  float* o = scratch_.get(n, s);
  conv1d(att, nullptr, w_.ptr(a + ".linear_out.weight"), w_.ptr(a + ".linear_out.bias"), o, nullptr, B, d_, T, d_, 1, 1, 0, -1.f, s);
  float* x1 = scratch_.get(n, s);
  ew(x, o, x1, n, EW_ADD, s);
  F32_LAUNCH(layernorm_nct_kernel, grid_t(T, 1, B), kTB, s, x1, w_.ptr(p + ".norm_ff.weight"), w_.ptr(p + ".norm_ff.bias"), nrm, d_, T,
             0, (const float*)nullptr, (const float*)nullptr);
  const int ff = (int)w_.shape(p + ".feed_forward.w_1.weight")[0];
  float* h = scratch_.get((size_t)B * ff * T, s);
  conv1d(nrm, nullptr, w_.ptr(p + ".feed_forward.w_1.weight"), w_.ptr(p + ".feed_forward.w_1.bias"), h, nullptr, B, d_, T, ff, 1, 1, 0,
         -1.f, s);
  ew(h, nullptr, h, (size_t)B * ff * T, EW_SILU, s);
  conv1d(h, nullptr, w_.ptr(p + ".feed_forward.w_2.weight"), w_.ptr(p + ".feed_forward.w_2.bias"), o, nullptr, B, ff, T, d_, 1, 1, 0,
         -1.f, s);
  float* x2 = scratch_.get(n, s);
  ew(x1, o, x2, n, EW_ADD, s);
  return x2;
}

// LinearNoSubsampling (subsampling.py:69-113) + the rel-pos encoding's input scale (embedding.py:268); pe = [2T-1][d]
float* FrontEngineF32::embed(const std::string& p, const float* x, int B, int T, float** pe, cudaStream_t s) {
  const size_t n = (size_t)B * d_ * T;
  float* y = scratch_.get(n, s);
  conv1d(x, nullptr, w_.ptr(p + ".out.0.weight"), w_.ptr(p + ".out.0.bias"), y, nullptr, B, d_, T, d_, 1, 1, 0, -1.f, s);
  float* z = scratch_.get(n, s);
  F32_LAUNCH(layernorm_nct_kernel, grid_t(T, 1, B), kTB, s, y, w_.ptr(p + ".out.1.weight"), w_.ptr(p + ".out.1.bias"), z, d_, T, 0,
             (const float*)nullptr, (const float*)nullptr);
  F32_LAUNCH(scale_kernel, blocks(n), 256, s, z, sqrtf((float)d_), n);
  *pe = scratch_.get((size_t)(2 * T - 1) * d_, s);
  F32_LAUNCH(rel_pos_emb_kernel, dim3((d_ / 2 + 127) / 128, 2 * T - 1), 128, s, *pe, T, d_);
  return z;
}

// CausalMaskedDiffWithXvec.inference front half (flow/flow.py:461-489), equal-length batch.  n_context > 0: the last
// n_context tokens are look-ahead context only (the finalize = False call, flow.py:482-489); streaming: block-causal
// attention with chunk_ tokens at 25 Hz and 2*chunk_ frames at 50 Hz.
void FrontEngineF32::encode(const long long* tokens, const float* embedding, float* mu, float* spks, int B, int T_all,
                            int n_context, bool streaming, const int* token_len, cudaStream_t s) {
  require(B > 0 && T_all - n_context > 0 && (n_context == 0 || n_context == 3), "B, T must be positive; context is 0 or 3 tokens");
  run(tokens, embedding, mu, spks, B, T_all, T_all - n_context, streaming, token_len, nullptr, s);
}

void FrontEngineF32::encode_sessions(const long long* tokens, const float* embedding, float* mu, float* spks, int B, int T_all,
                                     int T, const int* token_len, const int* n_context, bool streaming, cudaStream_t s) {
  require(B > 0 && T > 0 && T <= T_all && token_len && n_context, "B, T must be positive, T <= T_all, lengths given");
  run(tokens, embedding, mu, spks, B, T_all, T, streaming, token_len, n_context, s);
}

// T_all token rows per utterance in, T output tokens (2T frames) out; T_all > T: the rows past T are look-ahead context.
// n_context (session mode, with token_len): per-utterance context, see front_lens_kernel.
void FrontEngineF32::run(const long long* tokens, const float* embedding, float* mu, float* spks, int B, int T_all, int T,
                         bool streaming, const int* token_len, const int* n_context, cudaStream_t s) {
  LS_CUDA(cudaSetDevice(device_));
  scratch_.reset();
  // speaker embedding: normalise, project (flow.py:463, 469)
  float* en = scratch_.get((size_t)B * spk_, s);
  F32_LAUNCH(normalize_rows_kernel, B, 128, s, embedding, en, spk_);
  F32_LAUNCH(linear_rows_kernel, dim3((out_ + 127) / 128, B), 128, s, en, w_.ptr("spk_embed_affine_layer.weight"),
             w_.ptr("spk_embed_affine_layer.bias"), spks, B, spk_, out_, 0, 0);
  const size_t n_all = (size_t)B * d_ * T_all, n = (size_t)B * d_ * T;
  float* x0 = scratch_.get(n_all, s);
  int *lens0 = nullptr, *lens1 = nullptr;
  if (token_len) {
    lens0 = reinterpret_cast<int*>(scratch_.get((size_t)2 * B + 8, s));
    lens1 = lens0 + B;
    F32_LAUNCH(front_lens_kernel, (B + 127) / 128, 128, s, token_len, n_context, lens0, lens1, B, T_all, T);
  }
  F32_LAUNCH(embed_tokens_kernel, blocks(n_all), 256, s, tokens, w_.ptr("input_embedding.weight"), x0, d_, T_all, vocab_, n_all,
             token_len);
  // embed (Linear, LayerNorm, scale) is position-independent: tokens and context go through it together
  float* pe_all = nullptr;
  float* xe = embed("encoder.embed", x0, B, T_all, &pe_all, s);
  // session mode: the rows past a session's tokens are the zeros F.pad feeds the pre-lookahead layer of a call alone
  // (the reference's padded batch embeds them instead: bias and LayerNorm make them non-zero)
  if (n_context) F32_LAUNCH(zero_tail_nct_kernel, blocks(n_all), 256, s, xe, token_len, d_, T_all, n_all);
  float* x = xe;
  float* pe = pe_all;
  if (T_all > T) {
    x = scratch_.get(n, s);
    F32_LAUNCH(slice_time_kernel, blocks(n), 256, s, xe, x, T_all, T, n);
    pe = scratch_.get((size_t)(2 * T - 1) * d_, s);
    F32_LAUNCH(rel_pos_emb_kernel, dim3((d_ / 2 + 127) / 128, 2 * T - 1), 128, s, pe, T, d_);
  }
  {  // PreLookaheadLayer (upsample_encoder.py:66-107): [x | context or 3 zeros] -> conv k=4 -> leaky_relu -> causal conv k=3, + x
    float* a = scratch_.get(n, s);
    conv1d(xe, nullptr, w_.ptr("encoder.pre_lookahead_layer.conv1.weight"), w_.ptr("encoder.pre_lookahead_layer.conv1.bias"), a,
           nullptr, B, d_, T_all, d_, 4, 1, 0, 0.01f, s, 1, T);
    float* c = scratch_.get(n, s);
    conv1d(a, nullptr, w_.ptr("encoder.pre_lookahead_layer.conv2.weight"), w_.ptr("encoder.pre_lookahead_layer.conv2.bias"), c,
           nullptr, B, d_, T, d_, 3, 1, 2, -1.f, s);
    float* r = scratch_.get(n, s);
    ew(c, x, r, n, EW_ADD, s);
    x = r;
  }
  const int chunk = streaming ? chunk_ : 0;
  for (int i = 0; i < n_blocks_; ++i) x = layer("encoder.encoders." + std::to_string(i), x, pe, B, T, chunk, lens0, s);
  // Upsample1D (upsample_encoder.py:37-63): nearest x2, left-pad 4, conv k=5
  const int T2 = 2 * T;
  const size_t n2 = (size_t)B * d_ * T2;
  float* up = scratch_.get(n2, s);
  F32_LAUNCH(upsample2_nct_kernel, blocks(n2), 256, s, x, up, T, n2);
  float* uc = scratch_.get(n2, s);
  conv1d(up, nullptr, w_.ptr("encoder.up_layer.conv.weight"), w_.ptr("encoder.up_layer.conv.bias"), uc, nullptr, B, d_, T2, d_, 5, 1, 4,
         -1.f, s);
  x = embed("encoder.up_embed", uc, B, T2, &pe, s);
  for (int i = 0; i < n_up_; ++i) x = layer("encoder.up_encoders." + std::to_string(i), x, pe, B, T2, 2 * chunk, lens1, s);
  float* an = scratch_.get(n2, s);
  F32_LAUNCH(layernorm_nct_kernel, grid_t(T2, 1, B), kTB, s, x, w_.ptr("encoder.after_norm.weight"), w_.ptr("encoder.after_norm.bias"),
             an, d_, T2, 0, (const float*)nullptr, (const float*)nullptr);
  conv1d(an, nullptr, w_.ptr("encoder_proj.weight"), w_.ptr("encoder_proj.bias"), mu, nullptr, B, d_, T2, out_, 1, 1, 0, -1.f, s);
  if (lens1) F32_LAUNCH(zero_tail_nct_kernel, blocks((size_t)B * out_ * T2), 256, s, mu, lens1, out_, T2, (size_t)B * out_ * T2);
}

// ---------------------------------------------------------------------------------------------- speaker encoder (f-4)
SpeakerEngineF32::SpeakerEngineF32(const Weights& w, int device) : device_(device) {
  LS_CUDA(cudaSetDevice(device));
  upload_all(w, &w_);
  mel_ = (int)w_.shape("init.weight")[1];
  d_ = (int)w_.shape("init.weight")[0];
  out_ = (int)w_.shape("output_proj.weight")[0];
  require(d_ == heads_ * 64 && d_ % groups_ == 0, "fp32 speaker encoder: expected 8 heads of 64 channels", LS_ERR_UNSUPPORTED);
  while (w_.has("attn." + std::to_string(n_blocks_) + ".norm.weight")) ++n_blocks_;
}

// LearnableSpeakerEncoder.forward (llm.py:70-96): init conv -> AttentionBlocks (x + proj_out(attn(qkv(GroupNorm(x))))) ->
// first frame -> output_proj -> L2 normalise.  n_refs > 1: mel is [n_refs][B,mel,T]; the embeddings are averaged and
// normalised again (CausalMaskedDiffWithXvec.get_speaker_embedding, flow.py:336-366).
void SpeakerEngineF32::encode(const float* mel, float* emb, int B, int T, int n_refs, cudaStream_t s) {
  require(B > 0 && T > 0 && n_refs > 0, "B, T, n_refs must be positive");
  LS_CUDA(cudaSetDevice(device_));
  scratch_.reset();
  const int R = B * n_refs;  // every clip is an independent row of the batch
  const size_t n = (size_t)R * d_ * T;
  float* h = scratch_.get(n, s);
  conv1d(mel, nullptr, w_.ptr("init.weight"), w_.ptr("init.bias"), h, nullptr, R, mel_, T, d_, 1, 1, 0, -1.f, s);
  float* nrm = scratch_.get(n, s);
  float* qkv = scratch_.get(3 * n, s);
  float* att = scratch_.get(n, s);
  float* prj = scratch_.get(n, s);
  float* h2 = scratch_.get(n, s);
  for (int i = 0; i < n_blocks_; ++i) {
    const std::string p = "attn." + std::to_string(i);
    F32_LAUNCH(group_norm_nct_kernel, dim3(groups_, R), 256, s, h, w_.ptr(p + ".norm.weight"), w_.ptr(p + ".norm.bias"), nrm, d_, T,
               groups_);
    conv1d(nrm, nullptr, w_.ptr(p + ".qkv.weight"), w_.ptr(p + ".qkv.bias"), qkv, nullptr, R, d_, T, 3 * d_, 1, 1, 0, -1.f, s);
    F32_LAUNCH(qkv_legacy_attention_kernel, grid_t(T, heads_, R), kTB, s, qkv, att, heads_, T);
    conv1d(att, nullptr, w_.ptr(p + ".proj_out.weight"), w_.ptr(p + ".proj_out.bias"), prj, nullptr, R, d_, T, d_, 1, 1, 0, -1.f, s);
    ew(h, prj, h2, n, EW_ADD, s);
    std::swap(h, h2);
  }
  float* pooled = scratch_.get((size_t)R * d_, s);
  F32_LAUNCH(first_frame_kernel, blocks((size_t)R * d_), 256, s, h, pooled, T, (size_t)R * d_);
  float* proj = scratch_.get((size_t)R * out_, s);
  F32_LAUNCH(linear_rows_kernel, dim3((out_ + 127) / 128, R), 128, s, pooled, w_.ptr("output_proj.weight"), w_.ptr("output_proj.bias"),
             proj, R, d_, out_, 0, 0);
  if (n_refs == 1) {
    F32_LAUNCH(normalize_rows_kernel, R, 128, s, proj, emb, out_);
    return;
  }
  float* each = scratch_.get((size_t)R * out_, s);
  F32_LAUNCH(normalize_rows_kernel, R, 128, s, proj, each, out_);
  float* avg = scratch_.get((size_t)B * out_, s);
  F32_LAUNCH(mean_stack_kernel, blocks((size_t)B * out_), 256, s, each, avg, n_refs, (size_t)B * out_);
  F32_LAUNCH(normalize_rows_kernel, B, 128, s, avg, emb, out_);
}

// ---------------------------------------------------------------------------------------------- S3 tokenizer (f-4)
S3EngineF32::S3EngineF32(const Weights& w, int device) : device_(device) {
  LS_CUDA(cudaSetDevice(device));
  upload_all(w, &w_);
  mels_ = (int)w_.shape("encoder.conv1.weight")[1];
  d_ = (int)w_.shape("encoder.conv1.weight")[0];
  require(d_ % 64 == 0, "S3 tokenizer: n_audio_state must be a multiple of the 64-wide heads", LS_ERR_UNSUPPORTED);
  heads_ = d_ / 64;
  ksize_ = (int)w_.shape("encoder.blocks.0.attn.fsmn_block.weight")[2];
  while (w_.has("encoder.blocks." + std::to_string(n_blocks_) + ".attn.query.weight")) ++n_blocks_;
  require(w_.shape("quantizer._codebook.project_down.weight")[0] == 8, "S3 tokenizer: FSQ head must project to 8 dims",
          LS_ERR_UNSUPPORTED);
  // rotary table [len][32]: "rotary.cos" / "rotary.sin" when the caller supplies them (the Python module builds them with
  // the reference's own torch expressions), else precompute_freqs_cis(64, 2048) restated in double precision
  if (w_.has("rotary.cos") && w_.has("rotary.sin")) {
    table_len_ = (int)w_.shape("rotary.cos")[0];
    require(w_.shape("rotary.cos")[1] == 32 && w_.shape("rotary.sin")[0] == table_len_, "S3 tokenizer: rotary tables must be [len][32]");
  } else {
    table_len_ = 2048;
    std::vector<float> c((size_t)table_len_ * 32), sn((size_t)table_len_ * 32);
    for (int d = 0; d < 32; ++d) {
      const float inv = 1.0f / (float)std::pow(10000.0, (double)(2 * d) / 64.0);
      for (int t = 0; t < table_len_; ++t) {
        const float ang = (float)t * inv;
        c[(size_t)t * 32 + d] = (float)std::cos((double)ang), sn[(size_t)t * 32 + d] = (float)std::sin((double)ang);
      }
    }
    w_.add("rotary.cos", c.data(), c.size(), {table_len_, 32});
    w_.add("rotary.sin", sn.data(), sn.size(), {table_len_, 32});
  }
}

void S3EngineF32::code_frames(int T, int* T1, int* T2) {
  *T1 = (T - 1) / 2 + 1;
  *T2 = (*T1 - 1) / 2 + 1;
}

// S3TokenizerV2.quantize for clips of at most 30 s (model_v2.py:386-415) = AudioEncoderV2.forward (:320-351) + FSQ head
void S3EngineF32::quantize(const float* mel, const int* mel_len, int* codes, int* code_len, float* hidden_out, int B, int T,
                           cudaStream_t s) {
  require(B > 0 && T > 0, "B and T must be positive");
  require(T <= 3000, "S3 tokenizer: clips longer than 30 s (3000 mel frames) take the reference's sliding-window path, "
                     "which is not built", LS_ERR_UNSUPPORTED);
  LS_CUDA(cudaSetDevice(device_));
  scratch_.reset();
  int T1, T2;
  code_frames(T, &T1, &T2);
  require(T2 <= table_len_, "S3 tokenizer: rotary table too short");
  int* l1 = reinterpret_cast<int*>(scratch_.get((size_t)B, s));
  float* m0 = scratch_.get((size_t)B * T, s);
  float* m1 = scratch_.get((size_t)B * T1, s);
  float* m2 = scratch_.get((size_t)B * T2, s);
  F32_LAUNCH(s3_lens_kernel, B, 256, s, mel_len, l1, code_len, m0, m1, m2, T, T1, T2);
  const size_t n1 = (size_t)B * d_ * T1, n = (size_t)B * d_ * T2;
  float* c1 = scratch_.get(n1, s);
  conv1d(mel, m0, w_.ptr("encoder.conv1.weight"), w_.ptr("encoder.conv1.bias"), c1, nullptr, B, mels_, T, d_, 3, 1, 1, -1.f, s, 2, T1);
  float* g1 = scratch_.get(n1, s);
  ew(c1, nullptr, g1, n1, EW_GELU, s);
  float* c2 = scratch_.get(n, s);
  conv1d(g1, m1, w_.ptr("encoder.conv2.weight"), w_.ptr("encoder.conv2.bias"), c2, nullptr, B, d_, T1, d_, 3, 1, 1, -1.f, s, 2, T2);
  float* x = scratch_.get(n, s);
  ew(c2, nullptr, x, n, EW_GELU, s);
  float* nrm = scratch_.get(n, s);
  float* q = scratch_.get(n, s);
  float* k = scratch_.get(n, s);
  float* v = scratch_.get(n, s);
  float* mem = scratch_.get(n, s);
  float* att = scratch_.get(n, s);
  float* prj = scratch_.get(n, s);
  float* x1 = scratch_.get(n, s);
  float* h1 = scratch_.get(4 * n, s);
  float* h2 = scratch_.get(4 * n, s);
  const size_t n_pairs = (size_t)B * heads_ * 32 * T2;
  for (int i = 0; i < n_blocks_; ++i) {
    const std::string p = "encoder.blocks." + std::to_string(i);
    F32_LAUNCH(layernorm_nct_kernel, grid_t(T2, 1, B), kTB, s, x, w_.ptr(p + ".attn_ln.weight"), w_.ptr(p + ".attn_ln.bias"), nrm, d_,
               T2, 0, (const float*)nullptr, (const float*)nullptr, 1e-6f);
    conv1d(nrm, nullptr, w_.ptr(p + ".attn.query.weight"), w_.ptr(p + ".attn.query.bias"), q, nullptr, B, d_, T2, d_, 1, 1, 0, -1.f, s);
    conv1d(nrm, nullptr, w_.ptr(p + ".attn.key.weight"), nullptr, k, nullptr, B, d_, T2, d_, 1, 1, 0, -1.f, s);
    conv1d(nrm, nullptr, w_.ptr(p + ".attn.value.weight"), w_.ptr(p + ".attn.value.bias"), v, nullptr, B, d_, T2, d_, 1, 1, 0, -1.f, s);
    F32_LAUNCH(rotary_nct_kernel, blocks(n_pairs), 256, s, q, w_.ptr("rotary.cos"), w_.ptr("rotary.sin"), heads_, T2, n_pairs);
    F32_LAUNCH(rotary_nct_kernel, blocks(n_pairs), 256, s, k, w_.ptr("rotary.cos"), w_.ptr("rotary.sin"), heads_, T2, n_pairs);
    F32_LAUNCH(fsmn_nct_kernel, grid_t(T2, d_, B), kTB, s, v, m2, w_.ptr(p + ".attn.fsmn_block.weight"), mem, d_, T2, ksize_);
    // q and k each carry 64^-1/4 in the reference (model_v2.py:198,210,213): 1/8 on the scores; keys past the clip's
    // length get the -1e10 bias of mask_to_bias, i.e. weight exactly 0 after the softmax
    F32_LAUNCH(attention_nct_kernel, grid_t(T2, heads_, B), kTB, s, q, k, v, att, code_len, heads_, T2, 0, 0.125f);
    conv1d(att, nullptr, w_.ptr(p + ".attn.out.weight"), w_.ptr(p + ".attn.out.bias"), prj, nullptr, B, d_, T2, d_, 1, 1, 0, -1.f, s);
    ew(prj, mem, att, n, EW_ADD, s);
    ew(x, att, x1, n, EW_ADD, s);
    F32_LAUNCH(layernorm_nct_kernel, grid_t(T2, 1, B), kTB, s, x1, w_.ptr(p + ".mlp_ln.weight"), w_.ptr(p + ".mlp_ln.bias"), nrm, d_, T2,
               0, (const float*)nullptr, (const float*)nullptr, 1e-5f);
    conv1d(nrm, nullptr, w_.ptr(p + ".mlp.0.weight"), w_.ptr(p + ".mlp.0.bias"), h1, nullptr, B, d_, T2, 4 * d_, 1, 1, 0, -1.f, s);
    ew(h1, nullptr, h2, 4 * n, EW_GELU, s);
    conv1d(h2, nullptr, w_.ptr(p + ".mlp.2.weight"), w_.ptr(p + ".mlp.2.bias"), prj, nullptr, B, 4 * d_, T2, d_, 1, 1, 0, -1.f, s);
    ew(x1, prj, x, n, EW_ADD, s);
  }
  float* rows = hidden_out ? hidden_out : scratch_.get(n, s);
  F32_LAUNCH(nct_to_rows_kernel, blocks(n), 256, s, x, rows, d_, T2, n);
  LS_CUDA(launch_fsq_encode(rows, w_.ptr("quantizer._codebook.project_down.weight"), w_.ptr("quantizer._codebook.project_down.bias"),
                            codes, (long long)B * T2, d_, s));
}

}  // namespace ls
