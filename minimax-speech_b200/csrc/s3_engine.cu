// S3 tokenizer engine, bf16x3 mode (see s3_engine.h): log-mel [B,n_mels,T] -> 25 Hz FSQ tokens.
//
// Launch plan per call (model_v2.py:320-351 AudioEncoderV2.forward, :252-287 ResidualAttentionBlock, :152-249
// FSMNMultiHeadAttention; oracle/restatement.py s3_encode):
//   s3x_pack_mel      mel -> split rows [2*T1][3*n_mels], frames past mel_len selected to zero
//   conv1             conv_gemm, 2 taps over the [T1][2 * 3*n_mels] view (fp32 out)
//   s3x_split (GELU)  -> split rows [2*T2][3C], rows past l1 zero (the second conv's zero padding / input mask)
//   conv2             conv_gemm, 2 taps over the [T2][2 * 3C] view (fp32 out), s3x_gelu -> residual stream x
//   per block:  s3x_ln_split (attn_ln, 1e-6) -> QKV conv_gemm [3C][3C] (fp32 out) -> s3x_rope_fsmn (rotary on q, k in
//               place; FSMN memory over the masked v; addend x + mem) -> s3x_attention (fp32 flash attention, split
//               output) -> out-proj conv_gemm (+ addend) -> x1 -> s3x_ln_split (mlp_ln, 1e-5) -> FF1 conv_gemm (fp32
//               out) -> s3x_split (GELU) -> FF2 conv_gemm (+ x1) -> x
//   launch_fsq_encode on the fp32 rows.
// A stride-2 convolution over time-major rows is a 2-tap convolution over the same memory viewed as [T/2][2C] (see
// dac_enc_engine.cu): with k - pad = 2q + r, tap q+1 multiplies view row t+q, channel block r, W'[q+1][n][r*C + c] =
// W[n][c][2q + r + 1] (q in {-1, 0}; zero where k falls outside [0, 3)).  Here C is the 3C split columns.
//
// Mixed lengths: every GEMM skips the 128-row tiles starting at or past its clip's valid length and zero-fills the rows
// past it in the tiles it computes, so rows past a clip's length hold zeros or stale data.  Nothing valid reads them:
// the split kernels that feed the convolutions SELECT zero past the length (so the convolutions' zero padding is the
// clip's own), the FSMN memory selects v to zero past the length, attention never visits keys at or past it, and every
// other step is row-local.  A clip's valid rows therefore come out bitwise equal to a call with that clip alone, whatever
// the padding holds (NaN included) and whatever a larger earlier call left in the workspace.
#include <algorithm>
#include <cmath>

#include "f32_path.h"
#include "ptx.cuh"
#include "s3_engine.h"

namespace ls {
namespace {

constexpr int kAttQ = 64;        // queries per attention CTA
constexpr int kAttK = 64;        // keys per shared-memory tile
constexpr int kAttLd = 68;       // padded row stride (floats) of the attention tiles
constexpr int kAttThreads = 256;
constexpr int kAttSmem = 4 * kAttQ * kAttLd * 4;

__device__ __forceinline__ void split3(float v, __nv_bfloat16& hi, __nv_bfloat16& lo) {
  hi = __float2bfloat16_rn(v);
  lo = __float2bfloat16_rn(v - __bfloat162float(hi));
}
__device__ __forceinline__ float gelu_exact(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752f)); }

// write the 4 values v[0..3] of columns [n, n+4) of a split row [hi | lo | hi] (row of 3N bf16)
__device__ __forceinline__ void store_split4(__nv_bfloat16* row, int N, int n, const float (&v)[4]) {
  __nv_bfloat16 h[4], l[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) split3(v[i], h[i], l[i]);
  uint2 hv, lv;
  hv.x = (uint32_t)__bfloat16_as_ushort(h[0]) | ((uint32_t)__bfloat16_as_ushort(h[1]) << 16);
  hv.y = (uint32_t)__bfloat16_as_ushort(h[2]) | ((uint32_t)__bfloat16_as_ushort(h[3]) << 16);
  lv.x = (uint32_t)__bfloat16_as_ushort(l[0]) | ((uint32_t)__bfloat16_as_ushort(l[1]) << 16);
  lv.y = (uint32_t)__bfloat16_as_ushort(l[2]) | ((uint32_t)__bfloat16_as_ushort(l[3]) << 16);
  *reinterpret_cast<uint2*>(row + n) = hv;
  *reinterpret_cast<uint2*>(row + N + n) = lv;
  *reinterpret_cast<uint2*>(row + 2 * N + n) = hv;
}

// lengths after the two stride-2 convs (model_v2.py:330-334), as s3_lens_kernel of the fp32 path
__global__ void s3x_lens_kernel(const int* __restrict__ mel_len, int* __restrict__ l1, int* __restrict__ l2, int B) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const int n1 = (mel_len[b] - 1) / 2 + 1;
  l1[b] = n1, l2[b] = (n1 - 1) / 2 + 1;
}

// mel fp32 [B][M][T] -> split rows out [B][Tp][3M] (Tp >= T even); frames t >= min(mel_len[b], T) are zero
__global__ void s3x_pack_mel_kernel(const float* __restrict__ mel, const int* __restrict__ mel_len,
                                    __nv_bfloat16* __restrict__ out, int M, int T, int Tp, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int c = (int)(i % M);
  const int t = (int)((i / M) % Tp);
  const int b = (int)(i / ((size_t)M * Tp));
  const int len = min(mel_len[b], T);
  const float v = t < len ? mel[((size_t)b * M + c) * T + t] : 0.f;
  __nv_bfloat16 hi, lo;
  split3(v, hi, lo);
  __nv_bfloat16* row = out + ((size_t)b * Tp + t) * 3 * M;
  row[c] = hi, row[M + c] = lo, row[2 * M + c] = hi;
}

// src fp32 [B][rows_src][N] -> (GELU ->) split rows dst [B][rows_dst][3N]; rows t >= min(lens[b], rows_src) are zero
__global__ void s3x_split_kernel(const float* __restrict__ src, const int* __restrict__ lens, __nv_bfloat16* __restrict__ dst,
                                 int N, int rows_src, int rows_dst, int gelu, size_t n4) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n4) return;
  const int n = (int)(i % (N / 4)) * 4;
  const int t = (int)((i / (N / 4)) % rows_dst);
  const int b = (int)(i / ((size_t)(N / 4) * rows_dst));
  float v[4] = {0.f, 0.f, 0.f, 0.f};
  if (t < min(lens[b], rows_src)) {
    const float4 s = *reinterpret_cast<const float4*>(src + ((size_t)b * rows_src + t) * N + n);
    v[0] = s.x, v[1] = s.y, v[2] = s.z, v[3] = s.w;
    if (gelu) {
#pragma unroll
      for (int k = 0; k < 4; ++k) v[k] = gelu_exact(v[k]);
    }
  }
  store_split4(dst + ((size_t)b * rows_dst + t) * 3 * N, N, n, v);
}

// in-place exact GELU (F.gelu, approximate="none") on fp32 x [n]
__global__ void s3x_gelu_kernel(float* __restrict__ x, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) x[i] = gelu_exact(x[i]);
}

// LayerNorm of one fp32 row [C] per warp (two passes: mean, centred variance, as layernorm_nct_kernel) -> split row [3C]
__global__ void s3x_ln_split_kernel(const float* __restrict__ x, const float* __restrict__ g, const float* __restrict__ be,
                                    __nv_bfloat16* __restrict__ out, int C, float eps, long long R) {
  const long long r = (long long)blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (r >= R) return;
  const float* xr = x + r * C;
  float s = 0.f;
  for (int c = lane * 4; c < C; c += 128) {
    const float4 v = *reinterpret_cast<const float4*>(xr + c);
    s += (v.x + v.y) + (v.z + v.w);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const float mean = s / (float)C;
  float q = 0.f;
  for (int c = lane * 4; c < C; c += 128) {
    const float4 v = *reinterpret_cast<const float4*>(xr + c);
    const float d0 = v.x - mean, d1 = v.y - mean, d2 = v.z - mean, d3 = v.w - mean;
    q = fmaf(d0, d0, q), q = fmaf(d1, d1, q), q = fmaf(d2, d2, q), q = fmaf(d3, d3, q);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
  const float rstd = 1.0f / sqrtf(q / (float)C + eps);
  __nv_bfloat16* orow = out + r * 3 * C;
  for (int c = lane * 4; c < C; c += 128) {
    const float4 v = *reinterpret_cast<const float4*>(xr + c);
    const float4 gg = *reinterpret_cast<const float4*>(g + c);
    const float4 bb = *reinterpret_cast<const float4*>(be + c);
    float y[4] = {(v.x - mean) * rstd * gg.x + bb.x, (v.y - mean) * rstd * gg.y + bb.y, (v.z - mean) * rstd * gg.z + bb.z,
                  (v.w - mean) * rstd * gg.w + bb.w};
    store_split4(orow, C, c, y);
  }
}

// One thread per (b, t, head, d < 32), on qkv fp32 [B][T][3C] (q | k | v column blocks):
//   rotary (model_v2.py:51-70) in place on the pairs (d, d+32) of q and k, angle index d, position t;
//   FSMN memory (forward_fsmn, model_v2.py:177-189) of channels c = h*64 + d and c + 32: vm = v selected to zero at
//   frames >= len, mem = (depthwise conv(vm) + vm)[t], zero at t >= len;
//   addend xm = x + mem (the out-projection's residual: x + out(o) + mem, oracle s3_encode).
__global__ void s3x_rope_fsmn_kernel(float* __restrict__ qkv, const float* __restrict__ x, const int* __restrict__ lens,
                                     const float* __restrict__ cs, const float* __restrict__ sn, const float* __restrict__ fw,
                                     float* __restrict__ xm, int T, int C, int K, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int H = C / 64;
  const int d = (int)(i % 32);
  const int h = (int)((i / 32) % H);
  const int t = (int)((i / ((size_t)32 * H)) % T);
  const int b = (int)(i / ((size_t)32 * H * T));
  const int len = min(lens[b], T);
  const size_t ld = (size_t)3 * C;
  float* row = qkv + ((size_t)b * T + t) * ld;
  const int c0 = h * 64 + d, c1 = c0 + 32;
  const float co = cs[(size_t)t * 32 + d], si = sn[(size_t)t * 32 + d];
#pragma unroll
  for (int part = 0; part < 2; ++part) {
    float* lo = row + part * C + c0;
    float* hi = row + part * C + c1;
    const float a = *lo, bb = *hi;
    *lo = a * co + (-bb) * si;
    *hi = bb * co + a * si;
  }
  const float* vb = qkv + (size_t)b * T * ld + 2 * C;
  const int left = (K - 1) / 2;
  float m0 = 0.f, m1 = 0.f;
  if (t < len) {
    float a0 = 0.f, a1 = 0.f;
    for (int k = 0; k < K; ++k) {
      const int tt = t + k - left;
      if (tt >= 0 && tt < len) {
        a0 = fmaf(vb[(size_t)tt * ld + c0], fw[(size_t)c0 * K + k], a0);
        a1 = fmaf(vb[(size_t)tt * ld + c1], fw[(size_t)c1 * K + k], a1);
      }
    }
    m0 = a0 + vb[(size_t)t * ld + c0];
    m1 = a1 + vb[(size_t)t * ld + c1];
  }
  const size_t o = ((size_t)b * T + t) * C;
  xm[o + c0] = x[o + c0] + m0;
  xm[o + c1] = x[o + c1] + m1;
}

// fp32 flash attention on the CUDA cores, time-major q / k / v (column blocks of qkv [B][T][3C], 64-wide heads) ->
// split rows out [B][T][3C].  CTA = 64 queries x one head x one clip, 256 threads as 16 x 16: thread (ty, tx) holds the
// scores of queries ty + 16i and keys tx + 16j (i, j < 4) and the output columns 4tx .. 4tx+3 of queries ty + 16i.  Key
// tiles of 64 in shared memory, online softmax; keys at or past lens[b] are never visited (the reference's -1e10 bias
// gives them weight exactly 0).  Every query sums its keys in the same order whatever the grid, batch or T.
__global__ void __launch_bounds__(kAttThreads) s3x_attention_kernel(const float* __restrict__ qkv, const int* __restrict__ lens,
                                                                    __nv_bfloat16* __restrict__ out, int T, int C, float scale) {
  extern __shared__ float att_smem[];
  float* Qs = att_smem;
  float* Ks = Qs + kAttQ * kAttLd;
  float* Vs = Ks + kAttK * kAttLd;
  float* Ps = Vs + kAttK * kAttLd;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int q0 = blockIdx.x * kAttQ, h = blockIdx.y, b = blockIdx.z;
  const size_t ld = (size_t)3 * C;
  const float* base = qkv + (size_t)b * T * ld + h * 64;
  int n_keys = lens[b];
  if (n_keys > T) n_keys = T;
  if (n_keys <= 0) n_keys = T;
  for (int it = tid; it < kAttQ * 16; it += kAttThreads) {
    const int r = it >> 4, c4 = (it & 15) * 4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (q0 + r < T) v = *reinterpret_cast<const float4*>(base + (size_t)(q0 + r) * ld + c4);
    *reinterpret_cast<float4*>(Qs + r * kAttLd + c4) = v;
  }
  float o[4][4], m[4], l[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    m[i] = -INFINITY, l[i] = 0.f;
#pragma unroll
    for (int c = 0; c < 4; ++c) o[i][c] = 0.f;
  }
  for (int k0 = 0; k0 < n_keys; k0 += kAttK) {
    __syncthreads();  // the previous tile's K / V / P have been consumed (and Q is in place)
    for (int it = tid; it < kAttK * 16; it += kAttThreads) {
      const int r = it >> 4, c4 = (it & 15) * 4;
      float4 kv = make_float4(0.f, 0.f, 0.f, 0.f), vv = kv;
      if (k0 + r < n_keys) {
        kv = *reinterpret_cast<const float4*>(base + (size_t)(k0 + r) * ld + C + c4);
        vv = *reinterpret_cast<const float4*>(base + (size_t)(k0 + r) * ld + 2 * C + c4);
      }
      *reinterpret_cast<float4*>(Ks + r * kAttLd + c4) = kv;
      *reinterpret_cast<float4*>(Vs + r * kAttLd + c4) = vv;
    }
    __syncthreads();
    float s[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) s[i][j] = 0.f;
#pragma unroll 4
    for (int d = 0; d < 64; d += 4) {
      float4 qv[4], kv[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) qv[i] = *reinterpret_cast<const float4*>(Qs + (ty + 16 * i) * kAttLd + d);
#pragma unroll
      for (int j = 0; j < 4; ++j) kv[j] = *reinterpret_cast<const float4*>(Ks + (tx + 16 * j) * kAttLd + d);
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float a = s[i][j];
          a = fmaf(qv[i].x, kv[j].x, a);
          a = fmaf(qv[i].y, kv[j].y, a);
          a = fmaf(qv[i].z, kv[j].z, a);
          a = fmaf(qv[i].w, kv[j].w, a);
          s[i][j] = a;
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float mx = -INFINITY;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        s[i][j] = k0 + tx + 16 * j < n_keys ? s[i][j] * scale : -INFINITY;
        mx = fmaxf(mx, s[i][j]);
      }
#pragma unroll
      for (int off = 8; off > 0; off >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
      const float m_new = fmaxf(m[i], mx);  // finite: every tile holds at least one visible key
      const float corr = expf(m[i] - m_new);  // exp(-inf) = 0 on the first tile
      float rs = 0.f;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float p = expf(s[i][j] - m_new);
        Ps[(ty + 16 * i) * kAttLd + tx + 16 * j] = p;
        rs += p;
      }
#pragma unroll
      for (int off = 8; off > 0; off >>= 1) rs += __shfl_xor_sync(0xffffffffu, rs, off);
      l[i] = l[i] * corr + rs;
      m[i] = m_new;
#pragma unroll
      for (int c = 0; c < 4; ++c) o[i][c] *= corr;
    }
    __syncthreads();
    const int kn = min(kAttK, n_keys - k0);
    for (int kk = 0; kk < kn; kk += 4) {
      float4 pv[4], vv[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) pv[i] = *reinterpret_cast<const float4*>(Ps + (ty + 16 * i) * kAttLd + kk);
#pragma unroll
      for (int u = 0; u < 4; ++u) vv[u] = *reinterpret_cast<const float4*>(Vs + (kk + u) * kAttLd + tx * 4);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float pp[4] = {pv[i].x, pv[i].y, pv[i].z, pv[i].w};
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          o[i][0] = fmaf(pp[u], vv[u].x, o[i][0]);
          o[i][1] = fmaf(pp[u], vv[u].y, o[i][1]);
          o[i][2] = fmaf(pp[u], vv[u].z, o[i][2]);
          o[i][3] = fmaf(pp[u], vv[u].w, o[i][3]);
        }
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int q = q0 + ty + 16 * i;
    if (q >= T) continue;
    const float inv = 1.0f / l[i];
    float y[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) y[c] = o[i][c] * inv;
    store_split4(out + ((size_t)b * T + q) * 3 * C, C, h * 64 + tx * 4, y);
  }
}

inline unsigned blocks256(size_t n) { return (unsigned)((n + 255) / 256); }
#define S3X_LAUNCH(kernel, grid, block, smem, stream, ...)  \
  do {                                                      \
    count_launch();                                         \
    kernel<<<grid, block, smem, stream>>>(__VA_ARGS__);     \
    LS_CUDA(cudaGetLastError());                            \
  } while (0)

// fp32 -> bf16 hi / lo on the host (round to nearest even, as __float2bfloat16_rn)
inline void split_host(float v, __nv_bfloat16* hi, __nv_bfloat16* lo) {
  *hi = __float2bfloat16(v);
  *lo = __float2bfloat16(v - __bfloat162float(*hi));
}

// linear weight [N][K] -> split rows [W_hi | W_hi | W_lo] of 3K, written at rows [row0, row0 + N) of a reserved [.][3K] matrix
void put_split_rows(__nv_bfloat16* dst, const ls_tensor& w, int row0, int K) {
  const int N = (int)w.shape[0];
  for (int n = 0; n < N; ++n) {
    __nv_bfloat16* r = dst + (size_t)(row0 + n) * 3 * K;
    for (int k = 0; k < K; ++k) {
      __nv_bfloat16 hi, lo;
      split_host(w.data[(size_t)n * K + k], &hi, &lo);
      r[k] = hi, r[K + k] = hi, r[2 * K + k] = lo;
    }
  }
}

PackedLinear pack_split_linear(Arena& a, const Weights& w, const std::string& name, int N, int K, bool bias) {
  const ls_tensor& t = w.get(name + ".weight", {N, K});
  PackedLinear pl;
  pl.N = N, pl.K = 3 * K, pl.taps = 1, pl.block_n = pick_block_n(N);
  pl.w_off = a.reserve((size_t)N * 3 * K * 2);
  put_split_rows(reinterpret_cast<__nv_bfloat16*>(a.host(pl.w_off)), t, 0, K);
  std::vector<float> bv(N, 0.f);
  if (bias) {
    const ls_tensor& bt = w.get(name + ".bias", {N});
    for (int n = 0; n < N; ++n) bv[n] = bt.data[n];
  }
  pl.bias_off = a.put_f32(bv.data(), N);
  pl.has_bias = true;
  return pl;
}

// Conv1d(k = 3, stride 2, pad 1) weight [N][C][3] -> 2-tap split form [2][N][2 * 3C] over the [T/2][2 * 3C] view of
// split rows: tap q+1, channel block r holds [hi | hi | lo] of W[:, :, 2q + r + 1] (zero for k = -1)
PackedLinear pack_split_down(Arena& a, const Weights& w, const std::string& name, int N, int C) {
  const ls_tensor& t = w.get(name + ".weight", {N, C, 3});
  const ls_tensor& bt = w.get(name + ".bias", {N});
  PackedLinear pl;
  pl.N = N, pl.K = 2 * 3 * C, pl.taps = 2, pl.block_n = pick_block_n(N);
  pl.w_off = a.reserve((size_t)2 * N * pl.K * 2);
  __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(a.host(pl.w_off));
  for (size_t i = 0; i < (size_t)2 * N * pl.K; ++i) dst[i] = __float2bfloat16(0.f);
  for (int q = -1; q <= 0; ++q)
    for (int r = 0; r < 2; ++r) {
      const int k = 2 * q + r + 1;
      if (k < 0) continue;
      for (int n = 0; n < N; ++n) {
        __nv_bfloat16* row = dst + ((size_t)(q + 1) * N + n) * pl.K + (size_t)r * 3 * C;
        for (int c = 0; c < C; ++c) {
          __nv_bfloat16 hi, lo;
          split_host(t.data[((size_t)n * C + c) * 3 + k], &hi, &lo);
          row[c] = hi, row[C + c] = hi, row[2 * C + c] = lo;
        }
      }
    }
  pl.bias_off = a.put_f32(bt.data, N);
  pl.has_bias = true;
  return pl;
}

}  // namespace

struct S3Engine::Plan {
  CUtensorMap mel;  // mel_s viewed [T1][2 * 3 n_mels]
  CUtensorMap c1;   // h_s viewed [T2][2 * 3C] (conv2 input)
  CUtensorMap a;    // a_s [T2][3C]
  CUtensorMap h;    // h_s [T2][12C]
};

S3Engine::~S3Engine() {
  if (ws_base_) cudaFree(ws_base_);
}

S3Engine::S3Engine(const Weights& w, int device) : device_(device) {
  LS_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  LS_CUDA(cudaGetDeviceProperties(&prop, device));
  require(prop.major == 10, "this library only runs on sm_100 (B200) devices", LS_ERR_UNSUPPORTED);
  num_sms_ = prop.multiProcessorCount;
  const ls_tensor& c1 = w.get("encoder.conv1.weight");
  require(c1.ndim == 3 && c1.shape[2] == 3, "S3 tokenizer: conv1 must be a k = 3 Conv1d", LS_ERR_WEIGHTS);
  d_ = (int)c1.shape[0], mels_ = (int)c1.shape[1];
  require(d_ % 64 == 0 && mels_ % 64 == 0,
          "S3 tokenizer bf16x3: n_audio_state and n_mels must be multiples of 64 (GEMM K blocks)", LS_ERR_UNSUPPORTED);
  heads_ = d_ / 64;
  ksize_ = (int)w.get("encoder.blocks.0.attn.fsmn_block.weight").shape[2];
  const ls_tensor& pd = w.get("quantizer._codebook.project_down.weight");
  require(pd.shape[0] == 8 && pd.shape[1] == d_, "S3 tokenizer: FSQ head must project to 8 dims", LS_ERR_UNSUPPORTED);
  conv1_ = pack_split_down(arena_, w, "encoder.conv1", d_, mels_);
  conv2_ = pack_split_down(arena_, w, "encoder.conv2", d_, d_);
  for (int i = 0; w.has("encoder.blocks." + std::to_string(i) + ".attn.query.weight"); ++i) {
    const std::string p = "encoder.blocks." + std::to_string(i);
    BlockW bw;
    {  // fused Q | K | V: [3C][3 * C], bias [q_b | 0 | v_b]
      const int C = d_;
      bw.qkv.N = 3 * C, bw.qkv.K = 3 * C, bw.qkv.taps = 1, bw.qkv.block_n = pick_block_n(3 * C);
      bw.qkv.w_off = arena_.reserve((size_t)3 * C * 3 * C * 2);
      __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(arena_.host(bw.qkv.w_off));
      put_split_rows(dst, w.get(p + ".attn.query.weight", {C, C}), 0, C);
      put_split_rows(dst, w.get(p + ".attn.key.weight", {C, C}), C, C);
      put_split_rows(dst, w.get(p + ".attn.value.weight", {C, C}), 2 * C, C);
      std::vector<float> bv((size_t)3 * C, 0.f);
      const ls_tensor& qb = w.get(p + ".attn.query.bias", {C});
      const ls_tensor& vb = w.get(p + ".attn.value.bias", {C});
      for (int n = 0; n < C; ++n) bv[n] = qb.data[n], bv[2 * C + n] = vb.data[n];
      bw.qkv.bias_off = arena_.put_f32(bv.data(), bv.size());
      bw.qkv.has_bias = true;
    }
    bw.out = pack_split_linear(arena_, w, p + ".attn.out", d_, d_, true);
    bw.ff1 = pack_split_linear(arena_, w, p + ".mlp.0", 4 * d_, d_, true);
    bw.ff2 = pack_split_linear(arena_, w, p + ".mlp.2", d_, 4 * d_, true);
    bw.ln1_g = arena_.put_f32(w.get(p + ".attn_ln.weight", {d_}).data, d_);
    bw.ln1_b = arena_.put_f32(w.get(p + ".attn_ln.bias", {d_}).data, d_);
    bw.ln2_g = arena_.put_f32(w.get(p + ".mlp_ln.weight", {d_}).data, d_);
    bw.ln2_b = arena_.put_f32(w.get(p + ".mlp_ln.bias", {d_}).data, d_);
    bw.fsmn = arena_.put_f32(w.get(p + ".attn.fsmn_block.weight", {d_, 1, ksize_}).data, (size_t)d_ * ksize_);
    blocks_.push_back(bw);
  }
  require(!blocks_.empty(), "S3 tokenizer: no encoder blocks", LS_ERR_WEIGHTS);
  fsq_w_ = arena_.put_f32(pd.data, (size_t)8 * d_);
  fsq_b_ = arena_.put_f32(w.get("quantizer._codebook.project_down.bias", {8}).data, 8);
  // rotary table [len][32], as S3EngineF32: the caller's "rotary.cos" / "rotary.sin", else precompute_freqs_cis(64, 2048)
  if (w.has("rotary.cos") && w.has("rotary.sin")) {
    const ls_tensor& c = w.get("rotary.cos");
    table_len_ = (int)c.shape[0];
    require(c.ndim == 2 && c.shape[1] == 32, "S3 tokenizer: rotary tables must be [len][32]");
    cos_ = arena_.put_f32(c.data, (size_t)table_len_ * 32);
    sin_ = arena_.put_f32(w.get("rotary.sin", {table_len_, 32}).data, (size_t)table_len_ * 32);
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
    cos_ = arena_.put_f32(c.data(), c.size());
    sin_ = arena_.put_f32(sn.data(), sn.size());
  }
  arena_.upload();
  finalize_linear(arena_, conv1_);
  finalize_linear(arena_, conv2_);
  for (auto& bw : blocks_)
    finalize_linear(arena_, bw.qkv), finalize_linear(arena_, bw.out), finalize_linear(arena_, bw.ff1), finalize_linear(arena_, bw.ff2);
  static std::atomic<unsigned long long> optin{0};
  LS_CUDA(smem_optin_once(optin, reinterpret_cast<const void*>(s3x_attention_kernel), kAttSmem));
}

S3Engine::Layout S3Engine::layout(int B, int T, int mels, int d) {
  int T1, T2;
  S3EngineF32::code_frames(T, &T1, &T2);
  Layout L;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    const size_t o = off;
    off = (off + bytes + 1023) & ~size_t(1023);
    return o;
  };
  const size_t b = (size_t)B;
  L.l1 = take(b * 4);
  L.mel_s = take(b * 2 * T1 * 3 * mels * 2);   // [B][2 T1][3 n_mels] bf16
  L.x = take(b * T2 * d * 4);
  L.a_s = take(b * T2 * 3 * d * 2);
  L.qkv = take(b * T2 * 3 * d * 4);
  L.xm = take(b * T2 * d * 4);
  L.x1 = take(b * T2 * d * 4);
  L.h = take(b * std::max((size_t)T1, (size_t)4 * T2) * d * 4);     // conv1 output [T1][C], then FF1 output [T2][4C]
  L.h_s = take(b * std::max((size_t)2 * T2 * 3, (size_t)T2 * 12) * d * 2);  // conv2 input [2 T2][3C], then [T2][12C]
  L.total = off;
  return L;
}

const S3Engine::Plan& S3Engine::plan_for(int B, int T, const Layout& L) {
  auto key = std::make_pair(B, T);
  auto it = plans_.find(key);
  if (it != plans_.end()) return *it->second;
  int T1, T2;
  S3EngineF32::code_frames(T, &T1, &T2);
  auto pl = std::make_unique<Plan>();
  const bool halo = conv_halo_enabled();
  auto mk = [&](CUtensorMap* m, size_t off, int C, long long rows, int taps) {
    require(make_act_map(m, ws_base_ + off, C, (int)rows, B, C, rows * C, halo ? conv_halo_box_rows(taps, 1) : 128),
            "cuTensorMapEncodeTiled failed for an activation buffer", LS_ERR_CUDA);
  };
  mk(&pl->mel, L.mel_s, 6 * mels_, T1, 2);
  mk(&pl->c1, L.h_s, 6 * d_, T2, 2);
  mk(&pl->a, L.a_s, 3 * d_, T2, 1);
  mk(&pl->h, L.h_s, 12 * d_, T2, 1);
  const Plan& ref = *pl;
  plans_[key] = std::move(pl);
  return ref;
}

// S3TokenizerV2.quantize for clips of at most 30 s (model_v2.py:386-415)
void S3Engine::quantize(const float* mel, const int* mel_len, int* codes, int* code_len, float* hidden_out, int B, int T,
                        cudaStream_t s) {
  require(B > 0 && T > 0, "B and T must be positive");
  require(T <= 3000, "S3 tokenizer: clips longer than 30 s (3000 mel frames) take the reference's sliding-window path, "
                     "which is not built", LS_ERR_UNSUPPORTED);
  LS_CUDA(cudaSetDevice(device_));
  int T1, T2;
  S3EngineF32::code_frames(T, &T1, &T2);
  require(T2 <= table_len_, "S3 tokenizer: rotary table too short");
  const Layout L = layout(B, T, mels_, d_);
  if (L.total > ws_bytes_) {
    ws_release(ws_base_, s);
    plans_.clear();
    ws_alloc(ws_base_, L.total, s);
    ws_bytes_ = L.total;
  }
  const Plan& pl = plan_for(B, T, L);
  auto f32 = [&](size_t off) { return arena_.ptr<float>(off); };
  const bool halo = conv_halo_enabled();
  const int C = d_;
  int* l1 = ws<int>(L.l1);
  float* x = ws<float>(L.x);
  float* qkv = ws<float>(L.qkv);
  float* xm = ws<float>(L.xm);
  float* x1 = ws<float>(L.x1);
  float* h = ws<float>(L.h);
  __nv_bfloat16* a_s = ws<__nv_bfloat16>(L.a_s);
  __nv_bfloat16* h_s = ws<__nv_bfloat16>(L.h_s);
  const size_t R = (size_t)B * T2;

  // one conv_gemm launch: rows M per clip, lengths = valid rows per clip (tiles past them skipped, rows past them zeroed)
  auto gemm = [&](const CUtensorMap& a, const PackedLinear& w, int M, const int* lens, void* out, const float* addend,
                  int zero_skipped) {
    ConvGemmParams p{};
    p.B = B, p.M = M, p.N = w.N, p.block_n = w.block_n;
    p.taps = w.taps, p.dil = 1, p.pad = w.taps == 2 ? 1 : 0;
    p.kb_per_tap = w.K / 64, p.kb_split = p.kb_per_tap;
    p.lengths = lens, p.m_len_mul = 1, p.m_len_add = 0, p.skip_halo = 0, p.zero_skipped = zero_skipped;
    p.bias = w.bias, p.chan_mod = w.N, p.n_store = w.N, p.act = ACT_NONE;
    if (addend) p.addend = addend, p.addend_dtype = OUT_F32;
    p.out0 = out, p.out0_dtype = OUT_F32, p.out1_mode = OUT1_NONE;
    p.out_ld = w.N, p.out_shift = 0, p.out_bstride = (long long)M * w.N, p.out_alloc = (long long)M * w.N;
    p.out_valid_mul = w.N;
    p.k_true = w.K, p.tag = 1, p.halo_mode = halo ? conv_halo_mode() : 0;
    LS_CUDA(launch_conv_gemm(a, a, w.map, p, num_sms_, s));
  };
  auto split = [&](const float* src, const int* lens, __nv_bfloat16* dst, int N, int rows_src, int rows_dst, int gelu) {
    const size_t n4 = (size_t)B * rows_dst * (N / 4);
    S3X_LAUNCH(s3x_split_kernel, blocks256(n4), 256, 0, s, src, lens, dst, N, rows_src, rows_dst, gelu, n4);
  };
  auto ln_split = [&](const float* in, size_t g, size_t b, float eps) {
    S3X_LAUNCH(s3x_ln_split_kernel, (unsigned)((R + 7) / 8), 256, 0, s, in, f32(g), f32(b), a_s, C, eps, (long long)R);
  };

  S3X_LAUNCH(s3x_lens_kernel, (unsigned)((B + 127) / 128), 128, 0, s, mel_len, l1, code_len, B);
  {
    const size_t n = (size_t)B * 2 * T1 * mels_;
    S3X_LAUNCH(s3x_pack_mel_kernel, blocks256(n), 256, 0, s, mel, mel_len, ws<__nv_bfloat16>(L.mel_s), mels_, T, 2 * T1, n);
  }
  gemm(pl.mel, conv1_, T1, l1, h, nullptr, 0);
  split(h, l1, h_s, C, T1, 2 * T2, 1);  // GELU, rows past l1 zero: conv2's input mask and zero padding
  gemm(pl.c1, conv2_, T2, code_len, x, nullptr, 0);
  S3X_LAUNCH(s3x_gelu_kernel, blocks256(R * C), 256, 0, s, x, R * C);
  for (size_t i = 0; i < blocks_.size(); ++i) {
    const BlockW& bw = blocks_[i];
    const bool last = i + 1 == blocks_.size();
    ln_split(x, bw.ln1_g, bw.ln1_b, 1e-6f);
    gemm(pl.a, bw.qkv, T2, code_len, qkv, nullptr, 0);
    {
      const size_t n = R * heads_ * 32;
      S3X_LAUNCH(s3x_rope_fsmn_kernel, blocks256(n), 256, 0, s, qkv, x, code_len, f32(cos_), f32(sin_), f32(bw.fsmn), xm, T2,
                 C, ksize_, n);
    }
    // q and k each carry 64^-1/4 in the reference (model_v2.py:198,210,213): 1/8 on the scores
    S3X_LAUNCH(s3x_attention_kernel, dim3((unsigned)((T2 + kAttQ - 1) / kAttQ), (unsigned)heads_, (unsigned)B), kAttThreads,
               kAttSmem, s, qkv, code_len, a_s, T2, C, 0.125f);
    gemm(pl.a, bw.out, T2, code_len, x1, xm, 0);
    ln_split(x1, bw.ln2_g, bw.ln2_b, 1e-5f);
    gemm(pl.a, bw.ff1, T2, code_len, h, nullptr, 0);
    split(h, code_len, h_s, 4 * C, T2, T2, 1);
    gemm(pl.h, bw.ff2, T2, code_len, x, x1, last ? 1 : 0);  // the last block zeroes every row past code_len
  }
  if (hidden_out) LS_CUDA(cudaMemcpyAsync(hidden_out, x, R * C * 4, cudaMemcpyDeviceToDevice, s));
  LS_CUDA(launch_fsq_encode(x, f32(fsq_w_), f32(fsq_b_), codes, (long long)R, C, s));
}

}  // namespace ls
