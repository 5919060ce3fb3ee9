// Sample-rate conversion of right-padded batches of clips (torchaudio.functional.resample at its defaults:
// sinc_interp_hann, lowpass_filter_width 6, rolloff 0.99) and the linear stretch of DAC latents that CosyVoice2's
// token2wav(speed) applies (F.interpolate(mode='linear', align_corners=False)).
//
// Resampling: with the ratio reduced to O / N, output sample j = q*N + p of a clip is
//   y[j] = sum_i x[q*O + i] k_p(i),   k_p(i) = sinc(pi t) cos^2(pi t / 12) base / O,   t = base (i/O - p/N),
// base = min(O, N) * 0.99, x read as zero outside the clip.  torchaudio convolves with every i in [-width, width + O)
// and clamps t to +-6; a tap with |t| >= 6 is the product of two values that are almost zero (<= 1.5e-49 in double, 0
// in fp32), so the table keeps only the taps with |t| < 6: one contiguous run of i per phase p.  The table is built
// once on the host in double (the operations in torchaudio's order) and every tap is rounded once to fp32.
//
// One CTA per (clip, tile of output samples): the tap table and the tile's input span (with its halo, zero outside
// the clip) are staged in shared memory, then each thread sums one output's taps in increasing i, in fp32 (the first
// product, then fma).  An output's value depends only on the table and the clip's samples, never on the tile, grid or
// batch, so a clip is bitwise the same alone or in any padded batch.  Samples at or past audio_len[b] are never read.
// No allocation, no host synchronisation: a call can be captured in a CUDA graph.
#include <algorithm>
#include <cmath>
#include <numeric>

#include "../../include/ls_b200.h"
#include "kernels.h"
#include "profiler.h"

namespace ls {
namespace {

constexpr int kRsThreads = 256;
constexpr double kLowpassWidth = 6.0, kRolloff = 0.99;

__global__ void __launch_bounds__(kRsThreads) resample_kernel(const float* __restrict__ audio,
                                                              const int* __restrict__ audio_len,
                                                              const float* __restrict__ taps, const int2* __restrict__ fc,
                                                              float* __restrict__ out, int* __restrict__ out_len, int O,
                                                              int N, int stride, int min_first, int tile, int span,
                                                              int S_in, int S_out) {
  extern __shared__ __align__(16) float rs_smem[];
  float* st = rs_smem;                 // [N][stride] taps
  float* xs = rs_smem + N * stride;    // [span] input samples of the tile
  const int b = blockIdx.y, tid = threadIdx.x;
  const int len_raw = audio_len[b];
  const int len = (len_raw >= 1 && len_raw <= S_in) ? len_raw : 0;  // invalid lengths: an empty clip
  const int n_out = (int)(((long long)N * len + O - 1) / O);
  if (blockIdx.x == 0 && tid == 0) out_len[b] = n_out;
  const int j0 = blockIdx.x * tile;
  const int j_end = min(j0 + tile, S_out);
  float* dst = out + (long long)b * S_out;
  if (j0 >= n_out) {  // past the clip: zeros only
    for (int j = j0 + tid; j < j_end; j += kRsThreads) dst[j] = 0.f;
    return;
  }
  for (int i = tid; i < N * stride; i += kRsThreads) st[i] = __ldg(taps + i);
  const long long lo = (long long)(j0 / N) * O + min_first;
  const float* src = audio + (long long)b * S_in;
  for (int s = tid; s < span; s += kRsThreads) {
    const long long idx = lo + s;
    xs[s] = (idx >= 0 && idx < len) ? src[idx] : 0.f;
  }
  __syncthreads();
  for (int j = j0 + tid; j < j_end; j += kRsThreads) {
    float acc = 0.f;
    if (j < n_out) {
      const int q = j / N, p = j - q * N;
      const int2 f = __ldg(fc + p);  // first i, tap count
      const float* w = st + p * stride;
      const float* x = xs + ((long long)q * O + f.x - lo);
      if (f.y > 0) {
        acc = w[0] * x[0];
        for (int k = 1; k < f.y; ++k) acc = fmaf(w[k], x[k], acc);
      }
    }
    dst[j] = acc;
  }
}

// Row (b, c) of z [B][C][L_in]: its first len_in[b] frames stretched to len_out[b] frames (PyTorch's upsample_linear1d
// with align_corners=False and no scale factor), zeros from len_out[b] to L_out.  Invalid lengths give a zero row.
// The source coordinate and the blend are computed in double, as PyTorch does for float64 tensors: an output is then
// F.interpolate in float64 rounded once.  (PyTorch's fp32 path computes the coordinate in fp32, which moves the blend
// weights by up to about 1e-5 on a 100-frame row: 3e-6 rel-L2 from float64 at 100 -> 125 frames.)
__global__ void __launch_bounds__(256) latent_resize_kernel(const float* __restrict__ z, const int* __restrict__ len_in,
                                                            const int* __restrict__ len_out, float* __restrict__ out, int C,
                                                            int L_in, int L_out) {
  const long long row = blockIdx.x;
  const int b = (int)(row / C);
  const int Li = len_in[b], Lo = len_out[b];
  const bool ok = Li >= 1 && Li <= L_in && Lo >= 1 && Lo <= L_out;
  const double scale = ok ? (double)Li / Lo : 0.0;
  const float* x = z + row * L_in;
  float* y = out + row * L_out;
  for (int d = blockIdx.y * blockDim.x + threadIdx.x; d < L_out; d += gridDim.y * blockDim.x) {
    float v = 0.f;
    if (ok && d < Lo) {
      const double src = fmax(scale * (d + 0.5) - 0.5, 0.0);
      const int i0 = min((int)src, Li - 1), i1 = min(i0 + 1, Li - 1);
      const double l1 = src - i0, l0 = 1.0 - l1;
      v = (float)(l0 * x[i0] + l1 * x[i1]);
    }
    y[d] = v;
  }
}

}  // namespace

int resample_table(int orig_freq, int new_freq, ResampleTable* t, bool fill) {
  if (orig_freq <= 0 || new_freq <= 0) return LS_ERR_INVALID;
  *t = ResampleTable{};
  if (orig_freq == new_freq) {  // a copy: one tap of 1 (torchaudio returns the input unchanged)
    t->O = t->N = 1, t->width = 0, t->max_taps = 1;
    if (fill) t->first = {0}, t->count = {1}, t->taps = {1.0f};
    return LS_OK;
  }
  const int g = std::gcd(orig_freq, new_freq);
  const int O = orig_freq / g, N = new_freq / g;
  const double base = (double)std::min(O, N) * kRolloff;
  t->O = O, t->N = N, t->width = (int)std::ceil(kLowpassWidth * O / base);
  // every window position of every phase is visited once: bound the work before the exact size is known (any table
  // within kResampleMaxTableBytes needs far fewer visits than this)
  if ((long long)N * (2LL * t->width + O) > (64LL << 20)) return LS_ERR_UNSUPPORTED;
  std::vector<int> first(N), count(N, 0);
  std::vector<std::vector<double>> rows(fill ? N : 0);
  for (int p = 0; p < N; ++p) {
    const double ph = -(double)p / N;
    for (int i = -t->width; i < t->width + O; ++i) {
      const double tt = (ph + (double)i / O) * base;  // torchaudio: (arange(0, -N, -1) / N + arange(-w, w + O) / O) * base
      if (!(std::fabs(tt) < kLowpassWidth)) continue;
      if (count[p]++ == 0) first[p] = i;
      if (fill) {
        const double w = std::cos(tt * M_PI / kLowpassWidth / 2);
        const double a = tt * M_PI;
        const double k = a == 0.0 ? 1.0 : std::sin(a) / a;
        rows[p].push_back(k * (w * w * (base / O)));
      }
    }
  }
  t->max_taps = *std::max_element(count.begin(), count.end());
  if (resample_table_bytes(*t) > kResampleMaxTableBytes) return LS_ERR_UNSUPPORTED;
  if (fill) {
    t->first = first, t->count = count;
    t->taps.assign((size_t)N * t->max_taps, 0.0f);
    for (int p = 0; p < N; ++p)
      for (int k = 0; k < count[p]; ++k) t->taps[(size_t)p * t->max_taps + k] = (float)rows[p][k];
  }
  return LS_OK;
}

int resample_plan(const ResampleTable& t, ResamplePlan* plan) {
  plan->O = t.O, plan->N = t.N, plan->stride = t.max_taps | 1;  // odd row stride: the phases of a warp hit different banks
  int lo = t.first[0], hi = t.first[0] + t.count[0];
  for (int p = 0; p < t.N; ++p) lo = std::min(lo, t.first[p]), hi = std::max(hi, t.first[p] + t.count[p]);
  plan->min_first = lo;
  auto span = [&](long long tile) { return ((tile - 1) / t.N + 1) * t.O + (hi - lo); };
  const long long table_bytes = 4LL * t.N * plan->stride;
  long long tile = 2048;
  while (tile > 32 && span(tile) * 4 > (64 << 10)) tile /= 2;
  // a large table is staged per CTA: give it more outputs to serve
  while (tile < 16384 && table_bytes > 4 * tile && span(2 * tile) * 4 <= (96 << 10)) tile *= 2;
  plan->tile = (int)tile, plan->span = (int)span(tile);
  plan->smem = (size_t)(table_bytes + 4LL * plan->span);
  return plan->smem <= kResampleMaxSmem ? LS_OK : LS_ERR_UNSUPPORTED;
}

cudaError_t launch_resample(const ResamplePlan& p, const float* audio, const int* audio_len, float* out, int* out_len, int B,
                            long long S_in, long long S_out, cudaStream_t s) {
  if (B <= 0 || B > 65535 || S_in < 1 || S_in > INT32_MAX || S_out > INT32_MAX ||
      S_out < ((long long)p.N * S_in + p.O - 1) / p.O)
    return cudaErrorInvalidValue;
  static std::atomic<unsigned long long> optin{0};
  if (cudaError_t e = smem_optin_once(optin, reinterpret_cast<const void*>(resample_kernel), (int)kResampleMaxSmem);
      e != cudaSuccess)
    return e;
  const long long tiles = (S_out + p.tile - 1) / p.tile;
  const double taps = (double)p.stride;  // (upper bound of the taps per output)
  ProfScope prof(s, PK_ELEMENTWISE, 2.0 * B * S_out * taps, 4.0 * B * (S_in + S_out));
  resample_kernel<<<dim3((unsigned)std::max(tiles, 1LL), B), kRsThreads, p.smem, s>>>(
      audio, audio_len, p.taps, p.fc, out, out_len, p.O, p.N, p.stride, p.min_first, p.tile, p.span, (int)S_in, (int)S_out);
  count_launch();
  return cudaGetLastError();
}

cudaError_t launch_latent_resize_linear(const float* z, const int* len_in, const int* len_out, float* out, int B, int C,
                                        int L_in, int L_out, cudaStream_t s) {
  if (B <= 0 || C <= 0 || L_in < 1 || L_out < 1) return cudaErrorInvalidValue;
  const long long rows = (long long)B * C;
  if (rows > INT32_MAX) return cudaErrorInvalidValue;
  ProfScope prof(s, PK_ELEMENTWISE, 4.0 * rows * L_out, 4.0 * rows * ((double)L_in + L_out));
  const unsigned gy = (unsigned)std::min<long long>((L_out + 255) / 256, 65535);
  latent_resize_kernel<<<dim3((unsigned)rows, gy), 256, 0, s>>>(z, len_in, len_out, out, C, L_in, L_out);
  count_launch();
  return cudaGetLastError();
}

}  // namespace ls
