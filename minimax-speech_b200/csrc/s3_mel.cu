// Log-mel front end of the S3 speech tokenizer: s3tokenizer/utils.py log_mel_spectrogram (the Whisper front end) over a
// right-padded batch of 16 kHz clips, each clip transformed as if it were alone.
//
//   frames = reflect-padded 400-sample windows every 160 samples (torch.stft center=True), the last one dropped
//   power  = |rDFT(hann_periodic(400) * frame)|^2                 201 bins
//   mel    = log10(max(filters @ power, 1e-10))                   filters [n_mels][201]
//   out    = (max(mel, max(mel over the clip) - 8) + 4) / 4        [n_mels][len / 160]
//
// Pass 1 (s3_mel_frames_kernel): one CTA per (clip, tile of kTile frames).  The tile's frames are gathered with reflect
// indices about the clip's own ends (so nothing past audio_len[b] is ever read), windowed into shared memory, and
// transformed by a direct DFT on the CUDA cores in fp32: thread k owns bin k for all frames of the tile (register
// blocking over frames), with twiddles from a 400-entry table of cos / sin(2 pi j / 400) computed in double and rounded
// once.  The dense filter product follows in the same CTA; log10 is taken in double and rounded once.
// Pass 2 (s3_mel_norm_kernel): one cluster of kNormCta CTAs per clip reduces the clip's maximum over its valid frames
// (through distributed shared memory: no scratch memory), then applies the floor and the affine map in place and writes
// zeros past mel_len[b].  Max is exact, so the reduction order does not change a bit.
//
// Every frame is computed by the same instruction sequence whatever its tile, grid or batch, so a clip's mel is bitwise
// the same alone or in any padded batch.  No allocation, no host synchronisation: the call can be captured in a graph.
#include <cooperative_groups.h>

#include "kernels.h"
#include "profiler.h"

namespace cg = cooperative_groups;

namespace ls {
namespace {

constexpr int kFft = 400, kHop = 160, kBins = kFft / 2 + 1, kPad = kFft / 2;
constexpr int kTile = 16;          // frames per pass-1 CTA
constexpr int kThreads = 256;      // pass-1 CTA: bins 0..200 in the DFT; (mel, half tile) pairs in the filter product
constexpr int kMaxMels = kThreads / 2;
constexpr int kPStride = 204;      // power row stride (floats)
constexpr int kKChunk = 32;        // filter-bank columns staged per step
constexpr int kFsStride = kMaxMels + 1;
constexpr int kSmemA = kTile * kPStride + kKChunk * kFsStride;  // power + filter chunk; the frames alias it first
static_assert(kSmemA >= kTile * kFft, "frame tile must fit the shared region it shares with the power rows");
constexpr int kNormCta = 8;        // pass-2 cluster size (portable)
constexpr int kNormThreads = 512;

__device__ __forceinline__ int clip_frames(const int* audio_len, int b, long long S) {
  const int n = audio_len[b];
  return (n >= kPad + 1 && (long long)n <= S) ? n / kHop : 0;  // invalid lengths: no frames
}

__global__ void __launch_bounds__(kThreads) s3_mel_frames_kernel(const float* __restrict__ audio,
                                                                 const int* __restrict__ audio_len,
                                                                 const float* __restrict__ filters, int n_mels,
                                                                 float* __restrict__ mel, long long S, int T_out) {
  __shared__ __align__(16) float sa[kSmemA];
  __shared__ float2 tw[kFft];
  __shared__ float win[kFft];
  const int b = blockIdx.y, tid = threadIdx.x;
  const int len = audio_len[b];
  const int T_b = clip_frames(audio_len, b, S);
  const int t0 = blockIdx.x * kTile;
  if (t0 >= T_b) return;  // frames past mel_len are written by pass 2

  for (int j = tid; j < kFft; j += kThreads) {
    double s, c;
    sincospi((double)j / (kFft / 2), &s, &c);  // 2 pi j / 400
    tw[j] = make_float2((float)c, (float)s);
    win[j] = (float)(0.5 - 0.5 * c);           // periodic Hann (torch.hann_window(400))
  }
  __syncthreads();

  // gather: frame t covers samples t*160 - 200 + j, reflected about 0 and len - 1
  const float* src = audio + (long long)b * S;
  for (int i = tid; i < kTile * kFft; i += kThreads) {
    const int f = i / kFft, j = i - f * kFft, t = t0 + f;
    float v = 0.f;
    if (t < T_b) {
      int p = t * kHop - kPad + j;
      p = p < 0 ? -p : (p >= len ? 2 * (len - 1) - p : p);
      v = src[p] * win[j];
    }
    sa[i] = v;
  }
  __syncthreads();

  // direct real DFT: bin k of every frame of the tile
  float re[kTile], im[kTile];
#pragma unroll
  for (int f = 0; f < kTile; ++f) re[f] = im[f] = 0.f;
  const int k = tid;
  if (k < kBins) {
    int idx = 0;  // (k * n) mod 400
#pragma unroll 2
    for (int n = 0; n < kFft; n += 4) {
      float2 w[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        w[u] = tw[idx];
        idx += k;
        idx = idx >= kFft ? idx - kFft : idx;
      }
#pragma unroll
      for (int f = 0; f < kTile; ++f) {
        const float4 x = *reinterpret_cast<const float4*>(&sa[f * kFft + n]);
        re[f] = fmaf(x.x, w[0].x, re[f]); im[f] = fmaf(x.x, w[0].y, im[f]);
        re[f] = fmaf(x.y, w[1].x, re[f]); im[f] = fmaf(x.y, w[1].y, im[f]);
        re[f] = fmaf(x.z, w[2].x, re[f]); im[f] = fmaf(x.z, w[2].y, im[f]);
        re[f] = fmaf(x.w, w[3].x, re[f]); im[f] = fmaf(x.w, w[3].y, im[f]);
      }
    }
  }
  __syncthreads();  // the frames are dead: the power rows and the filter chunks reuse their memory
  float* pw = sa;
  float* fs = sa + kTile * kPStride;
  if (k < kBins) {
#pragma unroll
    for (int f = 0; f < kTile; ++f) pw[f * kPStride + k] = fmaf(re[f], re[f], im[f] * im[f]);
  }

  // filter product: thread (m, g) accumulates mel m of frames g*8 .. g*8+7, over the bins in a fixed order
  constexpr int kHalf = kTile / 2;
  const int m = tid % kMaxMels, g = tid / kMaxMels;
  float acc[kHalf];
#pragma unroll
  for (int j = 0; j < kHalf; ++j) acc[j] = 0.f;
  for (int k0 = 0; k0 < kBins; k0 += kKChunk) {
    __syncthreads();
    for (int i = tid; i < kKChunk * n_mels; i += kThreads) {
      const int mm = i / kKChunk, kk = i - mm * kKChunk;
      fs[kk * kFsStride + mm] = k0 + kk < kBins ? __ldg(filters + mm * kBins + k0 + kk) : 0.f;
    }
    __syncthreads();
    if (m < n_mels) {
      const int kn = min(kKChunk, kBins - k0);
      for (int kk = 0; kk < kn; ++kk) {
        const float w = fs[kk * kFsStride + m];
#pragma unroll
        for (int j = 0; j < kHalf; ++j) acc[j] = fmaf(w, pw[(g * kHalf + j) * kPStride + k0 + kk], acc[j]);
      }
    }
  }
  if (m < n_mels) {
    float* dst = mel + ((long long)b * n_mels + m) * T_out;
#pragma unroll
    for (int j = 0; j < kHalf; ++j) {
      const int t = t0 + g * kHalf + j;
      const float e = acc[j] < 1e-10f ? 1e-10f : acc[j];  // (NaN propagates, as in torch.clamp)
      if (t < T_b) dst[t] = (float)log10((double)e);
    }
  }
}

__global__ void __cluster_dims__(kNormCta, 1, 1) __launch_bounds__(kNormThreads)
    s3_mel_norm_kernel(const int* __restrict__ audio_len, float* __restrict__ mel, int* __restrict__ mel_len, int n_mels,
                       long long S, int T_out) {
  __shared__ float red[kNormThreads / 32];
  __shared__ float cta_max;
  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank(), b = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int kWarps = kNormThreads / 32, kUnroll = 8;
  const int T_b = clip_frames(audio_len, b, S);
  float* base = mel + (long long)b * n_mels * T_out;

  // rows are dealt to the cluster's warps; a warp streams a row with kUnroll loads in flight per lane
  float mx = -INFINITY;
  for (int r = rank * kWarps + warp; r < n_mels; r += kNormCta * kWarps) {
    const float* row = base + (long long)r * T_out;
    for (int t = lane; t < T_b; t += 32 * kUnroll) {
      float v[kUnroll];
#pragma unroll
      for (int u = 0; u < kUnroll; ++u) v[u] = t + 32 * u < T_b ? row[t + 32 * u] : -INFINITY;
#pragma unroll
      for (int u = 0; u < kUnroll; ++u) mx = fmaxf(mx, v[u]);
    }
  }
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if (lane == 0) red[warp] = mx;
  __syncthreads();
  if (threadIdx.x == 0) {
    float v = red[0];
    for (int w = 1; w < kWarps; ++w) v = fmaxf(v, red[w]);
    cta_max = v;
  }
  cluster.sync();
  float M = -INFINITY;
  for (int r = 0; r < kNormCta; ++r) M = fmaxf(M, *cluster.map_shared_rank(&cta_max, r));
  cluster.sync();  // no CTA leaves (and frees its shared memory) while another one still reads it

  const float floor_v = M - 8.0f;
  for (int r = rank * kWarps + warp; r < n_mels; r += kNormCta * kWarps) {
    float* row = base + (long long)r * T_out;
    for (int t = lane; t < T_out; t += 32 * kUnroll) {
      float v[kUnroll];
#pragma unroll
      for (int u = 0; u < kUnroll; ++u) v[u] = t + 32 * u < T_b ? row[t + 32 * u] : 0.f;
#pragma unroll
      for (int u = 0; u < kUnroll; ++u) {
        const int tu = t + 32 * u;
        if (tu < T_out) row[tu] = tu < T_b ? (fmaxf(v[u], floor_v) + 4.0f) / 4.0f : 0.f;
      }
    }
  }
  if (rank == 0 && threadIdx.x == 0) mel_len[b] = T_b;
}

}  // namespace

cudaError_t launch_s3_log_mel(const float* audio, const int* audio_len, const float* filters, int n_mels, float* mel,
                              int* mel_len, int B, long long S, cudaStream_t s) {
  if (B <= 0 || B > 65535 || S < 0 || n_mels < 1 || n_mels > kMaxMels || S / kHop > (1LL << 30))
    return cudaErrorInvalidValue;
  const int T_out = (int)(S / kHop);
  const unsigned tiles = (unsigned)((T_out + kTile - 1) / kTile);
  if (tiles > 0) {
    const double frames = (double)B * T_out;  // upper bound: frames past each clip's length exit at once
    ProfScope prof(s, PK_ELEMENTWISE, frames * 2.0 * ((double)kFft * (2 * kBins) + (double)kBins * n_mels),
                   (double)B * S * 4.0 + frames * n_mels * 4.0);
    s3_mel_frames_kernel<<<dim3(tiles, B), kThreads, 0, s>>>(audio, audio_len, filters, n_mels, mel, S, T_out);
    count_launch();
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
  }
  ProfScope prof(s, PK_ELEMENTWISE, 0.0, (double)B * n_mels * T_out * 12.0);
  s3_mel_norm_kernel<<<dim3(kNormCta, B), kNormThreads, 0, s>>>(audio_len, mel, mel_len, n_mels, S, T_out);
  count_launch();
  return cudaGetLastError();
}

}  // namespace ls
