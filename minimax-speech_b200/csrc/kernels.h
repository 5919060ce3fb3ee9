// Kernel-level interface shared by the engines (flow_engine.cu / dac_engine.cu) and the C-ABI test hooks.
#pragma once
#include <atomic>
#include <cstdint>
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <vector>

namespace ls {

extern std::atomic<long long> g_launch_count;  // kernels launched by this library
extern long long* g_debug_buffer;              // device buffer for kernel timelines (development aid), or nullptr
extern long long g_debug_bytes;
inline void count_launch() { g_launch_count.fetch_add(1, std::memory_order_relaxed); }

// Launch with programmatic dependent launch enabled: the kernel may start (up to its griddepcontrol.wait) while the
// previous kernel of the stream drains.  Only for kernels that execute pdl_wait() before touching global memory an
// earlier kernel wrote.  `cluster` > 1 adds a cluster dimension.  LS_NO_PDL=1 in the environment turns it off.
bool pdl_enabled();
bool conv_halo_enabled();
int conv_halo_mode();
bool conv_fuse_res_enabled();  // LS_CONV_FUSE_RES=0: the resnet's res_conv keeps its own launch (development aid)
bool conv_dual_enabled();  // LS_CONV_DUAL=0 switches the dual-issue mode of conv_gemm off (development aid)
bool conv_resident_enabled();
bool conv_tma_out_enabled();   // LS_CONV_TMA_OUT=0: epilogue stores through the LSU (development aid)  // LS_CONV_RESIDENT=0: always stream the weights through the ring (development aid)  // LS_CONV_HALO=0: fetch the activation box per tap instead of once with a halo
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                              int cluster, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid, cfg.blockDim = block, cfg.dynamicSmemBytes = smem, cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  int n = 0;
  if (cluster > 1) {
    attr[n].id = cudaLaunchAttributeClusterDimension;
    attr[n].val.clusterDim.x = cluster, attr[n].val.clusterDim.y = 1, attr[n].val.clusterDim.z = 1;
    ++n;
  }
  if (pdl_enabled()) {
    attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[n].val.programmaticStreamSerializationAllowed = 1;
    ++n;
  }
  cfg.attrs = attr, cfg.numAttrs = n;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
  return e != cudaSuccess ? e : cudaGetLastError();
}

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) applies to the CURRENT device only, and handles can be created on
// any device of the process: the opt-in is tracked per (kernel instance, device) in a bit mask owned by the caller
// (one static mask per kernel instance).  Racing threads may both set the attribute; that is idempotent.
inline cudaError_t smem_optin_once(std::atomic<unsigned long long>& done_mask, const void* func, int bytes) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  const unsigned long long bit = 1ull << (dev & 63);
  if (done_mask.load(std::memory_order_acquire) & bit) return cudaSuccess;
  e = cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e != cudaSuccess) return e;
  done_mask.fetch_or(bit, std::memory_order_release);
  return cudaSuccess;
}

enum Act : int { ACT_NONE = 0, ACT_LRELU = 1, ACT_GELU = 2, ACT_LN_MISH = 3, ACT_LRELU_TANH = 4,
                 ACT_SILU = 5, ACT_LRELU001 = 6 /* F.leaky_relu's default slope 0.01 */ };
enum OutDtype : int { OUT_NONE = 0, OUT_F32 = 1, OUT_BF16 = 2 /* the build's 16-bit operand type */,
                      OUT_F16 = 3 /* IEEE half whatever the operand type (conv_gemm out0 / addend only) */,
                      ADD_GEMM = 4 /* addend only: the residual is a second GEMM of this launch (ConvGemmParams::res_*) */ };
enum Out1Mode : int { OUT1_NONE = 0, OUT1_LN = 1, OUT1_COPY = 2, OUT1_SNAKE = 3 };

// Implicit-GEMM 1-D convolution on time-major activations:
//   D[b, t, n] = sum_tap sum_c A[b, t + tap*dil - pad, c] * W[tap][n][c]        (rows outside [0,T_in) read as 0)
// followed by a fused, row-local epilogue (see conv_gemm.cu).  Linear layers are taps=1.
struct ConvGemmParams {
  // iteration space
  int B;              // batch items (utterance x CFG half)
  int M;              // output rows per batch item in this launch's iteration space
  int N;              // total output columns (multiple of block_n)
  int block_n;        // tile width: multiple of 16, <= 256
  int taps, dil, pad;
  int kb_per_tap;     // 64-wide K blocks per tap (over both A sources)
  int kb_split;       // K blocks [0,kb_split) come from A source 0, the rest from A source 1
  const int* lengths; // [B] valid length units per batch item (device), or nullptr = everything valid
  int m_len_mul, m_len_add;  // rows that matter: lengths[b]*m_len_mul + m_len_add (+ skip_halo before tiles are skipped)
  int skip_halo;
  int zero_skipped;   // 1: skipped tiles still zero-fill their outputs
  // epilogue
  int chan_mod;       // per-channel vectors are indexed with (n % chan_mod)
  const float* bias;  // [chan_mod] or nullptr
  int act;
  const float* ln_g;  // ACT_LN_MISH: LayerNorm affine over the N(=block_n) columns, eps 1e-5
  const float* ln_b;
  const float* temb;  // optional [.. , N] vector added after the activation; row b uses temb + b*temb_bstride
  long long temb_bstride;
  const void* addend; // optional residual, same flat indexing as out0
  int addend_dtype;   // OUT_F32 / OUT_BF16
  // outputs: flat element index inside batch item = row*out_ld + n + out_shift; stored if in [0, valid),
  // zero-filled if in [valid, alloc), dropped otherwise.  valid = lengths ? lengths[b]*out_valid_mul : alloc.
  void* out0;
  int out0_dtype;
  void* out1;         // always bf16
  int out1_mode;
  const float* p1_a;  // OUT1_LN: gamma | OUT1_SNAKE: alpha
  const float* p1_b;  // OUT1_LN: beta  | OUT1_SNAKE: 1/(alpha+1e-9)
  int n_store;        // only columns n < n_store are stored (N padding)
  long long out_ld, out_shift, out_bstride, out_alloc, out_valid_mul;
  // accounting only (profiler): true K per tap and which engine launched it (0 flow, 1 DAC)
  int k_true, tag;
  int fp16;           // 1: the 16-bit operands and outputs of this launch are fp16 instead of bf16 (flow estimator only)
  // A-operand staging.  halo_mode 1: the caller's activation maps have boxes of 128 + (taps-1)*dil rows and the
  // kernel fetches each K block of the input ONCE, reading tap t through a descriptor shifted by t*dil rows;
  // halo_mode 0: 128-row boxes fetched per tap.  The remaining fields are filled in by launch_conv_gemm.
  int halo_mode;
  int a_box_rows, a_stages, b_stages;
  // b_resident: the whole weight tensor of the launch fits in the B ring (b_stages == taps*kb_per_tap, one N tile):
  // it is fetched once per CTA and stays in shared memory for every tile.
  int b_resident;
  int tma_out;  // dense [B][M][N] outputs are stored with cp.async.bulk.tensor (filled in by launch_conv_gemm)
  // per-channel epilogue vectors staged in shared memory (float offsets into the vector area, -1 = read from global)
  int sv_bias, sv_p1a, sv_p1b, sv_lng, sv_lnb, sv_floats;
  // dual: two MMA-issuing warps, one per accumulator, on alternating tiles; each weight box serves both (filled in by
  // launch_conv_gemm for streamed-or-resident halo launches with one N tile, see conv_gemm.cu)
  int dual;
  // Fused residual GEMM (addend_dtype == ADD_GEMM; single-tile launches only: B * ceil(M/128) <= SMs, N == block_n): after
  // the main GEMM the same CTA computes R[t, n] = sum_c A2[t, c] W2[n][c] + res_bias[n] (a 1x1 convolution of a second
  // input: the resnet's res_conv, decoder.py:84 / matcha decoder.py:60) into the SECOND TMEM accumulator, and the
  // epilogue adds it where it would have added a residual read from global memory.  res_kb 64-wide K blocks, the first
  // res_split of them from res_a0, the rest from res_a1 (128-row activation boxes).
  alignas(64) CUtensorMap res_a0, res_a1, res_w;
  int res_kb, res_split, res_k_true;
  const float* res_bias;
  int red_bytes;  // LayerNorm statistics exchange area (0 for launches without a LayerNorm: the operand rings get it)
  long long* timeline;  // development aid (ls_debug_set_buffer): [CTA][64] clock64 stamps of the first tile, or nullptr
};
// rows of the activation box a conv with this geometry needs in halo mode (make_act_map's box_rows)
inline int conv_halo_box_rows(int taps, int dil) { return 128 + (taps - 1) * dil; }
__host__ __device__ constexpr int ls_conv_a_stage_bytes(int box_rows) { return ((box_rows + 7) / 8) * 1024; }

// Tensor maps are created on the host (tma_host.cpp helpers) and passed by value.  The grid is at most num_sms CTAs.
// plan_out (optional, the kernel tests' hook): receives the plan the launch used, kConvPlanInts values:
// grid, the largest tile count of any CTA, dual, b_resident, a_stages, b_stages, tma_out, halo_mode (all 0 when there
// is nothing to launch).
constexpr int kConvPlanInts = 8;
cudaError_t launch_conv_gemm(const CUtensorMap& mapA0, const CUtensorMap& mapA1, const CUtensorMap& mapW,
                             const ConvGemmParams& p, int num_sms, cudaStream_t stream, int* plan_out = nullptr);
cudaError_t launch_conv_gemm_fp16(const CUtensorMap& mapA0, const CUtensorMap& mapA1, const CUtensorMap& mapW,
                                  const ConvGemmParams& p, int num_sms, cudaStream_t stream, int* plan_out = nullptr);

// Flash attention forward over a packed [B][T][3*H*64] bf16 QKV tensor (Q | K | V column blocks).
#ifndef ATTN_KV
#define ATTN_KV 64    /* keys per attention tile (64: three CTAs per SM, measured 37.1 vs 40.7 us at B=32, T=500) = box rows of the QKV tensor map handed to launch_attention */
#endif
struct AttnParams {
  int B, T, H;
  const int* lengths;   // [B] valid keys per batch item or nullptr (= T)
  int chunk;            // >0: block-causal mask, key j visible to query i iff j < (i/chunk+1)*chunk
  float scale_log2e;    // softmax scale * log2(e)
  __nv_bfloat16* out;   // [B][T][H*64]
  // optional additive score term (the conformer's relative-position term, front_engine.cu): score(i, j) gets
  // bias[(b*H + h)*bias_bh + i*bias_ld + (T-1-i) + j] before the softmax scale; nullptr = none
  const float* bias;
  long long bias_ld, bias_bh;
  long long* timeline;  // development aid (ls_debug_set_buffer): [CTA][64] clock64 stamps, or nullptr
  long long timeline_entries;
  int fp16;             // 1: Q / K / V and the output are fp16 instead of bf16
};
cudaError_t launch_attention(const CUtensorMap& mapQKV, const AttnParams& p, cudaStream_t stream);
cudaError_t launch_attention_fp16(const CUtensorMap& mapQKV, const AttnParams& p, cudaStream_t stream);

// Fused row-local tail of a transformer block (tblock.cu): out-proj + residual + LayerNorm + FF1 + GELU + FF2 +
// residual, then either the next block's LayerNorm + QKV projection (tail_mode 0) or a masked bf16 copy of the
// residual stream (tail_mode 1).  Fixed estimator geometry: C = 256, 8 heads x 64, FF = 1024.
#define TBLOCK_VEC_FLOATS 2560
#ifndef TBLOCK_PAIR
#define TBLOCK_PAIR 0                              /* 1: CTA pairs (tcgen05 cta_group::2): each CTA streams HALF of every weight box */
#endif
#if TBLOCK_PAIR
#undef TBLOCK_CLUSTER
#define TBLOCK_CLUSTER 2
#endif
#ifndef TBLOCK_CLUSTER
#define TBLOCK_CLUSTER 1                           /* CTAs per cluster sharing every weight box by TMA multicast */
#endif
#define TBLOCK_WBOX_ROWS (128 / TBLOCK_CLUSTER)    /* box rows of the weight tensor maps */
/* Pair mode weight maps: Wo / W2 (the pair's N = 256 operands) = 2-D, 128-row boxes; W1 / Wqkv (N = 128 chunks) = 3-D
   [64][rows][K/64] with boxes of 64 rows x 2 K blocks (make_weight_map_kb). */
#define TBLOCK_WIDE_BOX_ROWS (TBLOCK_PAIR ? 128 : TBLOCK_WBOX_ROWS)
struct TBlockParams {
  int R;               // rows = batch rows x T (time-major, flattened)
  int T;               // rows per batch row (only used with lengths)
  const int* lengths;  // [R / T] valid frames per batch row, or nullptr
  const float* vec;    // device, TBLOCK_VEC_FLOATS: bo[256] g3[256] be3[256] b1[1024] b2[256] g1n[256] be1n[256]
  int tail_mode;       // 0: u updated in place + next block's QKV written; 1: masked bf16 copy of u'' written;
                       // 2: "head" of a block group: only LayerNorm(u; g1n, be1n) + QKV (att, Wo, W1, W2 unused)
  long long* timeline; // development aid (ls_debug_set_buffer): [grid][64] clock64 stamps of the first tile, or nullptr
  int fp16;            // 1: every 16-bit operand / output is fp16 instead of bf16
  int no_skip;         // 1: tiles that are padding only are processed too (their rows come out as zeros): the non-causal
                       //    estimator's convolutions read the first padding row after an utterance
};
// Every global tensor is reached through TMA (loads and stores), 128-row boxes, 128-byte swizzle:
struct TBlockMaps {
  CUtensorMap att;       // bf16 [R][512]  attention output              (make_tile_map, box 64 x 128)
  CUtensorMap wo, w1, w2, wqkv;  // bf16 weights [N][K], K contiguous     (make_weight_map, box 64 x TBLOCK_WBOX_ROWS)
  CUtensorMap u;         // fp32 [R][256]  residual stream, in/out        (box 32 x 128)
  CUtensorMap qkv_out;   // bf16 [R][1536] next block's Q | K | V          (box 64 x 128)   tail_mode 0
  CUtensorMap tail_out;  // bf16 [R][256]  u'' masked                      (box 64 x 128)   tail_mode 1
};
// The grid is at most num_sms CTAs (fewer when clusters do not all fit at once).  plan_out (optional, the kernel tests'
// hook): receives the grid and the largest tile count of any CTA.
cudaError_t launch_tblock(const TBlockMaps& m, const TBlockParams& p, int num_sms, cudaStream_t stream,
                          int* plan_out = nullptr);
cudaError_t launch_tblock_fp16(const TBlockMaps& m, const TBlockParams& p, int num_sms, cudaStream_t stream,
                               int* plan_out = nullptr);

// ---- bandwidth kernels (elementwise.cu) ----
// NCT fp32 [B][C][T] -> time-major bf16 dst[b][t][c_off + c], dst row stride ld; rows >= len zeroed.
cudaError_t launch_pack_nct(const float* src, __nv_bfloat16* dst, int B, int C, int T, long long src_bstride,
                            int ld, int c_off, const int* lengths, cudaStream_t s, int fp16 = 0);
// broadcast a per-batch vector [B][C] over time into dst[b][t][c_off + c]
cudaError_t launch_pack_bcast(const float* src, __nv_bfloat16* dst, int B, int C, int T, int ld, int c_off,
                              const int* lengths, cudaStream_t s, int fp16 = 0);
// zero dst[b][t][c_off .. c_off+C)
cudaError_t launch_pack_zero(__nv_bfloat16* dst, int B, int C, int T, int ld, int c_off, cudaStream_t s);
// x_state[b][t][c] = noise[c][t] * temperature (noise row stride noise_ld); also writes bf16 copies into
// xin rows b and B+b (channel offset 0).
cudaError_t launch_init_state(const float* noise, int noise_ld, float temperature, float* x_state,
                              __nv_bfloat16* xin, int B, int C, int T, int ld, const int* lengths, cudaStream_t s,
                              int fp16 = 0);
// CFG combine + Euler update (flow_matching.py:118-120): x += dt*((1+w) v[b] - w v[B+b]); refresh bf16 copies.
cudaError_t launch_cfg_euler(const float* v, float* x_state, __nv_bfloat16* xin, int B, int C, int T, int ld,
                             float dt, float cfg_rate, cudaStream_t s, int fp16 = 0);
// time-major fp32 [B][T][C] -> NCT fp32 [B][C][T], rows >= len zeroed
cudaError_t launch_unpack_nct(const float* src, float* dst, int B, int C, int T, const int* lengths, cudaStream_t s);
// lengths[d*B + b] = number of non-zero entries of mask[b][0][:] for d < dup; *bad_flag (device-visible, optional) is set
// when a mask is not a prefix mask
cudaError_t launch_mask_to_lengths(const float* mask, int* lengths, int B, int T, int dup, cudaStream_t s,
                                   int* bad_flag = nullptr);
// GroupNorm(G) + Mish on time-major fp32 x [B][T][C] with per-row statistics over the valid frames (the non-causal
// ConditionalDecoder's blocks): stats [B][G] scratch; then + temb[b] (optional) + addend (optional fp32, same layout);
// fp32 and / or 16-bit outputs (either may be null); padding rows come out as exactly 0 (temb and addend are not added
// there).  Lengths above T count as T.
cudaError_t launch_groupnorm_mish(const float* x, float2* stats, const float* gamma, const float* beta, const float* temb,
                                  long long temb_bstride, const float* addend, float* out_f32, __nv_bfloat16* out_h, int B,
                                  int C, int T, int G, const int* lengths, int fp16, cudaStream_t s);
// FSQCodebook.encode of the S3 tokenizer: x fp32 [rows][D], w [8][D], bias [8] -> tokens int32 [rows] in [0, 3^8)
cudaError_t launch_fsq_encode(const float* x, const float* w, const float* bias, int* tokens, long long rows, int D,
                              cudaStream_t s);
// Log-mel front end of the S3 tokenizer (s3_mel.cu): right-padded audio fp32 [B][S] with audio_len [B], filters
// [n_mels][201] (n_mels <= 128) -> mel fp32 [B][n_mels][S/160] (zeros past mel_len[b]), mel_len [B] = audio_len / 160,
// or 0 (and an all-zero mel) when audio_len[b] < 201 or > S.  B <= 65535.
cudaError_t launch_s3_log_mel(const float* audio, const int* audio_len, const float* filters, int n_mels, float* mel,
                              int* mel_len, int B, long long S, cudaStream_t s);
// ---- sample-rate conversion and latent stretch (resample.cu) ----
// The taps of torchaudio.functional.resample (sinc_interp_hann, width 6, rolloff 0.99) with |t| < 6, one row per phase:
// output sample j = q*N + p is sum_k taps[p][k] * x[q*O + first[p] + k] for k < count[p].  taps: [N][max_taps], fp32.
struct ResampleTable {
  int O = 0, N = 0, width = 0, max_taps = 0;  // reduced ratio O / N (orig / new), torchaudio's window half-width
  std::vector<int> first, count;
  std::vector<float> taps;
};
constexpr long long kResampleMaxTableBytes = 96 << 10;
constexpr size_t kResampleMaxSmem = 200 << 10;
inline long long resample_table_bytes(const ResampleTable& t) { return 4LL * t.N * t.max_taps; }
// LS_OK, LS_ERR_INVALID (a rate <= 0) or LS_ERR_UNSUPPORTED (table over kResampleMaxTableBytes; O, N, width are set).
// fill = false computes the sizes only.  Host only.
int resample_table(int orig_freq, int new_freq, ResampleTable* t, bool fill = true);
struct ResamplePlan {
  const float* taps = nullptr;  // device [N][stride]
  const int2* fc = nullptr;     // device [N] (first, count)
  int O = 0, N = 0, stride = 0, min_first = 0, tile = 0, span = 0;
  size_t smem = 0;
};
// The launch geometry for a table (taps / fc are the caller's to set); LS_ERR_UNSUPPORTED if it needs too much shared memory.
int resample_plan(const ResampleTable& t, ResamplePlan* plan);
// audio [B][S_in] with audio_len [B] -> out [B][S_out] (zero past out_len[b] = ceil(N len / O); S_out >= ceil(N S_in / O)).
// A length < 1 or > S_in gives out_len 0 and a zero row.  B <= 65535, S_in and S_out < 2^31.
cudaError_t launch_resample(const ResamplePlan& p, const float* audio, const int* audio_len, float* out, int* out_len, int B,
                            long long S_in, long long S_out, cudaStream_t s);
// z [B][C][L_in] -> out [B][C][L_out]: row b's first len_in[b] frames linearly stretched to len_out[b] frames
// (align_corners=False), zero past len_out[b]; invalid lengths give a zero row.
cudaError_t launch_latent_resize_linear(const float* z, const int* len_in, const int* len_out, float* out, int B, int C,
                                        int L_in, int L_out, cudaStream_t s);
// timestep conditioning for nt time values: sinusoidal embedding -> MLP -> per-resnet projections
struct TimeEmbedParams {
  const float* t;        // [nt] device, or nullptr: the values come from t_host (nt <= 64) inside the kernel parameters
  const float* t_host;   // [nt] host (only read when t == nullptr)
  float* scratch;        // device, 2 * nt * hid floats (the two hidden layers of the MLP)
  const float* freqs;    // [in_dim/2]
  const float* w1; const float* b1;   // [hid][in_dim]
  const float* w2; const float* b2;   // [hid][hid]
  const float* wr; const float* br;   // [n_res][out_dim][hid], [n_res][out_dim]
  float* out;            // [nt][n_res][out_dim]
  int nt, in_dim, hid, n_res, out_dim;
};
cudaError_t launch_time_embed(const TimeEmbedParams& p, cudaStream_t s);

// ---- host helpers (tma_host.cu) ----
// bf16 activation [B][T][C] viewed through 64 x rows x 1 boxes with 128B swizzle (OOB -> zero)
// bf16 weights [rows][K] viewed as [64][rows][K/64]: one box = box_rows rows x box_kb 64-wide K blocks, landing in
// shared memory as box_kb consecutive 128B-swizzled tiles of box_rows rows
bool make_weight_map_kb(CUtensorMap* map, const void* base, int K, int rows, int box_rows, int box_kb);
// output tensor [B][M][N] (fp32 or bf16) for the conv epilogue's TMA stores: box 16 columns x 32 rows, 64 B / 32 B swizzle
bool make_out_map(CUtensorMap* map, const void* base, int elem_bytes, int N, int M, int B);
bool make_act_map(CUtensorMap* map, const void* base, int C, int T, int B, long long row_stride_elems,
                  long long batch_stride_elems, int box_rows);
// bf16 weight matrix [rows][K] with 64 x box_rows boxes
bool make_weight_map(CUtensorMap* map, const void* base, int K, int rows, int box_rows);
// row-major [rows][cols] matrix of bf16 (elem_bytes 2) or fp32 (4) with (128 B / elem_bytes) x box_rows boxes,
// 128-byte swizzle; usable for TMA loads (OOB rows read as zero) and TMA stores (OOB rows dropped)
bool make_tile_map(CUtensorMap* map, const void* base, int elem_bytes, long long cols, long long rows, int box_rows);

}  // namespace ls
