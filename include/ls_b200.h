/* ls_b200.h -- C ABI of the B200-native CFM-solve + DAC-VAE-decode hot path.
 *
 * Plain C: opaque handles, raw pointers, sizes, a CUDA stream passed as void*; no torch types.
 * Every entry point returns LS_OK (0) or a negative LS_ERR_* code and never throws; the message of
 * the last failure on the calling thread is available from ls_last_error().
 *
 * Reference interfaces these entry points replace (paths relative to the reference repo):
 *   ls_flow_estimator_forward  <- ConditionalCFM.forward_estimator, the nn.Module / TensorRT seam with
 *                                 inputs x, mask, mu, t, spks, cond -> estimator_out
 *                                 (speech/cosyvoice/flow/flow_matching.py:128-155;
 *                                  speech/cosyvoice/bin/export_onnx.py:84-85 names the tensors)
 *   ls_flow_solve              <- CausalConditionalCFM.forward + ConditionalCFM.solve_euler
 *                                 (speech/cosyvoice/flow/flow_matching.py:323-348, 74-126)
 *   ls_dac_decode              <- DACVAE.decode (dac-vae/model.py:485-488)
 *   ls_flow_create / ls_dac_create take the reference state_dict unchanged (key schema: SURVEY.md
 *                                 Appendix A/B); weight-norm folding and layout packing happen inside.
 *
 * Tensor layouts at the boundary are the reference's: float32, NCT contiguous
 * (x/mu/cond [rows,80,T], mask [rows,1,T], spks [rows,80], t [rows], latents z [B,80,L],
 * waveform [B,1,L*hop]).  Unless stated otherwise pointers are DEVICE pointers valid on `stream`.
 * One handle = one workspace (like one TensorRT execution context): calls on the same handle are serialised by the
 * library -- host threads by a per-handle mutex, streams by an event the next call waits for when the handle moves to
 * another stream -- so concurrent use is safe but does not overlap; use one handle per concurrent session.  Different
 * handles are independent.  The hot calls do not synchronise the device and allocate only when a shape larger than any
 * seen before arrives (stream-ordered cudaMallocAsync).  A mask that is not a prefix (right-padding) mask is detected on
 * the device and reported by the NEXT call on the handle (LS_ERR_INVALID): validating it in the call itself would cost a
 * host synchronisation.
 */
#ifndef LS_B200_H
#define LS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LS_OK 0
#define LS_ERR_INVALID (-1)     /* bad argument / shape */
#define LS_ERR_CUDA (-2)        /* CUDA runtime or driver failure */
#define LS_ERR_WEIGHTS (-3)     /* missing / mis-shaped state_dict entry */
#define LS_ERR_UNSUPPORTED (-4) /* configuration outside what the kernels cover */

#define LS_ABI_VERSION 1

/* One state_dict entry: host float32, C-contiguous. */
typedef struct ls_tensor {
  const char* name;
  const float* data;
  int32_t ndim;
  int64_t shape[4];
} ls_tensor;

typedef struct ls_flow ls_flow;
typedef struct ls_dac ls_dac;

int32_t ls_abi_version(void);
const char* ls_last_error(void);
/* Reports SM count and compute capability; LS_ERR_UNSUPPORTED unless the device is sm_100. */
int32_t ls_device_check(int32_t device, int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor);

/* ---- flow: CausalConditionalDecoder estimator + Euler/CFG solve ---- */
int32_t ls_flow_create(const ls_tensor* weights, int32_t n_weights, int32_t device, ls_flow** out);
/* fp16-operand mode: the same tensor-core kernels at the same speed with fp16 instead of bf16 GEMM operands (weights and
 * activations; accumulation, residual stream, LayerNorm, softmax statistics stay fp32).  fp16 is the format of the
 * reference's own half-precision path (speech/cosyvoice/cli/model.py:41-43 `.half()`; the TensorRT fp16 flag,
 * speech/cosyvoice/utils/file_utils.py:63-64,75); three more mantissa bits than bf16: a single estimator call is 1.5e-3
 * from the fp32 reference instead of 1.2e-2 (the bf16 rounding of the weights alone is 8.6e-3). */
int32_t ls_flow_create_fp16(const ls_tensor* weights, int32_t n_weights, int32_t device, ls_flow** out);
/* fp32 mode (north_star: latents within 1e-4 of the fp32 reference): the same handle type and calls, computed end to
 * end in fp32 on the CUDA cores with unfused kernels.  A validation mode, one to two orders of magnitude slower. */
int32_t ls_flow_create_fp32(const ls_tensor* weights, int32_t n_weights, int32_t device, ls_flow** out);
void ls_flow_destroy(ls_flow* h);

/* One estimator evaluation.  rows = batch rows as the reference passes them (2 for CFG at B=1).
 * out may alias x (the TensorRT path binds the output to x's buffer, flow_matching.py:136-152). */
int32_t ls_flow_estimator_forward(ls_flow* h, const float* x, const float* mask, const float* mu, const float* t,
                                  const float* spks, const float* cond, float* out, int32_t rows, int32_t T,
                                  int32_t streaming, void* stream);

/* Whole n_timesteps Euler solve with classifier-free guidance, B >= 1 utterances with per-utterance
 * semantics (equal to B reference calls at batch 1).  noise: [80][noise_stride] rows of the fixed-noise
 * buffer (CausalConditionalCFM.rand_noise); t_span_host: n_timesteps+1 HOST floats (the schedule the
 * caller computed exactly as the reference does).  out: [B,80,T], zero where mask == 0. */
int32_t ls_flow_solve(ls_flow* h, const float* mu, const float* mask, const float* spks, const float* cond,
                      const float* noise, int64_t noise_stride, const float* t_span_host, int32_t n_timesteps,
                      float temperature, float cfg_rate, int32_t streaming, float* out, int32_t B, int32_t T,
                      void* stream);

/* ---- DAC-VAE decoder ---- */
int32_t ls_dac_create(const ls_tensor* weights, int32_t n_weights, int32_t device, ls_dac** out);
/* fp16-operand mode of the DAC-VAE handle: the same tensor-core kernels with fp16 instead of bf16 GEMM operands (the
 * folded weights, z, and every Snake / LeakyReLU output a convolution consumes); accumulation stays fp32, the decoder's
 * residual stream fp16, the encoder's fp32, and the waveform and z / m / logs fp32.  Like ls_dac_create it builds the
 * decoder, the encoder, or both, from whatever the state dict holds, and the handle takes the same calls (including
 * ls_graph_create).  A folded weight outside fp16's range (|w| > 65504) fails with LS_ERR_UNSUPPORTED naming the layer. */
int32_t ls_dac_create_fp16(const ls_tensor* weights, int32_t n_weights, int32_t device, ls_dac** out);
int32_t ls_dac_create_fp32(const ls_tensor* weights, int32_t n_weights, int32_t device, ls_dac** out);
void ls_dac_destroy(ls_dac* h);
int32_t ls_dac_hop_length(const ls_dac* h);
/* z [B,80,L] -> wav [B,1,L*hop].  lengths (DEVICE int32 [B], may be NULL): valid latent frames per item;
 * each item is decoded as if alone at its own length, the rest of its row is zero. */
int32_t ls_dac_decode(ls_dac* h, const float* z, const int32_t* lengths, float* wav, int32_t B, int32_t L,
                      void* stream);

/* DACVAE.encode (dac-vae/model.py:469-483; bulk latent extraction, dac-vae/extract_dac_latents.py:20-54): audio
 * [B,1,S] with S a multiple of the hop -> z, m, logs, each [B,latent,S/hop]; z = m + noise * exp(logs) with the
 * caller's noise [B,latent,S/hop] (NULL: z = m).  The handle's weights must contain the encoder.* / en_conv_post.*
 * entries (ls_dac_create builds the decoder, the encoder, or both, from whatever the state dict holds). */
int32_t ls_dac_encode(ls_dac* h, const float* audio, const float* noise, float* z, float* m, float* logs, int32_t B,
                      int32_t S, void* stream);
/* ls_dac_encode for a right-padded batch of clips of different lengths.  lengths (DEVICE int32 [B], may be NULL =
 * ls_dac_encode): valid latent frames per clip, clamped to [0, S/hop]; clip b is the samples [0, lengths[b]*hop) of
 * its row and is encoded as if alone at that length (the samples after it are never read), noise is read over the
 * same frames, and z, m, logs are zero from frame lengths[b] on (a length of 0 gives an all-zero item). */
int32_t ls_dac_encode_lengths(ls_dac* h, const float* audio, const int32_t* lengths, const float* noise, float* z, float* m,
                              float* logs, int32_t B, int32_t S, void* stream);

/* ---- token -> mu front half (SURVEY section 8 f-1): CausalMaskedDiffWithXvec.inference up to the decoder call
 * (speech/cosyvoice/flow/flow.py:461-489): speaker-embedding normalise + affine, input embedding,
 * UpsampleConformerEncoder (speech/cosyvoice/transformer/upsample_encoder.py:266-318), encoder_proj.
 * ls_front_create: tensor-core path (bf16 operands, fp32 accumulate and residual stream); ls_front_create_fp32: fp32 mode.
 * token_len (device int32 [B], or NULL = every utterance has T tokens): token counts of a right-padded batch -- padded
 * token rows are embedded as zeros and masked as attention keys exactly as the reference's encoder does with `xs_lens`
 * (flow.py:475-476, upsample_encoder.py:293-301); mu is zero past 2 * token_len.  Prompt tokens are simply part of
 * `tokens` (flow.py:471-475 concatenates them).
 * tokens [B,T] int64 (25 Hz FSQ ids), embedding [B,192] -> mu [B,80,2(T - n_context)], spks [B,80] (the inputs of
 * ls_flow_solve).  n_context = 0: final chunk (finalize = True); n_context = 3: the last 3 tokens are look-ahead context
 * only (flow.py:482-489).  streaming != 0: block-causal attention (25 tokens / 50 frames, upsample_encoder.py:297,312). */
typedef struct ls_front ls_front;
int32_t ls_front_create(const ls_tensor* weights, int32_t n_weights, int32_t device, ls_front** out);
int32_t ls_front_create_fp32(const ls_tensor* weights, int32_t n_weights, int32_t device, ls_front** out);
void ls_front_destroy(ls_front* h);
int32_t ls_front_encode(ls_front* h, const int64_t* tokens, const float* embedding, float* mu, float* spks, int32_t B,
                        int32_t T, int32_t n_context, int32_t streaming, const int32_t* token_len, void* stream);
/* Session mode: a batch of independent calls, e.g. one streaming hop of each of B sessions.  Row b of tokens [B,T_all]
 * holds token_len[b] tokens (prompt tokens included), of which the last n_context[b] (0: finalize = True, 3: a
 * non-final hop) are look-ahead context, and comes out equal to ls_front_encode of that row alone with its own
 * n_context: T_b = token_len[b] - n_context[b] output tokens, mu [B,80,2T] with T = max T_b (the caller's), zero past
 * 2 T_b.  The padding after a row's tokens is never read.  token_len, n_context: DEVICE int32 [B].  A row with
 * n_context not 0 or 3, T_b < 1, token_len[b] > T_all or T_b > T gets an all-zero mu (no host synchronisation: the
 * entries are only read on the device).  Needs T <= T_all; B <= 512 on the tensor-core path. */
int32_t ls_front_encode_sessions(ls_front* h, const int64_t* tokens, const float* embedding, float* mu, float* spks, int32_t B,
                                 int32_t T_all, int32_t T, const int32_t* token_len, const int32_t* n_context, int32_t streaming,
                                 void* stream);

/* ---- speaker encoder (SURVEY section 8 f-4): LearnableSpeakerEncoder.forward (speech/cosyvoice/llm/llm.py:34-96, blocks:
 * speech/cosyvoice/transformer/arch_util.py:21-123) and the averaging over several reference clips of
 * CausalMaskedDiffWithXvec.get_speaker_embedding (speech/cosyvoice/flow/flow.py:336-366).  Equal-length clips.
 * mel [n_refs][B,80,T] -> embedding [B,192], L2-normalised (the `embedding` input of ls_front_encode). */
typedef struct ls_speaker ls_speaker;
int32_t ls_speaker_create(const ls_tensor* weights, int32_t n_weights, int32_t device, ls_speaker** out);      /* tensor cores */
int32_t ls_speaker_create_fp32(const ls_tensor* weights, int32_t n_weights, int32_t device, ls_speaker** out); /* fp32 mode */
void ls_speaker_destroy(ls_speaker* h);
int32_t ls_speaker_encode(ls_speaker* h, const float* mel, float* embedding, int32_t B, int32_t T, int32_t n_refs,
                          void* stream);

/* ---- S3 speech tokenizer (SURVEY section 8 f-4): S3TokenizerV2.quantize for clips of at most 30 s
 * (speech/tools/S3Tokenizer/s3tokenizer/model_v2.py:386-415) = AudioEncoderV2.forward (:320-351: two stride-2 convs,
 * FSMN attention blocks with rotary embedding :152-287) + FSQCodebook.encode (:97-112).  Two handle types share one call
 * surface: ls_s3_create_fp32 (fp32 arithmetic on the CUDA cores) and ls_s3_create (bf16x3: every dense linear /
 * convolution on the tensor cores as A_hi W_hi + A_lo W_hi + A_hi W_lo, hi = bf16(x), lo = bf16(x - hi), fp32
 * accumulation; residual stream, LayerNorm, rotary, FSMN and attention in fp32 -- fp32-level error, since a token is a
 * rounding decision; 716 MiB of weights at the shipped width against 470 MiB; encoder output rows past code_len[b] are zero).
 * mel [B,n_mels,T] (100 Hz log-mel, right-padded), mel_len [B] -> codes [B,T2] (ids < 3^8; frames past code_len[b] are
 * undefined, as in the reference), code_len [B]; T2 = ls_s3_code_frames(T); hidden (nullable): [B,T2,n_state], the
 * encoder output.  Weight names = the reference's state_dict keys; optional "rotary.cos" / "rotary.sin" [len][32] tables
 * (default: precompute_freqs_cis(64, 2048), model_v2.py:37-48).  All pointers are device pointers. */
typedef struct ls_s3 ls_s3;
int32_t ls_s3_create_fp32(const ls_tensor* weights, int32_t n_weights, int32_t device, ls_s3** out);
int32_t ls_s3_create(const ls_tensor* weights, int32_t n_weights, int32_t device, ls_s3** out);
void ls_s3_destroy(ls_s3* h);
int32_t ls_s3_code_frames(int32_t T);
int32_t ls_s3_quantize(ls_s3* h, const float* mel, const int32_t* mel_len, int32_t* codes, int32_t* code_len, float* hidden,
                       int32_t B, int32_t T, void* stream);

/* ---- log-mel front end of the S3 speech tokenizer: log_mel_spectrogram (speech/tools/S3Tokenizer/s3tokenizer/utils.py,
 * the Whisper front end) for a right-padded batch of 16 kHz clips, each clip computed as if it were alone:
 *   frames t = 0 .. audio_len[b]/160 - 1: samples t*160 - 200 + j, j < 400, reflected about the clip's own ends
 *     (i < 0 -> -i, i >= len -> 2(len-1) - i: torch.stft center=True, whose last frame the reference drops);
 *   power = |rDFT(hann_periodic(400) * frame)|^2 (201 bins), fp32 on the CUDA cores;
 *   e = log10(max(filters @ power, 1e-10)); mel = (max(e, max over the clip's mels and frames of e - 8) + 4) / 4.
 * audio [B,S] fp32, audio_len [B], filters [n_mels,201] fp32 (the reference's mel_filters.npz asset, key mel_<n_mels>;
 * n_mels in [1, 128]) -> mel [B,n_mels,S/160] fp32 (NCT: the mel input of ls_s3_quantize; frames at or past mel_len[b]
 * are zero), mel_len [B] = audio_len[b] / 160.  Samples at or past audio_len[b] are never read, so whatever the padding
 * holds (NaN included) a clip's mel is bitwise the same as computing it alone.  Invalid lengths: a clip with
 * audio_len[b] < 201 (reflect padding needs more than 200 samples) or > S gets mel_len[b] = 0 and an all-zero mel;
 * nothing out of bounds is read.  Stateless, no allocation and no host synchronisation (capturable in a CUDA graph).
 * B <= 65535.  All pointers are device pointers. */
int32_t ls_s3_log_mel(const float* audio, const int32_t* audio_len, const float* filters, int32_t n_mels, float* mel,
                      int32_t* mel_len, int32_t B, int64_t S, void* stream);

/* ---- sample-rate conversion: torchaudio.functional.resample(x, orig_freq, new_freq) at its defaults (sinc_interp_hann,
 * lowpass_filter_width 6, rolloff 0.99; the resampler of the S3 tokenizer's load_audio and CosyVoice's front end) for a
 * right-padded batch of clips, each converted as if it were alone.  With the ratio reduced to O / N (gcd), base =
 * min(O, N) * 0.99 and width = ceil(6 O / base), output sample j = q*N + p of a clip is
 *   sum_i x[q*O + i] k_p(i),  k_p(i) = sinc(pi t) cos^2(pi t / 12) base / O,  t = base (i/O - p/N),
 * with x zero outside the clip; torchaudio sums i over [-width, width + O) with t clamped to +-6, this library only the
 * taps with |t| < 6 (the others are below 1e-45).  The taps are computed once on the host in double and rounded once to
 * fp32; each output sums its taps in increasing i in fp32.  Output length ceil(N len / O).  orig == new is a copy.
 *
 * ls_resampler_create builds the table for one (orig, new) pair and uploads it to `device` (LS_ERR_UNSUPPORTED for a
 * table over 96 KiB, e.g. rates whose reduced ratio has thousands of phases); the handle is reused for any number of
 * calls, which copy nothing.  ls_resample: audio [B,S_in] fp32 with audio_len [B] -> out [B,S_out] fp32, out_len [B] =
 * ceil(N audio_len[b] / O); S_out >= ceil(N S_in / O) (the caller may pick a larger S_out, e.g. a multiple of a hop);
 * out is zero from out_len[b] to S_out.  Samples at or past audio_len[b] are never read, so whatever the padding holds a
 * clip's output is bitwise the same as converting it alone.  A length < 1 or > S_in gives out_len 0 and a zero row.
 * B <= 65535, S_in and S_out < 2^31.  No allocation and no host synchronisation (capturable in a CUDA graph); the calls
 * hold no per-call state, so one handle may serve several streams at once.  All pointers are device pointers.
 * ls_resample_taps (host only, no device needed): the reduced ratio, torchaudio's width, the largest tap count of a phase,
 * and (when the arrays are not NULL) the table ls_resample uses: first [N] (the first i of phase p), count [N], taps
 * [N][max_taps] (zero-padded).  NULL arrays: sizes only.  LS_ERR_UNSUPPORTED (sizes other than max_taps still written)
 * for a table over 96 KiB. */
typedef struct ls_resampler ls_resampler;
int32_t ls_resampler_create(int32_t orig_freq, int32_t new_freq, int32_t device, ls_resampler** out);
void ls_resampler_destroy(ls_resampler* h);
int32_t ls_resample(ls_resampler* h, const float* audio, const int32_t* audio_len, float* out, int32_t* out_len, int32_t B,
                    int64_t S_in, int64_t S_out, void* stream);
int32_t ls_resample_taps(int32_t orig_freq, int32_t new_freq, int32_t* orig_red, int32_t* new_red, int32_t* width,
                         int32_t* max_taps, int32_t* first, int32_t* count, float* taps);

/* ---- latent speed change: CosyVoice2's token2wav(speed) F.interpolate(feat, size=int(L / speed), mode='linear') on a
 * right-padded batch of DAC latents.  z [B,C,L_in] -> out [B,C,L_out]: row b's first len_in[b] frames go to len_out[b]
 * frames with PyTorch's align_corners=False arithmetic (scale = len_in / len_out, src = max(scale (d + 0.5) - 0.5, 0),
 * i0 = (int)src, i1 = min(i0 + 1, len_in - 1), lambda = src - i0, out = (1 - lambda) x[i0] + lambda x[i1]), evaluated in
 * double and rounded once to fp32 (= F.interpolate in float64, rounded); zero from len_out[b] to L_out.  len_in, len_out:
 * DEVICE int32 [B] (the caller computes len_out, e.g. int(L / speed) in Python).  A row with len_in outside [1, L_in] or
 * len_out outside [1, L_out] is all zero.  Stateless; all pointers are device pointers. */
int32_t ls_latent_resize_linear(const float* z, const int32_t* len_in, const int32_t* len_out, float* out, int32_t B, int32_t C,
                                int32_t L_in, int32_t L_out, void* stream);

/* ---- end to end with HOST buffers (pinned or pageable): H2D copies, solve, decode, D2H copy, and a
 * stream synchronise all happen inside the call.  wav_host: [B,1,T*hop]. */
int32_t ls_synthesize_host(ls_flow* flow, ls_dac* dac, const float* mu_host, const float* mask_host,
                           const float* spks_host, const float* cond_host, const float* noise_dev,
                           int64_t noise_stride, const float* t_span_host, int32_t n_timesteps, float temperature,
                           float cfg_rate, float* wav_host, int32_t B, int32_t T, void* stream);

/* ---- FSQ quantizer head of the S3 speech tokenizer (SURVEY section 8 f-4, second half): FSQCodebook.encode,
 * speech/tools/S3Tokenizer/s3tokenizer/model_v2.py:83-117 -- hidden [rows, dim] (the AudioEncoderV2 output, fp32) ->
 * tokens [rows] in [0, 3^8): round(tanh(project_down(h)) * 0.999) + 1 per digit, base-3 packed.  All pointers are device
 * pointers (project_down.weight [8, dim], project_down.bias [8]).  Stateless.  The encoder trunk in front of it
 * (model_v2.py:243-351) is not built. */
int32_t ls_fsq_encode(const float* hidden, const float* project_down_weight, const float* project_down_bias, int32_t* tokens,
                      int64_t rows, int32_t dim, void* stream);

/* lengths[b] = number of non-zero entries of mask[b,0,:] (device pointers; the glue between ls_flow_solve and
 * ls_dac_decode -- the reference builds the same information with make_pad_mask, speech/cosyvoice/flow/flow.py:478). */
int32_t ls_mask_to_lengths(const float* mask, int32_t* lengths, int32_t B, int32_t T, void* stream);

/* ---- CUDA-graph replay of one fixed shape: the n_timesteps loop of ConditionalCFM.solve_euler
 * (speech/cosyvoice/flow/flow_matching.py:103) plus, when dac != NULL, DACVAE.decode, captured once as a CUDA graph
 * (programmatic-dependent-launch edges kept) over buffers owned by the ls_graph object and replayed with one
 * cudaGraphLaunch: the form for launch-bound small batches (one 10 s utterance is ~1800 kernels of a few microseconds).
 * Tensor-core handles only; n_timesteps <= 64.  The caller writes the inputs into the static buffers (ls_graph_buffer:
 * 0 mu [B,80,T], 1 mask [B,1,T], 2 spks [B,80], 3 cond [B,80,T]), launches, and reads 4 latents [B,80,T] and 5 waveform
 * [B,1,T*hop] (NULL without a dac handle).  The flow / dac handles must outlive the graph; a launch re-captures by itself
 * when a larger eager call on the same handles has reallocated their workspace in between. */
typedef struct ls_graph ls_graph;
int32_t ls_graph_create(ls_flow* flow, ls_dac* dac, const float* noise_dev, int64_t noise_stride, const float* t_span_host,
                        int32_t n_timesteps, float temperature, float cfg_rate, int32_t streaming, int32_t B, int32_t T,
                        void* stream, ls_graph** out);
void* ls_graph_buffer(ls_graph* g, int32_t which);
int32_t ls_graph_launch(ls_graph* g, void* stream);
int64_t ls_graph_kernel_count(const ls_graph* g); /* kernels inside one replay */
void ls_graph_destroy(ls_graph* g);

/* Number of kernel launches issued by this library since load (all handles, all threads; a graph replay counts the
 * kernels it contains). */
int64_t ls_launch_count(void);

/* Per-kernel timing for bench.py's roofline figures: between ls_profile_begin() and ls_profile_end() every launch
 * is bracketed by CUDA events on its stream.  ls_profile_end synchronises the device and fills LS_PROFILE_KINDS
 * entries: 0 conv_gemm (estimator), 1 attention, 2 conv_gemm (DAC decoder), 3 bandwidth kernels,
 * 4 fused transformer-block kernel (estimator). */
#define LS_PROFILE_KINDS 5
typedef struct ls_profile_entry {
  int64_t launches;
  double ms;    /* summed device time of the launches */
  double flops; /* algorithmic FLOPs of the launches (2*M*N*K, unpadded K) */
  double bytes; /* algorithmic bytes (operands read once + outputs written once) */
} ls_profile_entry;
int32_t ls_profile_begin(void);
int32_t ls_profile_end(ls_profile_entry* out, int32_t n_entries);

/* Development aid: kernels that support it write clock64 timelines ([grid][64] int64) into this device buffer
 * while it is set (NULL clears it).  Not used by any product path. */
int32_t ls_debug_set_buffer(void* dev_ptr, int64_t bytes);

/* ---- kernel-level hooks used by the kernel tests (tests/test_kernels_gpu.py, tests/test_kernel_plans_gpu.py,
 * tests/test_estimator_kernels_gpu.py) ----
 * Test-only: not part of the product surface, no engine calls them.  num_sms: the SM count the launch plans for
 * (0 = the device's own; a value outside [0, device SMs] is refused with LS_ERR_INVALID), so that small shapes reach
 * the plans a full-size launch takes.  plan_out (may be NULL) receives the plan the launch used. */
typedef struct ls_conv_gemm_desc {
  const void* a0; /* bf16 [B][T_in][a0_C] */
  const void* a1; /* optional second K source (channel concat), bf16 [B][T_in][a1_C] */
  const void* w;  /* bf16 [taps*N][K], K = a0_C + a1_C */
  int32_t a0_C, a1_C, T_in, K;
  int32_t B, M, N, block_n, taps, dil, pad;
  const int32_t* lengths;
  int32_t m_len_mul, m_len_add, skip_halo;
  int32_t chan_mod;
  const float* bias;
  int32_t act; /* 0 none, 1 leaky-relu(0.1), 2 gelu(erf), 3 layernorm+mish, 4 leaky-relu then tanh */
  const float* ln_g;
  const float* ln_b;
  const float* temb;
  int64_t temb_bstride;
  const void* addend;
  int32_t addend_dtype; /* 1 f32, 2 bf16, 3 fp16 */
  void* out0;
  int32_t out0_dtype; /* 0 none, 1 f32, 2 bf16, 3 fp16 */
  void* out1;
  int32_t out1_mode; /* 0 none, 1 layernorm, 2 copy, 3 snake */
  const float* p1_a;
  const float* p1_b;
  int32_t n_store;
  int64_t out_ld, out_shift, out_bstride, out_alloc, out_valid_mul;
  int32_t fp16; /* 0: bf16 operands and 16-bit outputs (dtype 2), 1: fp16; fp16 outputs (dtype 3) are IEEE half either way */
  int32_t zero_skipped; /* 1: tiles that are all padding still store zeros at their output positions */
  /* Fused residual GEMM (res_w != NULL, no addend): the epilogue adds R = [res_a0 | res_a1] . res_w^T + res_bias, a
   * 1x1 convolution computed in the same launch.  res_a0 bf16 [B][T_in][res_a0_C], optional res_a1 [B][T_in][res_a1_C]
   * (res_a0_C % 64 == 0 then), res_w [N][res_K] with res_K = res_a0_C + res_a1_C, res_bias fp32 [N]. */
  const void* res_a0;
  const void* res_a1;
  int32_t res_a0_C, res_a1_C;
  const void* res_w;
  int32_t res_K;
  const float* res_bias;
} ls_conv_gemm_desc;
/* plan_out: int32[8] = grid, the largest tile count of any CTA, dual issue, resident weights, activation stages,
 * weight stages, TMA stores, halo mode (all 0 when there is nothing to launch) */
int32_t ls_test_conv_gemm(const ls_conv_gemm_desc* d, int32_t num_sms, int32_t* plan_out, void* stream);
/* qkv [B][T][3*H*64] -> out [B][T][H*64], bf16 (fp16 = 0) or IEEE half (fp16 = 1); softmax scale 0.125.
 * lengths int32[B] or NULL (= T); chunk > 0: key j visible to query i iff j < (i/chunk + 1)*chunk.
 * bias (NULL = none): fp32 relative-position term, score(i, j) += bias[(b*H + h)*bias_bh + i*bias_ld + (T-1-i) + j],
 * with bias_ld >= 2T-1 and bias_bh >= T*bias_ld (the reads then stay inside B*H*bias_bh floats). */
int32_t ls_test_attention(const void* qkv, void* out, const int32_t* lengths, int32_t B, int32_t T, int32_t H,
                          int32_t chunk, int32_t fp16, const float* bias, int64_t bias_ld, int64_t bias_bh,
                          void* stream);

/* Fused transformer-block tail (tblock.cu): att bf16 [R][512], u fp32 [R][256] (updated in place when
 * tail_mode == 0), bf16 weights wo [256][512], w1 [1024][256], w2 [256][1024], wqkv [1536][256], vec = 2560 floats
 * (bo, g3, be3, b1, b2, g1n, be1n).  tail_mode 0 -> qkv_out bf16 [R][1536]; 1 -> tail_out bf16 [R][256].
 * fp16 = 1: every 16-bit operand and output is IEEE half instead of bf16.  no_skip = 1: tiles that hold only padding
 * rows are processed too.  plan_out: int32[2] = grid, the largest tile count of any CTA. */
int32_t ls_test_tblock(const void* att, float* u, const void* wo, const void* w1, const void* w2, const void* wqkv,
                       const float* vec, void* qkv_out, void* tail_out, const int32_t* lengths, int32_t R, int32_t T,
                       int32_t tail_mode, int32_t fp16, int32_t no_skip, int32_t num_sms, int32_t* plan_out,
                       void* stream);
/* GroupNorm(G) + Mish (elementwise.cu) on fp32 x [B][T][C]: statistics per (batch row, group) over the row's valid frames
 * (lengths int32[B], clamped to T, or NULL = T) into stats (B*G float pairs of scratch), then on valid frames
 * y = mish(GroupNorm(x) * gamma + beta) + temb[b*temb_bstride + c] (temb may be NULL) + addend (fp32 [B][T][C], may be
 * NULL), and 0 on padding frames.  y goes to out_f32 and / or out_h (bf16, or IEEE half when fp16 = 1); either may be
 * NULL.  C must be a multiple of 4G and C/G of 32. */
int32_t ls_test_groupnorm_mish(const float* x, void* stats, const float* gamma, const float* beta, const float* temb,
                               int64_t temb_bstride, const float* addend, float* out_f32, void* out_h, int32_t B,
                               int32_t C, int32_t T, int32_t G, const int32_t* lengths, int32_t fp16, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LS_B200_H */
