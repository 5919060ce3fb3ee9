"""Voice conversion from raw speech: CosyVoice2's ``inference_vc(source_speech_16k, prompt_speech_16k, speed)`` -- source
tokens, prompt tokens + prompt features + speaker embedding -> ``token2wav`` -- batched over utterances of different
lengths, with the DAC-VAE where CosyVoice2 has its mel / HiFT pair.  No LLM is involved.

* ``VoiceConverter.prompts`` turns prompt recordings (any integer sample rate) into ``Prompt``s: the S3 tokens of the
  16 kHz signal, the DAC-VAE posterior mean of the 24 kHz signal, both cut to ``2 x tokens`` frames as CosyVoice2's
  ``frontend_zero_shot`` does, and the speaker embedding.  A ``Prompt`` holds exactly the tensors
  ``CausalMaskedDiffWithXvec.inference_batch``, ``StreamingSession`` and ``StreamingBatch.open`` take.
* ``synthesize``: tokens -> one padded flow solve -> the speed change (``F.interpolate(mode='linear')`` of token2wav, on
  the GPU) -> one length-masked DAC-VAE decode.
* ``convert``: source recordings -> S3 tokens (one padded ``quantize_audio`` call after the GPU resample) -> ``synthesize``.

The resampling runs on the GPU (``audio.resample``); a signal already at the rate a model wants skips it."""
from dataclasses import dataclass

import torch

from . import audio as _audio
from . import native

TOKEN_RATE = 16000  # the S3 tokenizer's sample rate


@dataclass
class Prompt:
    """token [1, Tp] int64, feat [1, 2 Tp, 80] (DAC-VAE latents, frame-major), embedding [1, 192] (as
    ``get_speaker_embedding`` returns it), all on the converter's device."""
    token: torch.Tensor
    feat: torch.Tensor
    embedding: torch.Tensor


def prompt_cut(n_frames, n_tokens):
    """CosyVoice2's ``frontend_zero_shot`` alignment: the prompt keeps n = min(frames // 2, tokens) tokens and 2n frames."""
    return min(int(n_frames) // 2, int(n_tokens))


def _speeds(speed, n):
    speeds = [float(speed)] * n if isinstance(speed, (int, float)) else [float(s) for s in speed]
    if len(speeds) != n or any(not s > 0 for s in speeds):
        raise ValueError(f"speed must be a positive number or {n} positive numbers")
    return speeds


def speed_lengths(lengths, speed):
    """token2wav's ``int(L / speed)`` per row; ``speed`` is a number or one number per row, each > 0."""
    return [int(int(L) / s) for L, s in zip(lengths, _speeds(speed, len(lengths)))]


def change_speed(z, lengths, speed):
    """token2wav's speed step on a right-padded batch of latents: row b's first ``lengths[b]`` frames of z [B, C, L] go
    to ``int(lengths[b] / speed_b)`` frames (linear, align_corners=False; zeros after).  Returns (z', new lengths as a host
    list).  Every speed 1: z itself, untouched (CosyVoice skips the interpolation then)."""
    lengths = [int(v) for v in lengths]
    if all(s == 1.0 for s in _speeds(speed, len(lengths))):
        return z, lengths
    new = speed_lengths(lengths, speed)
    if min(new) < 1:
        raise ValueError(f"speed leaves a row without frames (lengths {lengths} -> {new})")
    dev = z.device
    i32 = lambda v: torch.tensor(v, dtype=torch.int32, device=dev)  # noqa: E731
    return native.latent_resize_linear(z.to(torch.float32).contiguous(), i32(lengths), i32(new), max(new)), new


class VoiceConverter:
    """flow: ``front.CausalMaskedDiffWithXvec``; tokenizer: ``tokenizer.S3TokenizerV2``; dac_encoder / dac_decoder:
    ``dac.DACVAEEncoder`` / ``dac.DACVAEDecoder``.  ``device``: where everything runs (default: the current CUDA device).
    The caller serialises calls and splits large jobs into calls, as for ``StreamingBatch``."""

    def __init__(self, flow, tokenizer, dac_encoder, dac_decoder, device=None):
        self.flow, self.tokenizer, self.dac_encoder, self.dac_decoder = flow, tokenizer, dac_encoder, dac_decoder
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        if self.device.type != "cuda":
            raise RuntimeError("the B200 path runs on CUDA tensors only (no CPU fallback)")

    # -- helpers ---------------------------------------------------------------------------------------------------------
    def _batch(self, audio_list):
        """Right-padded [B, S] on the device and the host lengths."""
        clips = [torch.as_tensor(a).reshape(-1) for a in audio_list]
        if not clips or any(c.numel() < 1 for c in clips):
            raise ValueError("audio_list must hold at least one non-empty clip")
        lens = [c.numel() for c in clips]
        buf = torch.zeros(len(clips), max(lens), device=self.device)
        for b, c in enumerate(clips):
            buf[b, :lens[b]] = c.to(self.device, torch.float32)
        return buf, lens

    def _at(self, buf, lens, sample_rate, rate, out_samples=None):
        """The batch converted to ``rate`` (a no-op when it is there already) and its host lengths."""
        if int(sample_rate) == rate:
            if out_samples is not None and out_samples > buf.shape[1]:
                buf = torch.nn.functional.pad(buf, (0, out_samples - buf.shape[1]))
            return buf, lens
        out, _ = _audio.resample(buf, sample_rate, rate, lens, out_samples)
        return out, [_audio.output_length(n, sample_rate, rate) for n in lens]

    def _tokens(self, buf, lens, sample_rate):
        """S3 token lists [1, T_b] (int64) of the batch, one ``quantize_audio`` call."""
        a16, l16 = self._at(buf, lens, sample_rate, TOKEN_RATE)
        codes, code_len = self.tokenizer.quantize_audio(a16, l16)
        return [codes[b:b + 1, :n].to(torch.int64) for b, n in enumerate(code_len.tolist())]

    # -- public surface --------------------------------------------------------------------------------------------------
    @torch.inference_mode()
    def tokens(self, audio_list, sample_rate):
        """S3 tokens of each recording (GPU resample to 16 kHz, one padded ``quantize_audio``): list of [1, T_b] int64."""
        buf, lens = self._batch(audio_list)
        return self._tokens(buf, lens, sample_rate)

    @torch.inference_mode()
    def prompts(self, audio_list, sample_rate, embedding=None, reference_mels=None):
        """Prompt recordings -> [Prompt], one padded batch for each model.  The DAC-VAE encoder runs in ``lengths`` mode
        with zero noise (``feat`` is the posterior mean m); each clip is zero-padded to a whole number of hops, as
        ``DACVAE.preprocess`` pads it.  ``embedding``: [B, 192] x-vectors (or None); ``reference_mels``: None or one entry
        per prompt (what ``get_speaker_embedding`` takes, or None); neither: zero embeddings."""
        buf, lens = self._batch(audio_list)
        B = len(lens)
        toks = self._tokens(buf, lens, sample_rate)
        enc = self.dac_encoder
        hop = enc.hop_length
        S24 = _audio.output_length(buf.shape[1], sample_rate, enc.sample_rate)
        a24, l24 = self._at(buf, lens, sample_rate, enc.sample_rate, -(-S24 // hop) * hop)
        frames = [-(-n // hop) for n in l24]
        L = a24.shape[1] // hop
        _, m, _ = enc.encode(a24[:, None, :], torch.zeros(B, enc.latent_dim, L, device=self.device), lengths=frames)
        if embedding is not None and tuple(embedding.shape) != (B, self.flow.spk_embed_dim):
            raise ValueError(f"embedding must be [{B}, {self.flow.spk_embed_dim}]")
        if reference_mels is not None and len(reference_mels) != B:
            raise ValueError(f"reference_mels must hold one entry per prompt ({B})")
        out = []
        for b in range(B):
            n = prompt_cut(frames[b], toks[b].shape[1])
            token = toks[b][:, :n].contiguous()
            feat = m[b:b + 1, :, :2 * n].transpose(1, 2).contiguous()
            emb = self.flow.get_speaker_embedding({"embedding": None if embedding is None else embedding[b:b + 1],
                                                   "reference_mels": None if reference_mels is None else reference_mels[b],
                                                   "speech_token": token}, self.device)
            out.append(Prompt(token, feat, emb))
        return out

    @torch.inference_mode()
    def synthesize(self, tokens_list, prompts, speed=1.0):
        """tokens_list: B int tensors ([T_b] or [1, T_b]); prompts: one ``Prompt`` or B of them; speed: a number or B.
        One ``inference_batch`` (finalize=True), the speed change, one length-masked decode -> B 24 kHz waveforms (1-D)."""
        B = len(tokens_list)
        prompts = [prompts] * B if isinstance(prompts, Prompt) else list(prompts)
        if B < 1 or len(prompts) != B:
            raise ValueError("tokens_list and prompts must hold one entry per utterance")
        toks = [torch.as_tensor(t).reshape(1, -1).to(self.device, torch.int64) for t in tokens_list]
        lat, L = self.flow.inference_batch(toks, [p.token for p in prompts], [p.feat for p in prompts],
                                           torch.cat([p.embedding.to(self.device) for p in prompts], dim=0), [True] * B)
        z, lens = change_speed(lat, L.tolist(), speed)
        wav = self.dac_decoder.decode(z, torch.tensor(lens, dtype=torch.int32))
        hop = self.dac_decoder.hop_length
        return [wav[b, 0, :n * hop] for b, n in enumerate(lens)]

    @torch.inference_mode()
    def convert(self, source_list, sample_rate, prompts, speed=1.0):
        """``inference_vc`` for a batch: each source recording spoken with its prompt's voice -> B 24 kHz waveforms."""
        return self.synthesize(self.tokens(source_list, sample_rate), prompts, speed)
