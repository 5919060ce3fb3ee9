"""Sample-rate conversion on the GPU (csrc/resample.cu): ``torchaudio.functional.resample`` at its defaults
(``sinc_interp_hann``, ``lowpass_filter_width=6``, ``rolloff=0.99``) -- the resampler the S3 tokenizer's ``load_audio``
and CosyVoice's front end use -- for single clips and right-padded batches of clips of different lengths, each clip
converted as if it were alone.  The S3 tokenizer wants 16 kHz and the DAC-VAE 24 kHz; one recording at any integer rate
reaches both without a host-side resampler."""
import math

import numpy as np
import torch

from . import native

_HANDLES = {}


def reduced_ratio(orig_freq, new_freq):
    """(O, N): orig_freq / new_freq reduced by their gcd (1, 1 for equal rates)."""
    g = math.gcd(int(orig_freq), int(new_freq))
    return int(orig_freq) // g, int(new_freq) // g


def output_length(n_samples, orig_freq, new_freq):
    """Samples of a clip of ``n_samples`` at ``orig_freq`` after conversion to ``new_freq``: ceil(N n / O), as torchaudio
    computes it (its float64 ceil equals this integer form for any realistic length)."""
    O, N = reduced_ratio(orig_freq, new_freq)
    return -(-N * int(n_samples) // O)


def resampler(orig_freq, new_freq, device):
    """The ``native.ResamplerHandle`` of (orig_freq, new_freq) on ``device``, created once (one table upload) and reused."""
    device = torch.device(device)
    if device.type == "cuda" and device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    key = (int(orig_freq), int(new_freq), str(device))
    h = _HANDLES.get(key)
    if h is None:
        h = _HANDLES[key] = native.ResamplerHandle(orig_freq, new_freq, device)
    return h


def resample(audio, orig_freq, new_freq, audio_len=None, out_samples=None):
    """``torchaudio.functional.resample(audio, orig_freq, new_freq)`` on the GPU.

    A 1-D clip returns the converted 1-D clip.  A right-padded batch ``[B, S]`` returns ``(out [B, S_out], out_len [B]
    int32)`` (both on the audio's device): clip b is the first ``audio_len[b]`` samples of its row (host lengths, default
    all S) and is converted exactly as if alone, bitwise; ``out_len[b] = output_length(audio_len[b], ...)``, and ``out``
    is zero from there on.  ``out_samples`` (default ``output_length(S, ...)``, and never less) sets S_out, e.g. to a
    multiple of a hop.  The audio must be on a CUDA device: there is no CPU fallback."""
    if isinstance(audio, np.ndarray):
        audio = torch.from_numpy(audio)
    if not isinstance(audio, torch.Tensor) or audio.dim() not in (1, 2):
        raise ValueError(f"audio must be a 1-D clip or a [B, S] batch, got {getattr(audio, 'shape', type(audio))}")
    if audio.device.type != "cuda":
        raise RuntimeError("the B200 path runs on CUDA tensors only (no CPU fallback)")
    if int(orig_freq) != orig_freq or int(new_freq) != new_freq or orig_freq <= 0 or new_freq <= 0:
        raise ValueError(f"rates must be positive integers, got {orig_freq} -> {new_freq}")
    single = audio.dim() == 1
    x = audio.to(torch.float32).reshape(1 if single else audio.shape[0], audio.shape[-1]).contiguous()
    B, S = x.shape
    if S < 1:
        raise ValueError("audio must hold at least one sample")
    if single or audio_len is None:
        lens = [S] * B
    else:
        lens = [int(v) for v in (audio_len.tolist() if isinstance(audio_len, torch.Tensor) else audio_len)]
        if len(lens) != B:
            raise ValueError(f"audio_len has {len(lens)} entries for a batch of {B}")
        bad = [n for n in lens if not 1 <= n <= S]
        if bad:
            raise ValueError(f"every clip needs 1 <= length <= {S} samples, got {bad[:4]}")
    need = output_length(S, orig_freq, new_freq)
    S_out = need if out_samples is None else int(out_samples)
    if S_out < need:
        raise ValueError(f"out_samples must be at least {need} (ceil({new_freq} * {S} / {orig_freq}))")
    h = resampler(orig_freq, new_freq, x.device)
    out, out_len = h.resample(x, torch.tensor(lens, dtype=torch.int32, device=x.device), S_out)
    return out[0] if single else (out, out_len)
