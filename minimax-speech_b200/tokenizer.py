"""The S3 speech tokenizer (SURVEY.md section 8 f-4, second half): log-mel -> 25 Hz FSQ token ids.

Drop-ins for ``s3tokenizer.model_v2.S3TokenizerV2`` (speech/tools/S3Tokenizer/s3tokenizer/model_v2.py:354-415:
``quantize(mel [B, n_mels, T], mel_len [B]) -> (codes int32 [B, T'], code_len int32 [B])``), its ``AudioEncoderV2`` trunk
(:290-351: two stride-2 convolutions, six FSMN-attention blocks with rotary embedding) and its quantizer head
``FSQCodebook`` / ``FSQVectorQuantization`` (:83-147: ``encode(hidden [B, T, dim]) -> int32 tokens [B, T]``), with the
reference's parameter names, so a reference tokenizer checkpoint loads unchanged.  The tokens are the ids (vocabulary
3^8 = 6561) the flow's ``input_embedding`` consumes.  A token is a rounding decision, so the arithmetic is fp32-level in
both precisions of ``ls_s3_quantize``: ``"fp32"`` (default, CUDA cores) and ``"bf16x3"`` (tensor cores: every dense
linear / convolution as A_hi W_hi + A_lo W_hi + A_hi W_lo with hi = bf16(x), lo = bf16(x - hi), fp32 accumulation;
attention, FSMN, LayerNorm and the residual stream in fp32).  Plain bf16 / fp16 operands are refused.  Clips longer
than 30 s take the reference's sliding-window path (model_v2.py:417-588: host-side windowing and merging around one
batched device call).  The log-mel front end (utils.py ``log_mel_spectrogram``, the Whisper front end) is
``log_mel_spectrogram`` here, on the GPU (csrc/s3_mel.cu) for right-padded batches of clips of different lengths, and
``S3TokenizerV2.quantize_audio`` goes from 16 kHz audio to tokens.
"""
import functools
import math

import numpy as np
import torch
import torch.nn as nn

from . import native

SAMPLE_RATE, N_FFT, HOP_LENGTH = 16000, 400, 160
N_BINS = N_FFT // 2 + 1
MIN_SAMPLES = N_FFT // 2 + 1  # torch.stft's reflect padding of 200 samples needs more than 200


def _hz_to_mel(f):
    """librosa.hz_to_mel, Slaney scale (htk=False): linear below 1 kHz, logarithmic above."""
    f = np.asarray(f, dtype=np.float64)
    f_sp, min_log_hz, logstep = 200.0 / 3, 1000.0, np.log(6.4) / 27.0
    mels = f / f_sp
    return np.where(f >= min_log_hz, min_log_hz / f_sp + np.log(np.maximum(f, 1e-300) / min_log_hz) / logstep, mels)


def _mel_to_hz(m):
    """librosa.mel_to_hz, Slaney scale."""
    m = np.asarray(m, dtype=np.float64)
    f_sp, min_log_hz, logstep = 200.0 / 3, 1000.0, np.log(6.4) / 27.0
    min_log_mel = min_log_hz / f_sp
    return np.where(m >= min_log_mel, min_log_hz * np.exp(logstep * (m - min_log_mel)), f_sp * m)


def mel_band_edges(n_mels=128):
    """The n_mels + 2 Slaney-scale frequencies (Hz) that bound and centre the triangles: band m spans edges[m] ..
    edges[m + 2] and peaks at edges[m + 1]."""
    return _mel_to_hz(np.linspace(_hz_to_mel(0.0), _hz_to_mel(SAMPLE_RATE / 2), n_mels + 2))


@functools.lru_cache(maxsize=None)
def _mel_filters_cached(n_mels):
    fft_freqs = np.arange(N_BINS, dtype=np.float64) * (SAMPLE_RATE / N_FFT)
    edges = mel_band_edges(n_mels)
    fdiff = np.diff(edges)
    ramps = edges[:, None] - fft_freqs[None, :]
    weights = np.zeros((n_mels, N_BINS), dtype=np.float32)  # librosa's default dtype: each triangle is stored as
    for i in range(n_mels):                                   # float32, then scaled in place (as librosa does)
        weights[i] = np.maximum(0.0, np.minimum(-ramps[i] / fdiff[i], ramps[i + 2] / fdiff[i + 1]))
    weights *= (2.0 / (edges[2:n_mels + 2] - edges[:n_mels]))[:, None]  # norm="slaney": constant energy per band
    weights.setflags(write=False)
    return weights


def mel_filters(n_mels=128):
    """The Whisper / S3 tokenizer filter bank, float32 [n_mels, 201]: librosa.filters.mel(sr=16000, n_fft=400,
    n_mels=n_mels) -- Slaney mel scale, norm="slaney", fmin 0, fmax 8000 -- restated in float64.  The reference ships it
    as an asset (s3tokenizer/assets/mel_filters.npz, saved from that librosa call); ``load_mel_filters`` reads the asset
    itself for callers who have it."""
    return torch.from_numpy(_mel_filters_cached(int(n_mels)).copy())


def load_mel_filters(path, n_mels=128):
    """The reference's ``mel_filters.npz`` (key ``mel_{n_mels}``) as float32 [n_mels, 201]."""
    with np.load(path, allow_pickle=False) as f:
        w = torch.from_numpy(np.ascontiguousarray(f[f"mel_{n_mels}"], dtype=np.float32))
    if tuple(w.shape) != (n_mels, N_BINS):
        raise ValueError(f"{path}: mel_{n_mels} has shape {tuple(w.shape)}, expected ({n_mels}, {N_BINS})")
    return w


_FILTERS_ON = {}


def _filters_on(n_mels, device):
    key = (int(n_mels), str(device))
    if key not in _FILTERS_ON:
        _FILTERS_ON[key] = mel_filters(n_mels).to(device)
    return _FILTERS_ON[key]


def log_mel_spectrogram(audio, n_mels=128, padding=0, device=None, audio_len=None, filters=None):
    """utils.py ``log_mel_spectrogram`` on the GPU (csrc/s3_mel.cu).

    A 1-D clip (tensor or numpy array) returns ``[n_mels, len // 160]`` like the reference.  A right-padded batch
    ``[B, S]`` returns ``(mel [B, n_mels, S // 160], mel_len [B] int32)``; clip b is computed from its first
    ``audio_len[b]`` samples alone (default: all S), exactly as a call with that clip alone would, and frames at or past
    ``mel_len[b] = audio_len[b] // 160`` are zero.  ``padding`` appends that many zeros to every clip, as the reference
    does.  ``filters``: [n_mels, 201] (default ``mel_filters(n_mels)``; ``load_mel_filters`` gives the reference's
    asset).  ``device``: where to compute (the audio is moved there); without it the audio must already be on a CUDA
    device.  Lengths are checked on the host: every clip needs 201 <= length <= S."""
    if isinstance(audio, np.ndarray):
        audio = torch.from_numpy(audio)
    if not isinstance(audio, torch.Tensor) or audio.dim() not in (1, 2):
        raise ValueError(f"audio must be a 1-D clip or a [B, S] batch, got {getattr(audio, 'shape', type(audio))}")
    if device is not None:
        audio = audio.to(device)
    if audio.device.type != "cuda":
        raise RuntimeError("the B200 path runs on CUDA tensors only (no CPU fallback)")
    if not 1 <= int(n_mels) <= 128:
        raise ValueError(f"n_mels must be in [1, 128], got {n_mels}")
    dev = audio.device
    single = audio.dim() == 1
    audio = audio.to(torch.float32).reshape(-1 if single else audio.shape[0], audio.shape[-1])
    B, S = audio.shape
    if audio_len is None:
        lens = [S] * B
    else:
        lens = [int(v) for v in (audio_len.tolist() if isinstance(audio_len, torch.Tensor) else audio_len)]
        if len(lens) != B:
            raise ValueError(f"audio_len has {len(lens)} entries for a batch of {B}")
    bad = [n for n in lens if not MIN_SAMPLES <= n <= S]
    if bad:
        raise ValueError(f"every clip needs {MIN_SAMPLES} <= length <= {S} samples (reflect padding of {N_FFT // 2}), "
                         f"got {bad[:4]}")
    if padding > 0:
        keep = torch.arange(S, device=dev)[None, :] < torch.tensor(lens, device=dev)[:, None]
        audio = torch.nn.functional.pad(torch.where(keep, audio, torch.zeros((), device=dev)), (0, int(padding)))
        lens = [n + int(padding) for n in lens]
        S += int(padding)
    if filters is None:
        filters = _filters_on(n_mels, dev)
    if tuple(filters.shape) != (n_mels, N_BINS):
        raise ValueError(f"filters must be [{n_mels}, {N_BINS}], got {tuple(filters.shape)}")
    filters = filters.to(device=dev, dtype=torch.float32).contiguous()
    mel, mel_len = native.s3_log_mel(audio.contiguous(), torch.tensor(lens, dtype=torch.int32, device=dev), filters)
    return mel[0] if single else (mel, mel_len)


class FSQCodebook(nn.Module):
    def __init__(self, dim=1280, level=3, weight_seed=0):
        super().__init__()
        if level != 3:
            raise NotImplementedError("level 3 (codebook size 3^8), the reference's only configuration")
        self.level = level
        g = torch.Generator().manual_seed(weight_seed)
        bound = 1.0 / math.sqrt(dim)  # nn.Linear's default initialiser
        self.project_down = nn.Linear(dim, 8)
        with torch.no_grad():
            self.project_down.weight.copy_((torch.rand(8, dim, generator=g) * 2 - 1) * bound)
            self.project_down.bias.copy_((torch.rand(8, generator=g) * 2 - 1) * bound)
        for p in self.parameters():
            p.requires_grad_(False)

    @torch.inference_mode()
    def encode(self, x):
        if x.dim() != 3 or x.shape[-1] != self.project_down.in_features:
            raise ValueError(f"hidden must be [B, T, {self.project_down.in_features}], got {tuple(x.shape)}")
        if x.device.type != "cuda":
            raise RuntimeError("the B200 path runs on CUDA tensors only (no CPU fallback)")
        dev = x.device
        w = self.project_down.weight.to(device=dev, dtype=torch.float32).contiguous()
        b = self.project_down.bias.to(device=dev, dtype=torch.float32).contiguous()
        return native.fsq_encode(x.to(torch.float32).contiguous(), w, b)

    def decode(self, embed_ind):
        raise NotImplementedError("There is no official up project component provided")  # model_v2.py:114-117


class FSQVectorQuantization(nn.Module):
    """model_v2.py:120-147."""

    def __init__(self, dim=1280, codebook_size=3 ** 8, weight_seed=0):
        super().__init__()
        assert 3 ** 8 == codebook_size
        self._codebook = FSQCodebook(dim=dim, level=3, weight_seed=weight_seed)
        self.codebook_size = codebook_size

    def encode(self, x):
        return self._codebook.encode(x)


def precompute_rotary(dim=64, end=2048, theta=10000.0):
    """precompute_freqs_cis (model_v2.py:37-48) with the reference's own torch expressions -> (cos, sin) [end, dim/2]."""
    freqs = 1.0 / (theta ** (torch.arange(0, dim, 2)[:(dim // 2)].float() / dim))
    ang = torch.outer(torch.arange(end), freqs).float()
    cis = torch.polar(torch.ones_like(ang), ang)
    real = torch.view_as_real(cis)
    return real[..., 0].contiguous(), real[..., 1].contiguous()


class _Block(nn.Module):
    """Parameter container with ResidualAttentionBlock's names (model_v2.py:252-273)."""

    def __init__(self, n_state, kernel_size=31):
        super().__init__()
        self.attn = nn.Module()
        self.attn.query = nn.Linear(n_state, n_state)
        self.attn.key = nn.Linear(n_state, n_state, bias=False)
        self.attn.value = nn.Linear(n_state, n_state)
        self.attn.out = nn.Linear(n_state, n_state)
        self.attn.fsmn_block = nn.Conv1d(n_state, n_state, kernel_size, groups=n_state, bias=False)
        self.attn_ln = nn.LayerNorm(n_state, eps=1e-6)
        self.mlp = nn.Sequential(nn.Linear(n_state, 4 * n_state), nn.GELU(), nn.Linear(4 * n_state, n_state))
        self.mlp_ln = nn.LayerNorm(n_state)


class S3TokenizerV2(nn.Module):
    """model_v2.py:354-415.  ``S3TokenizerV2(name, config)`` like the reference; ``config`` may be the reference's
    ``ModelConfig`` or anything with its attribute names (n_mels, n_audio_state, n_audio_head, n_audio_layer)."""

    def __init__(self, name="speech_tokenizer_v2_25hz", config=None, weight_seed=None, precision="fp32"):
        super().__init__()
        self.name = name
        self.precision = native.check_s3_precision(precision)
        g = lambda k, d: getattr(config, k, d) if config is not None else d
        self.n_mels, self.n_state = g("n_mels", 128), g("n_audio_state", 1280)
        self.n_head, self.n_layer = g("n_audio_head", 20), g("n_audio_layer", 6)
        if self.n_state != 64 * self.n_head:
            raise NotImplementedError("64-wide heads: the reference precomputes its rotary table for them (model_v2.py:307)")
        self.encoder = nn.Module()
        self.encoder.conv1 = nn.Conv1d(self.n_mels, self.n_state, 3, stride=2, padding=1)
        self.encoder.conv2 = nn.Conv1d(self.n_state, self.n_state, 3, stride=2, padding=1)
        self.encoder.blocks = nn.ModuleList([_Block(self.n_state) for _ in range(self.n_layer)])
        self.quantizer = FSQVectorQuantization(self.n_state, 3 ** 8)
        if weight_seed is not None:
            from . import synth
            self.load_state_dict(synth.s3_tokenizer_state_dict(weight_seed, self.n_mels, self.n_state, self.n_head, self.n_layer))
        for p in self.parameters():
            p.requires_grad_(False)
        # the front end's filter bank: not a reference weight, so kept out of state_dict() (strict loads still work)
        self.register_buffer("mel_filters", mel_filters(self.n_mels), persistent=False)
        self._handle = None

    def load_state_dict(self, state_dict, strict=True, **kw):
        self._handle = None
        return super().load_state_dict(state_dict, strict=strict, **kw)

    def handle(self, device):
        device = torch.device(device)
        native.check_s3_precision(self.precision)  # (the attribute may have been changed since)
        if self._handle is None or self._handle.device != device or self._handle.precision != self.precision:
            sd = {k: v.detach().to(torch.float32).contiguous() for k, v in self.state_dict().items()}
            sd["rotary.cos"], sd["rotary.sin"] = precompute_rotary(64, 1024 * 2)  # model_v2.py:307
            self._handle = native.S3Handle(sd, device, self.precision)
        return self._handle

    @torch.inference_mode()
    def quantize(self, mel, mel_len, return_hidden=False):
        if mel.dim() != 3 or mel.shape[1] != self.n_mels:
            raise ValueError(f"mel must be [B, {self.n_mels}, T], got {tuple(mel.shape)}")
        if mel.device.type != "cuda":
            raise RuntimeError("the B200 path runs on CUDA tensors only (no CPU fallback)")
        dev = mel.device
        lens = [int(v) for v in mel_len.tolist()]  # (the reference reads the lengths on the host as well: .any(), .item())
        if max(lens) > self.MAX_FRAMES:
            if return_hidden:
                raise ValueError("return_hidden is only defined for batches without clips longer than 30 s")
            return self._quantize_mixed_batch(mel.to(torch.float32), lens)
        return self.handle(dev).quantize(mel.to(torch.float32).contiguous(),
                                         torch.tensor(lens, dtype=torch.int32, device=dev), want_hidden=return_hidden)

    @torch.inference_mode()
    def quantize_audio(self, audio, audio_len):
        """16 kHz audio to tokens: ``log_mel_spectrogram`` (on the GPU, per-clip lengths) then ``quantize``.
        audio [B, S] (right-padded, on a CUDA device), audio_len [B] host lengths in samples (201 <= len <= S) ->
        the outputs of ``quantize`` for mel_len = audio_len // 160 (clips over 30 s take the sliding-window path).
        mel_len is computed on the host, so nothing is read back from the device before ``quantize``."""
        if audio.dim() != 2:
            raise ValueError(f"audio must be [B, S], got {tuple(audio.shape)}")
        lens = [int(v) for v in (audio_len.tolist() if isinstance(audio_len, torch.Tensor) else audio_len)]
        mel, _ = log_mel_spectrogram(audio, self.n_mels, audio_len=lens, filters=self._filters_on(audio.device))
        return self.quantize(mel, torch.tensor([n // HOP_LENGTH for n in lens], dtype=torch.int32))

    def _filters_on(self, device):
        """The filter bank on ``device``: the buffer itself when the module lives there, else a copy kept until the
        buffer changes (no host-to-device copy per call)."""
        f = self.mel_filters
        if f.device == torch.device(device):
            return f
        key = (str(device), id(f), f._version)
        if getattr(self, "_filters_copy", (None,))[0] != key:
            self._filters_copy = (key, f.to(device))
        return self._filters_copy[1]

    MAX_FRAMES = 3000       # 30 s of 100 Hz mel frames (model_v2.py:399-401)
    WINDOW, OVERLAP = 3000, 400  # 30 s windows overlapping by 4 s (model_v2.py:436-445)

    def _quantize_mixed_batch(self, mel, lens):
        """model_v2.py:417-588: clips longer than 30 s are cut into 30 s windows every 26 s, every window (and every short
        clip, padded to 30 s) goes through the encoder in ONE batch, and a long clip's token lists are joined by dropping
        half of each overlap on either side of a seam (utils.py merge_tokenized_segments).  int64 ids, like the reference's."""
        dev = mel.device
        stride = self.WINDOW - self.OVERLAP
        segs, seg_lens, owner = [], [], []
        for b, n in enumerate(lens):
            starts = [0] if n <= self.MAX_FRAMES else list(range(0, n, stride))
            for st in starts:
                piece = mel[b, :, st:min(st + self.WINDOW, n)]
                seg_lens.append(piece.shape[1])
                segs.append(torch.nn.functional.pad(piece, (0, self.WINDOW - piece.shape[1])))
                owner.append(b)
        codes, code_len = self.handle(dev).quantize(torch.stack(segs).contiguous(),
                                                    torch.tensor(seg_lens, dtype=torch.int32, device=dev))
        codes, code_len = codes.cpu(), code_len.tolist()
        half = (self.OVERLAP // 100 // 2) * 25  # tokens in half of the overlap: (4 s // 2) * 25 Hz
        merged = [[] for _ in lens]
        for b in range(len(lens)):
            mine = [i for i, o in enumerate(owner) if o == b]
            for j, i in enumerate(mine):
                toks = codes[i, :code_len[i]].tolist()
                if lens[b] > self.MAX_FRAMES:
                    toks = toks[(0 if j == 0 else half):(len(toks) - half if j != len(mine) - 1 else len(toks))]
                merged[b].extend(toks)
        out = torch.zeros(len(lens), max(len(m) for m in merged), dtype=torch.long)
        for b, m in enumerate(merged):
            out[b, :len(m)] = torch.tensor(m, dtype=torch.long)
        return out.to(dev), torch.tensor([len(m) for m in merged], dtype=torch.long, device=dev)

    def forward(self, mel, mel_len):
        return self.quantize(mel, mel_len)
