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
batched device call).  Not built: the log-mel front end (utils.py ``log_mel_spectrogram``: an STFT with
a filter bank shipped as an asset file).
"""
import math

import torch
import torch.nn as nn

from . import native


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
