"""Token -> mu front half of ``CausalMaskedDiffWithXvec.inference`` (speech/cosyvoice/flow/flow.py:437-511; SURVEY.md
section 8 row f-1): speaker-embedding normalise + ``spk_embed_affine_layer``, ``input_embedding``, the
``UpsampleConformerEncoder`` (transformer/upsample_encoder.py) and ``encoder_proj``.  Parameters are registered under the
reference's state_dict keys, so the flow checkpoint loads unchanged.  ``precision="bf16"`` (default): tensor-core path
(csrc/front_engine.cu); ``"fp32"``: CUDA-core kernels of csrc/f32_path.cu.  Equal-length or right-padded batches; final chunks
(finalize=True) and non-final chunks (3 look-ahead context tokens), optional block-causal streaming attention; ``encode_sessions``
batches independent calls with a per-row look-ahead.  ``CausalMaskedDiffWithXvec`` is the drop-in for the reference's
pipeline class: the same ``inference`` signature (prompt tokens, prompt latents, x-vector or reference mels), and
``inference_batch`` for many utterances in one call."""
import torch
import torch.nn as nn

from . import native, synth
from .flow import _as_f32, _register_tree
from .speaker import LearnableSpeakerEncoder


_FRONT_PREFIXES = ("input_embedding.", "encoder.", "encoder_proj.", "spk_embed_affine_layer.")


class TokenToMu(nn.Module):
    def __init__(self, input_size=512, output_size=80, spk_embed_dim=192, vocab_size=6561, attention_heads=8,
                 linear_units=2048, num_blocks=6, weight_seed=7, precision="bf16", **_ignored):
        super().__init__()
        precision = native.check_precision(precision)
        if input_size != attention_heads * 64:
            raise NotImplementedError("head dim 64 only (config.yaml:73-88: 512 / 8)")
        self.precision, self.output_size, self.spk_embed_dim, self.vocab_size = precision, output_size, spk_embed_dim, vocab_size
        _register_tree(self, synth.conformer_encoder_state_dict(weight_seed, d=input_size, heads=attention_heads, ff=linear_units,
                                                                num_blocks=num_blocks, out_dim=output_size, vocab=vocab_size,
                                                                spk_dim=spk_embed_dim))
        self._handle = None

    def load_state_dict(self, state_dict, strict=True, **kw):
        self._handle = None
        keep = {k: v for k, v in state_dict.items() if k.startswith(_FRONT_PREFIXES)}
        return super().load_state_dict(keep, strict=strict, **kw)

    def handle(self, device):
        device = torch.device(device)
        if device.type != "cuda":
            raise RuntimeError("the B200 hot path runs on CUDA tensors only (no CPU fallback)")
        if self._handle is None or self._handle.device != device or self._handle.precision != self.precision:
            sd = {k: v for k, v in self.state_dict().items() if k.startswith(_FRONT_PREFIXES)}
            self._handle = native.FrontHandle(sd, device, self.precision)
        return self._handle

    pre_lookahead_len = 3

    @torch.inference_mode()
    def forward(self, token, embedding, finalize=True, streaming=False, token_len=None):
        """token [B,T] int64, embedding [B,192] -> (mu [B,80,2T'], spks [B,80]): the ``mu`` / ``spks`` the reference hands to
        ``self.decoder`` (flow.py:501-508).  finalize=False: the last 3 tokens are look-ahead context (T' = T - 3).
        token_len [B] (optional): token counts of a right-padded batch, handled like the reference encoder's ``xs_lens``
        (zero embeddings and masked keys past the length); mu is zero past ``2 * token_len``."""
        n_ctx = 0 if finalize else self.pre_lookahead_len
        if token.dim() != 2 or token.shape[1] < 1 + n_ctx or token.dtype != torch.int64:
            raise ValueError(f"token must be an int64 tensor [B, T >= {1 + n_ctx}]")
        if tuple(embedding.shape) != (token.shape[0], self.spk_embed_dim):
            raise ValueError(f"embedding must be [{token.shape[0]}, {self.spk_embed_dim}]")
        dev = token.device
        if token_len is not None:
            token_len = torch.as_tensor(token_len).reshape(-1)
            if token_len.numel() != token.shape[0] or int(token_len.min()) < 1 or int(token_len.max()) > token.shape[1]:
                raise ValueError("token_len must hold one count in [1, T] per utterance")
            if n_ctx:
                raise NotImplementedError("right-padded batches of non-final chunks (the reference call is batch 1)")
            token_len = token_len.to(device=dev, dtype=torch.int32).contiguous()
        return self.handle(dev).encode(token.contiguous(), _as_f32(embedding, dev), n_ctx, streaming, token_len)

    @torch.inference_mode()
    def encode_sessions(self, token, token_len, n_context, embedding, streaming=False):
        """A batch of independent calls in one launch sequence (e.g. one streaming hop of each of B sessions).
        token [B,T_all] int64, right-padded; token_len [B]: tokens of each row, look-ahead included; n_context [B]: 0
        (finalize=True) or 3 (the last 3 tokens are look-ahead context) per row; embedding [B,192].  Row b comes out
        exactly as ``forward`` of that row alone with its own ``finalize``: -> (mu [B,80,2T], spks [B,80]) with
        T = max(token_len - n_context), mu zero past ``2 * (token_len[b] - n_context[b])``.  The padding is never read."""
        if token.dim() != 2 or token.shape[1] < 1 or token.dtype != torch.int64:
            raise ValueError("token must be an int64 tensor [B, T_all >= 1]")
        B, T_all = token.shape
        if tuple(embedding.shape) != (B, self.spk_embed_dim):
            raise ValueError(f"embedding must be [{B}, {self.spk_embed_dim}]")
        n = torch.as_tensor(token_len).detach().cpu().reshape(-1)
        c = torch.as_tensor(n_context).detach().cpu().reshape(-1)
        if n.numel() != B or c.numel() != B or n.is_floating_point() or c.is_floating_point():
            raise ValueError(f"token_len and n_context must be {B} integers each")
        if bool(((c != 0) & (c != self.pre_lookahead_len)).any()):
            raise ValueError(f"n_context must be 0 or {self.pre_lookahead_len} per row")
        if bool(((n - c < 1) | (n > T_all)).any()):
            raise ValueError(f"token_len must leave at least one token after the context and be at most {T_all}")
        dev = token.device
        i32 = lambda t: t.to(dtype=torch.int32).to(dev)  # noqa: E731
        return self.handle(dev).encode_sessions(token.contiguous(), _as_f32(embedding, dev), int((n - c).max()), i32(n), i32(c),
                                                streaming)

    @torch.inference_mode()
    def inference(self, token, embedding, decoder, n_timesteps=10, streaming=False, finalize=True):
        """``CausalMaskedDiffWithXvec.inference`` without prompt (flow.py:437-511): tokens -> latents [B,80,2T']."""
        mu, spks = self.forward(token, embedding, finalize=finalize, streaming=streaming)
        mask = torch.ones(mu.shape[0], 1, mu.shape[2], device=mu.device)
        feat, _ = decoder(mu=mu, mask=mask, spks=spks, cond=torch.zeros_like(mu), n_timesteps=n_timesteps, streaming=streaming)
        return feat.float(), None


class UpsampleConformerEncoder:
    """Constructor-argument holder with the signature of ``cosyvoice.transformer.upsample_encoder.UpsampleConformerEncoder``
    (upsample_encoder.py:110-180), so that speech/config.yaml:73-88 can name this class for the ``encoder:`` entry of the
    drop-in ``CausalMaskedDiffWithXvec``.  The parameters live on the pipeline module (keys ``encoder.*``); only the
    configuration of config.yaml is built (rel-pos self-attention, linear input layer, no macaron / CNN module)."""

    def __init__(self, input_size=512, output_size=512, attention_heads=8, linear_units=2048, num_blocks=6, dropout_rate=0.1,
                 positional_dropout_rate=0.1, attention_dropout_rate=0.1, input_layer="linear", pos_enc_layer_type="rel_pos_espnet",
                 normalize_before=True, static_chunk_size=25, use_dynamic_chunk=False, global_cmvn=None,
                 use_dynamic_left_chunk=False, positionwise_conv_kernel_size=1, macaron_style=False,
                 selfattention_layer_type="rel_selfattn", activation_type="swish", use_cnn_module=False, cnn_module_kernel=15,
                 causal=False, cnn_module_norm="batch_norm", key_bias=True, gradient_checkpointing=False):
        if (input_size != output_size or input_layer != "linear" or pos_enc_layer_type != "rel_pos_espnet" or not normalize_before
                or macaron_style or use_cnn_module or selfattention_layer_type != "rel_selfattn" or activation_type != "swish"
                or static_chunk_size != 25 or not key_bias or global_cmvn is not None):
            raise NotImplementedError("B200 token encoder covers config.yaml:73-88's UpsampleConformerEncoder only")
        self.kwargs = dict(input_size=input_size, attention_heads=attention_heads, linear_units=linear_units, num_blocks=num_blocks)

    def output_size(self):
        return self.kwargs["input_size"]


class CausalMaskedDiffWithXvec(TokenToMu):
    """Drop-in for ``cosyvoice.flow.flow.CausalMaskedDiffWithXvec`` (speech/cosyvoice/flow/flow.py:201-511), inference only:
    same constructor keywords as speech/config.yaml:61-116 (``encoder`` = an ``UpsampleConformerEncoder`` holder, its keyword dict or None, ``decoder`` = a
    ``CausalConditionalCFM``), same ``inference(...)`` signature and return value, same state_dict keys
    (``input_embedding.*``, ``encoder.*``, ``encoder_proj.*``, ``spk_embed_affine_layer.*``, ``speaker_encoder.*``,
    ``decoder.estimator.*``), so the reference's flow checkpoint loads with ``load_state_dict`` unchanged.  ``forward`` (the
    training losses) is out of scope."""

    def __init__(self, input_size=512, output_size=80, spk_embed_dim=192, output_type="mel", vocab_size=6561, input_frame_rate=25,
                 only_mask_loss=True, token_latent_ratio=2, pre_lookahead_len=3, use_speaker_encoder=False,
                 freeze_speaker_encoder=False, max_conditioning_inputs=2, speaker_encoder_path=None, encoder=None, decoder=None,
                 precision="bf16", **_ignored):
        if decoder is None:
            raise ValueError("decoder (a CausalConditionalCFM) is required")
        if pre_lookahead_len != TokenToMu.pre_lookahead_len:
            raise NotImplementedError("pre_lookahead_len = 3 only (config.yaml:70)")
        enc = dict(encoder.kwargs if isinstance(encoder, UpsampleConformerEncoder) else (encoder or {}))
        if enc.pop("input_size", input_size) != input_size:
            raise ValueError("encoder input_size must equal the pipeline's input_size")
        super().__init__(input_size=input_size, output_size=output_size, spk_embed_dim=spk_embed_dim, vocab_size=vocab_size,
                         precision=precision, **enc)
        self.input_size, self.input_frame_rate, self.token_latent_ratio = input_size, input_frame_rate, token_latent_ratio
        self.use_speaker_encoder = use_speaker_encoder
        self.decoder = decoder
        if use_speaker_encoder:
            self.speaker_encoder = LearnableSpeakerEncoder(mel_dim=80, model_dim=512, output_dim=spk_embed_dim, num_blocks=6,
                                                           num_heads=8, precision=precision)
            if speaker_encoder_path is not None:  # flow.py:270-305: the speaker_encoder.* entries of an LLM checkpoint
                ck = torch.load(speaker_encoder_path, map_location="cpu")
                sd = ck["state_dict"] if "state_dict" in ck else {k: v for k, v in ck.items() if k not in ("epoch", "step")}
                sub = {k.replace("module.", "").replace("speaker_encoder.", ""): v for k, v in sd.items() if "speaker_encoder." in k}
                if sub:
                    self.speaker_encoder.load_state_dict(sub, strict=True)

    def load_state_dict(self, state_dict, strict=True, **kw):
        self._handle = None
        if self.use_speaker_encoder:
            self.speaker_encoder._handle = None
        return nn.Module.load_state_dict(self, state_dict, strict=strict, **kw)

    def get_speaker_embedding(self, batch, device):
        """flow.py:327-378 (inference branches): reference mels -> speaker encoder, else the given x-vector, else zeros."""
        if self.use_speaker_encoder and batch.get("reference_mels") is not None:
            emb = self.speaker_encoder.encode_references(batch["reference_mels"].to(device))
            return torch.nn.functional.normalize(emb, dim=1)
        if batch.get("embedding") is not None:
            return torch.nn.functional.normalize(batch["embedding"].to(device).float(), dim=1)
        return torch.zeros(batch["speech_token"].shape[0], self.spk_embed_dim, device=device)

    @torch.inference_mode()
    def inference(self, token, token_len, prompt_token, prompt_token_len, prompt_feat, prompt_feat_len, embedding=None,
                  reference_mels=None, reference_mel_lengths=None, reference_mel_masks=None, streaming=False, finalize=False):
        """flow.py:437-511.  token [1,T] / prompt_token [1,Tp] int, prompt_feat [1,Fp,80] -> (latents [1,80,2(T [-3])] fp32, None).
        The lengths must equal the tensors' extents (the reference's batch-1 call always passes them that way)."""
        if token.shape[0] != 1:
            raise AssertionError("batch 1 only, as in the reference (flow.py:453)")
        dev = token.device
        for name, t, n in (("token", token, token_len), ("prompt_token", prompt_token, prompt_token_len)):
            if n is not None and int(torch.as_tensor(n).reshape(-1)[0]) != t.shape[1]:
                raise ValueError(f"{name}_len must equal {name}.shape[1] (padded single utterances are not supported)")
        embedding = self.get_speaker_embedding({"reference_mels": reference_mels, "embedding": embedding, "speech_token": token}, dev)
        tok = torch.cat([prompt_token.to(dev), token], dim=1).to(torch.int64)
        # the front half normalises its input again: a no-op on the unit vector, and the all-zero vector stays zero
        mu, spks = TokenToMu.forward(self, tok, embedding, finalize=finalize, streaming=streaming)
        mel_len1 = prompt_feat.shape[1]
        if mu.shape[2] < mel_len1:
            raise ValueError("prompt_feat is longer than the encoded token sequence")
        cond = torch.zeros_like(mu)
        cond[:, :, :mel_len1] = _as_f32(prompt_feat, dev).transpose(1, 2)
        mask = torch.ones(1, 1, mu.shape[2], device=dev)
        feat, _ = self.decoder(mu=mu, mask=mask, spks=spks, cond=cond, n_timesteps=10, streaming=streaming)
        return feat[:, :, mel_len1:].float(), None

    @torch.inference_mode()
    def inference_batch(self, token, prompt_token, prompt_feat, embedding, finalize, streaming=False):
        """Padded-batch form of ``inference``: B independent utterances in one front call and one ``self.decoder`` call,
        each equal to ``inference`` on it alone.  token, prompt_token: lists of B int tensors [1,T_b] / [1,Tp_b];
        prompt_feat: list of B [1,Fp_b,80]; embedding [B,192]: each utterance's speaker embedding as
        ``get_speaker_embedding`` returns it (used as is: normalising a unit vector again can change its last bits);
        finalize: B bools (False: the last 3 tokens are look-ahead context).
        -> (latents [B,80,max L] fp32, L [B] int64 on the host) with L_b = 2 (Tp_b + T_b [- 3]) - Fp_b; zero past L_b."""
        B = len(token)
        if B < 1 or not len(prompt_token) == len(prompt_feat) == len(finalize) == B:
            raise ValueError("token, prompt_token, prompt_feat and finalize must hold one entry per utterance")
        dev = embedding.device
        rows = [torch.cat([p.reshape(-1).to(dev, torch.int64), t.reshape(-1).to(dev, torch.int64)]) for p, t in zip(prompt_token, token)]
        n = torch.tensor([r.numel() for r in rows])
        ctx = torch.tensor([0 if f else self.pre_lookahead_len for f in finalize])
        mu, spks = self.encode_sessions(torch.nn.utils.rnn.pad_sequence(rows, batch_first=True), n, ctx, embedding, streaming)
        frames = 2 * (n - ctx)
        pf = torch.tensor([p.shape[1] for p in prompt_feat])
        if bool((frames < pf).any()):
            raise ValueError("prompt_feat is longer than the encoded token sequence")
        T2 = mu.shape[2]
        mask = (torch.arange(T2)[None, :] < frames[:, None]).float()[:, None, :].to(dev)
        cond = torch.zeros_like(mu)
        for b, p in enumerate(prompt_feat):
            cond[b, :, :p.shape[1]] = _as_f32(p, dev)[0].transpose(0, 1)
        feat, _ = self.decoder(mu=mu, mask=mask, spks=spks, cond=cond, n_timesteps=10, streaming=streaming)
        # per-utterance cut at its prompt: frame Fp_b + t of row b -> frame t
        L = frames - pf
        t = torch.arange(int(L.max()))[None, :]
        idx = (pf[:, None] + t).clamp(max=T2 - 1).to(dev)
        out = feat.float().gather(2, idx[:, None, :].expand(B, feat.shape[1], -1))
        return torch.where((t < L[:, None]).to(dev)[:, None, :], out, 0.0), L

    def forward(self, batch, device):
        raise NotImplementedError("training (flow.py:380-435) is out of scope; inference only")
