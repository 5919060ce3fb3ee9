"""Drop-in DAC-VAE decoder: ``decode(z [B,latent,L]) -> [B,1,L*hop]`` (dac-vae/model.py:485-488).

``DACVAEDecoder`` carries the ``decoder.*`` / ``de_conv_pre.*`` half of the reference ``DACVAE``
state_dict (weight_g / weight_v / bias / alpha keys, SURVEY.md Appendix B) and loads reference
checkpoints (``ckpt['generator']``, dac-vae/inference.py:42-46) with ``strict=False`` semantics for the
encoder keys it does not own.  ``patch_reference_model`` swaps ``decode`` on an instance of the reference
class instead.  The encoder (``encode``) is out of scope (SURVEY.md section 8f-3).
"""
import torch
import torch.nn as nn

from . import native, ops, synth
from .flow import _as_f32, _register_tree


class DACVAEDecoder(nn.Module):
    def __init__(self, latent_dim=80, decoder_dim=1536, decoder_rates=(5, 4, 4, 3, 2), sample_rate=24000,
                 d_out=1, weight_seed=0, precision="bf16", **_ignored):
        super().__init__()
        self.precision = native.check_precision(precision, fp16_ok=True)
        if d_out != 1:
            raise NotImplementedError("mono output only (configx2.yml: d_out=1)")
        self.latent_dim, self.decoder_dim, self.decoder_rates = latent_dim, decoder_dim, list(decoder_rates)
        self.sample_rate = sample_rate
        self.hop_length = 1
        for r in decoder_rates:
            self.hop_length *= r
        _register_tree(self, synth.dac_decoder_state_dict(weight_seed, "reference", latent_dim=latent_dim,
                                                          decoder_dim=decoder_dim, decoder_rates=decoder_rates))
        self._handle = None
        self._register_load_state_dict_pre_hook(lambda *a, **k: self.invalidate())

    @property
    def device(self):
        return next(self.parameters()).device

    def invalidate(self):
        self._handle = None

    def load_state_dict(self, state_dict, strict=True, **kw):
        own = {k: v for k, v in state_dict.items() if k.startswith(("decoder.", "de_conv_pre."))}
        return super().load_state_dict(own, strict=strict, **kw)

    def handle(self, device):
        device = torch.device(device)
        if device.type != "cuda":
            raise RuntimeError("the B200 hot path runs on CUDA tensors only (no CPU fallback)")
        if self._handle is None or self._handle.device != device or self._handle.precision != self.precision:
            self._handle = native.DacHandle(self.state_dict(), device, self.precision)
        return self._handle

    @torch.inference_mode()
    def decode(self, z, lengths=None):
        """``lengths`` (optional int tensor [B]): valid latent frames per item of a right-padded batch; each item
        is then decoded exactly as if alone (the reference decodes one utterance per call)."""
        return self.run(z, lengths)

    def run(self, z, lengths=None):
        """``decode`` without the inference_mode decorator (the form torch.compile traces)."""
        dev = z.device
        if z.dim() != 3 or z.shape[1] != self.latent_dim or z.shape[2] < 1:
            raise ValueError(f"z must be [B, {self.latent_dim}, L >= 1], got {tuple(z.shape)}")
        if lengths is not None:
            if lengths.numel() != z.shape[0]:
                raise ValueError(f"lengths must have {z.shape[0]} entries")
            lengths = lengths.to(device=dev, dtype=torch.int32).contiguous()
        return torch.ops.ls_b200.dac_decode(self.handle(dev).key, _as_f32(z, dev), lengths, self.hop_length)

    forward = decode


class DACVAEEncoder(nn.Module):
    """``DACVAE.encode`` (dac-vae/model.py:469-483) -- SURVEY section 8 row f-3, the path the reference's multi-GPU
    latent extraction tool runs (extract_dac_latents.py:20-54).  precision="bf16": tensor-core path (every
    ResidualUnit and downsampling convolution is an implicit-GEMM launch); "fp16": the same path with fp16 GEMM
    operands; "fp32": validation mode."""

    def __init__(self, encoder_dim=64, encoder_rates=(2, 3, 4, 4, 5), latent_dim=80, sample_rate=24000, d_in=1,
                 weight_seed=0, precision="bf16", **_ignored):
        super().__init__()
        native.check_precision(precision, fp16_ok=True)
        if d_in != 1:
            raise NotImplementedError("mono input only (configx2.yml: d_in=1)")
        self.precision, self.latent_dim, self.sample_rate = precision, latent_dim, sample_rate
        self.hop_length = 1
        for r in encoder_rates:
            self.hop_length *= r
        _register_tree(self, synth.dac_encoder_state_dict(weight_seed, "reference", encoder_dim=encoder_dim,
                                                          encoder_rates=encoder_rates, latent_dim=latent_dim))
        self._handle = None

    def load_state_dict(self, state_dict, strict=True, **kw):
        self._handle = None
        keep = {k: v for k, v in state_dict.items() if k.startswith(("encoder.", "en_conv_post."))}
        return super().load_state_dict(keep, strict=strict, **kw)

    def handle(self, device):
        device = torch.device(device)
        if device.type != "cuda":
            raise RuntimeError("the B200 hot path runs on CUDA tensors only (no CPU fallback)")
        if self._handle is None or self._handle.device != device or self._handle.precision != self.precision:
            self._handle = native.DacHandle(self.state_dict(), device, self.precision)
        return self._handle

    def preprocess(self, audio_data):
        """Right-pad to a multiple of the hop (model.py:455-462)."""
        pad = (-audio_data.shape[-1]) % self.hop_length
        return torch.nn.functional.pad(audio_data, (0, pad))

    @torch.inference_mode()
    def encode(self, audio_data, noise=None, lengths=None):
        """audio [B,1,S] (S a multiple of the hop) -> (z, m, logs).  ``noise`` ([B,latent,S/hop]) injects the sample
        the reference draws with torch.randn_like; by default it is drawn here the same way.

        ``lengths`` (optional list or tensor of B latent-frame counts in [1, S/hop]) encodes a right-padded batch of
        clips of different lengths: clip b is ``audio_data[b, :, :lengths[b] * hop]`` and is encoded exactly as if
        alone at that length (the samples after it are never read); z, m and logs are zero from frame lengths[b] on."""
        dev = audio_data.device
        if audio_data.dim() != 3 or audio_data.shape[1] != 1 or audio_data.shape[2] % self.hop_length or \
                audio_data.shape[2] < self.hop_length:
            raise ValueError(f"audio must be [B, 1, S] with S a positive multiple of {self.hop_length}")
        B, _, S = audio_data.shape
        L = S // self.hop_length
        if lengths is not None:
            host = torch.as_tensor(lengths).detach().cpu().reshape(-1)  # one copy per call: not a per-step call
            if host.numel() != B or host.is_floating_point() or host.is_complex() or \
                    bool(((host < 1) | (host > L)).any()):
                raise ValueError(f"lengths must be {B} integer latent-frame counts in [1, {L}]")
            lengths = host.to(device=dev, dtype=torch.int32)
        if noise is None:
            noise = torch.randn(B, self.latent_dim, L, device=dev)
        elif tuple(noise.shape) != (B, self.latent_dim, L):
            raise ValueError("noise must be [B, latent, S / hop]")
        return self.handle(dev).encode(_as_f32(audio_data, dev), _as_f32(noise, dev), lengths)


def patch_reference_model(model):
    """Replace ``decode`` of a reference ``DACVAE`` instance by the B200 path (weights taken from it)."""
    sd = {k: v for k, v in model.state_dict().items() if k.startswith(("decoder.", "de_conv_pre."))}
    dec = DACVAEDecoder(latent_dim=model.latent_dim, decoder_dim=model.decoder_dim,
                        decoder_rates=tuple(model.decoder_rates), sample_rate=model.sample_rate)
    dec.load_state_dict(sd)
    model.decode = dec.decode
    model._b200_decoder = dec
    return model
