"""DAC-VAE encoder on right-padded batches of clips of different lengths (``DACVAEEncoder.encode(..., lengths=)``,
``ls_dac_encode_lengths``) and the batched latent extraction built on it, tensor-core path and fp32 mode.  Each clip
must come out exactly as if encoded alone at its own length: no kernel's summation order depends on the grid or on
the batch, so the comparisons with per-clip calls are bitwise."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

if not torch.cuda.is_available():
    pytest.skip("needs a CUDA device", allow_module_level=True)

import minimax_speech_b200.synth as synth  # noqa: E402
from minimax_speech_b200 import pipeline  # noqa: E402
from minimax_speech_b200.dac import DACVAEDecoder, DACVAEEncoder  # noqa: E402
from oracle import restatement as O  # noqa: E402

DEV = torch.device("cuda:0")
HOP = 480
TOL = {"bf16": 1e-2, "fp32": 1e-4}
LENS = [20, 1, 7, 13, 20, 3]
torch.set_num_threads(os.cpu_count() or 1)


@pytest.fixture(scope="module", params=["bf16", "fp32"])
def enc(golden_dir, request):
    g = np.load(os.path.join(golden_dir, "dac_enc_golden.npz"))
    sd = synth.dac_encoder_state_dict(int(g["weights_seed"]), init="test")
    e = DACVAEEncoder(precision=request.param)
    e.load_state_dict(sd)
    return sd, e


def _batch(lengths, first=60, fill=0.0, seed=11):
    """Right-padded audio [B,1,max*hop] (padding = ``fill``) and noise [B,80,max] (padding = ``fill`` too)."""
    L = max(lengths)
    audio = torch.full((len(lengths), 1, L * HOP), fill)
    noise = torch.full((len(lengths), 80, L), fill)
    gen = torch.Generator().manual_seed(seed)
    for b, n in enumerate(lengths):
        audio[b, :, :n * HOP] = synth.audio_clip(first + b, n * HOP)[0]
        noise[b, :, :n] = torch.randn(80, n, generator=gen)
    return audio, noise


def _encode(e, audio, noise, lengths=None):
    return [t.cpu() for t in e.encode(audio.to(DEV), noise.to(DEV), lengths=lengths)]


def _check_per_clip(e, audio, noise, lengths, outs):
    for b, n in enumerate(lengths):
        alone = _encode(e, audio[b:b + 1, :, :n * HOP], noise[b:b + 1, :, :n])
        for name, o, a in zip(("z", "m", "logs"), outs, alone):
            d = float((o[b:b + 1, :, :n] - a).abs().max())
            assert torch.equal(o[b:b + 1, :, :n], a), f"clip {b} ({n} frames) {name}: max |diff| {d:.3e}"
            assert not bool(o[b, :, n:].any()), f"clip {b}: {name} not zero past its length"


def test_batch_equals_per_clip(enc):
    sd, e = enc
    audio, noise = _batch(LENS)
    outs = _encode(e, audio, noise, LENS)
    assert all(o.shape == (len(LENS), 80, max(LENS)) for o in outs)
    _check_per_clip(e, audio, noise, LENS, outs)


def test_padding_is_never_read(enc):
    """NaN or huge padding, noise included, on a handle whose workspace holds a larger batch's activations."""
    sd, e = enc
    ref = _encode(e, *_batch(LENS), LENS)
    big = torch.cat([synth.audio_clip(90 + b, 32 * HOP) for b in range(8)], 0)
    for fill in (float("nan"), 1e4):
        _encode(e, big, torch.randn(8, 80, 32))  # stale workspace
        outs = _encode(e, *_batch(LENS, fill=fill), LENS)
        for o, r in zip(outs, ref):
            assert torch.equal(o, r), f"padding {fill} changed the output"


def test_batch_vs_oracle(enc):
    sd, e = enc
    audio, noise = _batch(LENS)
    z, m, logs = _encode(e, audio, noise, LENS)
    tol = TOL[e.precision]
    for b in (0, 3):
        n = LENS[b]
        with torch.inference_mode():
            zr, mr, lr = O.dac_encode(sd, audio[b:b + 1, :, :n * HOP], noise[b:b + 1, :, :n])
        errs = [O.rel_l2(x[b:b + 1, :, :n], r) for x, r in ((z, zr), (m, mr), (logs, lr))]
        print(f"mixed batch [{e.precision}] clip {b} ({n} frames): z {errs[0]:.3e} m {errs[1]:.3e} logs {errs[2]:.3e}")
        assert max(errs) < tol


def test_full_lengths_equal_no_lengths(enc):
    sd, e = enc
    audio, noise = _batch([16, 16, 16])
    a = _encode(e, audio, noise)
    b = _encode(e, audio, noise, torch.tensor([16, 16, 16]))
    for x, y in zip(a, b):
        assert torch.equal(x, y)


def test_bad_lengths_rejected(enc):
    sd, e = enc
    audio = torch.zeros(3, 1, 10 * HOP, device=DEV)
    for bad in ([10, 10], [10, 0, 10], [10, 11, 10], [10, -1, 10], torch.tensor([10.0, 5.0, 2.0])):
        with pytest.raises(ValueError):
            e.encode(audio, lengths=bad)
    e.encode(audio, lengths=torch.tensor([10, 5, 1], device=DEV))  # a CUDA tensor is accepted


def test_round_trip_mixed(enc):
    """Mixed-length encode -> mixed-length decode equals encode -> decode of each clip alone."""
    sd, e = enc
    dec = DACVAEDecoder(precision=e.precision)
    dec.load_state_dict(synth.dac_decoder_state_dict(5, init="test"))
    audio, noise = _batch(LENS)
    z, _, _ = e.encode(audio.to(DEV), noise.to(DEV), lengths=LENS)
    wav = dec.decode(z, torch.tensor(LENS)).cpu()
    for b, n in enumerate(LENS):
        z1, _, _ = e.encode(audio[b:b + 1, :, :n * HOP].to(DEV), noise[b:b + 1, :, :n].to(DEV))
        w1 = dec.decode(z1).cpu()
        d = float((wav[b:b + 1, :, :n * HOP] - w1).abs().max())
        assert torch.equal(wav[b:b + 1, :, :n * HOP], w1), f"clip {b}: max |diff| {d:.3e}"
        assert not bool(wav[b, :, n * HOP:].any())


def test_realistic_mixed_batch_tensor_core(golden_dir):
    """8 clips of 2-30 s (synth.mixed_lengths) in one call: every clip equals its own call; the shortest vs the
    oracle."""
    g = np.load(os.path.join(golden_dir, "dac_enc_golden.npz"))
    sd = synth.dac_encoder_state_dict(int(g["weights_seed"]), init="test")
    e = DACVAEEncoder()
    e.load_state_dict(sd)
    lengths = synth.mixed_lengths(8)
    audio, noise = _batch(lengths, first=200)
    outs = _encode(e, audio, noise, lengths)
    _check_per_clip(e, audio, noise, lengths, outs)
    b = int(np.argmin(lengths))
    n = lengths[b]
    with torch.inference_mode():
        _, mr, lr = O.dac_encode(sd, audio[b:b + 1, :, :n * HOP])
    em, el = O.rel_l2(outs[1][b:b + 1, :, :n], mr), O.rel_l2(outs[2][b:b + 1, :, :n], lr)
    print(f"mixed 8 clips, clip {b} ({n} frames) vs oracle: m {em:.3e} logs {el:.3e}")
    assert em < 1e-2 and el < 1e-2


@pytest.mark.parametrize("world", [1, 2])
def test_batched_extraction_equals_per_file(enc, tmp_path, world):
    sd, e = enc
    paths = []
    for i, n in enumerate([5 * HOP + 17, 12 * HOP, 3 * HOP - 100, 20 * HOP + 1, 8 * HOP, 15 * HOP - 7]):
        p = tmp_path / f"clip{i}.pt"
        torch.save(synth.audio_clip(300 + i, n).reshape(-1) * 1.5, p)  # (clamped to [-1, 1] by extract_latents)
        paths.append(str(p))
    for rank in range(world):
        kw = dict(rank=rank, world_size=world, save=False)
        ref = pipeline.extract_latents(paths, torch.load, e, DEV, generator=torch.Generator().manual_seed(5), **kw)
        out = pipeline.extract_latents(paths, torch.load, e, DEV, generator=torch.Generator().manual_seed(5),
                                       max_batch_samples=3 * 13 * HOP, **kw)
        assert [r["original_path"] for _, r in out] == [r["original_path"] for _, r in ref]
        for (_, r), (_, q) in zip(out, ref):
            for k in ("z", "mu", "logs"):
                assert torch.equal(r[k], q[k]), (world, rank, r["original_path"], k)
            assert r["latent_shape"] == q["latent_shape"]
