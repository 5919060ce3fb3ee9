"""Sample-rate conversion on the GPU (csrc/resample.cu) against torchaudio.functional.resample in float64, mixed-length
batches against each clip converted alone (bitwise), invalid lengths from a C caller, equal rates, and the latent speed
change against F.interpolate in float64."""
import ctypes
import math
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

if not torch.cuda.is_available():
    pytest.skip("needs a CUDA device", allow_module_level=True)

import torchaudio.functional as AF  # noqa: E402

import minimax_speech_b200.native as native  # noqa: E402
from minimax_speech_b200 import audio, vc  # noqa: E402

DEV = torch.device("cuda:0")
torch.set_num_threads(os.cpu_count() or 1)
RATIOS = [(16000, 24000), (24000, 16000), (48000, 24000), (48000, 16000), (44100, 24000), (44100, 16000),
          (11025, 16000), (96000, 16000)]


def speech_like(n, seed, rate=16000):
    """A voiced harmonic signal with vibrato plus noise, driven into clipping at +-1."""
    rng = np.random.default_rng(seed)
    t = np.arange(n) / rate
    f0 = 150 + 50 * np.sin(2 * np.pi * 0.3 * t)
    ph = np.cumsum(2 * np.pi * f0 / rate)
    x = 0.1 * sum(np.sin(h * ph) / h for h in range(1, 30)) + 0.01 * rng.standard_normal(n)
    return torch.from_numpy(np.clip(3 * x, -1, 1).astype(np.float32))


def clipped_tone(n, rate):
    t = np.arange(n) / rate
    return torch.from_numpy(np.clip(1.5 * np.sin(2 * np.pi * 997.0 * t), -1, 1).astype(np.float32))


def reference(x, orig, new):
    return AF.resample(x.double(), orig, new)


def check_close(y, ref, what):
    y = y.double().cpu()
    assert y.shape == ref.shape, f"{what}: length {y.shape[-1]} vs torchaudio {ref.shape[-1]}"
    err = (y - ref).abs().max().item()
    rel = ((y - ref).norm() / ref.norm()).item() if ref.norm() > 0 else 0.0
    assert rel <= 3e-7 and err <= 1e-6, f"{what}: rel-L2 {rel:.2e}, max abs {err:.2e}"
    return rel, err


@pytest.mark.parametrize("orig,new", RATIOS)
def test_against_torchaudio_float64(orig, new):
    O, N = audio.reduced_ratio(orig, new)
    width = native.resample_taps(orig, new)["width"]
    short = sorted({n for n in (1, 2, O - 1, O, O + 1, width + 1, 3 * orig + 77) if n >= 1})
    worst = [0.0, 0.0]
    for n in short + [30 * orig]:
        for name, x in (("speech", speech_like(n, n, orig)), ("tone", clipped_tone(n, orig))):
            rel, err = check_close(audio.resample(x.to(DEV), orig, new), reference(x, orig, new), f"{name} {n}")
            worst = [max(worst[0], rel), max(worst[1], err)]
    x = speech_like(600 * orig, 7, orig)  # 10 minutes
    rel, err = check_close(audio.resample(x.to(DEV), orig, new), reference(x, orig, new), "speech 10 min")
    silence = audio.resample(torch.zeros(orig, device=DEV), orig, new)
    assert silence.shape[0] == N * orig // O and not silence.any()
    print(f"{orig} -> {new}: worst rel-L2 {max(worst[0], rel):.2e}, max abs {max(worst[1], err):.2e} (10 min: {rel:.2e})")


def _call(h, x, lens, S_out, out=None):
    """ls_resample on a raw batch with device lengths (anything the C ABI accepts) and an optional pre-filled output."""
    B, S_in = x.shape
    out = torch.empty(B, S_out, device=DEV) if out is None else out
    out_len = torch.full((B,), -7, dtype=torch.int32, device=DEV)
    native.check(native.load().ls_resample(h._h, native.ptr(x), native.ptr(lens), native.ptr(out), native.ptr(out_len), B,
                                           S_in, S_out, native.current_stream_ptr(DEV)), "ls_resample")
    return out, out_len


@pytest.mark.parametrize("orig,new", [(44100, 16000), (44100, 24000), (16000, 24000), (48000, 16000), (11025, 16000)])
def test_mixed_batch_bitwise_equals_each_clip_alone(orig, new):
    O, N = audio.reduced_ratio(orig, new)
    lens = [orig + 311, 1, 7 * orig // 3, O + 1, 5, 3 * orig]
    S = max(lens) + 123
    clips = [speech_like(n, 40 + b, orig) for b, n in enumerate(lens)]
    alone = [audio.resample(c.to(DEV), orig, new) for c in clips]
    h = audio.resampler(orig, new, DEV)
    S_out = audio.output_length(S, orig, new) + 1000  # a caller-chosen longer row
    for fill in (0.0, 1e4, float("nan")):
        x = torch.full((len(lens), S), fill)
        for b, c in enumerate(clips):
            x[b, :lens[b]] = c
        out, out_len = _call(h, x.to(DEV), torch.tensor(lens, dtype=torch.int32, device=DEV), S_out,
                             torch.full((len(lens), S_out), float("nan"), device=DEV))
        assert out_len.tolist() == [audio.output_length(n, orig, new) for n in lens]
        for b, n in enumerate(out_len.tolist()):
            assert torch.equal(out[b, :n], alone[b]), f"clip {b} (padding {fill}) differs from the clip alone"
            assert torch.equal(out[b, n:], torch.zeros_like(out[b, n:])), f"clip {b}: not zero past out_len"
    got, got_len = audio.resample(x.to(DEV), orig, new, lens)  # the Python batch form
    assert got.shape == (len(lens), audio.output_length(S, orig, new)) and torch.equal(got_len.cpu(), out_len.cpu())
    assert all(torch.equal(got[b, :n], alone[b]) for b, n in enumerate(out_len.tolist()))


def test_invalid_lengths_give_zero_rows_and_equal_rates_copy():
    h = audio.resampler(44100, 16000, DEV)
    S = 5000
    x = torch.randn(5, S, device=DEV)
    lens = torch.tensor([0, -5, S + 1, 2000, S], dtype=torch.int32, device=DEV)
    out, out_len = _call(h, x, lens, audio.output_length(S, 44100, 16000), torch.full((5, 1815), float("nan"), device=DEV))
    assert out_len.tolist() == [0, 0, 0, audio.output_length(2000, 44100, 16000), audio.output_length(S, 44100, 16000)]
    assert not out[:3].any() and not out[:3].isnan().any()
    assert torch.equal(out[3, :726], audio.resample(x[3, :2000].contiguous(), 44100, 16000))
    with pytest.raises(RuntimeError):  # S_out below ceil(N S_in / O)
        _call(h, x, lens, audio.output_length(S, 44100, 16000) - 1)
    for rate in (16000, 22050):
        y = torch.randn(12345, device=DEV)
        y[7] = -0.0
        got = audio.resample(y, rate, rate)
        assert torch.equal(got, y) and got.data_ptr() != y.data_ptr() and math.copysign(1.0, float(got[7])) < 0


def test_latent_speed_against_interpolate():
    B, C, L = 5, 80, 100
    lens = [37, 100, 64, 9, 80]
    speeds = [0.5, 0.8, 1.3, 2.0, 1.0]
    g = torch.Generator().manual_seed(3)
    z = torch.zeros(B, C, L)
    for b, n in enumerate(lens):
        z[b, :, :n] = torch.randn(C, n, generator=g)
        z[b, :, n:] = 1e4  # padding is never read
    out, new = vc.change_speed(z.to(DEV), lens, speeds)
    assert new == [int(n / s) for n, s in zip(lens, speeds)] and out.shape == (B, C, max(new))
    for b, (n, m) in enumerate(zip(lens, new)):
        ref = torch.nn.functional.interpolate(z[b:b + 1, :, :n].double(), size=m, mode="linear")
        e = ((out[b:b + 1, :, :m].double().cpu() - ref).norm() / ref.norm()).item()
        print(f"speed {speeds[b]}: {n} -> {m} frames, rel-L2 vs F.interpolate (float64) {e:.2e}")
        assert e <= 1e-6
        assert not out[b, :, m:].any()
    assert torch.equal(out[4, :, :80], z[4, :, :80].to(DEV))  # a speed-1 row inside a batch is returned unchanged
    zd = z.to(DEV)
    same, lens1 = vc.change_speed(zd, lens, 1.0)
    assert same is zd and lens1 == lens
