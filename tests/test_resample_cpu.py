"""CPU checks of the sample-rate converter's host side: the tap table ls_resample uses against torchaudio's own float64
kernel, the output-length formula against torchaudio's output lengths, the refusal of oversized tables, and the host
arithmetic of the voice-conversion path (prompt cut, speed lengths)."""
import ctypes
import math

import numpy as np
import pytest
import torch

torchaudio_functional = pytest.importorskip("torchaudio.functional")
from torchaudio.functional.functional import _get_sinc_resample_kernel  # noqa: E402

import minimax_speech_b200.native as native  # noqa: E402
from minimax_speech_b200 import audio, vc  # noqa: E402

RATIOS = [(16000, 24000), (24000, 16000), (48000, 24000), (48000, 16000), (44100, 24000), (44100, 16000),
          (11025, 16000), (96000, 16000)]


@pytest.mark.parametrize("orig,new", RATIOS)
def test_tap_table_matches_torchaudio_float64(orig, new):
    t = native.resample_taps(orig, new)
    g = math.gcd(orig, new)
    kernel, width = _get_sinc_resample_kernel(orig, new, g, dtype=torch.float64)
    kernel = kernel[:, 0, :].numpy()  # [N][2 width + O]: column c is i = c - width
    assert (t["O"], t["N"], t["width"]) == (orig // g, new // g, width)
    assert t["taps"].shape == (t["N"], t["max_taps"]) and t["max_taps"] == int(t["count"].max())
    for p in range(t["N"]):
        f, c = int(t["first"][p]), int(t["count"][p])
        kept = np.zeros(kernel.shape[1], bool)
        kept[f + width:f + width + c] = True
        assert kept.sum() == c and c > 0, f"phase {p}: taps outside torchaudio's window"
        np.testing.assert_array_equal(t["taps"][p, :c], kernel[p, kept].astype(np.float32), err_msg=f"phase {p}")
        assert not t["taps"][p, c:].any(), "padding of a row must be zero"
        assert np.abs(kernel[p, ~kept]).max(initial=0.0) < 1e-45, f"phase {p}: a dropped tap is not negligible"


@pytest.mark.parametrize("orig,new", RATIOS)
def test_output_length_matches_torchaudio(orig, new):
    rng = np.random.default_rng(orig + new)
    O, N = audio.reduced_ratio(orig, new)
    lengths = sorted(set([1, 2, O - 1, O, O + 1, 1000] + rng.integers(1, 20000, 300).tolist()) - {0})
    for n in lengths:
        # torchaudio's own formula (_apply_sinc_resample_kernel), evaluated without running the convolution
        want = int(torch.ceil(torch.as_tensor(N * n / O)).long())
        assert audio.output_length(n, orig, new) == want, n
    # long clips: the exact ceil.  torchaudio's expression makes a float32 tensor of the Python float, which loses the
    # last sample of some long clips (28 800 001 samples at 48 -> 16 kHz: 9 600 000 instead of 9 600 001)
    for n in (30 * orig, 600 * orig, 600 * orig + 1, 600 * orig + O - 1):
        assert audio.output_length(n, orig, new) == math.ceil(N * n / O)


def test_equal_rates_are_a_copy_table():
    t = native.resample_taps(22050, 22050)
    assert (t["O"], t["N"], t["width"], t["max_taps"]) == (1, 1, 0, 1)
    assert t["first"].tolist() == [0] and t["count"].tolist() == [1] and t["taps"].tolist() == [[1.0]]


def test_tables_over_96_kib_are_refused():
    lib = native.load()
    # the largest table among the common rates (11.025 -> 96 kHz, 66.5 kB) is accepted
    t = native.resample_taps(11025, 96000)
    assert 4 * t["N"] * t["max_taps"] == 66560
    O, N, W, M = (ctypes.c_int32(-1) for _ in range(4))
    for orig, new in [(16000, 16001), (1000, 4999), (99991, 1000), (1000, 99991)]:
        code = lib.ls_resample_taps(orig, new, ctypes.byref(O), ctypes.byref(N), ctypes.byref(W), ctypes.byref(M),
                                    None, None, None)
        assert code == -4, (orig, new)  # LS_ERR_UNSUPPORTED
        g = math.gcd(orig, new)
        assert (O.value, N.value, M.value) == (orig // g, new // g, 0)
        h = ctypes.c_void_p()
        assert lib.ls_resampler_create(orig, new, 0, ctypes.byref(h)) == -4 and not h.value  # refused before any CUDA call
    assert lib.ls_resample_taps(0, 16000, None, None, None, None, None, None, None) == -1


def test_resample_rejects_cpu_tensors():
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        audio.resample(torch.zeros(1000), 44100, 16000)


def test_prompt_cut_and_speed_lengths():
    # frontend_zero_shot: n = min(frames // 2, tokens); 2n frames, n tokens
    assert vc.prompt_cut(301, 150) == 150 and vc.prompt_cut(301, 151) == 150 and vc.prompt_cut(200, 120) == 100
    assert vc.prompt_cut(1, 5) == 0
    lengths = [100, 37, 1, 250]
    for s in (0.5, 0.8, 1.0, 1.3, 2.0, 1 / 3):
        assert vc.speed_lengths(lengths, s) == [int(L / s) for L in lengths]
    assert vc.speed_lengths(lengths, [0.5, 0.8, 1.3, 2.0]) == [200, int(37 / 0.8), 0, 125]
    for bad in (0.0, -1.0, [1.0, 2.0]):
        with pytest.raises(ValueError):
            vc.speed_lengths(lengths, bad)
    z = torch.zeros(2, 80, 10)
    out, lens = vc.change_speed(z, [10, 7], 1.0)
    assert out is z and lens == [10, 7]  # speed 1: nothing is launched
