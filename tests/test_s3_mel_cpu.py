"""The S3 tokenizer's log-mel front end on the host: the conventions of the reference restatement the GPU tests check
against (profiles/s3_mel_reference.py: frame count, reflect padding, periodic Hann window, dropped last frame, per-clip
floor) against an independent float64 numpy statement, the restated librosa filter bank, and pipeline.extract_tokens'
bookkeeping with a stand-in tokenizer."""
import os

import numpy as np
import pytest
import torch

from minimax_speech_b200 import pipeline
from minimax_speech_b200 import tokenizer as tk
from profiles import s3_mel_reference as R


def numpy_log_mel(audio, filters):
    """float64: reflect pad 200 each side, periodic Hann, 201-bin DFT of every 400-sample frame at hop 160, last frame
    dropped, |X|^2, filter bank, log10 with the 1e-10 clamp, floor 8 below the clip's maximum, (x + 4) / 4."""
    a = np.asarray(audio, dtype=np.float64)
    padded = np.concatenate([a[1:201][::-1], a, a[-201:-1][::-1]])
    n_frames = 1 + (len(padded) - 400) // 160
    win = 0.5 - 0.5 * np.cos(2 * np.pi * np.arange(400) / 400)
    frames = np.stack([padded[t * 160:t * 160 + 400] for t in range(n_frames)]) * win
    n = np.arange(400)
    k = np.arange(201)
    ang = 2 * np.pi * np.outer(n, k) / 400
    re, im = frames @ np.cos(ang), frames @ np.sin(ang)
    power = (re ** 2 + im ** 2)[:-1].T
    log = np.log10(np.maximum(np.asarray(filters, np.float64) @ power, 1e-10))
    log = np.maximum(log, log.max() - 8.0)
    return (log + 4.0) / 4.0


def _clip(n, seed):
    g = torch.Generator().manual_seed(seed)
    t = torch.arange(n, dtype=torch.float64) / 16000
    return 0.3 * torch.sin(2 * np.pi * 440 * t) + 0.05 * torch.randn(n, generator=g, dtype=torch.float64)


@pytest.mark.parametrize("n", [201, 400, 16000, 16159, 16160, 45 * 16000])
def test_reference_matches_numpy(n):
    filt = tk.mel_filters(128).double()
    a = _clip(n, n)
    ref = numpy_log_mel(a.numpy(), filt.numpy())
    out = R.s3_log_mel(a, filt).numpy()
    assert out.shape == (128, n // 160) == ref.shape
    assert np.abs(out - ref).max() < 1e-9


def test_reference_frame_count_and_short_clip():
    filt = tk.mel_filters(128).double()
    for n in (201, 400, 16000, 16159, 16160):
        assert R.s3_log_mel(_clip(n, 1), filt).shape[1] == n // 160
    with pytest.raises(RuntimeError):
        R.s3_log_mel(_clip(200, 1), filt)  # reflect padding of 200 needs more than 200 samples


def test_mel_filters_are_slaney_triangles():
    f = tk.mel_filters(128).numpy()
    assert f.shape == (128, 201) and f.dtype == np.float32
    assert (f >= 0).all()
    edges = tk.mel_band_edges(128)
    freqs = np.arange(201) * 40.0
    assert abs(edges[0]) < 1e-9 and abs(edges[-1] - 8000.0) < 1e-6
    for m in range(128):
        row = f[m]
        support = np.nonzero(row)[0]
        assert 1 <= len(support) <= 9
        assert (freqs[support] > edges[m]).all() and (freqs[support] < edges[m + 2]).all()  # inside its band
        assert np.all(np.diff(support) == 1)  # one contiguous triangle
        peak = int(row.argmax())
        assert abs(freqs[peak] - edges[m + 1]) < 40.0  # a bin next to the centre frequency
        # rising then falling about the centre
        assert np.all(np.diff(row[:peak + 1]) >= 0) and np.all(np.diff(row[peak:]) <= 0)
        # height at the samples: 2 / (f[m+2] - f[m]) times the triangle, so the area (Hz) of the continuous triangle is 1
        height = 2.0 / (edges[m + 2] - edges[m])
        tri = np.maximum(0, np.minimum((freqs - edges[m]) / (edges[m + 1] - edges[m]),
                                       (edges[m + 2] - freqs) / (edges[m + 2] - edges[m + 1])))
        np.testing.assert_allclose(row, height * tri, rtol=1e-6, atol=1e-9)
        assert row.max() <= height * (1 + 1e-6)
        if len(support) >= 5:  # sampled finely enough for a Riemann sum
            assert abs(row.sum() * 40.0 - 1.0) < 0.05
    assert tk.mel_filters(80).shape == (80, 201)


def test_mel_filters_against_reference_asset():
    path = os.environ.get("LS_S3_MEL_FILTERS")
    if not path:
        pytest.skip("set LS_S3_MEL_FILTERS to the reference's mel_filters.npz to compare against it")
    for n_mels in (80, 128):
        asset = tk.load_mel_filters(path, n_mels)
        mine = tk.mel_filters(n_mels)
        print(f"mel_{n_mels}: {int((asset != mine).sum())} entries differ in bits, max abs "
              f"{float((asset - mine).abs().max()):.2e}")
        assert torch.allclose(asset, mine, rtol=1e-6, atol=1e-9)


def test_load_mel_filters_reads_npz(tmp_path):
    p = tmp_path / "mel_filters.npz"
    np.savez(p, mel_128=tk.mel_filters(128).numpy(), mel_80=tk.mel_filters(80).numpy())
    assert torch.equal(tk.load_mel_filters(str(p)), tk.mel_filters(128))
    assert torch.equal(tk.load_mel_filters(str(p), 80), tk.mel_filters(80))


def test_log_mel_rejects_cpu():
    with pytest.raises(RuntimeError):
        tk.log_mel_spectrogram(torch.zeros(16000))


# ---- extract_tokens with a stand-in tokenizer -----------------------------------------------------------------------
class StandInTokenizer:
    """Tokens = the first sample of every 640-sample block, scaled; records every call."""

    def __init__(self):
        self.calls = []

    def quantize_audio(self, audio, audio_len):
        B, S = audio.shape
        self.calls.append((B, S, list(audio_len)))
        n_tok = [n // 640 for n in audio_len]
        codes = torch.zeros(B, max(max(n_tok), 1), dtype=torch.long)
        for b, n in enumerate(n_tok):
            codes[b, :n] = (audio[b, :n * 640:640] * 1000).round().long()
            codes[b, n:] = -1  # garbage past the length
        return codes, torch.tensor(n_tok)


SIZES = [48000, 16000, 112000, 8000, 40000, 153600, 19200, 64000]


def _clips(tmp_path, sizes):
    paths = []
    for i, n in enumerate(sizes):
        p = tmp_path / f"clip{i}.pt"
        torch.save(torch.sin(torch.arange(n, dtype=torch.float32) * (0.001 * (i + 1))), p)
        paths.append(str(p))
    return paths


def test_extract_tokens_batched_matches_per_file(tmp_path):
    paths = _clips(tmp_path, SIZES)
    ref_tok = StandInTokenizer()
    ref = pipeline.extract_tokens(paths, torch.load, ref_tok, "cpu", save=False)
    assert [c[0] for c in ref_tok.calls] == [1] * len(paths)  # one file per call by default
    assert [c[2] for c in ref_tok.calls] == [[n] for n in SIZES]  # in file order
    for budget in [100000, 400000, 10 ** 9]:
        tok = StandInTokenizer()
        out = pipeline.extract_tokens(paths, torch.load, tok, "cpu", save=False, max_batch_samples=budget)
        assert len(out) == len(paths)
        plan = pipeline.plan_micro_batches(SIZES, budget)
        assert [c[2] for c in tok.calls] == [[SIZES[i] for i in b] for b in plan]  # one call per micro-batch
        for (_, r), (_, q), n, p in zip(out, ref, SIZES, paths):
            assert r["original_path"] == q["original_path"] == p  # file order
            assert r["original_samples"] == n and r["sample_rate"] == 16000
            assert r["tokens"].dtype == torch.int64 and r["token_len"] == r["tokens"].shape[0] == n // 640
            assert torch.equal(r["tokens"], q["tokens"])
        for B, S, lens in tok.calls:
            assert B == 1 or B * S <= budget
            assert S == max(lens)
        assert any(c[0] > 1 for c in tok.calls)


def test_extract_tokens_save_and_sharding(tmp_path):
    paths = _clips(tmp_path, SIZES[:6])
    out = pipeline.extract_tokens(paths, torch.load, StandInTokenizer(), "cpu", rank=1, world_size=2,
                                  max_batch_samples=300000)
    assert [os.path.basename(p) for p, _ in out] == ["clip3_fsq.pt", "clip4_fsq.pt", "clip5_fsq.pt"]
    for p, rec in out:
        saved = torch.load(p)
        assert torch.equal(saved["tokens"], rec["tokens"]) and saved["token_len"] == rec["token_len"]
        assert saved["tokens"].untyped_storage().nbytes() == saved["tokens"].numel() * 8  # not a view of the batch
