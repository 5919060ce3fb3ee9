"""The S3 tokenizer's log-mel front end on the B200 (csrc/s3_mel.cu, ls_s3_log_mel): agreement with the reference function
restated in float64 (profiles/s3_mel_reference.py), bitwise per-clip batch invariance, audio-to-token agreement with the
oracle chain (that restatement in fp32, then oracle.s3_encode / s3_quantize) in both precisions, batched
extract_tokens against per-file calls, argument errors and state_dict compatibility."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

if not torch.cuda.is_available():
    pytest.skip("needs a CUDA device", allow_module_level=True)

import minimax_speech_b200.native as native  # noqa: E402
import minimax_speech_b200.synth as synth  # noqa: E402
from minimax_speech_b200 import pipeline  # noqa: E402
from minimax_speech_b200 import tokenizer as tk  # noqa: E402
from minimax_speech_b200.tokenizer import S3TokenizerV2  # noqa: E402
from oracle import restatement as O  # noqa: E402
from profiles import s3_mel_reference as R  # noqa: E402
from profiles.emulate_s3_precision import fsq_margin  # noqa: E402

DEV = torch.device("cuda")
MARGIN = 1e-4
FILT = tk.mel_filters(128)


def speech_like(n, seed):
    """A voiced-speech stand-in: harmonics of a gliding 100-200 Hz pitch under a syllable-rate envelope, plus noise."""
    g = torch.Generator().manual_seed(seed)
    t = torch.arange(n, dtype=torch.float64) / 16000
    f0 = 150 + 50 * torch.sin(2 * math.pi * (0.3 + 0.1 * (seed % 7)) * t)
    phase = torch.cumsum(2 * math.pi * f0 / 16000, 0)
    sig = sum(torch.sin(h * phase) / h for h in range(1, 16))
    env = 0.5 + 0.5 * torch.sin(2 * math.pi * 4 * t + seed)
    return (0.1 * sig * env + 0.01 * torch.randn(n, generator=g, dtype=torch.float64)).float()


def _test_clips():
    t = torch.arange(160000, dtype=torch.float64) / 16000
    g = torch.Generator().manual_seed(5)
    tone_noise = (0.3 * torch.sin(2 * math.pi * 440 * t) + 0.05 * torch.randn(160000, generator=g, dtype=torch.float64))
    quiet = 0.5 * torch.sin(2 * math.pi * 1000 * t)
    quiet[48000:112000] *= 1e-3  # a -60 dB stretch
    clipped = torch.clamp(3.0 * torch.sin(2 * math.pi * 220 * t), -1.0, 1.0)
    return {"tone+noise": tone_noise.float(), "tone with -60 dB stretch": quiet.float(),
            "full-scale clipped": clipped.float(), "all zero": torch.zeros(32000),
            "201 samples": speech_like(201, 1), "16159 samples": speech_like(16159, 2),
            "16160 samples": speech_like(16160, 3), "60 s": speech_like(60 * 16000, 4)}


@pytest.mark.parametrize("name", list(_test_clips()))
def test_log_mel_vs_float64_oracle(name):
    a = _test_clips()[name]
    ref = R.s3_log_mel(a.double(), FILT.double())
    mine = tk.log_mel_spectrogram(a.to(DEV)).cpu()
    assert mine.shape == (128, a.shape[0] // 160) == ref.shape
    e, mx = O.rel_l2(mine, ref), float((mine.double() - ref).abs().max())
    t32 = R.s3_log_mel(a, FILT)
    print(f"{name}: kernel rel-L2 {e:.2e} max abs {mx:.2e}; torch.stft fp32 rel-L2 {O.rel_l2(t32, ref):.2e} "
          f"max abs {float((t32.double() - ref).abs().max()):.2e}")
    assert e <= 2e-5 and mx <= 1e-3
    if name == "all zero":
        assert torch.all(mine == -1.5)


def test_batch_invariance_and_padding():
    lens = [201, 16159, 16160, 48000, 5000, 160000, 1000]
    S = max(lens) + 1234
    clips = [speech_like(n, 20 + i) for i, n in enumerate(lens)]
    alone = [tk.log_mel_spectrogram(c.to(DEV)) for c in clips]
    for pad in (0.0, 1e4, float("nan")):
        audio = torch.full((len(lens), S), pad)
        for b, c in enumerate(clips):
            audio[b, :c.shape[0]] = c
        mel, mel_len = tk.log_mel_spectrogram(audio.to(DEV), audio_len=lens)
        assert mel.shape == (len(lens), 128, S // 160) and mel_len.dtype == torch.int32
        assert mel_len.tolist() == [n // 160 for n in lens]
        for b, n in enumerate(lens):
            T = n // 160
            assert torch.equal(mel[b, :, :T], alone[b]), f"pad {pad}: clip {b} differs from the clip alone"
            assert torch.all(mel[b, :, T:] == 0)


def test_invalid_lengths_from_c_callers():
    """ls_s3_log_mel with lengths the Python layer refuses: mel_len 0 and an all-zero mel, nothing else touched."""
    S = 4000
    audio = torch.randn(4, S, device=DEV)
    lens = torch.tensor([100, S + 1, 200, 3000], dtype=torch.int32, device=DEV)
    mel, mel_len = native.s3_log_mel(audio, lens, FILT.to(DEV))
    assert mel_len.tolist() == [0, 0, 0, 3000 // 160]
    assert torch.all(mel[:3] == 0)
    assert torch.equal(mel[3, :, :18], tk.log_mel_spectrogram(audio[3, :3000]))
    assert torch.all(mel[3, :, 18:] == 0)


def test_drop_in_and_errors():
    a = speech_like(16000 * 3 + 77, 9)
    out = tk.log_mel_spectrogram(a, device=DEV)
    assert out.shape == (128, (16000 * 3 + 77) // 160) and out.device.type == "cuda"
    assert torch.equal(out, tk.log_mel_spectrogram(a.numpy(), device="cuda"))
    padded = tk.log_mel_spectrogram(a, padding=480, device=DEV)  # zeros appended, like the reference
    assert torch.equal(padded, tk.log_mel_spectrogram(torch.cat([a, torch.zeros(480)]).to(DEV)))
    with pytest.raises(RuntimeError):
        tk.log_mel_spectrogram(a)  # CPU tensors are rejected, not emulated
    batch = torch.zeros(2, 1000, device=DEV)
    with pytest.raises(ValueError):
        tk.log_mel_spectrogram(batch, audio_len=[200, 1000])
    with pytest.raises(ValueError):
        tk.log_mel_spectrogram(batch, audio_len=[1001, 1000])
    with pytest.raises(ValueError):
        tk.log_mel_spectrogram(batch, audio_len=[1000])
    with pytest.raises(ValueError):
        tk.log_mel_spectrogram(batch, filters=torch.zeros(128, 200, device=DEV))
    with pytest.raises(ValueError):
        tk.log_mel_spectrogram(batch, n_mels=80, filters=FILT.to(DEV))
    with pytest.raises(ValueError):
        tk.log_mel_spectrogram(batch, n_mels=129)
    with pytest.raises(ValueError):
        tk.log_mel_spectrogram(torch.zeros(200, device=DEV))
    m80, _ = tk.log_mel_spectrogram(batch + 0.1, n_mels=80, audio_len=[1000, 500])
    assert m80.shape == (2, 80, 6)


# ---- audio to tokens ------------------------------------------------------------------------------------------------
_TOK = {}


def _tok(precision):
    if precision not in _TOK:
        _TOK[precision] = S3TokenizerV2(weight_seed=33, precision=precision)
    return _TOK[precision]


def _padded(clips):
    S = max(c.shape[0] for c in clips)
    audio = torch.zeros(len(clips), S)
    for b, c in enumerate(clips):
        audio[b, :c.shape[0]] = c
    return audio


_ORACLE = {}


def _oracle_short(seed):
    """Per clip: the reference log-mel in fp32 on the CPU, then the oracle's encoder and FSQ head (tokens, hidden)."""
    if seed not in _ORACLE:
        lens = synth.mixed_lengths(16, 2, 30, frame_rate=16000, seed=seed)
        clips = [speech_like(n, 100 + i) for i, n in enumerate(lens)]
        sd = {k: v.clone() for k, v in _tok("fp32").state_dict().items()}
        w, bias = sd["quantizer._codebook.project_down.weight"], sd["quantizer._codebook.project_down.bias"]
        ref = []
        with torch.inference_mode():
            for c in clips:
                mel = R.s3_log_mel(c, FILT)[None]
                h, l2 = O.s3_encode(sd, mel, torch.tensor([mel.shape[-1]]))
                ref.append((O.fsq_encode(w, bias, h)[0], h, int(l2[0])))
        _ORACLE[seed] = (lens, clips, sd, ref)
    return _ORACLE[seed]


@pytest.mark.parametrize("precision", ["bf16x3", "fp32"])
def test_audio_to_tokens_vs_oracle_chain(precision):
    lens, clips, sd, ref = _oracle_short(6)
    codes, code_len = _tok(precision).quantize_audio(_padded(clips).to(DEV), lens)
    diff = 0
    for b, (rc, rh, n) in enumerate(ref):
        assert int(code_len[b]) == n
        mine = codes[b, :n].cpu()
        safe = fsq_margin(sd, rh)[0] > MARGIN
        assert torch.equal(mine[safe], rc[safe].to(mine.dtype)), f"{precision} clip {b}: a token away from every boundary differs"
        diff += int((mine != rc.to(mine.dtype)).sum())
    print(f"{precision}: {diff} of {sum(r[2] for r in ref)} tokens differ from the oracle chain")
    assert diff <= 1


@pytest.mark.parametrize("precision", ["bf16x3", "fp32"])
def test_audio_to_tokens_long_clip_vs_oracle_chain(precision):
    """A batch holding a 47 s clip: the sliding-window path behind quantize_audio."""
    lens = [47 * 16000 + 333, 7 * 16000, 31 * 16000]
    clips = [speech_like(n, 300 + i) for i, n in enumerate(lens)]
    tok = _tok(precision)
    sd = {k: v.clone() for k, v in tok.state_dict().items()}
    codes, code_len = tok.quantize_audio(_padded(clips).to(DEV), lens)
    with torch.inference_mode():
        mels = [R.s3_log_mel(c, FILT) for c in clips]
        mel = torch.zeros(len(clips), 128, max(m.shape[1] for m in mels))
        for b, m in enumerate(mels):
            mel[b, :, :m.shape[1]] = m
        rc, rl = O.s3_quantize(sd, mel, torch.tensor([m.shape[1] for m in mels]))
    assert code_len.tolist() == rl.tolist()
    diff = sum(int((codes[b, :n].cpu() != rc[b, :n]).sum()) for b, n in enumerate(rl.tolist()))
    print(f"{precision} long-clip batch: {diff} of {int(rl.sum())} tokens differ from the oracle chain")
    assert diff <= 1


@pytest.mark.parametrize("precision", ["bf16x3", "fp32"])
def test_extract_tokens_batched_equals_per_file(tmp_path, precision):
    sizes = [16000 * s + 17 * i for i, s in enumerate([3, 12, 7, 29, 2, 35, 18, 9])]
    paths = []
    for i, n in enumerate(sizes):
        p = tmp_path / f"utt{i}.pt"
        torch.save(speech_like(n, 500 + i), p)
        paths.append(str(p))
    tok = _tok(precision)
    per_file = pipeline.extract_tokens(paths, torch.load, tok, DEV, save=False)
    for budget in (16000 * 60, 10 ** 9):
        batched = pipeline.extract_tokens(paths, torch.load, tok, DEV, save=False, max_batch_samples=budget)
        for (_, r), (_, q), n in zip(batched, per_file, sizes):
            assert r["original_samples"] == n and r["original_path"] == q["original_path"]
            assert torch.equal(r["tokens"], q["tokens"]), f"{precision}: {r['original_path']} differs from the per-file call"


def test_state_dict_unchanged_and_strict_load():
    tok = S3TokenizerV2(precision="bf16x3")
    sd = synth.s3_tokenizer_state_dict(33, 128, 1280, 20, 6)
    assert set(tok.state_dict()) == set(sd)  # the filter bank is not a weight
    tok.load_state_dict(sd, strict=True)
    assert torch.equal(tok.mel_filters, FILT)
    tok = tok.to(DEV)
    assert tok.mel_filters.device.type == "cuda"
    a = speech_like(16000 * 4, 7)
    c1, l1 = tok.quantize_audio(a[None].to(DEV), [a.shape[0]])
    mel = tk.log_mel_spectrogram(a, device=DEV)
    c2, l2 = tok.quantize(mel[None], torch.tensor([mel.shape[1]]))
    assert torch.equal(c1, c2) and l1.tolist() == l2.tolist()
