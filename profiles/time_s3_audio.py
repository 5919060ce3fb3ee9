"""Time the S3 tokenizer's log-mel front end (csrc/s3_mel.cu, tokenizer.log_mel_spectrogram) and audio-to-token
extraction on the GPU:
  1. the log-mel call alone: 16 clips x 10 s, 64 clips of synth.mixed_lengths (2-30 s) in one padded call, and one
     10-minute clip; achieved FLOP/s from the shape formula (400*402 + 201*n_mels multiply-adds per valid frame);
  2. the same 64 clips through the reference function (profiles/s3_mel_reference.py: torch.stft in fp32 on the GPU),
     one call per clip -- what correct mixed-length mels cost without the kernel;
  3. audio to tokens (bf16x3) for the 64 clips: quantize_audio in one padded call, against per-clip torch mels padded
     into one quantize call;
  4. pipeline.extract_tokens per file against length-sorted micro-batches;
  5. per-kernel times of the two front-end passes (torch.profiler, after the timed sections).
Device events after warm-up; the card's name and power limit are read in the same run.

    python -m profiles.time_s3_audio [--reps 20]

Log: profiles/r05_time_s3_audio.log.
"""
import argparse
import math
import os
import sys
import time
from collections import defaultdict

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import minimax_speech_b200.synth as synth  # noqa: E402
from minimax_speech_b200 import pipeline  # noqa: E402
from minimax_speech_b200 import tokenizer as tk  # noqa: E402
from profiles import s3_mel_reference as R  # noqa: E402
from profiles.time_tokenizer import gpu_info, time_ms  # noqa: E402


def mel_flops(lens, n_mels=128):
    return sum(2.0 * (400 * 402 + 201 * n_mels) * (n // 160) for n in lens)


def clips(lens, seed=0):
    g = torch.Generator().manual_seed(seed)
    out = []
    for i, n in enumerate(lens):
        t = torch.arange(n, dtype=torch.float32) / 16000
        f0 = 150 + 50 * torch.sin(2 * math.pi * 0.3 * t + i)
        ph = torch.cumsum(2 * math.pi * f0 / 16000, 0)
        out.append(0.1 * sum(torch.sin(h * ph) / h for h in range(1, 12)) + 0.01 * torch.randn(n, generator=g))
    return out


def padded(cs):
    a = torch.zeros(len(cs), max(c.shape[0] for c in cs))
    for b, c in enumerate(cs):
        a[b, :c.shape[0]] = c
    return a.cuda()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs the GPU"
    print(f"GPU: {gpu_info()}  (name, power limit, max SM clock)")
    filt = tk.mel_filters(128).cuda()
    tok = tk.S3TokenizerV2(weight_seed=33, precision="bf16x3")
    tok.handle(torch.device("cuda"))

    # 1. the front end alone
    eq = [160000] * 16
    audio_eq = padded(clips(eq))
    ms_eq = time_ms(lambda: tk.log_mel_spectrogram(audio_eq, audio_len=eq, filters=filt), a.reps)
    mel_eq, _ = tk.log_mel_spectrogram(audio_eq, audio_len=eq, filters=filt)
    ms_q = time_ms(lambda: tok.quantize(mel_eq, torch.tensor([1000] * 16)), a.reps)
    print(f"log-mel 16 x 10 s: {ms_eq:.3f} ms, {mel_flops(eq) / 1e9:.2f} GFLOP -> {mel_flops(eq) / (ms_eq * 1e-3) / 1e12:.1f} "
          f"TFLOP/s fp32; bf16x3 quantize of the same mels {ms_q:.2f} ms: the front end is "
          f"{100 * ms_eq / ms_q:.1f} % of it")

    mixed = synth.mixed_lengths(64, 2, 30, frame_rate=16000, seed=0)
    cs = clips(mixed, seed=1)
    audio_mx = padded(cs)
    ms_mx = time_ms(lambda: tk.log_mel_spectrogram(audio_mx, audio_len=mixed, filters=filt), a.reps)
    audio_s = sum(mixed) / 16000
    print(f"log-mel 64 mixed clips (2-30 s, {audio_s:.0f} s of audio, padded to {max(mixed) / 16000:.0f} s), one call: "
          f"{ms_mx:.3f} ms, {mel_flops(mixed) / (ms_mx * 1e-3) / 1e12:.1f} TFLOP/s on the valid frames")

    long = [600 * 16000]
    audio_long = padded(clips(long, seed=2))
    ms_long = time_ms(lambda: tk.log_mel_spectrogram(audio_long, audio_len=long, filters=filt), max(3, a.reps // 4))
    print(f"log-mel one 10-minute clip: {ms_long:.3f} ms, {mel_flops(long) / (ms_long * 1e-3) / 1e12:.1f} TFLOP/s")

    # 2. the reference function per clip on the same GPU
    cs_dev = [c.cuda() for c in cs]

    def ref_per_clip():
        return [R.s3_log_mel(c, filt) for c in cs_dev]
    ms_ref = time_ms(ref_per_clip, max(3, a.reps // 4))
    print(f"reference log_mel_spectrogram (torch.stft fp32), 64 calls, one per clip: {ms_ref:.3f} ms "
          f"({ms_ref / ms_mx:.1f}x the one kernel call)")

    # 3. audio to tokens
    ms_at = time_ms(lambda: tok.quantize_audio(audio_mx, mixed), max(3, a.reps // 2))
    ml = torch.tensor([n // 160 for n in mixed], dtype=torch.int32)

    def torch_then_quantize():
        mels = ref_per_clip()
        mel = torch.zeros(len(mels), 128, max(m.shape[1] for m in mels), device="cuda")
        for b, m in enumerate(mels):
            mel[b, :, :m.shape[1]] = m
        return tok.quantize(mel, ml)
    ms_tq = time_ms(torch_then_quantize, max(3, a.reps // 2))
    print(f"audio -> tokens, 64 mixed clips, bf16x3: quantize_audio (one padded call) {ms_at:.2f} ms "
          f"= {audio_s / (ms_at * 1e-3):.0f} audio-s/s; torch mels per clip + one quantize {ms_tq:.2f} ms")

    # 4. extract_tokens
    store = {f"clip{i}.wav": c for i, c in enumerate(cs)}
    paths = list(store)
    for budget in (None, 64 * 30 * 16000):
        pipeline.extract_tokens(paths[:4], store.__getitem__, tok, "cuda", save=False, max_batch_samples=budget)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        pipeline.extract_tokens(paths, store.__getitem__, tok, "cuda", save=False, max_batch_samples=budget)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        print(f"extract_tokens, 64 files, max_batch_samples={budget}: {dt * 1e3:.1f} ms "
              f"= {audio_s / dt:.0f} audio-s/s (host clock, audio already in memory)")

    # 5. per-kernel split of the front end
    for label, audio, lens in (("16 x 10 s", audio_eq, eq), ("64 mixed", audio_mx, mixed), ("10-minute clip", audio_long, long)):
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for _ in range(5):
                tk.log_mel_spectrogram(audio, audio_len=lens, filters=filt)
            torch.cuda.synchronize()
        per = defaultdict(float)
        for e in prof.events():
            if e.device_type == torch.autograd.DeviceType.CUDA and "s3_mel" in e.name:
                per["frames (pass 1)" if "frames" in e.name else "normalise (pass 2)"] += e.device_time_total / 1e3 / 5
        print(f"kernels, {label}: " + ", ".join(f"{k} {v:.3f} ms" for k, v in per.items()))


if __name__ == "__main__":
    main()
