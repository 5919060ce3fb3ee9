"""Time the S3 tokenizer (S3TokenizerV2.quantize, shipped width: 1280 wide, 20 heads, 6 blocks) on the GPU, fp32 mode
against the bf16x3 tensor-core mode:
  1. 16 clips x 10 s (one call), the two modes alternating;
  2. 64 clips of synth.mixed_lengths (2-30 s) through quantize, one right-padded call;
  3. one batch of 30 s windows (clips longer than 30 s: the sliding-window path around one device call);
  4. per-kernel shares of one bf16x3 16 x 10 s call (torch.profiler, a run of its own), with the achieved TFLOP/s of the
     attention kernel and of the GEMMs (operations counted from the shapes below).
The GPU's name and power limit are read in the same run.

    python -m profiles.time_tokenizer [--reps 20]

Log: profiles/r04_time_tokenizer.log.
"""
import argparse
import os
import subprocess
import sys
from collections import defaultdict

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import minimax_speech_b200.synth as synth  # noqa: E402
from minimax_speech_b200.tokenizer import S3TokenizerV2  # noqa: E402


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[torch.cuda.current_device()] if q else "unknown"
    except Exception as e:  # the timings stand without it, but say so
        return f"nvidia-smi failed: {e}"


def batch(lens, first=10):
    mel = torch.zeros(len(lens), 128, max(lens))
    for i, n in enumerate(lens):
        mel[i, :, :n] = synth.s3_mel(first + i, n)[0]
    return mel.cuda(), torch.tensor(lens)


def time_ms(fn, reps):
    fn()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(reps):
        fn()
    ev[1].record()
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1]) / reps


def flops(B, T, n_mels=128, C=1280, H=20, n_blocks=6):
    """bf16x3 MMA operations (2 per multiply-add, over the 3K-wide split operands, both conv taps) and fp32 attention
    operations (QK^T and PV over every key) of one equal-length call."""
    T1 = (T - 1) // 2 + 1
    T2 = (T1 - 1) // 2 + 1
    R = B * T2
    gemm = 2.0 * B * T1 * C * (2 * 6 * n_mels) + 2.0 * B * T2 * C * (2 * 6 * C)
    gemm += n_blocks * 2.0 * R * (3 * C * 3 * C + C * 3 * C + 4 * C * 3 * C + C * 12 * C)
    att = n_blocks * 4.0 * B * H * T2 * T2 * 64
    return gemm, att


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs the GPU"
    print(f"GPU: {gpu_info()}  (name, power limit, max SM clock)")
    toks = {p: S3TokenizerV2(weight_seed=33, precision=p) for p in ("fp32", "bf16x3")}
    for p, t in toks.items():
        t.handle(torch.device("cuda"))

    mel, ml = batch([1000] * 16)
    res = defaultdict(list)
    for _ in range(3):  # alternate the modes
        for p, t in toks.items():
            res[p].append(time_ms(lambda: t.quantize(mel, ml), a.reps if p == "bf16x3" else max(2, a.reps // 4)))
    f32, f3 = min(res["fp32"]), min(res["bf16x3"])
    print(f"16 x 10 s: fp32 {f32:.2f} ms (runs {', '.join(f'{v:.2f}' for v in res['fp32'])}), "
          f"bf16x3 {f3:.2f} ms (runs {', '.join(f'{v:.2f}' for v in res['bf16x3'])}): {f32 / f3:.1f}x")
    gemm, att = flops(16, 1000)
    print(f"  bf16x3: {gemm / 1e12:.2f} TFLOP of bf16 MMA work + {att / 1e9:.1f} GFLOP fp32 attention; "
          f"whole call {(gemm + att) / (f3 * 1e-3) / 1e12:.0f} TFLOP/s")

    lens = synth.mixed_lengths(64, 2, 30, frame_rate=100, seed=0)
    mel, ml = batch(lens, first=300)
    audio_s = sum(lens) / 100.0
    for p, t in toks.items():
        ms = time_ms(lambda: t.quantize(mel, ml), 3 if p == "fp32" else a.reps // 2)
        print(f"64 mixed clips (2-30 s, {audio_s:.0f} s of audio, padded to {max(lens) / 100:.0f} s): {p} {ms:.1f} ms "
              f"= {audio_s / (ms * 1e-3):.0f} audio-s/s")

    lens = [9000, 6000, 4500, 3100]  # 90 / 60 / 45 / 31 s -> 4 + 3 + 2 + 2 = 11 windows of 30 s in one device call
    mel, ml = batch(lens, first=400)
    for p, t in toks.items():
        ms = time_ms(lambda: t.quantize(mel, ml), 2 if p == "fp32" else a.reps // 2)
        print(f"30 s windows of clips {[n / 100 for n in lens]} s (11 windows, one call): {p} {ms:.1f} ms")

    mel, ml = batch([1000] * 16)
    t = toks["bf16x3"]
    t.quantize(mel, ml)
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(5):
            t.quantize(mel, ml)
        torch.cuda.synchronize()
    per = defaultdict(lambda: [0, 0.0])
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            name = e.name.replace("(anonymous namespace)::", "").replace("void ", "").split("<")[0].split("(")[0]
            name = name.split("::")[-1]
            per[name][0] += 1
            per[name][1] += e.device_time_total / 1e3 / 5  # ms per call
    total = sum(v[1] for v in per.values())
    print(f"per-kernel shares of one bf16x3 16 x 10 s call (torch.profiler, {total:.2f} ms of kernel time per call):")
    for name, (n, ms) in sorted(per.items(), key=lambda kv: -kv[1][1]):
        extra = ""
        if name.startswith("conv_gemm"):
            extra = f"  {gemm / (ms * 1e-3) / 1e12:.0f} TFLOP/s (bf16 MMA work)"
        elif "attention" in name:
            extra = f"  {att / (ms * 1e-3) / 1e12:.1f} TFLOP/s (fp32)"
        print(f"  {name:32s} {n // 5:4d} launches {ms:8.3f} ms {100 * ms / total:5.1f} %{extra}")


if __name__ == "__main__":
    main()
