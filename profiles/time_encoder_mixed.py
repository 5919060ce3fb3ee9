"""Timing aid: DAC-VAE encoder (tensor-core path) on 256 clips of mixed length (synth.mixed_lengths: 2-30 s, the
bulk-latent-extraction workload), one encode call per clip against length-sorted micro-batches with per-clip
``lengths`` at three sample budgets, on device-resident audio and through pipeline.extract_latents (which adds the
host work: loading, padding, noise, read-back).  Ends with profiles/time_encoder.py (16 x 10 s, equal lengths).
Prints the device name and power limit first; needs a GPU."""
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import minimax_speech_b200.synth as synth  # noqa: E402
from minimax_speech_b200 import pipeline  # noqa: E402
from minimax_speech_b200.dac import DACVAEEncoder  # noqa: E402

DEV = torch.device("cuda:0")
SR, HOP = 24000, 480
BUDGETS = [16 * 240000, 32 * 240000, 64 * 240000]  # padded samples per micro-batch: 16, 32, 64 x 10 s
PASSES = 3


def device_line():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "nvidia-smi unavailable"
    return f"device: {torch.cuda.get_device_name(DEV)} | nvidia-smi name, power.limit, clocks.max.sm: {q}"


def timed(fn, passes=PASSES):
    """ms per pass of fn() (CUDA events, synchronised), every pass; fn was warmed up by the caller."""
    out = []
    for _ in range(passes):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1))
    return out


def report(name, ms, audio_s):
    best, mean = min(ms), sum(ms) / len(ms)
    print(f"{name:<44s} {best:9.1f} ms best, {mean:9.1f} ms mean of {len(ms)}  ->  {audio_s / (best / 1000):8.0f} audio-s/s "
          f"(best), {audio_s / (mean / 1000):8.0f} (mean)", flush=True)


def main():
    print(device_line(), flush=True)
    lengths = synth.mixed_lengths(256)  # latent frames (50 Hz)
    audio_s = sum(lengths) * HOP / SR
    print(f"workload: {len(lengths)} clips, {min(lengths) * HOP / SR:g}-{max(lengths) * HOP / SR:g} s, {audio_s:g} s of audio",
          flush=True)
    e = DACVAEEncoder()
    gen = torch.Generator(device=DEV).manual_seed(0)
    clips = [torch.rand(1, 1, n * HOP, device=DEV, generator=gen) * 0.2 - 0.1 for n in lengths]
    noise = [torch.randn(1, 80, n, device=DEV, generator=gen) for n in lengths]

    # (a) one call per clip
    ref = [None] * len(clips)

    def per_clip(keep=False):
        for i, (a, z) in enumerate(zip(clips, noise)):
            r = e.encode(a, z)
            if keep:
                ref[i] = r

    per_clip(keep=True)  # warm-up: every shape once
    report("per clip (256 calls)", timed(per_clip), audio_s)

    # (b) length-sorted micro-batches, lengths passed per clip
    for budget in BUDGETS:
        plan = pipeline.plan_micro_batches([n * HOP for n in lengths], budget)
        batches = []
        for idx in plan:
            L = max(lengths[i] for i in idx)
            a = torch.zeros(len(idx), 1, L * HOP, device=DEV)
            z = torch.zeros(len(idx), 80, L, device=DEV)
            for b, i in enumerate(idx):
                a[b, :, :lengths[i] * HOP] = clips[i][0]
                z[b, :, :lengths[i]] = noise[i][0]
            batches.append((idx, a, z, [lengths[i] for i in idx]))
        outs = []

        def batched(keep=False):
            for idx, a, z, ln in batches:
                r = e.encode(a, z, lengths=ln)
                if keep:
                    outs.append((idx, ln, r))

        batched(keep=True)
        same = all(torch.equal(r[k][b:b + 1, :, :n], ref[i][k])
                   for idx, ln, r in outs for b, (i, n) in enumerate(zip(idx, ln)) for k in range(3))
        padded = sum(len(idx) * max(lengths[i] for i in idx) for idx in plan) / sum(lengths)
        report(f"batched, budget {budget / SR:g} s ({len(plan)} calls)", timed(batched), audio_s)
        print(f"    padded / valid frames {padded:.3f}; every clip identical to its per-clip call: {same}", flush=True)
        del batches, outs
    del ref

    # (c) pipeline.extract_latents end to end (files on local disk, torch.load, noise from a CPU generator)
    with tempfile.TemporaryDirectory() as tmp:
        paths = []
        for i, a in enumerate(clips):
            p = os.path.join(tmp, f"clip{i:03d}.pt")
            torch.save(a.reshape(-1).cpu(), p)
            paths.append(p)
        for budget in [None] + BUDGETS:
            def run():
                pipeline.extract_latents(paths, torch.load, e, DEV, save=False, generator=torch.Generator().manual_seed(0),
                                         max_batch_samples=budget)
            run()  # warm-up
            ms = []
            for _ in range(2):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                run()
                torch.cuda.synchronize()
                ms.append((time.perf_counter() - t0) * 1000)
            report("extract_latents, " + ("per file" if budget is None else f"budget {budget / SR:g} s"), ms, audio_s)

    print("equal lengths (profiles/time_encoder.py):", flush=True)
    subprocess.run([sys.executable, os.path.join(ROOT, "profiles", "time_encoder.py")], check=True)


if __name__ == "__main__":
    main()
