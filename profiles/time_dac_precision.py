"""Timing aid: the DAC-VAE decoder and encoder with bf16 against fp16 GEMM operands (precision="bf16" / "fp16": the
same kernels compiled for the two 16-bit formats), and each against fp32 mode on the same inputs.

Cases: decode 64 x 30 s (the configs[2] shape) and 16 x 10 s on the trained-scale decoder weights
(synth.dac_decoder_state_dict(init="trained"): Snake alpha in [0.5, 2], activations O(10)); encode 16 x 10 s and one
call on 64 mixed 2-30 s clips (per-clip lengths) on the encoder's test weights.  The two precisions run alternately in
one process, REPS passes each, with a 512 MB buffer overwritten before every timed pass (nothing of the previous pass
is left in the 126 MB L2).  Reported per case: median, min and max ms per call, the spread (max - min) / median, and
the SNR of the output against fp32 mode (for the encoder: of m and of logs; fp32 mode runs REF_ITEMS items per call).
Prints the device name and power limit first; needs a GPU."""
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import minimax_speech_b200.synth as synth  # noqa: E402
from minimax_speech_b200.dac import DACVAEDecoder, DACVAEEncoder  # noqa: E402

DEV = torch.device("cuda:0")
SR, HOP = 24000, 480
REPS = 7
REF_ITEMS = 4  # fp32 mode runs this many items per call (its unfused workspace for 64 x 30 s does not fit in 180 GB)
PRECISIONS = ("bf16", "fp16")


def device_line():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "nvidia-smi unavailable"
    return f"device: {torch.cuda.get_device_name(DEV)} | nvidia-smi name, power.limit, clocks.max.sm: {q}"


_scrub = None


def scrub_l2():
    global _scrub
    if _scrub is None:
        _scrub = torch.empty(512 * 2 ** 20 // 4, device=DEV)
    _scrub.fill_(1.0)


def time_once(fn):
    scrub_l2()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def snr_db(y, ref):
    y, ref = y.double(), ref.double()
    return float(10.0 * torch.log10((ref ** 2).sum() / ((y - ref) ** 2).sum().clamp_min(1e-300)))


def compare(name, audio_s, calls, snrs):
    """calls: precision -> fn; alternates the precisions (the starting one too) for REPS rounds."""
    for fn in calls.values():
        fn()  # warm-up: workspace, plans, module load
    ms = {p: [] for p in calls}
    for r in range(REPS):
        order = list(calls) if r % 2 == 0 else list(reversed(list(calls)))
        for p in order:
            ms[p].append(time_once(calls[p]))
    print(f"{name}  ({audio_s:g} s of audio)", flush=True)
    for p, v in ms.items():
        med = statistics.median(v)
        print(f"  {p:5s} median {med:8.2f} ms  min {min(v):8.2f}  max {max(v):8.2f}  spread {(max(v) - min(v)) / med * 100:5.1f} %"
              f"  -> {audio_s / (med / 1000):8.0f} audio-s/s   SNR vs fp32 mode: {snrs[p]}", flush=True)
    b, h = statistics.median(ms["bf16"]), statistics.median(ms["fp16"])
    print(f"  fp16 / bf16 median time {h / b:.4f}", flush=True)


def decode_case(name, B, seconds, sd):
    L = int(seconds * SR) // HOP
    z = torch.cat([synth.dac_latents(1000 + b, L) for b in range(B)], 0).to(DEV)
    decs = {}
    for p in PRECISIONS + ("fp32",):
        decs[p] = DACVAEDecoder(precision=p)
        decs[p].load_state_dict(sd)
    ref = torch.cat([decs["fp32"].decode(z[i:i + REF_ITEMS]) for i in range(0, B, REF_ITEMS)], 0)
    snrs = {p: f"{snr_db(decs[p].decode(z), ref):.1f} dB" for p in PRECISIONS}
    del ref, decs["fp32"]
    torch.cuda.empty_cache()
    compare(name, B * seconds, {p: (lambda d=decs[p]: d.decode(z)) for p in PRECISIONS}, snrs)
    del decs, z
    torch.cuda.empty_cache()


def encode_case(name, lengths, sd, equal):
    L = max(lengths)
    audio = torch.zeros(len(lengths), 1, L * HOP)
    for b, n in enumerate(lengths):
        audio[b, :, :n * HOP] = synth.audio_clip(2000 + b, n * HOP)[0]
    audio = audio.to(DEV)
    noise = torch.zeros(len(lengths), 80, L, device=DEV)
    ln = None if equal else lengths
    encs = {}
    for p in PRECISIONS + ("fp32",):
        encs[p] = DACVAEEncoder(precision=p)
        encs[p].load_state_dict(sd)
    ref = [encs["fp32"].encode(audio[i:i + REF_ITEMS], noise[i:i + REF_ITEMS], lengths=ln and ln[i:i + REF_ITEMS])
           for i in range(0, len(lengths), REF_ITEMS)]
    m32, l32 = torch.cat([r[1] for r in ref], 0), torch.cat([r[2] for r in ref], 0)
    del ref
    snrs = {}
    for p in PRECISIONS:
        _, m, lg = encs[p].encode(audio, noise, lengths=ln)
        snrs[p] = f"m {snr_db(m, m32):.1f} dB, logs {snr_db(lg, l32):.1f} dB"
    del encs["fp32"], m32, l32
    torch.cuda.empty_cache()
    compare(name, sum(lengths) * HOP / SR, {p: (lambda e=encs[p]: e.encode(audio, noise, lengths=ln)) for p in PRECISIONS},
            snrs)
    del encs, audio
    torch.cuda.empty_cache()


def main():
    print(device_line(), flush=True)
    print(f"{REPS} alternating passes per precision, L2 overwritten (512 MB) before each timed pass", flush=True)
    dsd = synth.dac_decoder_state_dict(0, init="trained")
    decode_case("decode 64 x 30 s (trained-scale weights)", 64, 30.0, dsd)
    decode_case("decode 16 x 10 s (trained-scale weights)", 16, 10.0, dsd)
    esd = synth.dac_encoder_state_dict(0, init="test")
    encode_case("encode 16 x 10 s (test weights)", [500] * 16, esd, equal=True)
    mixed = synth.mixed_lengths(64)
    encode_case(f"encode 64 mixed {min(mixed) * HOP / SR:g}-{max(mixed) * HOP / SR:g} s clips, one call (test weights)",
                mixed, esd, equal=False)


if __name__ == "__main__":
    main()
