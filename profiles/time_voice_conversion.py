"""Time sample-rate conversion (csrc/resample.cu, audio.resample) and voice conversion (vc.VoiceConverter) on the GPU:
  1. the resampler: 64 clips of 30 s at 44.1 kHz -> 24 kHz and -> 16 kHz in one padded call; GB/s (audio read + written
     once) against a measured device-to-device copy of the same input; torchaudio.functional.resample on the same GPU
     over the zero-padded batch (one conv1d) for comparison;
  2. convert: 64 sources of 2-30 s (synth.mixed_lengths) at 44.1 kHz with 8 prompts of 3-10 s, the reference-size
     models with synthetic weights (flow bf16, S3 tokenizer bf16x3, DAC-VAE bf16); audio-s/s and a per-stage split
     (resample, tokens, prompt latents, flow, speed, decode, each timed alone with device events), against one convert
     call per source.
Inputs are larger than L2 (126 MB) where the kernel is bandwidth-bound; device events after warm-up; the card's name
and power limit are read in the same run.

    python -m profiles.time_voice_conversion [--reps 20]

Log: profiles/r07_time_voice_conversion.log.
"""
import argparse
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import minimax_speech_b200.synth as synth  # noqa: E402
from minimax_speech_b200 import audio, vc  # noqa: E402
from minimax_speech_b200.dac import DACVAEDecoder, DACVAEEncoder  # noqa: E402
from minimax_speech_b200.flow import CausalConditionalCFM, CausalConditionalDecoder  # noqa: E402
from minimax_speech_b200.front import CausalMaskedDiffWithXvec  # noqa: E402
from minimax_speech_b200.tokenizer import S3TokenizerV2  # noqa: E402
from profiles.time_tokenizer import gpu_info, time_ms  # noqa: E402

DEV = torch.device("cuda:0")
RATE = 44100


def clip(n, seed):
    g = torch.Generator().manual_seed(seed)
    t = torch.arange(n, dtype=torch.float64) / RATE
    x = 0.3 * torch.sin(2 * torch.pi * (140 + 40 * torch.sin(2 * torch.pi * 0.3 * t)) * t) + 0.02 * torch.randn(n, generator=g, dtype=torch.float64)
    return x.float()


def timed(fn):
    """(result, ms) of one call between device events."""
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    torch.cuda.synchronize()
    ev[0].record()
    r = fn()
    ev[1].record()
    torch.cuda.synchronize()
    return r, ev[0].elapsed_time(ev[1])


def resampler_section(reps):
    import torchaudio.functional as AF
    B, S = 64, 30 * RATE
    x = torch.randn(B, S, device=DEV).clamp_(-1, 1)
    lens = [S] * B
    copy_dst = torch.empty_like(x)
    t_copy = time_ms(lambda: copy_dst.copy_(x), reps)
    gbs_copy = 2 * x.numel() * 4 / t_copy / 1e6
    print(f"device copy of the {x.numel() * 4 / 1e6:.0f} MB input: {t_copy:.3f} ms, {gbs_copy:.0f} GB/s (read + write)")
    for new in (24000, 16000):
        t_k = time_ms(lambda: audio.resample(x, RATE, new, lens), reps)
        out, _ = audio.resample(x, RATE, new, lens)
        gbs = (x.numel() + out.numel()) * 4 / t_k / 1e6
        t_ta = time_ms(lambda: AF.resample(x, RATE, new), max(2, reps // 4))
        ref = AF.resample(x, RATE, new)
        d = ((out - ref).norm() / ref.norm()).item()
        print(f"resample 64 x 30 s 44.1k -> {new // 1000}k: {t_k:.3f} ms, {gbs:.0f} GB/s ({gbs / gbs_copy:.2f} of the copy); "
              f"torchaudio (conv1d, fp32) {t_ta:.3f} ms ({t_ta / t_k:.1f}x); rel-L2 vs torchaudio fp32 {d:.1e}; "
              f"{B * S / RATE / (t_k / 1e3):.0f} audio-s/s")


def build():
    est = CausalConditionalDecoder(precision="bf16")
    cfm = CausalConditionalCFM(240, dict(t_scheduler="cosine", inference_cfg_rate=0.7), 1, 80, est)
    flow = CausalMaskedDiffWithXvec(decoder=cfm, precision="bf16")
    return vc.VoiceConverter(flow, S3TokenizerV2(weight_seed=33, precision="bf16x3"), DACVAEEncoder(), DACVAEDecoder(), DEV)


def convert_section(speed):
    vcv = build()
    secs = [f // 50 for f in synth.mixed_lengths(64, 2, 30, seed=3)]
    sources = [clip(s * RATE, 100 + i) for i, s in enumerate(secs)]
    prompt_secs = [3, 4, 5, 6, 7, 8, 9, 10]
    prompts = vcv.prompts([clip(s * RATE, 200 + i) for i, s in enumerate(prompt_secs)], RATE,
                          embedding=torch.randn(8, 192, generator=torch.Generator().manual_seed(0)).to(DEV))
    which = [prompts[i % 8] for i in range(64)]
    audio_s = float(sum(secs))
    vcv.convert(sources, RATE, which, speed)  # warm-up: workspaces, plans, handles
    _, t_all = timed(lambda: vcv.convert(sources, RATE, which, speed))
    out_s = sum(w.shape[0] for w in vcv.convert(sources, RATE, which, speed)) / 24000
    print(f"convert, 64 sources ({audio_s:.0f} s of 44.1 kHz input, {out_s:.0f} s of output at speed {speed}), 8 prompts: "
          f"{t_all:.1f} ms, {audio_s / (t_all / 1e3):.1f} source-audio-s/s")

    # per-stage split (each stage alone, same inputs)
    buf, lens = vcv._batch(sources)
    (a16, l16), t_rs = timed(lambda: vcv._at(buf, lens, RATE, 16000))
    toks, t_tok = timed(lambda: vcv._tokens(a16, l16, 16000))
    pbuf, plens = vcv._batch([clip(s * RATE, 200 + i) for i, s in enumerate(prompt_secs)])
    _, t_prs = timed(lambda: vcv._at(pbuf, plens, RATE, 16000))
    _, t_ptok = timed(lambda: vcv._tokens(pbuf, plens, RATE))
    _, t_prompt = timed(lambda: vcv.prompts([clip(s * RATE, 200 + i) for i, s in enumerate(prompt_secs)], RATE))
    (lat, L), t_flow = timed(lambda: vcv.flow.inference_batch(toks, [p.token for p in which], [p.feat for p in which],
                                                              torch.cat([p.embedding for p in which]), [True] * 64))
    (z, zl), t_speed = timed(lambda: vc.change_speed(lat, L.tolist(), speed))
    _, t_dec = timed(lambda: vcv.dac_decoder.decode(z, torch.tensor(zl, dtype=torch.int32)))
    print(f"  stages: resample (sources -> 16k) {t_rs:.1f} ms | tokens {t_tok:.1f} ms | flow {t_flow:.1f} ms | speed "
          f"{t_speed:.2f} ms | decode {t_dec:.1f} ms | (8 prompts, separately: prompts() {t_prompt:.1f} ms, of which "
          f"resample to 16k {t_prs:.2f} ms and tokens with resample {t_ptok:.1f} ms)")
    total = t_rs + t_tok + t_flow + t_speed + t_dec
    print(f"  resample share of the source path: {t_rs / total:.2%}; speed share {t_speed / total:.2%}")

    one = lambda: [vcv.convert([s], RATE, p, speed) for s, p in zip(sources, which)]  # noqa: E731
    one()
    _, t_one = timed(one)
    print(f"one convert per source: {t_one:.1f} ms, {audio_s / (t_one / 1e3):.1f} source-audio-s/s; batched is "
          f"{t_one / t_all:.2f}x faster")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--speed", type=float, default=1.1)
    args = ap.parse_args()
    print(f"GPU: {torch.cuda.get_device_name(0)} | nvidia-smi name, power limit, max SM clock: {gpu_info()}")
    t0 = time.time()
    # (no inference_mode around model construction: the tokenizer's filter bank must stay an ordinary tensor)
    resampler_section(args.reps)
    convert_section(args.speed)
    print(f"(wall {time.time() - t0:.0f} s)")


if __name__ == "__main__":
    main()
