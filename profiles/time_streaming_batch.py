"""Timing aid: streaming synthesis of N concurrent sessions, N in {1, 4, 16, 64}, advanced one after another through N
``StreamingSession``s against one ``StreamingBatch``.  Each session has a 3 s prompt (75 tokens, 150 latent frames)
and 10 s of tokens (250) pushed in 25-token pieces, as fast as the synthesis takes them (no LLM in the loop).  Full-size
synthetic weights, tensor-core path, 10 Euler steps with CFG, DAC context 16 frames.

Per configuration, one untimed pass warms up every shape, then one timed pass reports:
  * audio-s/s: N x 10 s over the wall time of the whole pass;
  * first-chunk latency: from the start of the pass to a session's first chunk (p50 and max over the sessions);
  * per-hop latency: from the push of a round of pieces to a session's chunk of that round (p50 and max over all chunks;
    one after another, session k also waits for sessions 0 .. k-1).
Every time is host wall time after torch.cuda.synchronize().  Prints the device name and power limit first; needs a GPU."""
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import minimax_speech_b200.synth as synth  # noqa: E402
from minimax_speech_b200.dac import DACVAEDecoder  # noqa: E402
from minimax_speech_b200.flow import CausalConditionalCFM, CausalConditionalDecoder  # noqa: E402
from minimax_speech_b200.front import CausalMaskedDiffWithXvec  # noqa: E402
from minimax_speech_b200.streaming import StreamingBatch, StreamingSession  # noqa: E402

DEV = torch.device("cuda:0")
N_PROMPT, N_TOKENS, PIECE, AUDIO_S = 75, 250, 25, 10.0


def device_line():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "nvidia-smi unavailable"
    return f"device: {torch.cuda.get_device_name(DEV)} | nvidia-smi name, power.limit, clocks.max.sm: {q}"


def build():
    est = CausalConditionalDecoder()
    cfm = CausalConditionalCFM(240, dict(t_scheduler="cosine", inference_cfg_rate=0.7), 1, 80, est)
    return CausalMaskedDiffWithXvec(decoder=cfm), DACVAEDecoder()


def inputs(n):
    out = []
    for i in range(n):
        tok, emb = synth.token_inputs(800 + i, N_TOKENS)
        ptok, _ = synth.token_inputs(900 + i, N_PROMPT)
        pfeat = synth.dac_latents(1000 + i, 2 * N_PROMPT).transpose(1, 2).contiguous()
        out.append((tok[0].tolist(), ptok.to(DEV), pfeat.to(DEV), emb.to(DEV)))
    return out


def now():
    torch.cuda.synchronize()
    return time.perf_counter()


def run_sequential(flow, dac, ins):
    """-> (wall s, first-chunk latencies, per-hop latencies, samples per session)"""
    t0 = now()
    sess = [StreamingSession(flow, dac, p, f, embedding=e) for _, p, f, e in ins]
    first, hops, samples = [None] * len(ins), [], [0] * len(ins)
    for k in range(0, N_TOKENS, PIECE):
        tr = now()
        for i, (toks, *_) in enumerate(ins):
            chunks = sess[i].push(toks[k:k + PIECE])
            if chunks:
                t = now()
                hops.append(t - tr)
                first[i] = first[i] or t - t0
                samples[i] += sum(c.shape[1] for c in chunks)
    tr = now()
    for i, s in enumerate(sess):
        c = s.finish()
        t = now()
        hops.append(t - tr)
        first[i] = first[i] or t - t0
        samples[i] += c.shape[1]
    return now() - t0, first, hops, samples


def run_batched(flow, dac, ins):
    t0 = now()
    batch = StreamingBatch(flow, dac)
    ids = [batch.open(p, f, embedding=e) for _, p, f, e in ins]
    first, hops, samples = {}, [], {sid: 0 for sid in ids}

    def step(tr):
        out = batch.step()
        t = now()
        for sid, chunks in out.items():
            hops.append(t - tr)
            first.setdefault(sid, t - t0)
            samples[sid] += sum(c.shape[1] for c in chunks)

    for k in range(0, N_TOKENS, PIECE):
        tr = now()
        for sid, (toks, *_) in zip(ids, ins):
            batch.push(sid, toks[k:k + PIECE])
        step(tr)
    tr = now()
    for sid in ids:
        batch.finish(sid)
    step(tr)
    return now() - t0, [first[sid] for sid in ids], hops, [samples[sid] for sid in ids]


def report(name, n, res):
    wall, first, hops, samples = res
    ms = lambda v: 1000 * v  # noqa: E731
    print(f"N={n:3d} {name:<10s} {n * AUDIO_S / wall:8.1f} audio-s/s  (wall {wall:7.3f} s)  first chunk p50 {ms(statistics.median(first)):7.1f} "
          f"max {ms(max(first)):7.1f} ms  per hop p50 {ms(statistics.median(hops)):7.1f} max {ms(max(hops)):7.1f} ms  "
          f"({len(hops)} chunks)", flush=True)
    return samples


def main():
    print(device_line(), flush=True)
    print(f"workload per session: {N_PROMPT}-token / {2 * N_PROMPT}-frame prompt, {N_TOKENS} tokens ({AUDIO_S:g} s) in pieces of "
          f"{PIECE}; bf16 tensor-core path, full-size synthetic weights", flush=True)
    flow, dac = build()
    with torch.inference_mode():
        for n in (1, 4, 16, 64):
            ins = inputs(n)
            run_sequential(flow, dac, ins), run_batched(flow, dac, ins)  # warm-up: every shape of the timed passes
            a = report("sequential", n, run_sequential(flow, dac, ins))
            b = report("batched", n, run_batched(flow, dac, ins))
            assert a == b == [int(AUDIO_S * 24000)] * n, "sample counts differ"


if __name__ == "__main__":
    main()
