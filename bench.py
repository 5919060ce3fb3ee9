#!/usr/bin/env python
"""Headline benchmark: seconds of 24 kHz audio synthesised per second (BASELINE.json metric) on the
configuration the metric is quoted on -- configs[1]: 16 x 10 s utterances per GPU, 10-step Euler + CFG through
the CausalConditionalDecoder estimator, then DAC-VAE decode, bf16 tensor-core operands with fp32 accumulation.

  python bench.py --gpus N --steps K --warmup W                 (N > 1: launched by torch.distributed.run)
  python bench.py --impl reference --gpus N --steps K --warmup W  (the reference algorithm on the host CPU cores)

One JSON line on stdout (rank 0).  A step = one pass of the whole hot path over one batch of synthetic inputs.
The inputs and weights are seeded, so ``--dump-outputs DIR`` (the waveforms of the last timed step as float32 .npy)
lets two builds run with the same arguments be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "audio-sec synthesized/sec (24 kHz)"
UNIT = "audio-s/s"
FRAME_RATE = 50


_OUT = None


def claim_stdout():
    """The contract is ONE JSON line on stdout: keep a private handle on the real stdout and point fd 1 at stderr, so that
    whatever libraries print (NCCL's version / INFO lines go to stdout) cannot end up next to it."""
    global _OUT
    if _OUT is None:
        sys.stdout.flush()
        _OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(rec):
    claim_stdout()
    _OUT.write(json.dumps(rec) + "\n")
    _OUT.flush()


DUMP_BYTES = 60 * 10 ** 6  # data written by --dump-outputs, all arrays together (below 64 MB with the .npy headers)


def dump_outputs(directory, arrays):
    """Write each array as ``directory/<name>.npy`` in float32.  An array larger than its share of DUMP_BYTES is replaced
    by a fixed, seeded sample of its elements (flattened; the same positions for the same shape), so that outputs of
    two runs with the same arguments still line up element for element."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    budget = DUMP_BYTES // 4 // len(arrays)
    for name, t in arrays.items():
        t = t.detach().float()
        if t.numel() > budget:
            idx = np.unique(np.random.default_rng(0).integers(0, t.numel(), budget))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(directory, name + ".npy"), t.cpu().numpy())


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=16, help="utterances per GPU")
    ap.add_argument("--seconds", type=float, default=10.0, help="utterance length")
    ap.add_argument("--n-timesteps", type=int, default=10)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the configs[2..4] / batch-1 latency legs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned to DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    return a


def config_of(a):
    return {"workload": f"configs[1]: flow (CausalConditionalDecoder, {a.n_timesteps}-step Euler + CFG) + DAC-VAE "
                        f"decode, {a.batch} x {a.seconds:g} s utterances per GPU, 24 kHz",
            "utterances_per_gpu": a.batch, "utterance_seconds": a.seconds, "n_timesteps": a.n_timesteps,
            "cfg_rate": 0.7, "latent_rate_hz": FRAME_RATE, "sharding": "utterances per rank, no data-path collective; "
            "one waveform gather", "l2": "256 MiB scratch write between steps (inside the timed region); the "
            "per-step working set (> 1 GB activations + 212 MB weights) also exceeds the 126 MB L2"}


# ------------------------------------------------------------------------------------------ CPU / reference arm
class ReferenceModules:
    """The reference's OWN modules through its own call surface -- ``CausalConditionalCFM.forward``
    (speech/cosyvoice/flow/flow_matching.py:323-348, batch 1 like its solve_euler) then ``DACVAE.decode``
    (dac-vae/model.py:236-257) -- imported unmodified from /root/reference in the build container or from the copy
    oracle/stage_ref.py staged under baseline/_ref (git-ignored, travels to the GPU box); third-party packages absent
    from the image are the stubs of oracle/ref_import.py.  None of this repo's kernels or modules are on this path."""

    def __init__(self, esd, dsd, dev="cpu"):
        from oracle import ref_import as R
        self.root = R.REF_ROOT
        self.cfm = R.build_reference_flow()
        self.cfm.estimator.load_state_dict(esd, strict=True)
        self.dac = R.build_reference_dac()
        missing, unexpected = self.dac.load_state_dict(dsd, strict=False)
        assert not unexpected and all(k.startswith(("encoder.", "en_conv_post.")) for k in missing), (missing[:3], unexpected[:3])
        self.cfm.to(dev).eval()
        self.dac.to(dev).eval()

    def __call__(self, mu, mask, spks, cond, n_timesteps):
        lat, _ = self.cfm(mu=mu, mask=mask, n_timesteps=n_timesteps, temperature=1.0, spks=spks, cond=cond)
        return self.dac.decode(lat.float())


def reference_modules(esd, dsd, dev="cpu"):
    """-> ReferenceModules, or None when no copy of the reference is importable here (then the oracle port is timed)."""
    try:
        from oracle import ref_import as R
        if not R.reference_available():
            return None
        return ReferenceModules(esd, dsd, dev)
    except Exception as e:  # a reference that does not import is reported, not fatal: the port stands in
        sys.stderr.write(f"bench: reference modules not importable ({type(e).__name__}: {e}); timing the oracle port\n")
        return None


def oracle_sample(seconds, n_timesteps, esd, dsd, ref=None):
    """One utterance through the reference's CPU path (fp32, all host threads): the reference's own modules when a copy
    is importable (``ref``), else the oracle restatement."""
    import minimax_speech_b200.synth as synth
    from oracle import restatement as O
    T = int(round(seconds * FRAME_RATE))
    mu, mask, spks, cond = synth.batch_inputs([T])
    t0 = time.perf_counter()
    with torch.inference_mode():
        if ref is not None:
            wav = ref(mu, mask, spks, cond, n_timesteps)
        else:
            lat = O.cfm_forward(esd, synth.fixed_noise(), mu, mask, n_timesteps, 1.0, spks, cond)
            wav = O.dac_decode(dsd, lat)
    dt = time.perf_counter() - t0
    return dt, float(wav.abs().max())


def _ref_kind(ref):
    if ref is None:
        return "port", "oracle/restatement.py (restatement of the reference's PyTorch CPU path; no copy of the reference is importable on this box)"
    return "reference", (f"the reference's own CausalConditionalCFM.forward -> DACVAE.decode, unmodified modules from {ref.root} "
                         f"(third-party imports stubbed by oracle/ref_import.py)")


def cpu_baseline(a, esd, dsd):
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    ref = reference_modules(esd, dsd)
    kind, what = _ref_kind(ref)
    oracle_sample(0.32, 1, esd, dsd, ref)  # thread-pool / allocator warm-up
    n, total = 0, 0.0
    while n < a.batch and (n == 0 or total < 12.0):  # about 10-30 s of CPU work
        dt, _ = oracle_sample(a.seconds, a.n_timesteps, esd, dsd, ref)
        n, total = n + 1, total + dt
    return {"value": n * a.seconds / total, "unit": UNIT, "cores": cores, "kind": kind,
            "sample": f"{n} of {a.batch} utterances ({a.seconds:g} s, {a.n_timesteps} steps CFG + DAC decode), one at a "
                      f"time (the reference's solve_euler is batch-1), {what}, fp32 torch-CPU, "
                      f"{torch.get_num_threads()} threads, {total:.2f} s"}


def gpu_eager_baseline(a, esd, dsd, dev):
    """The denominator north_star names: the reference as eager PyTorch ON THE GPU (fp32 and bf16 autocast), one
    utterance at a time like the reference's solve_euler -- the reference's own modules when a copy is importable
    (baseline/_ref, staged by oracle/stage_ref.py), else the oracle restatement (plain torch ops) on cuda."""
    import minimax_speech_b200.synth as synth
    from oracle import restatement as O
    T = int(round(a.seconds * FRAME_RATE))
    e_gpu = {k: v.to(dev) for k, v in esd.items()}
    d_gpu = {k: v.to(dev) for k, v in dsd.items()}
    noise = synth.fixed_noise().to(dev)
    inputs = [[t.to(dev) for t in synth.batch_inputs([T], first_index=i)] for i in range(2)]
    ref = reference_modules(esd, dsd, dev)
    kind, what = _ref_kind(ref)
    out = {"unit": UNIT, "kind": kind, "sample": f"2 of {a.batch} utterances, batch 1 each, {what} as eager "
           f"PyTorch on cuda ({a.n_timesteps} steps CFG + DAC decode), best of 2 passes"}
    for name, ctx in (("fp32", None), ("bf16_autocast", torch.bfloat16)):
        best = None
        for _ in range(3):  # pass 0 = warm-up (cuDNN / cuBLAS heuristics)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            with torch.inference_mode(), torch.autocast("cuda", dtype=ctx, enabled=ctx is not None):
                for mu, mask, spks, cond in inputs:
                    if ref is not None:
                        ref(mu, mask, spks, cond, a.n_timesteps)
                    else:
                        lat = O.cfm_forward(e_gpu, noise, mu, mask, a.n_timesteps, 1.0, spks, cond)
                        O.dac_decode(d_gpu, lat.float())
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            best = ms if best is None or _ == 1 else min(best, ms)
        out[name] = len(inputs) * a.seconds / (best / 1000.0)
    del ref
    # fairness figure (SURVEY section 8d ii): the same eager algorithm with the whole batch in one call (the estimator
    # itself is batch-agnostic; the reference's solve_euler is not)
    mu, mask, spks, cond = [t.to(dev) for t in synth.batch_inputs([T] * a.batch)]
    for name, ctx in (("batched_fp32", None), ("batched_bf16_autocast", torch.bfloat16)):
        best = None
        for it in range(2):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            with torch.inference_mode(), torch.autocast("cuda", dtype=ctx, enabled=ctx is not None):
                lat = O.cfm_forward(e_gpu, noise, mu, mask, a.n_timesteps, 1.0, spks, cond)
                for b0 in range(0, a.batch, 4):  # decode in groups of 4: the eager decoder's activations are large
                    O.dac_decode(d_gpu, lat[b0:b0 + 4].float())
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            best = ms if it == 0 else min(best, ms)
        out[name] = a.batch * a.seconds / (best / 1000.0)
    out["sample"] += (f"; batched_*: all {a.batch} utterances in one call (DAC decode in groups of 4) through "
                      f"oracle/restatement.py (kind port: the reference's solve_euler cannot batch)")
    return out


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import minimax_speech_b200.synth as synth
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    esd = synth.estimator_state_dict(1986, "reference")
    dsd = synth.dac_decoder_state_dict(0, "reference")
    ref = reference_modules(esd, dsd)
    kind, what = _ref_kind(ref)
    oracle_sample(0.32, 1, esd, dsd, ref)
    seconds = a.seconds
    probe, _ = oracle_sample(seconds, a.n_timesteps, esd, dsd, ref)
    note = ""
    if probe * (a.steps + a.warmup) > 240.0 and seconds > 2.0:
        seconds, note = 2.0, " (sample shortened to 2 s utterances to bound the run)"
    for _ in range(max(a.warmup - 1, 0)):
        oracle_sample(seconds, a.n_timesteps, esd, dsd, ref)
    times = [oracle_sample(seconds, a.n_timesteps, esd, dsd, ref)[0] for _ in range(a.steps)]
    total = sum(times)
    value = seconds * a.steps / total
    cb = {"value": value, "unit": UNIT, "cores": cores, "kind": kind,
          "sample": f"each step = 1 utterance ({seconds:g} s, {a.n_timesteps} steps CFG + DAC decode) of the "
                    f"{a.batch}-utterance batch, {what}, fp32, {cores} threads{note}"}
    emit({"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
          "warmup": a.warmup, "ms_per_step": 1000.0 * total / a.steps, "higher_is_better": True,
          "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
          "config": config_of(a), "impl": "reference", "cpu_baseline": cb,
          "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            pass

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            out = self.p.communicate(timeout=5)[0]
        except subprocess.TimeoutExpired:
            self.p.kill()
            out = self.p.communicate()[0]
        sm, mx, pw, reasons = [], 0, [], set()
        for line in out.splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])), pw.append(float(f[2]))
                mx = max(mx, float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        busy = [c for c, w in zip(sm, pw) if w > 0.5 * max(pw)] if pw else sm
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": mx or None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}



# ------------------------------------------------------------------------------------------ BASELINE.json configs[2..4]
def extra_legs(a, syn, cfm, dac, dev, world, rank, sync_all, esd=None):
    """Throughput of the other configurations BASELINE.json lists, next to the unchanged headline (configs[1]):
    configs[2] DAC-VAE decoder only (64 x 30 s), configs[3] 32-step solve of 32 x 30 s utterances sharded by utterance,
    configs[4] 256 mixed-length (2-30 s) utterances, length-balanced over the ranks, one waveform gather at the end --
    the last two are STRONG scaling (fixed total work split over the ranks) -- and the batch-1 latency of configs[0]'s
    shape (one 10 s utterance, 10 steps) with eager launches and as one CUDA-graph replay.  Device time, max over ranks."""
    import torch.distributed as dist
    import minimax_speech_b200.synth as synth
    from minimax_speech_b200.pipeline import PlannedGather, gather_plan, shard_utterances, utterance_cost
    hop = dac.hop_length
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn, iters):
        sync_all()
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        sync_all()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()) / iters

    out = {}
    # ---- configs[2]: decoder only, 64 x 30 s of latents, 64 / world per rank
    n2 = 64 // world
    if n2 >= 1:
        z = torch.cat([synth.dac_latents(100 + rank * n2 + b, 1500) for b in range(n2)], 0).to(dev)
        dac.decode(z)
        ms = timed(lambda: dac.decode(z), 3)
        out["configs[2]"] = {"workload": f"DAC-VAE decoder only, 64 x 30 s latents ({n2} per GPU)", "value": world * n2 * 30.0 / (ms / 1000.0),
                             "unit": UNIT, "ms_per_step": ms, "scaling": "strong", "n_gpus": world}
        del z
    # ---- configs[3]: n_timesteps = 32, 30 s utterances, batch 32 sharded by utterance
    n3 = 32 // world
    if n3 >= 1:
        inp = [t.to(dev) for t in synth.batch_inputs([1500] * n3, first_index=300 + rank * n3)]
        step3 = lambda: syn(*inp, n_timesteps=32)
        step3()
        ms = timed(step3, 2)
        out["configs[3]"] = {"workload": f"flow (32-step Euler + CFG) + DAC decode, 32 x 30 s utterances ({n3} per GPU)",
                             "value": world * n3 * 30.0 / (ms / 1000.0), "unit": UNIT, "ms_per_step": ms, "scaling": "strong",
                             "n_gpus": world}
        del inp
    # ---- configs[4]: 256 mixed-length utterances; cost-model bin packing over the ranks, micro-batches of <= 32 sorted by
    # length, one gather of every rank's waveforms to rank 0
    lengths_all = synth.mixed_lengths(256)
    shards = shard_utterances(lengths_all, world)
    mine = sorted(shards[rank], key=lambda i: lengths_all[i])
    groups = [mine[i:i + 32] for i in range(0, len(mine), 32)]
    batches = [[t.to(dev) for t in synth.batch_inputs([lengths_all[i] for i in g], first_index=1000 + g[0])] for g in groups]
    plan = gather_plan(shards, [n * hop for n in lengths_all])
    order = {uid: k for k, uid in enumerate(plan[rank][1])}
    smax = max(n for p_ in plan for n in p_[0])
    local = torch.zeros(len(mine), 1, smax, device=dev)
    gatherer = PlannedGather(plan, dev, dst=0) if world > 1 else None
    busy0, busy1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def step4():
        busy0.record()
        for g, inp in zip(groups, batches):
            wav = syn(*inp, n_timesteps=a.n_timesteps)
            rows = torch.tensor([order[i] for i in g], device=dev)
            local[rows, :, :wav.shape[-1]] = wav
        busy1.record()
        return gatherer(local) if gatherer else local

    step4()
    ms = timed(step4, 1)
    busy = torch.tensor([busy0.elapsed_time(busy1)], device=dev)
    if world > 1:
        allb = [torch.zeros_like(busy) for _ in range(world)]
        dist.all_gather(allb, busy)
        busy_ms = [float(b.item()) for b in allb]
    else:
        busy_ms = [float(busy.item())]
    audio = sum(lengths_all) / FRAME_RATE
    cost = [sum(utterance_cost(lengths_all[i]) for i in s_) for s_ in shards]
    out["configs[4]"] = {"workload": "256 mixed-length (2-30 s) utterances, padded + masked micro-batches of <= 32, flow "
                                     f"({a.n_timesteps}-step Euler + CFG) + DAC decode, one waveform gather",
                         "value": audio / (ms / 1000.0), "unit": UNIT, "ms_per_step": ms, "audio_seconds": audio,
                         "scaling": "strong", "n_gpus": world, "utterances_per_rank": [len(s_) for s_ in shards],
                         "rank_busy_ms": busy_ms, "imbalance_max_over_mean": max(busy_ms) / (sum(busy_ms) / len(busy_ms)),
                         "cost_model_max_over_mean": max(cost) / (sum(cost) / len(cost)),
                         "gather_bytes_to_rank0": int(sum(n for p_ in plan for n in p_[0]) * 4) if world > 1 else 0}
    del batches, local
    # ---- batch-1 latency (configs[0]'s shape on the GPU): eager launches vs one CUDA-graph replay
    if rank == 0:
        one = [t.to(dev) for t in synth.batch_inputs([int(round(a.seconds * FRAME_RATE))], first_index=7)]
        lat = {}
        for name, fn in (("eager_launches", lambda: syn(*one, n_timesteps=a.n_timesteps)),
                         ("cuda_graph", lambda: syn.graphed(*one, n_timesteps=a.n_timesteps))):
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
            ts = []
            for _ in range(10):
                t0 = time.perf_counter()
                fn()
                torch.cuda.synchronize()
                ts.append((time.perf_counter() - t0) * 1000.0)
            lat[name + "_ms"] = statistics.median(ts)
        g = next(iter(syn._graphs.values()))
        lat.update({"workload": f"one {a.seconds:g} s utterance, {a.n_timesteps}-step Euler + CFG + DAC decode (configs[0]'s shape), "
                                "host wall clock per call incl. synchronise, median of 10", "kernels_per_call": g.kernels,
                    "audio_s_per_s_graph": a.seconds / (lat["cuda_graph_ms"] / 1000.0)})
        out["latency_b1"] = lat
    # ---- the headline workload with fp16 operands (same kernels, 3 more mantissa bits: DESIGN section 2) -- speed and the
    # distance of the two operand types' waveforms from each other
    if rank == 0 and esd is not None:
        from minimax_speech_b200.flow import CausalConditionalCFM, CausalConditionalDecoder
        est16 = CausalConditionalDecoder(precision="fp16")
        est16.load_state_dict(esd)
        cfm16 = CausalConditionalCFM(240, dict(t_scheduler="cosine", inference_cfg_rate=0.7), 1, 80, est16)
        T = int(round(a.seconds * FRAME_RATE))
        inp = [t.to(dev) for t in synth.batch_inputs([T] * a.batch, first_index=0)]
        f16 = lambda: cfm16(mu=inp[0], mask=inp[1], n_timesteps=a.n_timesteps, spks=inp[2], cond=inp[3])[0]
        b16 = lambda: cfm(mu=inp[0], mask=inp[1], n_timesteps=a.n_timesteps, spks=inp[2], cond=inp[3])[0]
        y16, yb = f16().clone(), b16().clone()
        torch.cuda.synchronize()
        ms16, msb = [], []
        for _ in range(3):
            e0.record(); f16(); e1.record(); torch.cuda.synchronize(); ms16.append(e0.elapsed_time(e1))
            e0.record(); b16(); e1.record(); torch.cuda.synchronize(); msb.append(e0.elapsed_time(e1))
        out["fp16_operands"] = {"workload": f"flow solve only, {a.batch} x {a.seconds:g} s, {a.n_timesteps} steps, same weights, interleaved",
                                "solve_ms_fp16": statistics.median(ms16), "solve_ms_bf16": statistics.median(msb),
                                "max_abs_diff_mel_fp16_vs_bf16": float((y16 - yb).abs().max()),
                                "note": "parity of each against the fp32 oracle: tests/test_parity_gpu.py (bf16 <= 1e-2, fp16 ~1.5e-3)"}
        del est16, cfm16, inp
    if world > 1:
        dist.barrier()
    return out

# ------------------------------------------------------------------------------------------ B200 arm
def run_b200(a):
    import torch.distributed as dist
    import minimax_speech_b200.native as native
    import minimax_speech_b200.synth as synth
    from minimax_speech_b200.dac import DACVAEDecoder
    from minimax_speech_b200.flow import CausalConditionalCFM, CausalConditionalDecoder
    from minimax_speech_b200.pipeline import PlannedGather, Synthesizer, gather_plan

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device: the hot path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    assert world == a.gpus or world == 1, f"--gpus {a.gpus} but WORLD_SIZE={world}"
    gatherer = None

    esd = synth.estimator_state_dict(1986, "reference")
    dsd = synth.dac_decoder_state_dict(0, "reference")
    est = CausalConditionalDecoder()
    est.load_state_dict(esd)
    cfm = CausalConditionalCFM(240, dict(t_scheduler="cosine", inference_cfg_rate=0.7), 1, 80, est)
    dac = DACVAEDecoder()
    dac.load_state_dict(dsd)
    syn = Synthesizer(cfm, dac)

    T = int(round(a.seconds * FRAME_RATE))
    B = a.batch
    lengths = [T] * B
    ids = list(range(rank * B, rank * B + B))
    mu_h, mask_h, spks_h, cond_h = [t.pin_memory() for t in synth.batch_inputs(lengths, first_index=rank * B)]
    mu, mask, spks, cond = [t.to(dev) for t in (mu_h, mask_h, spks_h, cond_h)]
    n_samples = [T * dac.hop_length] * B
    # the shard assignment is host knowledge on every rank (rank r holds utterances [r*B, (r+1)*B)): no metadata exchange
    plan = gather_plan([list(range(r * B, r * B + B)) for r in range(world)], [T * dac.hop_length] * (world * B))
    if world > 1:
        gatherer = PlannedGather(plan, dev, dst=0)
    scratch = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def step():
        scratch.zero_()  # L2 flush
        wav = syn(mu, mask, spks, cond, n_timesteps=a.n_timesteps)
        if world > 1:
            return gatherer(wav)
        return wav

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # warm-up: at least W (>= 3) steps AND at least ~4 s of work -- on a box that has just been handed out the first
    # seconds run below the sustained rate (measured: 96 vs 80 ms per step with 3 warm-up steps only, and still 84.9 ms
    # after 1.5 s of warm-up when the same step measured 79.6-80.6 ms later in the same process)
    n_warm, t_warm = 0, time.perf_counter()
    for _ in range(max(a.warmup, 3)):
        step()
        n_warm += 1
    torch.cuda.synchronize()
    t_one = time.perf_counter()
    step()  # one more, timed on its own: the first steps carry one-time costs (workspaces, tensor maps)
    n_warm += 1
    torch.cuda.synchronize()
    now = time.perf_counter()
    spent, one = now - t_warm, max(now - t_one, 1e-3)
    extra = int(min(128 - n_warm, (4.0 - spent) / one + 1)) if spent < 4.0 else 0
    if world > 1:  # every rank must run the same number of steps: step() ends in a collective
        ex = torch.tensor([extra], device=dev)
        dist.all_reduce(ex, op=dist.ReduceOp.MAX)
        extra = int(ex.item())
    for _ in range(max(extra, 0)):
        step()
        n_warm += 1
    sync_all()
    clocks = ClockSampler(local) if rank == 0 else None
    l0 = native.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ncu_range = os.environ.get("LS_NCU_RANGE") == "1"  # ncu --profile-from-start off: capture the timed region only
    if ncu_range:
        torch.cuda.cudart().cudaProfilerStart()
    e0.record()
    for _ in range(a.steps):
        out = step()
    e1.record()
    sync_all()
    if ncu_range:
        torch.cuda.cudart().cudaProfilerStop()
    launches = native.launch_count() - l0
    if a.dump_outputs and rank == 0:  # before any later call can reuse the output buffers
        wav = out if world == 1 else torch.stack([out[uid] for uid in sorted(out)]).unsqueeze(1)
        dump_outputs(a.dump_outputs, {"wav": wav})
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item())
    audio_per_step = world * B * a.seconds
    value = audio_per_step * a.steps / (ms / 1000.0)

    # ---- end to end through the host-buffer C-ABI call (H2D of inputs + D2H of the waveform inside) ----
    wav_h = torch.empty(B, 1, T * dac.hop_length, dtype=torch.float32).pin_memory()
    for _ in range(2):
        syn.synthesize_host(mu_h, mask_h, spks_h, cond_h, a.n_timesteps, wav_out=wav_h, device=dev)
    sync_all()
    t0 = time.perf_counter()
    e0.record()
    for _ in range(a.steps):
        scratch.zero_()
        syn.synthesize_host(mu_h, mask_h, spks_h, cond_h, a.n_timesteps, wav_out=wav_h, device=dev)
    e1.record()
    sync_all()
    wall_ms = (time.perf_counter() - t0) * 1000.0
    ems = torch.tensor([max(e0.elapsed_time(e1), 0.0)], device=dev)
    if world > 1:
        dist.all_reduce(ems, op=dist.ReduceOp.MAX)
    ems = float(ems.item())
    clock_rec = clocks.stop() if clocks else None
    h2d = sum(t.numel() * 4 for t in (mu_h, mask_h, spks_h, cond_h))
    d2h = wav_h.numel() * 4
    e2e = {"value": audio_per_step * a.steps / (ems / 1000.0), "unit": UNIT, "h2d_bytes_per_step": h2d,
           "d2h_bytes_per_step": d2h, "ms_per_step": ems / a.steps, "wall_ms_per_step_rank0": wall_ms / a.steps,
           "api": "Synthesizer.synthesize_host -> ls_synthesize_host (pinned host buffers)"}

    # ---- per-kernel device time (CUDA events around every launch, separate pass) -> roofline ----
    roofline, kernels = None, None
    if rank == 0 and not a.no_profile:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except (OSError, ValueError):
            pass
        peak_tf = peaks.get("bf16_tflops_sustained")
        peak_src = "measured (MEASURED_PEAKS.json bf16_tflops_sustained: kernel timed inside a long step)"
        if not peak_tf:
            peak_tf, peak_src = 1400.0, "fallback (B200_PROFILING.md sustained figure)"
        peak_bw = peaks.get("hbm_gbs") or 6650.0
        native.profile_begin()
        for _ in range(a.steps):
            syn(mu, mask, spks, cond, n_timesteps=a.n_timesteps)
        prof = native.profile_end()
        tot = sum(v["ms"] for v in prof.values()) or 1.0
        kernels = {}
        for k, v in prof.items():
            if not v["launches"]:
                continue
            sec = v["ms"] / 1000.0
            kernels[k] = {"launches_per_step": v["launches"] / a.steps, "ms_per_step": v["ms"] / a.steps,
                          "share_of_kernel_time": v["ms"] / tot,
                          "tflops": v["flops"] / sec / 1e12 if sec else None,
                          "gbs": v["bytes"] / sec / 1e9 if sec else None}
        dom = max(("conv_gemm_estimator", "attention", "conv_gemm_dac", "tblock_estimator"), key=lambda k: prof[k]["ms"])
        ach = prof[dom]["flops"] / (prof[dom]["ms"] / 1000.0) / 1e12
        traffic = None
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(dom)
        except (OSError, ValueError):
            pass
        roofline = {"kernel": dom, "bound": "tensor", "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s",
                    "frac": ach / peak_tf, "traffic": traffic, "peak_source": peak_src,
                    "flops_per_launch": prof[dom]["flops"] / prof[dom]["launches"],
                    "avg_launch_us": 1000.0 * prof[dom]["ms"] / prof[dom]["launches"],
                    "hbm_peak_gbs": peak_bw}

    # north_star: ">= 60 % of HBM peak on the fused elementwise kernels": the stand-alone bandwidth kernels of the step
    # (layout packing, CFG combine + Euler update, time embedding) against the measured copy bandwidth; every other
    # row-local op is fused into a GEMM epilogue and has no pass of its own.  Algorithmic bytes / event time per launch.
    hbm = None
    if kernels and "bandwidth" in kernels:
        k = kernels["bandwidth"]
        hbm = {"kernel_kind": "bandwidth (pack / unpack / cfg_euler / time embedding)", "achieved_gbs": k["gbs"], "peak_gbs": peak_bw,
               "frac": (k["gbs"] or 0.0) / peak_bw, "launches_per_step": k["launches_per_step"], "ms_per_step": k["ms_per_step"],
               "note": "launch-latency sized at this workload (a few MB per launch): see configs[3] for the larger shape"}
        dk = kernels.get("conv_gemm_dac")
        if dk:
            hbm["dac_decode_gbs"] = dk["gbs"]
            hbm["dac_decode_frac"] = (dk["gbs"] or 0.0) / peak_bw

    # ---- the same step started from FSQ tokens (SURVEY section 8 f-1): token -> mu front half (tensor-core path) in front ----
    from_tokens = None
    if rank == 0 and world == 1 and int(round(a.seconds * 25)) * 2 == T:
        from minimax_speech_b200.front import TokenToMu
        front = TokenToMu()
        toks, embs = zip(*[synth.token_inputs(b, T // 2) for b in range(B)])
        tok, emb = torch.cat(toks, 0).to(dev), torch.cat(embs, 0).to(dev)

        def step_tokens():
            scratch.zero_()
            mu_t, spks_t = front(tok, emb)
            return syn(mu_t, mask, spks_t, cond, n_timesteps=a.n_timesteps)

        for _ in range(3):
            step_tokens()
        torch.cuda.synchronize()
        e0.record()
        for _ in range(a.steps):
            step_tokens()
        e1.record()
        torch.cuda.synchronize()
        tms = e0.elapsed_time(e1) / a.steps
        e0.record()
        for _ in range(a.steps):
            front(tok, emb)
        e1.record()
        torch.cuda.synchronize()
        from_tokens = {"value": B * a.seconds / (tms / 1000.0), "unit": UNIT, "ms_per_step": tms,
                       "front_ms_per_step": e0.elapsed_time(e1) / a.steps,
                       "workload": f"{B} x {T // 2} FSQ tokens (25 Hz) -> UpsampleConformerEncoder -> mu, then the step above"}

    configs = None
    if not a.no_extra:
        configs = extra_legs(a, syn, cfm, dac, dev, world, rank, sync_all, esd)

    cb, eager = None, None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        eager = gpu_eager_baseline(a, esd, dsd, dev)
        cb = cpu_baseline(a, esd, dsd)
        # north_star's ">= 20x the reference's GPU-eager PyTorch throughput": kept inside cpu_baseline so that the driver's
        # record carries it (literal = one utterance at a time like the reference's solve_euler; batched = fairness figure)
        cb["gpu_eager"] = dict(eager, speedup_vs_fp32_literal=value / eager["fp32"],
                               speedup_vs_best_batched=value / max(eager["batched_fp32"], eager["batched_bf16_autocast"]))

    if rank == 0:
        rec = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps,
               "warmup": n_warm, "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak",
               "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": config_of(a),
               "e2e": e2e, "gpu_launches": int(launches), "clocks": clock_rec, "roofline": roofline,
               "kernels": kernels, "from_tokens": from_tokens, "cpu_baseline": cb, "gpu_eager_baseline": eager,
               "configs": configs, "hbm": hbm, "audio_seconds_per_step": audio_per_step,
               "weights": "synthetic numpy draws with the reference initialisers' distributions and the reference state_dict "
                          "schema (synth.py), loaded into both arms (strict load into the reference's own modules when they are "
                          "timed), not the reference constructors' own random tensors"}
        emit(rec)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    args = parse()
    claim_stdout()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)
