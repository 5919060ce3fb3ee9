"""Flow -> DAC-VAE glue (the reference never wires the two together: SURVEY.md section 0) and the
utterance sharding used at N > 1 GPUs (one utterance group per rank, one gather of waveforms at the end,
mirroring dac-vae/extract_dac_latents.py:146-150's contiguous per-rank slices)."""
import numpy as np
import torch

from . import native


class Synthesizer:
    """latents = cfm(mu, mask, n_timesteps, spks=, cond=)[0];  wav = dac.decode(latents)."""

    def __init__(self, cfm, dac):
        self.cfm, self.dac = cfm, dac
        self._graphs = {}

    @torch.inference_mode()
    def __call__(self, mu, mask, spks, cond, n_timesteps=10, temperature=1.0, streaming=False):
        return self.run(mu, mask, spks, cond, n_timesteps, temperature, streaming)

    def run(self, mu, mask, spks, cond, n_timesteps=10, temperature=1.0, streaming=False):
        """``__call__`` without the inference_mode decorator: three ``torch.ops.ls_b200`` calls and nothing else on the
        device (the form ``torch.compile(fullgraph=True)`` traces)."""
        lat, _ = self.cfm.run(mu, mask, n_timesteps, temperature, spks, cond, streaming)
        lengths = torch.ops.ls_b200.mask_to_lengths(mask.to(dtype=torch.float32).contiguous())
        return self.dac.run(lat, lengths)

    @torch.inference_mode()
    def synthesize_host(self, mu, mask, spks, cond, n_timesteps=10, temperature=1.0, wav_out=None, device=None):
        """Host tensors in, host waveform out; host<->device copies happen inside the C call."""
        device = torch.device(device or "cuda:%d" % torch.cuda.current_device())
        B, _, T = mu.shape
        if wav_out is None:
            wav_out = torch.empty(B, 1, T * self.dac.hop_length, dtype=torch.float32).pin_memory()
        flow_h = self.cfm.estimator.handle(device)
        dac_h = self.dac.handle(device)
        return native.synthesize_host(flow_h, dac_h, mu, mask, spks, cond, self.cfm._noise_on(device)[0],
                                      self.cfm._t_span(n_timesteps).numpy(), temperature,
                                      self.cfm.inference_cfg_rate, wav_out)

    @torch.inference_mode()
    def graphed(self, mu, mask, spks, cond, n_timesteps=10, temperature=1.0, streaming=False):
        """The same result as ``__call__`` through a CUDA graph captured once per (B, T, n_timesteps, temperature,
        streaming): ~1800 kernel launches become one cudaGraphLaunch (the form for launch-bound small batches, e.g.
        one 10 s utterance).  Inputs are copied into the graph's static buffers; the returned waveform is a view of
        its static output buffer, overwritten by the next call with the same shape."""
        dev = mu.device
        B, _, T = mu.shape
        key = (str(dev), B, T, int(n_timesteps), float(temperature), bool(streaming))
        g = self._graphs.get(key)
        if g is None:
            if self.cfm.estimator.precision == "fp32" or self.dac.precision == "fp32":
                raise NotImplementedError("CUDA-graph replay covers the tensor-core path (precision 'bf16' / 'fp16')")
            g = native.GraphHandle(self.cfm.estimator.handle(dev), self.dac.handle(dev), self.cfm._noise_on(dev)[0],
                                   self.cfm._t_span(n_timesteps).numpy(), temperature, self.cfm.inference_cfg_rate,
                                   streaming, B, T)
            self._graphs[key] = g
        g_mu, g_mask, g_spks, g_cond, _, g_wav = g.buffers
        g_mu.copy_(mu), g_mask.copy_(mask), g_spks.copy_(spks), g_cond.copy_(cond)
        g.launch()
        return g_wav


def utterance_cost(frames):
    """Relative cost model of one utterance (SURVEY.md section 8e): linear + attention FLOPs per step."""
    return frames * (132.2e6 + 114688.0 * frames)


def shard_utterances(lengths, world_size):
    """Length-balanced assignment (greedy longest-first); returns per-rank lists of utterance indices."""
    order = sorted(range(len(lengths)), key=lambda i: -lengths[i])
    loads = [0.0] * world_size
    shards = [[] for _ in range(world_size)]
    for i in order:
        r = min(range(world_size), key=lambda k: loads[k])
        shards[r].append(i)
        loads[r] += utterance_cost(lengths[i])
    return [sorted(s) for s in shards]


def gather_plan(shards, n_samples_all):
    """Host-side description of a gather, known on every rank before the step (the shard assignment is computed from the
    utterance lengths, so every rank knows what every other rank will contribute): per rank (sample counts, utterance ids).
    ``shards``: per-rank lists of utterance ids (``shard_utterances``); ``n_samples_all[i]``: valid samples of utterance i."""
    return [([int(n_samples_all[i]) for i in s], [int(i) for i in s]) for s in shards]


class PlannedGather:
    """``gather_waveforms`` with a plan and persistent staging buffers: nothing is allocated, exchanged as metadata or read back
    per call, so the host thread keeps launching the next step (allocating the padded buffers per step makes the caching
    allocator wait on the communication stream's use of the previous ones).  The returned views alias the receive buffer and
    are overwritten by the next call."""

    def __init__(self, plan, device, dst=0, group=None):
        import torch.distributed as dist
        self.plan, self.dst, self.group = plan, dst, group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        if len(plan) != self.world:
            raise ValueError("gather plan must have one entry per rank")
        self.bmax = max(len(p[0]) for p in plan)
        self.smax = max([n for p in plan for n in p[0]] + [1])
        self.pad = torch.zeros(self.bmax, self.smax, device=device, dtype=torch.float32)
        self.out = torch.empty(self.world, self.bmax, self.smax, device=device, dtype=torch.float32) if self.rank == dst else None
        self.nccl = dist.get_backend(group) == "nccl"

    def __call__(self, wav):
        import torch.distributed as dist
        b, S = wav.shape[0], min(wav.shape[-1], self.smax)
        if b != len(self.plan[self.rank][0]):
            raise ValueError("gather plan does not describe this rank's contribution")
        self.pad[:b, :S].copy_(wav[:, 0, :S])
        if self.nccl:
            dist.gather(self.pad, list(self.out.unbind(0)) if self.rank == self.dst else None, dst=self.dst, group=self.group)
        else:
            bufs = [torch.zeros_like(self.pad) for _ in range(self.world)] if self.rank == self.dst else None
            dist.gather(self.pad, bufs, dst=self.dst, group=self.group)
            if self.rank == self.dst:
                self.out.copy_(torch.stack(bufs))
        if self.rank != self.dst:
            return None
        return {uid: self.out[r, i, :n] for r, (counts, ids) in enumerate(self.plan) for i, (n, uid) in enumerate(zip(counts, ids))}


def gather_waveforms(wav, n_samples, index, dst=0, group=None, plan=None):
    """Variable-length gather to ``dst``: every rank contributes ``wav [b,1,S_r]`` with per-item valid sample
    counts ``n_samples`` and global utterance ids ``index``.  Returns {utterance id: 1-D tensor} on ``dst``.
    One collective for the payload (padded gather over NCCL/NVLink, or gloo on CPU).  With ``plan`` (``gather_plan``) the
    sizes are host knowledge and the call neither exchanges metadata nor reads anything back from the device, so the host
    keeps launching the next step; without it a tiny metadata all_gather and a read-back of the counts come first."""
    import torch.distributed as dist
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    dev = wav.device
    b = wav.shape[0]

    def exchange(pad, bmax, width):
        out = torch.empty(world, bmax, width, device=dev, dtype=torch.float32) if rank == dst else None
        if dist.get_backend(group) == "nccl":
            dist.gather(pad, list(out.unbind(0)) if rank == dst else None, dst=dst, group=group)
        else:
            bufs = [torch.zeros_like(pad) for _ in range(world)] if rank == dst else None
            dist.gather(pad, bufs, dst=dst, group=group)
            if rank == dst:
                out = torch.stack(bufs)
        return out

    if plan is not None:
        if len(plan) != world or list(plan[rank][1]) != [int(i) for i in index] or len(plan[rank][0]) != b:
            raise ValueError("gather plan does not describe this rank's contribution")
        bmax = max(len(p[0]) for p in plan)
        smax = max([n for p in plan for n in p[0]] + [1])
        if wav.shape[-1] > smax:
            wav = wav[..., :smax]
        pad = torch.zeros(bmax, smax, device=dev, dtype=torch.float32)
        pad[:b, :wav.shape[-1]] = wav[:, 0, :]
        out = exchange(pad, bmax, smax)
        if rank != dst:
            return None
        return {uid: out[r, i, :n] for r, (counts, ids) in enumerate(plan) for i, (n, uid) in enumerate(zip(counts, ids))}

    meta = torch.tensor([wav.shape[0], wav.shape[-1]], device=dev, dtype=torch.int64)
    metas = [torch.zeros_like(meta) for _ in range(world)]
    dist.all_gather(metas, meta, group=group)
    bmax = int(max(m[0] for m in metas))
    smax = int(max(m[1] for m in metas))
    pad = torch.zeros(bmax, smax + 2, device=dev, dtype=torch.float32)
    pad[:b, :wav.shape[-1]] = wav[:, 0, :]
    # counts and ids travel bit-cast as int32 inside the float payload (a float32 VALUE would round above 2^24)
    pad_i = pad.view(torch.int32)
    pad_i[:b, smax] = torch.as_tensor(n_samples, device=dev, dtype=torch.int32)
    pad_i[:b, smax + 1] = torch.as_tensor(index, device=dev, dtype=torch.int32)
    out = exchange(pad, bmax, smax + 2)
    if rank != dst:
        return None
    res = {}
    out_i = out.view(torch.int32)
    for r in range(world):
        for i in range(int(metas[r][0])):
            n = int(out_i[r, i, smax])
            res[int(out_i[r, i, smax + 1])] = out[r, i, :n]
    return res


# ---------------------------------------------------------------------------------------------------------------------
# Bulk latent extraction: the reference's multi-GPU tool around DACVAE.encode (dac-vae/extract_dac_latents.py)
# ---------------------------------------------------------------------------------------------------------------------
def shard_files(n_files, rank, world_size):
    """Contiguous per-rank slice, the last rank taking the remainder (extract_dac_latents.py:146-150)."""
    per = n_files // world_size
    start = rank * per
    end = start + per if rank < world_size - 1 else n_files
    return start, end


def latent_record(z, mu, logs, sample_rate, n_samples, n_padded, path):
    """The ``*_latent2x.pt`` dict of extract_dac_latents.py:184-196 (batch dim removed, CPU tensors)."""
    z, mu, logs = z.squeeze(0).cpu(), mu.squeeze(0).cpu(), logs.squeeze(0).cpu()
    return {"z": z, "mu": mu, "logs": logs, "sample_rate": sample_rate, "compression_ratio": n_padded // z.shape[-1],
            "original_duration": n_samples / sample_rate, "original_samples": n_samples, "latent_shape": list(z.shape),
            "original_path": path}


def plan_micro_batches(n_samples, max_batch_samples=None):
    """Group items of ``n_samples`` (padded sample counts) into micro-batches of at most ``max_batch_samples`` padded
    samples (batch size x longest item): items sorted by length (stable), filled greedily; an item longer than the
    budget gets a batch of its own.  ``None``: one item per batch, in order.  Returns lists of item indices."""
    if max_batch_samples is None:
        return [[i] for i in range(len(n_samples))]
    batches, cur = [], []
    for i in sorted(range(len(n_samples)), key=lambda i: n_samples[i]):
        if cur and (len(cur) + 1) * n_samples[i] > max_batch_samples:  # sorted: item i is the longest so far
            batches.append(cur)
            cur = []
        cur.append(i)
    if cur:
        batches.append(cur)
    return batches


def _load_at(load_audio, path, sample_rate, rate, device):
    """load_audio(path) as a 1-D float32 tensor at ``rate``: converted on the GPU (``audio.resample``) when ``sample_rate``
    names another rate, returned on the host either way."""
    a = torch.as_tensor(load_audio(path), dtype=torch.float32).reshape(-1)
    if sample_rate is None or int(sample_rate) == rate:
        return a
    from . import audio as _audio
    return _audio.resample(a.to(device), sample_rate, rate).cpu()


def extract_latents(paths, load_audio, encoder, device, rank=0, world_size=1, save=True, generator=None,
                    max_batch_samples=None, sample_rate=None):
    """Encode this rank's share of ``paths`` and write ``<stem>_latent2x.pt`` next to each input.
    ``load_audio(path) -> 1-D float tensor`` at ``encoder.sample_rate`` (the reference uses librosa, which is not a
    dependency here), or at ``sample_rate`` when given: the audio is then converted to ``encoder.sample_rate`` on the GPU
    (``audio.resample``, torchaudio's resampler; the reference tool resamples with librosa, whose result this does not
    reproduce) and the records describe the converted signal.  Audio is clamped to [-1, 1] (:31) and right-padded to a
    multiple of the hop (DACVAE.preprocess, model.py:455-462; the reference tool feeds the unpadded signal, so its last
    latent frame can differ).

    By default each file is encoded on its own (like the reference).  ``max_batch_samples`` encodes length-sorted
    micro-batches of at most that many padded samples (batch size x longest file, see ``plan_micro_batches``) with
    per-file ``lengths``, which gives every file the latents it gets alone; the share is loaded into host memory first.
    Noise is drawn from ``generator`` in file order either way.  Returns the list of records (and output paths when
    saved) in file order."""
    import os
    start, end = shard_files(len(paths), rank, world_size)
    mine = paths[start:end]
    padded, n_orig, noise = [], [], []
    for path in mine:
        audio = torch.clamp(_load_at(load_audio, path, sample_rate, encoder.sample_rate, device).reshape(1, 1, -1), -1.0, 1.0)
        n_orig.append(audio.shape[-1])
        padded.append(encoder.preprocess(audio))
        L = padded[-1].shape[-1] // encoder.hop_length
        noise.append(torch.randn(1, encoder.latent_dim, L, generator=generator))
    recs = [None] * len(mine)
    for batch in plan_micro_batches([a.shape[-1] for a in padded], max_batch_samples):
        if len(batch) == 1:
            i = batch[0]
            z, mu, logs = encoder.encode(padded[i].to(device), noise[i].to(device))
            recs[i] = latent_record(z, mu, logs, encoder.sample_rate, n_orig[i], padded[i].shape[-1], mine[i])
            continue
        s_max = max(padded[i].shape[-1] for i in batch)
        audio = torch.zeros(len(batch), 1, s_max)
        nz = torch.zeros(len(batch), encoder.latent_dim, s_max // encoder.hop_length)
        lengths = []
        for b, i in enumerate(batch):
            audio[b, :, :padded[i].shape[-1]] = padded[i][0]
            nz[b, :, :noise[i].shape[-1]] = noise[i][0]
            lengths.append(noise[i].shape[-1])
        z, mu, logs = (t.cpu() for t in encoder.encode(audio.to(device), nz.to(device), lengths=lengths))
        for b, i in enumerate(batch):  # (copies: a saved view would carry the whole batch's storage)
            n = lengths[b]
            recs[i] = latent_record(z[b:b + 1, :, :n].clone(), mu[b:b + 1, :, :n].clone(), logs[b:b + 1, :, :n].clone(),
                                    encoder.sample_rate, n_orig[i], padded[i].shape[-1], mine[i])
    out = []
    for path, rec in zip(mine, recs):
        if save:
            rec_path = os.path.splitext(path)[0] + "_latent2x.pt"
            torch.save(rec, rec_path)
            out.append((rec_path, rec))
        else:
            out.append((None, rec))
    return out


# ---------------------------------------------------------------------------------------------------------------------
# Bulk token extraction: 16 kHz audio -> S3 tokenizer ids (the tokens the flow's input_embedding consumes)
# ---------------------------------------------------------------------------------------------------------------------
def token_record(tokens, n_samples, path, sample_rate=16000):
    """The ``*_fsq.pt`` dict written by ``extract_tokens`` (CPU tensors).  This layout is this project's choice, modelled
    on ``latent_record``; it has not been checked against what the reference's data loader reads."""
    tokens = tokens.to(torch.int64).cpu()
    return {"tokens": tokens, "token_len": int(tokens.shape[0]), "sample_rate": sample_rate,
            "original_samples": n_samples, "original_path": path}


def extract_tokens(paths, load_audio, tokenizer, device, rank=0, world_size=1, save=True, max_batch_samples=None,
                   sample_rate=None):
    """Tokenize this rank's share of ``paths`` (``shard_files``) with an ``S3TokenizerV2`` and write
    ``<stem>_fsq.pt`` (``token_record``) next to each input.  ``load_audio(path) -> 1-D float tensor`` of 16 kHz mono
    audio, or of audio at ``sample_rate`` when given: it is then converted to 16 kHz on the GPU (``audio.resample``) and
    the records describe the converted signal.  Decoding stays with the caller.

    By default each file is one ``quantize_audio`` call.  ``max_batch_samples`` tokenizes length-sorted micro-batches of
    at most that many padded samples (batch size x longest file, see ``plan_micro_batches``) in one call each, with
    per-file lengths, so every file's mel is the one it gets alone; the share is loaded into host memory first.  Returns
    the list of (output path or None, record) in file order."""
    import os
    start, end = shard_files(len(paths), rank, world_size)
    mine = paths[start:end]
    from .tokenizer import SAMPLE_RATE
    audio = [_load_at(load_audio, path, sample_rate, SAMPLE_RATE, device) for path in mine]
    recs = [None] * len(mine)
    for batch in plan_micro_batches([a.shape[0] for a in audio], max_batch_samples):
        lens = [audio[i].shape[0] for i in batch]
        buf = torch.zeros(len(batch), max(lens))
        for b, i in enumerate(batch):
            buf[b, :lens[b]] = audio[i]
        codes, code_len = tokenizer.quantize_audio(buf.to(device), lens)
        codes, code_len = codes.cpu(), code_len.tolist()
        for b, i in enumerate(batch):  # (copies: a saved view would carry the whole batch's storage)
            recs[i] = token_record(codes[b, :code_len[b]].clone(), lens[b], mine[i])
    out = []
    for path, rec in zip(mine, recs):
        if save:
            rec_path = os.path.splitext(path)[0] + "_fsq.pt"
            torch.save(rec, rec_path)
            out.append((rec_path, rec))
        else:
            out.append((None, rec))
    return out
