"""pipeline.extract_latents with length-sorted micro-batches (``max_batch_samples``): the planner and the bookkeeping
around it, with a stand-in encoder that takes ``lengths`` (the real one needs a GPU)."""
import os

import torch

from minimax_speech_b200 import pipeline

HOP, LATENT = 480, 4


class LengthsEncoder:
    """Frame means of the audio as m, z = m + noise; zero past each clip's length.  Records every call."""
    hop_length, latent_dim, sample_rate = HOP, LATENT, 24000

    def __init__(self):
        self.calls = []

    def preprocess(self, a):
        return torch.nn.functional.pad(a, (0, (-a.shape[-1]) % self.hop_length))

    def encode(self, audio, noise, **kw):
        B, _, S = audio.shape
        L = S // self.hop_length
        lengths = kw.get("lengths")
        self.calls.append((B, S, None if lengths is None else list(lengths), "lengths" in kw))
        m = audio.reshape(B, 1, L, self.hop_length).mean(-1).expand(B, self.latent_dim, L).clone()
        if lengths is not None:
            for b, n in enumerate(lengths):
                m[b, :, n:] = 0.0
                noise[b, :, n:] = 0.0
        return m + noise, m, torch.zeros_like(m)


def _clips(tmp_path, sizes):
    paths = []
    for i, n in enumerate(sizes):
        p = tmp_path / f"clip{i}.pt"
        torch.save(torch.sin(torch.arange(n, dtype=torch.float32) * (0.001 * (i + 1))), p)
        paths.append(str(p))
    return paths


SIZES = [3000, 1000, 7000, 480, 2500, 9600, 1200, 4000]  # samples; padded to 3360, 1440, 7200, 480, 2880, 9600, 1440, 4320


def test_planner_budget_and_coverage():
    n = [((s + HOP - 1) // HOP) * HOP for s in SIZES]
    for budget in [480, 2000, 5000, 10000, 40000, 10 ** 9]:
        batches = pipeline.plan_micro_batches(n, budget)
        assert sorted(i for b in batches for i in b) == list(range(len(n)))  # every item exactly once
        for b in batches:
            assert len(b) == 1 or len(b) * max(n[i] for i in b) <= budget
        for i in range(len(n)):
            if n[i] > budget:
                assert [i] in batches  # an oversized item gets a batch of its own
    assert pipeline.plan_micro_batches(n, 10 ** 9) == [sorted(range(len(n)), key=lambda i: n[i])]
    assert pipeline.plan_micro_batches(n, None) == [[i] for i in range(len(n))]


def test_batched_records_match_per_file(tmp_path):
    paths = _clips(tmp_path, SIZES)
    ref_enc = LengthsEncoder()
    ref = pipeline.extract_latents(paths, torch.load, ref_enc, "cpu", save=False, generator=torch.Generator().manual_seed(3))
    assert all(not has for *_, has in ref_enc.calls)  # budget None never passes lengths
    assert [c[0] for c in ref_enc.calls] == [1] * len(paths)
    for budget in [5000, 20000, 10 ** 9]:
        enc = LengthsEncoder()
        out = pipeline.extract_latents(paths, torch.load, enc, "cpu", save=False,
                                       generator=torch.Generator().manual_seed(3), max_batch_samples=budget)
        assert len(out) == len(paths)
        for (_, r), (_, q) in zip(out, ref):
            assert r["original_path"] == q["original_path"]  # file order
            assert r["latent_shape"] == q["latent_shape"] and r["compression_ratio"] == HOP
            for k in ("z", "mu", "logs"):
                assert torch.equal(r[k], q[k]), (budget, r["original_path"], k)  # same noise as the per-file path
        assert sum(c[0] for c in enc.calls) == len(paths)
        for B, S, lengths, has in enc.calls:
            assert B == 1 or B * S <= budget
            assert (lengths is not None) == (B > 1) and has == (B > 1)
        assert any(c[0] > 1 for c in enc.calls)


def test_batched_save_and_sharding(tmp_path):
    paths = _clips(tmp_path, SIZES[:6])
    out = pipeline.extract_latents(paths, torch.load, LengthsEncoder(), "cpu", rank=1, world_size=2,
                                   generator=torch.Generator().manual_seed(0), max_batch_samples=30000)
    assert [os.path.basename(p) for p, _ in out] == ["clip3_latent2x.pt", "clip4_latent2x.pt", "clip5_latent2x.pt"]
    for p, rec in out:
        saved = torch.load(p)
        assert torch.equal(saved["z"], rec["z"]) and saved["z"].shape == (LATENT, rec["latent_shape"][1])
        assert saved["z"].untyped_storage().nbytes() == saved["z"].numel() * 4  # not a view of the whole batch
