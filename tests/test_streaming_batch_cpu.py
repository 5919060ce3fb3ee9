"""Host logic of the batched streaming scheduler (``StreamingBatch``) with stand-in flow / decoder objects on CPU: every
session's chunks must equal, chunk by chunk, those of a lone ``StreamingSession`` fed the same pushes.  The stand-ins
depend on the prompt, the speaker embedding, the look-ahead and the decode window the way the real modules do, so a
row mix-up, a wrong prompt cut or a wrong window shows up as a different chunk."""
import pytest
import torch

from minimax_speech_b200.streaming import StreamingBatch, StreamingSession


class FakeFlow:
    pre_lookahead_len, token_latent_ratio, output_size = 3, 2, 4

    def __init__(self):
        self.batch_sizes = []

    def get_speaker_embedding(self, batch, device):
        if batch.get("reference_mels") is not None:
            return batch["reference_mels"].float().mean().reshape(1, 1).repeat(1, 2)
        return batch["embedding"].float() * 0.5  # stands for the normalise

    def _latents(self, tok, n_prompt_feat, emb, finalize):
        t = tok[:tok.numel() - (0 if finalize else self.pre_lookahead_len)].float()
        frames = torch.repeat_interleave(t, 2) + 0.5 * torch.arange(2 * t.numel()).remainder(2) + float(emb[0, 0])
        return frames[n_prompt_feat:].reshape(1, 1, -1).repeat(1, self.output_size, 1)

    def inference(self, token, token_len, prompt_token, prompt_token_len, prompt_feat, prompt_feat_len, embedding=None,
                  reference_mels=None, streaming=False, finalize=False):
        assert streaming and int(token_len[0]) == token.shape[1]
        emb = self.get_speaker_embedding({"embedding": embedding, "reference_mels": reference_mels}, None)
        return self._latents(torch.cat([prompt_token[0], token[0]]), prompt_feat.shape[1], emb, finalize), None

    def inference_batch(self, token, prompt_token, prompt_feat, embedding, finalize, streaming=False):
        assert streaming and embedding.shape[0] == len(token) == len(prompt_token) == len(prompt_feat) == len(finalize)
        self.batch_sizes.append(len(token))
        lats = [self._latents(torch.cat([p.reshape(-1), t.reshape(-1)]), f.shape[1], embedding[b:b + 1], fin)
                for b, (t, p, f, fin) in enumerate(zip(token, prompt_token, prompt_feat, finalize))]
        L = torch.tensor([x.shape[2] for x in lats])
        out = torch.full((len(lats), self.output_size, int(L.max())), float("nan"))  # the real one pads with zeros
        for b, x in enumerate(lats):
            out[b, :, :x.shape[2]] = x[0]
        return out, L


class FakeDac:
    hop_length = 4

    def __init__(self):
        self.batch_sizes = []

    def _one(self, z):
        x = torch.nn.functional.pad(z[:, :1], (3, 3))  # reach of 3 frames either side: not causal
        y = sum(x[:, :, k:k + z.shape[2]] * (k + 1) for k in range(7))
        return torch.repeat_interleave(y, self.hop_length, dim=2) + torch.arange(self.hop_length).repeat(z.shape[2])

    def decode(self, z, lengths=None):
        if lengths is None:
            return self._one(z)
        self.batch_sizes.append(z.shape[0])
        out = torch.zeros(z.shape[0], 1, z.shape[2] * self.hop_length)
        for b, n in enumerate(lengths.tolist()):  # each item alone at its own length, as DACVAEDecoder.decode(z, lengths)
            out[b, :, :n * self.hop_length] = self._one(z[b:b + 1, :, :n])[0]
        return out


def _session_inputs(i, n_prompt, n_feat=None):
    ptok = torch.arange(n_prompt, dtype=torch.int64).reshape(1, -1) * 3 + 7 * i
    pfeat = torch.zeros(1, 2 * n_prompt if n_feat is None else n_feat, 4)
    return ptok, pfeat, torch.tensor([[float(i + 1), 0.0]])


def run_schedule(sessions, n_steps):
    """sessions: dicts with n_prompt, (n_feat), tokens, events {step: ("push", k) | ("finish",) | ("open",)}.  Returns
    per-session chunk lists from the batch and from lone sessions, and the fakes."""
    flow, dac = FakeFlow(), FakeDac()
    batch = StreamingBatch(flow, dac, dac_context=3)
    solo_flow, solo_dac = FakeFlow(), FakeDac()
    ids, solo, pos = {}, {}, {}
    got = {i: [] for i in range(len(sessions))}
    want = {i: [] for i in range(len(sessions))}
    for step in range(n_steps):
        for i, s in enumerate(sessions):
            for ev in s["events"].get(step, []):
                ptok, pfeat, emb = _session_inputs(i, s["n_prompt"], s.get("n_feat"))
                if ev[0] == "open":
                    if s.get("ref"):
                        mels = torch.full((1, 80, 10), float(i + 1))
                        ids[i] = batch.open(ptok, pfeat, reference_mels=mels)
                        solo[i] = StreamingSession(solo_flow, solo_dac, ptok, pfeat, reference_mels=mels, dac_context=3)
                    else:
                        ids[i] = batch.open(ptok, pfeat, embedding=emb)
                        solo[i] = StreamingSession(solo_flow, solo_dac, ptok, pfeat, embedding=emb, dac_context=3)
                    pos[i] = 0
                elif ev[0] == "push":
                    piece = s["tokens"][pos[i]:pos[i] + ev[1]]
                    pos[i] += ev[1]
                    batch.push(ids[i], piece)
                    want[i] += solo[i].push(piece)
                else:
                    batch.finish(ids[i])
                    want[i].append(solo[i].finish())
        for sid, chunks in batch.step().items():
            got[next(i for i, v in ids.items() if v == sid)] += chunks
    return got, want, flow, dac, batch


def _assert_same(got, want):
    for i in want:
        assert len(got[i]) == len(want[i]), f"session {i}: {len(got[i])} chunks, alone {len(want[i])}"
        for a, b in zip(got[i], want[i]):
            assert a.shape == b.shape and torch.equal(a, b)


def test_staggered_sessions_equal_lone_sessions():
    sessions = [
        # several hops ready at once (one big push), then finish in the same step as others' mid-stream hops
        dict(n_prompt=10, tokens=list(range(100, 203)), events={0: [("open",), ("push", 90)], 3: [("push", 13)], 5: [("finish",)]}),
        # opened later, small pieces, odd prompt feature length (the cut is not at a token boundary)
        dict(n_prompt=25, n_feat=49, tokens=list(range(300, 380)),
             events={2: [("open",)], **{3 + k: [("push", 8)] for k in range(10)}, 13: [("finish",)]}),
        # shorter than its first hop: everything goes out in the finishing round
        dict(n_prompt=3, tokens=list(range(500, 509)), events={1: [("open",), ("push", 4)], 4: [("push", 5)], 5: [("finish",)]}),
        # reference mels instead of an x-vector; exact multiple of the hop with no look-ahead left at the end
        dict(n_prompt=25, tokens=list(range(700, 775)), ref=True, events={0: [("open",)], 1: [("push", 75)], 5: [("finish",)]}),
    ]
    got, want, flow, dac, batch = run_schedule(sessions, 16)
    _assert_same(got, want)
    assert len(batch) == 0
    assert max(flow.batch_sizes) >= 3 and max(dac.batch_sizes) >= 3  # the rounds did batch several sessions
    for i, s in enumerate(sessions):  # all audio handed out (where the prompt features cover the prompt tokens exactly)
        if "n_feat" not in s:
            assert sum(c.shape[1] for c in got[i]) == 2 * len(s["tokens"]) * 4


@pytest.mark.parametrize("piece", [1, 7, 25, 28, 200])
def test_piece_sizes(piece):
    toks = list(range(1000, 1137))
    sessions = [dict(n_prompt=n, tokens=toks, events={0: [("open",)], **{1 + k: [("push", piece)] for k in range(-(-137 // piece))},
                                                    1 + -(-137 // piece): [("finish",)]}) for n in (0, 7, 30)]
    got, want, *_ = run_schedule(sessions, 3 + -(-137 // piece))
    _assert_same(got, want)


def test_finish_without_new_tokens_and_errors():
    flow, dac = FakeFlow(), FakeDac()
    batch = StreamingBatch(flow, dac, dac_context=3)
    ptok, pfeat, emb = _session_inputs(0, 25)
    a = batch.open(ptok, pfeat, embedding=emb)
    b = batch.open(ptok, pfeat, embedding=emb)
    batch.push(a, range(28))
    out = batch.step()
    assert list(out) == [a] and sum(c.shape[1] for c in out[a]) == (50 - 3) * 4  # tail of dac_context frames held back
    batch.finish(a)
    with pytest.raises(RuntimeError):
        batch.push(a, [1])  # finishing
    with pytest.raises(RuntimeError):
        batch.finish(a)
    out = batch.step()
    assert [c.shape[1] for c in out[a]] == [(3 + 6) * 4] and b not in out  # the held tail and the finalize call's frames
    with pytest.raises(RuntimeError):
        batch.push(a, [1])  # closed
    with pytest.raises(KeyError):
        batch.push(99, [1])
    with pytest.raises(KeyError):
        batch.finish("x")
    batch.finish(b)
    out = batch.step()
    assert [c.shape for c in out[b]] == [(1, 0)] and len(batch) == 0  # nothing pushed: one empty last chunk
    assert batch.step() == {}
