"""Batched streaming on the GPU: the token encoder's session mode (each row of a padded batch equals that row encoded
alone with its own look-ahead), ``CausalMaskedDiffWithXvec.inference_batch`` against ``inference`` per utterance, and
``StreamingBatch`` against the same sessions run alone through ``StreamingSession``."""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu

if not torch.cuda.is_available():
    pytest.skip("needs a CUDA device", allow_module_level=True)

import minimax_speech_b200.synth as synth  # noqa: E402
from minimax_speech_b200.dac import DACVAEDecoder  # noqa: E402
from minimax_speech_b200.flow import CausalConditionalCFM, CausalConditionalDecoder  # noqa: E402
from minimax_speech_b200.front import CausalMaskedDiffWithXvec, TokenToMu  # noqa: E402
from minimax_speech_b200.streaming import StreamingBatch, StreamingSession  # noqa: E402
from oracle import restatement as O  # noqa: E402

DEV = torch.device("cuda:0")
torch.set_num_threads(os.cpu_count() or 1)
ORACLE_TOL = {"bf16": 1e-2, "fp32": 1e-5}


@pytest.fixture(scope="module", params=["bf16", "fp32"])
def front(request):
    sd = synth.conformer_encoder_state_dict(7)
    f = TokenToMu(precision=request.param)
    f.load_state_dict(sd)
    return request.param, sd, f


def _pack(rows, T_all, pad):
    """Right-padded [B, T_all] int64 with `pad(b, k)` in the padding."""
    tok = torch.empty(len(rows), T_all, dtype=torch.int64)
    for b, t in enumerate(rows):
        tok[b, :t.shape[1]] = t[0]
        for k in range(t.shape[1], T_all):
            tok[b, k] = pad(b, k)
    return tok


# (tokens, look-ahead) per row: mid-stream hops (3 context tokens) and final calls (none) in one batch
ROWS = [(60, 3), (23, 0), (4, 3), (1, 0), (131, 3), (50, 0), (28, 3)]
GARBAGE = [lambda b, k: 10 ** 9 + k, lambda b, k: -5 - k, lambda b, k: (b * 7919 + k * 104729) % 6561]


@pytest.mark.parametrize("streaming", [False, True])
def test_session_mu_equals_each_row_alone(front, streaming):
    precision, sd, f = front
    toks, embs = zip(*[synth.token_inputs(200 + b, n) for b, (n, _) in enumerate(ROWS)])
    n = torch.tensor([r[0] for r in ROWS])
    c = torch.tensor([r[1] for r in ROWS])
    emb = torch.cat(embs, 0).to(DEV)
    # a larger call first leaves its data in the workspace
    big, _ = zip(*[synth.token_inputs(300 + b, 150) for b in range(9)])
    f.encode_sessions(torch.cat(big, 0).to(DEV), torch.full((9,), 150), torch.full((9,), 3), torch.randn(9, 192, device=DEV), streaming)
    for i, pad in enumerate(GARBAGE):
        tok = _pack(toks, 140, pad).to(DEV)
        mu, spks = f.encode_sessions(tok, n, c, emb, streaming)
        T = int((n - c).max())
        assert mu.shape == (len(ROWS), 80, 2 * T)
        for b, (nb, cb) in enumerate(ROWS):
            one, s1 = f(toks[b].to(DEV), embs[b].to(DEV), finalize=cb == 0, streaming=streaming)
            Tb = nb - cb
            assert torch.equal(mu[b:b + 1, :, :2 * Tb], one), f"row {b} ({nb} tokens, {cb} context) differs from its call alone"
            assert torch.equal(spks[b:b + 1], s1)
            assert not mu[b, :, 2 * Tb:].any()
            if i == 0:
                with torch.inference_mode():
                    mr, _ = O.tokens_to_mu(sd, toks[b], embs[b], finalize=cb == 0, streaming=streaming)
                e = O.rel_l2(mu[b:b + 1, :, :2 * Tb].cpu(), mr)
                print(f"session mode ({precision}, streaming={streaming}) row {b}: {nb} tokens, {cb} context: rel-L2 vs oracle {e:.2e}")
                assert e < ORACLE_TOL[precision]


def test_invalid_rows_and_host_checks(front):
    precision, sd, f = front
    T_all = 40
    toks, embs = zip(*[synth.token_inputs(400 + b, 30) for b in range(6)])
    tok = _pack(toks, T_all, lambda b, k: 3).to(DEV)
    emb = torch.cat(embs, 0).to(DEV)
    # valid (30, 3); n_context 2; nothing after the context; more tokens than T_all; more output tokens than T; valid (30, 0)
    n = torch.tensor([30, 30, 3, T_all + 1, 30, 30], dtype=torch.int32, device=DEV)
    c = torch.tensor([3, 2, 3, 0, 0, 0], dtype=torch.int32, device=DEV)
    T = 29  # row 4 has T_b = 30 > T
    n[5] = 29
    mu, _ = f.handle(DEV).encode_sessions(tok, emb, T, n, c, False)
    assert mu.shape == (6, 80, 2 * T)
    for b in (1, 2, 3, 4):
        assert not mu[b].any(), f"invalid row {b} is not all zero"
    one, _ = f(toks[0].to(DEV), embs[0].to(DEV), finalize=False)
    assert torch.equal(mu[0:1, :, :54], one) and not mu[0, :, 54:].any()
    one, _ = f(toks[5][:, :29].to(DEV), embs[5].to(DEV), finalize=True)
    assert torch.equal(mu[5:6], one)
    bad = [([30, 30], [3, 1]), ([30, 3], [3, 3]), ([30, T_all + 1], [0, 0]), ([30], [0])]
    for nn, cc in bad:
        with pytest.raises(ValueError):
            f.encode_sessions(tok[:2], torch.tensor(nn), torch.tensor(cc), emb[:2])


def build_flow(precision):
    fsd, esd, ssd = synth.pipeline_state_dicts()
    est = CausalConditionalDecoder(precision=precision, **synth.PIPE_EST)
    cfm = CausalConditionalCFM(240, dict(t_scheduler="cosine", inference_cfg_rate=0.7), 1, 80, est)
    flow = CausalMaskedDiffWithXvec(use_speaker_encoder=True, decoder=cfm, precision=precision)
    full = dict(fsd)
    full.update({"decoder.estimator." + k: v for k, v in esd.items()})
    full.update({"speaker_encoder." + k: v for k, v in ssd.items()})
    flow.load_state_dict(full, strict=True)
    dac = DACVAEDecoder(precision=precision)
    dac.load_state_dict(synth.dac_decoder_state_dict(5, init="test"))
    return flow, dac


@pytest.fixture(scope="module", params=["bf16", "fp32"])
def pipeline(request):
    return (request.param,) + build_flow(request.param)


def test_inference_batch_equals_inference_alone(pipeline):
    precision, flow, dac = pipeline
    # (prompt tokens, tokens, finalize)
    rows = [(10, 43, False), (25, 3, True), (0, 29, False), (40, 100, True), (7, 61, False)]
    n = lambda t: torch.tensor([t.shape[1]], dtype=torch.int32)  # noqa: E731
    toks, ptoks, pfeats, embs, alone = [], [], [], [], []
    for b, (np_, nt, fin) in enumerate(rows):
        tok, emb = synth.token_inputs(500 + b, nt)
        ptok, _ = synth.token_inputs(520 + b, np_)
        pfeat = synth.dac_latents(540 + b, 2 * np_).transpose(1, 2).contiguous()
        toks.append(tok.to(DEV)), ptoks.append(ptok.to(DEV)), pfeats.append(pfeat.to(DEV))
        embs.append(flow.get_speaker_embedding({"embedding": emb.to(DEV)}, DEV))
        lat, _ = flow.inference(toks[-1], n(tok), ptoks[-1], n(ptok), pfeats[-1], n(pfeat), embedding=emb.to(DEV), streaming=True,
                                finalize=fin)
        alone.append(lat)
    lat, L = flow.inference_batch(toks, ptoks, pfeats, torch.cat(embs, 0), [r[2] for r in rows], streaming=True)
    assert lat.shape[2] == int(L.max())
    for b, one in enumerate(alone):
        assert int(L[b]) == one.shape[2]
        e = O.rel_l2(lat[b:b + 1, :, :one.shape[2]].cpu(), one.cpu())
        print(f"inference_batch ({precision}) row {b}: rel-L2 vs inference alone {e:.2e}, bitwise "
              f"{torch.equal(lat[b:b + 1, :, :one.shape[2]], one)}")
        assert e <= 1e-5
        assert not lat[b, :, one.shape[2]:].any()


def test_scheduler_equals_lone_sessions(pipeline):
    precision, flow, dac = pipeline
    specs = []  # (prompt tokens, tokens, piece, step opened, reference mels?)
    for i, (np_, nt, piece, t0) in enumerate([(10, 103, 7, 0), (25, 80, 25, 0), (3, 20, 9, 1), (40, 131, 13, 2),
                                              (0, 57, 57, 0), (17, 90, 4, 3), (25, 75, 75, 1), (8, 64, 11, 0)]):
        specs.append((np_, nt, piece, t0, i == 3))
    inputs = []
    for i, (np_, nt, piece, t0, ref) in enumerate(specs):
        tok, emb = synth.token_inputs(600 + i, nt)
        ptok, _ = synth.token_inputs(620 + i, np_)
        pfeat = synth.dac_latents(640 + i, 2 * np_).transpose(1, 2).contiguous().to(DEV)
        kw = dict(reference_mels=torch.stack([synth.reference_mel(660 + i, 40)], dim=1).to(DEV)) if ref else dict(embedding=emb.to(DEV))
        inputs.append((tok[0].tolist(), ptok.to(DEV), pfeat, kw))

    batch = StreamingBatch(flow, dac)
    ids, sess, got = {}, {}, {i: [] for i in range(len(specs))}
    pos = [0] * len(specs)
    for step in range(60):
        for i, (np_, nt, piece, t0, ref) in enumerate(specs):
            toks, ptok, pfeat, kw = inputs[i]
            if step == t0:
                ids[i] = batch.open(ptok, pfeat, **kw)
                sess[i] = batch._sessions[ids[i]]
            elif step > t0 and pos[i] < nt:
                batch.push(ids[i], toks[pos[i]:pos[i] + piece])
                pos[i] += piece
            elif step > t0 and pos[i] >= nt and i in ids and ids[i] in batch._sessions and ids[i] not in batch._finishing:
                batch.finish(ids[i])
        for sid, chunks in batch.step().items():
            got[next(i for i, v in ids.items() if v == sid)] += chunks
        if step > 0 and len(batch) == 0:
            break
    assert len(batch) == 0

    for i, (np_, nt, piece, t0, ref) in enumerate(specs):
        toks, ptok, pfeat, kw = inputs[i]
        lone = StreamingSession(flow, dac, ptok, pfeat, **kw)
        want = []
        for k in range(0, nt, piece):
            want += lone.push(toks[k:k + piece])
        want.append(lone.finish())
        assert [c.shape[1] for c in got[i]] == [c.shape[1] for c in want], f"session {i}: chunk boundaries differ"
        e = O.rel_l2(sess[i].latents.cpu(), lone.latents.cpu())
        wav, ref_wav = torch.cat(got[i], 1), torch.cat(want, 1)
        s = O.snr_db(wav.cpu(), ref_wav.cpu())
        print(f"scheduler ({precision}) session {i}: {len(want)} chunks, latents rel-L2 {e:.2e} (bitwise "
              f"{torch.equal(sess[i].latents, lone.latents)}), audio SNR {s:.1f} dB (bitwise {torch.equal(wav, ref_wav)})")
        assert e <= 1e-5 and s >= 60.0
