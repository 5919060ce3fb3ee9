"""Voice conversion from raw speech (``vc.VoiceConverter``) with synthetic weights: prompt preparation against the same
steps called by hand, a batched ``convert`` against each conversion alone, the whole chain against the CPU oracle
(torchaudio float64 resample -> log-mel -> S3 tokens; DAC-VAE encoder mean; flow inference; DAC-VAE decode), a
``Prompt`` opening a streaming session, and the ``sample_rate`` keyword of the bulk extraction tools."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

if not torch.cuda.is_available():
    pytest.skip("needs a CUDA device", allow_module_level=True)

import torchaudio.functional as AF  # noqa: E402

import minimax_speech_b200.synth as synth  # noqa: E402
from minimax_speech_b200 import audio, pipeline  # noqa: E402
from minimax_speech_b200.dac import DACVAEDecoder, DACVAEEncoder  # noqa: E402
from minimax_speech_b200.flow import CausalConditionalCFM, CausalConditionalDecoder  # noqa: E402
from minimax_speech_b200.front import CausalMaskedDiffWithXvec  # noqa: E402
from minimax_speech_b200.streaming import StreamingSession  # noqa: E402
from minimax_speech_b200.tokenizer import S3TokenizerV2  # noqa: E402
from minimax_speech_b200.vc import Prompt, VoiceConverter, prompt_cut  # noqa: E402
from oracle import restatement as O  # noqa: E402
from profiles import s3_mel_reference as R  # noqa: E402

DEV = torch.device("cuda:0")
torch.set_num_threads(os.cpu_count() or 1)
ENC_SEED, DEC_SEED = 4, 5
_TOK = {}


def speech_like(n, seed, rate):
    rng = np.random.default_rng(seed)
    t = np.arange(n) / rate
    f0 = 120 + 80 * np.sin(2 * np.pi * (0.2 + 0.05 * (seed % 5)) * t)
    ph = np.cumsum(2 * np.pi * f0 / rate)
    x = 0.1 * sum(np.sin(h * ph) / h for h in range(1, 25)) * (1 + 0.5 * np.sin(2 * np.pi * 3 * t))
    x = x + 0.01 * rng.standard_normal(n)
    return torch.from_numpy(np.clip(2 * x, -1, 1).astype(np.float32))


def tokenizer():
    if "fp32" not in _TOK:
        _TOK["fp32"] = S3TokenizerV2(weight_seed=33, precision="fp32")
    return _TOK["fp32"]


def build(precision):
    fsd, esd, ssd = synth.pipeline_state_dicts()
    est = CausalConditionalDecoder(precision=precision, **synth.PIPE_EST)
    cfm = CausalConditionalCFM(240, dict(t_scheduler="cosine", inference_cfg_rate=0.7), 1, 80, est)
    flow = CausalMaskedDiffWithXvec(use_speaker_encoder=True, decoder=cfm, precision=precision)
    full = dict(fsd)
    full.update({"decoder.estimator." + k: v for k, v in esd.items()})
    full.update({"speaker_encoder." + k: v for k, v in ssd.items()})
    flow.load_state_dict(full, strict=True)
    enc = DACVAEEncoder(precision=precision)
    enc.load_state_dict(synth.dac_encoder_state_dict(ENC_SEED, init="test"))
    dec = DACVAEDecoder(precision=precision)
    dec.load_state_dict(synth.dac_decoder_state_dict(DEC_SEED, init="test"))
    return VoiceConverter(flow, tokenizer(), enc, dec, DEV)


@pytest.fixture(scope="module", params=["bf16", "fp32"])
def conv(request):
    return request.param, build(request.param)


def test_prompts_equal_the_steps_by_hand(conv):
    precision, vcv = conv
    rate = 44100
    clips = [speech_like(int(s * rate), 10 + i, rate) for i, s in enumerate((3.2, 5.05, 4.0))]
    emb = torch.randn(3, 192, generator=torch.Generator().manual_seed(1)).to(DEV)
    got = vcv.prompts(clips, rate, embedding=emb)
    for b, c in enumerate(clips):
        a16 = audio.resample(c.to(DEV), rate, 16000)
        codes, code_len = vcv.tokenizer.quantize_audio(a16[None], [a16.shape[0]])
        a24 = audio.resample(c.to(DEV), rate, 24000)
        a24 = vcv.dac_encoder.preprocess(a24[None, None])
        L = a24.shape[-1] // 480
        _, m, _ = vcv.dac_encoder.encode(a24, torch.zeros(1, 80, L, device=DEV))
        n = prompt_cut(L, int(code_len[0]))
        assert torch.equal(got[b].token, codes[:, :n].to(torch.int64)), f"prompt {b}: tokens"
        assert torch.equal(got[b].feat, m[:, :, :2 * n].transpose(1, 2)), f"prompt {b}: features"
        assert torch.equal(got[b].embedding, vcv.flow.get_speaker_embedding({"embedding": emb[b:b + 1]}, DEV))
        assert got[b].feat.shape == (1, 2 * n, 80) and got[b].token.dtype == torch.int64


def test_convert_batch_equals_each_alone(conv):
    precision, vcv = conv
    rate = 24000
    prompts = vcv.prompts([speech_like(int(s * rate), 20 + i, rate) for i, s in enumerate((3.0, 4.4, 3.7))], rate,
                          embedding=torch.randn(3, 192, generator=torch.Generator().manual_seed(2)).to(DEV))
    secs = (2.3, 4.1, 3.0, 2.0, 5.2, 3.3)
    sources = [speech_like(int(s * 16000), 30 + i, 16000) for i, s in enumerate(secs)]
    which = [prompts[i % 3] for i in range(len(sources))]
    speeds = [1.0, 1.3, 0.8, 1.0, 2.0, 0.5]
    wav = vcv.convert(sources, 16000, which, speed=speeds)
    toks = vcv.tokens(sources, 16000)
    for b, src in enumerate(sources):
        one_tok = vcv.tokens([src], 16000)[0]
        assert torch.equal(one_tok, toks[b]), f"source {b}: tokens differ alone"
        one = vcv.convert([src], 16000, which[b], speed=speeds[b])[0]
        assert wav[b].shape == one.shape, f"source {b}: length {wav[b].shape} vs {one.shape} alone"
        s = O.snr_db(wav[b].cpu(), one.cpu())
        print(f"convert ({precision}) source {b}: {wav[b].shape[0]} samples, audio SNR vs alone {s:.1f} dB")
        assert s >= 60.0
    # latents of the batched solve against the solve alone
    lat, L = vcv.flow.inference_batch([t for t in toks], [p.token for p in which], [p.feat for p in which],
                                      torch.cat([p.embedding for p in which]), [True] * len(toks))
    for b in range(len(toks)):
        one, _ = vcv.flow.inference_batch([toks[b]], [which[b].token], [which[b].feat], which[b].embedding, [True])
        e = O.rel_l2(lat[b:b + 1, :, :int(L[b])].cpu(), one.cpu())
        assert e <= 1e-5, f"source {b}: latents rel-L2 {e:.2e} vs alone"
    # speed 1 given as a number or per row is the same as no speed at all
    a = vcv.convert(sources[:2], 16000, which[:2])
    b_ = vcv.convert(sources[:2], 16000, which[:2], speed=[1.0, 1.0])
    assert all(torch.equal(x, y) for x, y in zip(a, b_))


ORACLE_RATE = 22050


def oracle_inputs():
    """Prompt recording, two sources and an x-vector, all at 22.05 kHz."""
    rate = ORACLE_RATE
    return (speech_like(int(3.1 * rate), 50, rate), [speech_like(int(2.4 * rate), 51, rate), speech_like(int(3.6 * rate), 52, rate)],
            torch.randn(1, 192, generator=torch.Generator().manual_seed(3)))


_ORACLE = {}


def oracle_chain():
    """The chain on the CPU: torchaudio float64 resample -> log-mel restated in float64 -> S3 tokens; DAC-VAE encoder mean
    of the 24 kHz prompt, cut as CosyVoice2 cuts it; flow inference; DAC-VAE decode.  Computed once for both precisions."""
    if not _ORACLE:
        rate = ORACLE_RATE
        prompt_audio, sources, emb = oracle_inputs()
        fsd, esd, _ = synth.pipeline_state_dicts()
        tok_sd = {k: v.clone() for k, v in tokenizer().state_dict().items()}
        filt = tokenizer().mel_filters.double()

        def ref_tokens(x):
            mel = R.s3_log_mel(AF.resample(x.double(), rate, 16000), filt).float()
            codes, n = O.s3_quantize(tok_sd, mel[None], torch.tensor([mel.shape[1]]))
            return codes[:, :int(n[0])].to(torch.int64)

        with torch.inference_mode():
            ptok = ref_tokens(prompt_audio)
            a24 = AF.resample(prompt_audio.double(), rate, 24000).float()
            a24 = torch.nn.functional.pad(a24, (0, (-a24.shape[0]) % 480))[None, None]
            _, m, _ = O.dac_encode(synth.dac_encoder_state_dict(ENC_SEED, init="test"), a24)
            n = prompt_cut(m.shape[2], ptok.shape[1])
            ptok, pfeat = ptok[:, :n], m[:, :, :2 * n].transpose(1, 2).contiguous()
            toks, lats, wavs = [], [], []
            for x in sources:
                toks.append(ref_tokens(x))
                lats.append(O.flow_inference(fsd, esd, synth.fixed_noise(), toks[-1], ptok, pfeat, embedding=emb, finalize=True))
                wavs.append(O.dac_decode(synth.dac_decoder_state_dict(DEC_SEED, init="test"), lats[-1])[0, 0])
        _ORACLE.update(ptok=ptok, pfeat=pfeat, toks=toks, lats=lats, wavs=wavs)
    return _ORACLE


def test_end_to_end_against_oracle_chain(conv):
    precision, vcv = conv
    prompt_audio, sources, emb = oracle_inputs()
    p = vcv.prompts([prompt_audio], ORACLE_RATE, embedding=emb.to(DEV))[0]
    wav = vcv.convert(sources, ORACLE_RATE, p)
    toks = vcv.tokens(sources, ORACLE_RATE)
    ref = oracle_chain()
    tol = 1e-4 if precision == "fp32" else 1e-2
    assert torch.equal(p.token.cpu(), ref["ptok"]), "prompt tokens differ from the oracle chain"
    e = O.rel_l2(p.feat.cpu(), ref["pfeat"])
    print(f"oracle chain ({precision}): {p.token.shape[1]} prompt tokens, prompt features rel-L2 {e:.2e}")
    assert e <= tol
    for b in range(len(sources)):
        assert torch.equal(toks[b].cpu(), ref["toks"][b]), f"source {b}: tokens differ from the oracle chain"
        lat, _ = vcv.flow.inference_batch([toks[b]], [p.token], [p.feat], p.embedding, [True])
        e = O.rel_l2(lat.cpu(), ref["lats"][b])
        s = O.snr_db(wav[b].cpu(), ref["wavs"][b])
        print(f"oracle chain ({precision}) source {b}: {toks[b].shape[1]} tokens, latents rel-L2 {e:.2e}, waveform {s:.1f} dB")
        assert e <= tol and s >= (80.0 if precision == "fp32" else 30.0)


def test_prompt_opens_a_streaming_session(conv):
    precision, vcv = conv
    if precision != "bf16":
        pytest.skip("the session path is the same in both precisions")
    p = vcv.prompts([speech_like(48000, 60, 16000)], 16000)[0]
    toks = synth.token_inputs(61, 70)[0][0].tolist()
    outs = []
    for prompt in (p, Prompt(p.token.clone(), p.feat.clone(), p.embedding.clone())):
        s = StreamingSession(vcv.flow, vcv.dac_decoder, prompt.token, prompt.feat, embedding=prompt.embedding)
        chunks = s.push(toks)
        chunks.append(s.finish())
        outs.append(torch.cat(chunks, 1))
    s = O.snr_db(outs[1].cpu(), outs[0].cpu())
    print(f"streaming session from a Prompt: {outs[0].shape[1]} samples, bitwise {torch.equal(outs[0], outs[1])}, {s:.1f} dB")
    assert outs[0].shape == outs[1].shape and outs[0].shape[1] > 0 and (torch.equal(outs[0], outs[1]) or s >= 100.0)


def test_extraction_sample_rate_keyword(tmp_path, conv):
    precision, vcv = conv
    if precision != "bf16":
        pytest.skip("one precision is enough for the resampling step")
    paths = []
    for i, s in enumerate((2.5, 3.7, 1.9)):
        f = tmp_path / f"clip{i}.pt"
        torch.save(speech_like(int(s * 44100), 70 + i, 44100), f)
        paths.append(str(f))

    def by_hand(rate):
        return lambda path: audio.resample(torch.load(path).to(DEV), 44100, rate).cpu()

    for mbs in (None, 10 ** 6):
        got = pipeline.extract_tokens(paths, torch.load, vcv.tokenizer, DEV, save=False, max_batch_samples=mbs, sample_rate=44100)
        want = pipeline.extract_tokens(paths, by_hand(16000), vcv.tokenizer, DEV, save=False, max_batch_samples=mbs)
        for (_, r1), (_, r2) in zip(got, want):
            assert torch.equal(r1["tokens"], r2["tokens"]) and r1["original_samples"] == r2["original_samples"]
    g1, g2 = torch.Generator().manual_seed(9), torch.Generator().manual_seed(9)
    got = pipeline.extract_latents(paths, torch.load, vcv.dac_encoder, DEV, save=False, generator=g1, sample_rate=44100)
    want = pipeline.extract_latents(paths, by_hand(24000), vcv.dac_encoder, DEV, save=False, generator=g2)
    for (_, r1), (_, r2) in zip(got, want):
        assert torch.equal(r1["z"], r2["z"]) and torch.equal(r1["mu"], r2["mu"])
        assert r1["original_samples"] == r2["original_samples"]
    # 24 kHz sources for the tokenizer
    got = pipeline.extract_tokens(paths[:1], torch.load, vcv.tokenizer, DEV, save=False, sample_rate=24000)
    want = pipeline.extract_tokens(paths[:1], lambda path: audio.resample(torch.load(path).to(DEV), 24000, 16000).cpu(),
                                   vcv.tokenizer, DEV, save=False)
    assert torch.equal(got[0][1]["tokens"], want[0][1]["tokens"])
