"""DAC-VAE decoder and encoder with fp16 GEMM operands (precision="fp16", ``ls_dac_create_fp16``): the tensor-core
kernels compiled for fp16 instead of bf16 operands -- the folded weights, z, and every Snake / LeakyReLU output a
convolution consumes -- with fp32 accumulation, the decoder's residual stream in fp16 and the encoder's in fp32.

Checks: parity with the reference's golden outputs next to bf16 on the same input (the trained-scale decode must gain
at least 10 dB), batch invariance of both halves (bitwise), streaming and CUDA-graph replay (bitwise), the kernel's
launch plans for the DAC shapes with fp16 operands (bitwise across plans, per tile against float64), and the refusal
of weights outside fp16's range."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

if not torch.cuda.is_available():
    pytest.skip("needs a CUDA device", allow_module_level=True)

import minimax_speech_b200.native as native  # noqa: E402
import minimax_speech_b200.synth as synth  # noqa: E402
import test_kernel_plans_gpu as KP  # noqa: E402  (the launch-plan test machinery: geometry, references, plan checks)
from minimax_speech_b200.dac import DACVAEDecoder, DACVAEEncoder  # noqa: E402
from minimax_speech_b200.flow import CausalConditionalCFM, CausalConditionalDecoder  # noqa: E402
from minimax_speech_b200.front import CausalMaskedDiffWithXvec  # noqa: E402
from minimax_speech_b200.pipeline import Synthesizer  # noqa: E402
from minimax_speech_b200.streaming import StreamingSession  # noqa: E402
from oracle import restatement as O  # noqa: E402

DEV = torch.device("cuda:0")
HOP = 480
SNR_MIN_DB = 30.0
torch.set_num_threads(os.cpu_count() or 1)


def _decoder(sd, precision):
    d = DACVAEDecoder(precision=precision)
    d.load_state_dict(sd)
    return d


def _encoder(sd, precision):
    e = DACVAEEncoder(precision=precision)
    e.load_state_dict(sd)
    return e


# ------------------------------------------------------------------------------------------------ decoder parity
@pytest.fixture(scope="module")
def dac_test(golden_dir):
    g = np.load(os.path.join(golden_dir, "dac_golden.npz"))
    sd = synth.dac_decoder_state_dict(int(g["weights_seed"]), init="test")
    return g, sd, _decoder(sd, "bf16"), _decoder(sd, "fp16")


@pytest.mark.parametrize("case", ["a", "b", "c"])
def test_decode_vs_reference_golden(dac_test, case):
    g, sd, d16b, d16 = dac_test
    z = synth.dac_latents(int(g[f"dac_{case}_index"]), int(g[f"dac_{case}_frames"])).to(DEV)
    ref = torch.from_numpy(g[f"dac_{case}_y"])
    s_b, s_h = O.snr_db(d16b.decode(z).cpu(), ref), O.snr_db(d16.decode(z).cpu(), ref)
    print(f"dac {case}: SNR bf16 {s_b:.1f} dB, fp16 {s_h:.1f} dB")
    assert s_h > SNR_MIN_DB


@pytest.mark.parametrize("case", ["a", "b"])
def test_trained_scale_decode_gains_10_db(golden_dir, case):
    """Trained-scale weights (Snake alpha in [0.5, 2], activations O(10)): where the bf16 decoder's margin is thinnest."""
    g = np.load(os.path.join(golden_dir, "dac_trained_golden.npz"))
    sd = synth.dac_decoder_state_dict(int(g["weights_seed"]), init="trained")
    z = synth.dac_latents(int(g[f"dac_{case}_index"]), int(g[f"dac_{case}_frames"])).to(DEV)
    ref = torch.from_numpy(g[f"dac_{case}_y"])
    s_b = O.snr_db(_decoder(sd, "bf16").decode(z).cpu(), ref)
    s_h = O.snr_db(_decoder(sd, "fp16").decode(z).cpu(), ref)
    print(f"dac trained-scale {case}: SNR bf16 {s_b:.1f} dB, fp16 {s_h:.1f} dB (gain {s_h - s_b:.1f} dB)")
    assert s_h > SNR_MIN_DB
    assert s_h >= s_b + 10.0


def test_decode_3s_vs_oracle(dac_test):
    g, sd, _, d16 = dac_test
    z = synth.dac_latents(3, 150)
    y = d16.decode(z.to(DEV)).cpu()
    with torch.inference_mode():
        ref = O.dac_decode(sd, z)
    s = O.snr_db(y, ref)
    print(f"dac fp16 3 s SNR {s:.1f} dB")
    assert s > SNR_MIN_DB and float(y.abs().max()) <= 1.0


# ------------------------------------------------------------------------------------------------ encoder parity
@pytest.fixture(scope="module")
def enc_test(golden_dir):
    g = np.load(os.path.join(golden_dir, "dac_enc_golden.npz"))
    sd = synth.dac_encoder_state_dict(int(g["weights_seed"]), init="test")
    return g, sd, _encoder(sd, "bf16"), _encoder(sd, "fp16")


@pytest.mark.parametrize("case", ["a", "b"])
def test_encode_vs_reference_golden(enc_test, case):
    g, sd, ebf, e16 = enc_test
    frames = int(g[f"enc_{case}_frames"])
    audio = synth.audio_clip(int(g[f"enc_{case}_index"]), frames * HOP).to(DEV)
    noise = torch.zeros(1, 80, frames, device=DEV)
    m_ref, l_ref = torch.from_numpy(g[f"enc_{case}_m"]), torch.from_numpy(g[f"enc_{case}_logs"])
    errs = {}
    for name, e in (("bf16", ebf), ("fp16", e16)):
        z, m, logs = [t.cpu() for t in e.encode(audio, noise)]
        assert torch.equal(z, m)
        errs[name] = (O.rel_l2(m, m_ref), O.rel_l2(logs, l_ref))
    print(f"encode {case}: m rel-L2 bf16 {errs['bf16'][0]:.3e} fp16 {errs['fp16'][0]:.3e}; "
          f"logs rel-L2 bf16 {errs['bf16'][1]:.3e} fp16 {errs['fp16'][1]:.3e}")
    assert errs["fp16"][0] < errs["bf16"][0] and errs["fp16"][1] < errs["bf16"][1]


def test_encode_decode_round_trip(enc_test):
    g, esd, _, e16 = enc_test
    dsd = synth.dac_decoder_state_dict(5, init="test")
    audio = synth.audio_clip(3, 40 * HOP)
    z, _, _ = e16.encode(audio.to(DEV), torch.zeros(1, 80, 40, device=DEV))
    wav = _decoder(dsd, "fp16").decode(z).cpu()
    with torch.inference_mode():
        wav_ref = O.dac_decode(dsd, O.dac_encode(esd, audio)[0])
    s = O.snr_db(wav, wav_ref)
    print(f"fp16 encode -> decode round trip vs oracle: {s:.1f} dB")
    assert wav.shape == (1, 1, 40 * HOP) and s > SNR_MIN_DB


# ------------------------------------------------------------------------------------------------ batch invariance
LENS = [20, 1, 7, 13, 20, 3]


def _audio_batch(lengths, fill, seed=11):
    L = max(lengths)
    audio = torch.full((len(lengths), 1, L * HOP), fill)
    noise = torch.full((len(lengths), 80, L), fill)
    gen = torch.Generator().manual_seed(seed)
    for b, n in enumerate(lengths):
        audio[b, :, :n * HOP] = synth.audio_clip(60 + b, n * HOP)[0]
        noise[b, :, :n] = torch.randn(80, n, generator=gen)
    return audio, noise


def test_encoder_mixed_batch_bitwise_per_clip_any_padding(enc_test):
    """Padding 0, 1e4 or NaN (noise included), each on a workspace left stale by a larger call: every clip comes out
    bitwise as if encoded alone at its own length, and zero past it."""
    _, _, _, e16 = enc_test
    audio0, noise0 = _audio_batch(LENS, 0.0)
    alone = [[t.cpu() for t in e16.encode(audio0[b:b + 1, :, :n * HOP].to(DEV), noise0[b:b + 1, :, :n].to(DEV))]
             for b, n in enumerate(LENS)]
    big = torch.cat([synth.audio_clip(90 + b, 32 * HOP) for b in range(8)], 0).to(DEV)
    for fill in (0.0, 1e4, float("nan")):
        e16.encode(big, torch.randn(8, 80, 32, device=DEV))  # stale workspace
        audio, noise = _audio_batch(LENS, fill)
        outs = [t.cpu() for t in e16.encode(audio.to(DEV), noise.to(DEV), lengths=LENS)]
        for b, n in enumerate(LENS):
            for name, o, a in zip(("z", "m", "logs"), outs, alone[b]):
                assert torch.equal(o[b:b + 1, :, :n], a), f"padding {fill}: clip {b} {name}"
                assert not bool(o[b, :, n:].any()), f"padding {fill}: clip {b} {name} not zero past its length"


def test_decoder_mixed_batch_bitwise_per_item_garbage_padding(dac_test):
    """Latents past ``lengths`` are garbage (huge values, NaN): every item decodes bitwise as if alone, zero past it."""
    _, _, _, d16 = dac_test
    lengths = [60, 33, 5, 41]
    z = torch.full((4, 80, 60), float("nan"))
    z[1] = 1e4
    for b, n in enumerate(lengths):
        z[b, :, :n] = synth.dac_latents(10 + b, n)[0]
    y = d16.decode(z.to(DEV), torch.tensor(lengths)).cpu()
    for b, n in enumerate(lengths):
        y1 = d16.decode(z[b:b + 1, :, :n].to(DEV)).cpu()
        assert torch.equal(y[b:b + 1, :, :n * HOP], y1), f"item {b}"
        assert not bool(y[b, :, n * HOP:].any()), f"item {b} not zero past its length"


# ------------------------------------------------------------------------------------------------ streaming and graphs
def test_streaming_session_chunks_bitwise_one_decode():
    fsd, esd, _ = synth.pipeline_state_dicts()
    est = CausalConditionalDecoder(**synth.PIPE_EST)
    cfm = CausalConditionalCFM(240, dict(t_scheduler="cosine", inference_cfg_rate=0.7), 1, 80, est)
    flow = CausalMaskedDiffWithXvec(decoder=cfm)
    full = dict(fsd)
    full.update({"decoder.estimator." + k: v for k, v in esd.items()})
    flow.load_state_dict(full, strict=True)
    dac = _decoder(synth.dac_decoder_state_dict(5, init="test"), "fp16")
    tok, emb = synth.token_inputs(60, 103)
    ptok, _ = synth.token_inputs(61, 10)
    pfeat = synth.dac_latents(62, 20).transpose(1, 2).contiguous()
    sess = StreamingSession(flow, dac, ptok.to(DEV), pfeat.to(DEV), embedding=emb.to(DEV))
    chunks = []
    for i in range(0, 103, 7):
        chunks += sess.push(tok[0, i:i + 7].tolist())
    chunks.append(sess.finish())
    wav = torch.cat(chunks, dim=1)
    ref = dac.decode(sess.latents)[:, 0, :]
    print(f"fp16 DAC streaming: {len(chunks)} chunks, {wav.shape[1]} samples")
    assert len(chunks) >= 3 and wav.shape == ref.shape
    assert torch.equal(wav, ref)


def test_graphed_fp16_flow_and_dac_bitwise_eager():
    est = CausalConditionalDecoder(precision="fp16")
    est.load_state_dict(synth.estimator_state_dict(7, "test"))
    cfm = CausalConditionalCFM(240, dict(t_scheduler="cosine", inference_cfg_rate=0.7), 1, 80, est)
    dac = _decoder(synth.dac_decoder_state_dict(11, "test"), "fp16")
    syn = Synthesizer(cfm, dac)
    mu, mask, spks, cond = (t.to(DEV) for t in synth.batch_inputs([90, 37, 64], first_index=60))
    eager = syn(mu, mask, spks, cond, n_timesteps=3).clone()
    wav = syn.graphed(mu, mask, spks, cond, n_timesteps=3)
    assert torch.equal(wav, eager)
    assert next(iter(syn._graphs.values())).kernels > 100


# ------------------------------------------------------------------------------------------------ kernel level
@pytest.fixture
def fp16_launches(monkeypatch):
    """Every conv_gemm launch of the launch-plan machinery goes out with fp16 = 1 (fp16 operands)."""
    native.load()  # sets the hook's argtypes from the real descriptor type before it is replaced below
    desc = native.ConvGemmDesc

    def fp16_desc():
        d = desc()
        d.fp16 = 1
        return d
    monkeypatch.setattr(native, "ConvGemmDesc", fp16_desc)


def h16(t):
    return t.half()


def _snake_out(y, mag, alpha, ialpha):
    """A 16-bit Snake output checked in ulps: the rounded float64 Snake of the float64 pre-activation.  Its slack term
    (where the value cancels) bounds the fp32 accumulation error carried through Snake (slope <= 2) and the error of
    the kernel's sine (__sinf, growing with |alpha * y|)."""
    ia = ialpha.double()
    return KP.snake(y, alpha, ialpha), 2.0 * mag + 2.0 * ia * (1.0 + (alpha.double() * y).abs())


def _conv7_case(Cc, dil, seed):
    def case():
        rn = KP._gen(seed)
        a = h16(rn(KP.DAC_B, KP.DAC_M, Cc))
        w = h16(rn(7, Cc, Cc, scale=(7 * Cc) ** -0.5))
        bias, alpha = rn(Cc, scale=0.1), rn(Cc, scale=0.5) + 1.0
        ialpha = 1.0 / (alpha + 1e-9)
        lengths = KP._lens(KP.DAC_LENS)
        pad = 3 * dil
        y = KP.lrelu(KP.conv64(a, w, dil, pad) + bias.double())
        mag = KP.conv64(a.abs(), w.abs(), dil, pad) + bias.double().abs()
        geo = KP.Geometry((KP.DAC_B, KP.DAC_M, Cc), KP.DAC_B, KP.DAC_M, Cc, Cc, lengths, skip_halo=64)
        return dict(name=f"fp16 dac conv7 C={Cc} dil={dil}",
                    launch=dict(a0=a, w=w, dil=dil, pad=pad, lengths=lengths, skip_halo=64, bias=bias,
                                act=native.ACT_LRELU, out1_mode=native.OUT1_SNAKE, p1=(alpha, ialpha)),
                    outputs={"out1": (KP._nan(KP.DAC_B, KP.DAC_M, Cc, dtype=torch.float16), geo, "ulp",
                                      *_snake_out(y, mag, alpha, ialpha))})
    return case


def test_fp16_conv7_resident(fp16_launches):
    """conv7 at C = 48: resident weights from 3 tiles per CTA on."""
    def expect(sms, geo):
        tpc = -(-geo.n_all // min(geo.n_all, sms))
        if tpc >= 3:
            return dict(dual=0, b_resident=1, b_stages=7, a_stages=6, tma_out=1)
        return dict(dual=0, b_resident=0, tma_out=1)
    plans = KP.run_conv_case(_conv7_case(48, 3, 1101), KP.DAC_SMS, expect)
    assert any(p["b_resident"] for _, p, _ in plans) and any(not p["b_resident"] for _, p, _ in plans)
    KP._check_edges(plans, "b_resident")


def test_fp16_conv7_dual(fp16_launches):
    """conv7 at C = 96, dilation 9: two MMA-issuing warps from 4 tiles per CTA on."""
    def expect(sms, geo):
        tpc = -(-geo.n_all // min(geo.n_all, sms))
        if tpc >= 4:
            return dict(dual=1, b_resident=0, a_stages=4, b_stages=6, tma_out=1)
        return dict(dual=0, b_resident=0, tma_out=1)
    plans = KP.run_conv_case(_conv7_case(96, 9, 1296), KP.DAC_SMS, expect)
    assert any(p["dual"] for _, p, _ in plans) and any(not p["dual"] for _, p, _ in plans)
    KP._check_edges(plans, "dual")


def test_fp16_conv1_inplace_residual(fp16_launches):
    """1x1 conv1 (C = 96): LeakyReLU + the fp16 residual stream read and written in place, Snake of the result."""
    Cc = 96

    def case():
        rn = KP._gen(1300)
        a = h16(rn(KP.DAC_B, KP.DAC_M, Cc))
        w = h16(rn(1, Cc, Cc, scale=Cc ** -0.5))
        bias, alpha = rn(Cc, scale=0.1), rn(Cc, scale=0.5) + 1.0
        ialpha = 1.0 / (alpha + 1e-9)
        x = rn(KP.DAC_B, KP.DAC_M, Cc, scale=2.0).half()
        lengths = KP._lens(KP.DAC_LENS)
        y = KP.lrelu(KP.conv64(a, w, 1, 0) + bias.double()) + x.double()
        mag = KP.lrelu(KP.conv64(a.abs(), w.abs(), 1, 0) + bias.double().abs()) + x.double().abs()
        geo = KP.Geometry((KP.DAC_B, KP.DAC_M, Cc), KP.DAC_B, KP.DAC_M, Cc, Cc, lengths, skip_halo=64)
        return dict(name="fp16 dac conv1 in-place x", inplace=True,
                    launch=dict(a0=a, w=w, lengths=lengths, skip_halo=64, bias=bias, act=native.ACT_LRELU,
                                out1_mode=native.OUT1_SNAKE, p1=(alpha, ialpha)),
                    outputs={"out0": (x, geo, "ulp", y, mag),
                             "out1": (KP._nan(KP.DAC_B, KP.DAC_M, Cc, dtype=torch.float16), geo, "ulp",
                                      *_snake_out(y, mag, alpha, ialpha))})

    def expect(sms, geo):
        tpc = -(-geo.n_all // min(geo.n_all, sms))
        return dict(dual=0, b_resident=1, a_stages=6, b_stages=2, tma_out=1) if tpc >= 3 else dict(dual=0, b_resident=0,
                                                                                                   tma_out=1)
    plans = KP.run_conv_case(case, KP.DAC_SMS, expect)
    assert any(p["b_resident"] for _, p, _ in plans)
    KP._check_edges(plans, "b_resident")


@pytest.mark.parametrize("cin,cout,s,L,lens,sm_counts", [
    (96, 48, 2, 500, [0, 150, 0, 260], [0, 1, 3, 5, 8]),
    (384, 192, 4, 300, [300, 0, 90], [0, 1, 4, 7]),
])
def test_fp16_transposed_conv(fp16_launches, cin, cout, s, L, lens, sm_counts):
    """Up-sampling ConvTranspose1d as a two-tap GEMM (negative out_shift, LSU stores): fp16 residual + fp16 Snake."""
    import torch.nn.functional as F
    B, N = len(lens), s * cout
    block_n = max(b for b in range(16, 257, 16) if N % b == 0)
    padT, rows = (s + 1) // 2, L * s

    def case():
        rn = KP._gen(1600 + s)
        x = h16(rn(B, L, cin))
        wt = h16(rn(cin, cout, 2 * s, scale=cin ** -0.5))
        bias, alpha = rn(cout, scale=0.1), rn(cout, scale=0.5) + 1.0
        ialpha = 1.0 / (alpha + 1e-9)
        w = torch.zeros(2, N, cin, device=DEV, dtype=torch.float16)  # polyphase packing (dac_engine.cu)
        for phi in range(s):
            w[1, phi * cout:(phi + 1) * cout] = wt[:, :, phi].t()
            w[0, phi * cout:(phi + 1) * cout] = wt[:, :, phi + s].t()
        lengths = KP._lens(lens)
        ct = lambda xx, ww, bb: F.conv_transpose1d(xx.double().transpose(1, 2), ww.double(), bb, stride=s, padding=padT,
                                                   output_padding=s % 2).transpose(1, 2)
        y = ct(x, wt, bias.double())
        mag = ct(x.abs(), wt.abs(), bias.double().abs())
        geo = KP.Geometry((B, rows, cout), B, L + 1, N, block_n, lengths, m_len_add=1, skip_halo=64,
                          out_shift=-padT * cout, out_valid_mul=s * cout)
        return dict(name=f"fp16 transposed conv s={s}",
                    launch=dict(a0=x, w=w, M=L + 1, block_n=block_n, pad=1, lengths=lengths, m_len_add=1, skip_halo=64,
                                chan_mod=cout, bias=bias, out1_mode=native.OUT1_SNAKE, p1=(alpha, ialpha),
                                out_ld=N, out_shift=-padT * cout, out_bstride=rows * cout, out_alloc=rows * cout,
                                out_valid_mul=s * cout),
                    outputs={"out0": (KP._nan(B, rows, cout, dtype=torch.float16), geo, "ulp", y, mag),
                             "out1": (KP._nan(B, rows, cout, dtype=torch.float16), geo, "ulp",
                                      *_snake_out(y, mag, alpha, ialpha))})

    def expect(sms, geo):
        tpc = -(-geo.n_all // min(geo.n_all, sms))
        if N == block_n and tpc >= 3:
            return dict(dual=0, b_resident=1, tma_out=0)
        return dict(dual=0, b_resident=0, tma_out=0)
    plans = KP.run_conv_case(case, sm_counts, expect)
    assert max(p["tiles_per_cta"] for _, p, _ in plans) >= 4


def test_fp16_final_conv_tanh(fp16_launches):
    """Final conv7 (C = 48 -> 1, padded to one 16-wide tile): LeakyReLU + tanh, fp32 mono output."""
    B, T, Cc = 3, 1000, 48

    def case():
        rn = KP._gen(1700)
        a = h16(rn(B, T, Cc))
        w = torch.zeros(7, 16, Cc, device=DEV, dtype=torch.float16)
        w[:, :1] = h16(rn(7, 1, Cc, scale=(7 * Cc) ** -0.5))
        bias = torch.zeros(16, device=DEV)
        bias[0] = 0.05
        lengths = KP._lens([1000, 0, 400])
        ref = torch.tanh(KP.lrelu(KP.conv64(a, w[:, :1], 1, 3)[..., 0] + 0.05))
        geo = KP.Geometry((B, T), B, T, 16, 16, lengths, skip_halo=64, n_store=1, out_ld=1, out_valid_mul=1)
        return dict(name="fp16 final conv tanh mono",
                    launch=dict(a0=a, w=w, block_n=16, pad=3, lengths=lengths, skip_halo=64, chan_mod=16, bias=bias,
                                act=native.ACT_LRELU_TANH, n_store=1, out_ld=1, out_bstride=T, out_alloc=T,
                                out_valid_mul=1),
                    outputs={"out0": (KP._nan(B, T), geo, "tanh_f32", ref, None)})

    def expect(sms, geo):
        tpc = -(-geo.n_all // min(geo.n_all, sms))
        return dict(dual=0, b_resident=int(tpc >= 3), tma_out=0)
    plans = KP.run_conv_case(case, [0, 1, 3, 5], expect)
    assert max(p["tiles_per_cta"] for _, p, _ in plans) >= 3


# ------------------------------------------------------------------------------------------------ errors
def test_weight_outside_fp16_range_is_refused():
    dsd = synth.dac_decoder_state_dict(5, init="test")
    layer = "decoder.model.2.block.3.block.1.0"
    dsd[layer + ".weight_g"] = dsd[layer + ".weight_g"] * 1e7
    with pytest.raises(RuntimeError, match=r"code -4\).*" + layer.replace(".", r"\.") + ".*fp16"):
        _decoder(dsd, "fp16").handle(DEV)
    _decoder(dsd, "bf16").handle(DEV)  # bf16's range holds it
    esd = synth.dac_encoder_state_dict(5, init="test")
    layer = "encoder.block.3.block.4.0"  # a downsampling conv (the polyphase re-pack)
    esd[layer + ".weight_g"] = esd[layer + ".weight_g"] * 1e7
    with pytest.raises(RuntimeError, match=r"code -4\).*" + layer.replace(".", r"\.") + ".*fp16"):
        _encoder(esd, "fp16").handle(DEV)


def test_other_precisions_still_refused():
    for cls in (DACVAEDecoder, DACVAEEncoder):
        with pytest.raises(ValueError):
            cls(precision="bf16x3")
