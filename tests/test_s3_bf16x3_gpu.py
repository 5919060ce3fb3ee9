"""S3 tokenizer, precision="bf16x3" (tensor cores, split bf16 operands, csrc/s3_engine.cu) on the B200: fp32-level
agreement with the reference goldens, the oracle and fp32 mode; bitwise batch invariance; edge shapes; argument errors."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

if not torch.cuda.is_available():
    pytest.skip("needs a CUDA device", allow_module_level=True)

import minimax_speech_b200.synth as synth  # noqa: E402
from minimax_speech_b200.tokenizer import S3TokenizerV2  # noqa: E402
from oracle import restatement as O  # noqa: E402
from profiles.emulate_s3_precision import fsq_margin  # noqa: E402

DEV = torch.device("cuda")
HIDDEN_TOL = 5e-5
MARGIN = 1e-4


def _small(g, precision="bf16x3"):
    n_mels, n_state, n_head, n_layer = [int(v) for v in g["cfg"]]

    class Cfg:
        pass
    Cfg.n_mels, Cfg.n_audio_state, Cfg.n_audio_head, Cfg.n_audio_layer = n_mels, n_state, n_head, n_layer
    return S3TokenizerV2("speech_tokenizer_v2_25hz", Cfg(), weight_seed=int(g["weights_seed"]), precision=precision)


_FULL = {}


def _full(precision):
    if precision not in _FULL:
        _FULL[precision] = S3TokenizerV2(weight_seed=33, precision=precision)
    return _FULL[precision]


def _batch(lens, first=10, T=None):
    T = T or max(lens)
    mel = torch.zeros(len(lens), 128, T)
    for i, n in enumerate(lens):
        mel[i, :, :n] = synth.s3_mel(first + i, n)[0]
    return mel


def _check_against(sd, hidden, codes, ref_h, ref_c, code_len, label, max_diff=1):
    """hidden rel-L2 < 5e-5 per clip; tokens identical wherever every fp32 decision is > 1e-4 from a boundary; at most
    `max_diff` tokens differ overall"""
    diff = 0
    for b, n in enumerate(code_len):
        e = O.rel_l2(hidden[b, :n].cpu(), ref_h[b, :n].cpu())
        print(f"{label} clip {b}: hidden rel-L2 {e:.2e}")
        assert e < HIDDEN_TOL
        mine, ref = codes[b, :n].cpu(), ref_c[b, :n].cpu()
        safe = fsq_margin(sd, ref_h[b:b + 1, :n].cpu())[0] > MARGIN
        assert torch.equal(mine[safe], ref[safe]), f"{label} clip {b}: a token away from every rounding boundary differs"
        diff += int((mine != ref).sum())
    print(f"{label}: {diff} tokens differ")
    assert diff <= max_diff


def test_bf16x3_vs_reference_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "s3_golden.npz"))
    tok = _small(g)
    lens = [int(v) for v in g["mel_len"]]
    mel = torch.cat([synth.s3_mel(i, int(g["frames"])) for i in range(len(lens))], 0)
    codes, code_len, hidden = tok.quantize(mel.to(DEV), torch.tensor(lens), return_hidden=True)
    assert codes.dtype == torch.int32 and code_len.tolist() == g["code_len"].tolist()
    ref_h, ref_c = torch.from_numpy(g["hidden"]), torch.from_numpy(g["codes"])
    for b, n in enumerate(code_len.tolist()):
        e = O.rel_l2(hidden[b, :n].cpu(), ref_h[b, :n])
        print(f"bf16x3 golden clip {b}: hidden rel-L2 {e:.2e}")
        assert e < HIDDEN_TOL
        assert torch.equal(codes[b, :n].cpu(), ref_c[b, :n])


@pytest.mark.parametrize("lens", [[400, 263], [1000, 760, 520]])
def test_bf16x3_full_width_vs_oracle(lens):
    tok = _full("bf16x3")
    sd = {k: v.clone() for k, v in tok.state_dict().items()}
    mel = _batch(lens)
    codes, code_len, hidden = tok.quantize(mel.to(DEV), torch.tensor(lens), return_hidden=True)
    with torch.inference_mode():
        ref_h, ref_l = O.s3_encode(sd, mel, torch.tensor(lens))
        ref_c = O.fsq_encode(sd["quantizer._codebook.project_down.weight"], sd["quantizer._codebook.project_down.bias"], ref_h)
    assert code_len.tolist() == ref_l.tolist()
    _check_against(sd, hidden, codes, ref_h, ref_c, ref_l.tolist(), "bf16x3 vs oracle")


def test_bf16x3_vs_fp32_mode_mixed_lengths():
    fast, ref = _full("bf16x3"), _full("fp32")
    sd = {k: v.clone() for k, v in fast.state_dict().items()}
    lens = synth.mixed_lengths(16, 2, 30, frame_rate=100, seed=4)
    mel = _batch(lens, first=100).to(DEV)
    ml = torch.tensor(lens)
    codes, code_len, hidden = fast.quantize(mel, ml, return_hidden=True)
    rc, rl, rh = ref.quantize(mel, ml, return_hidden=True)
    assert code_len.tolist() == rl.tolist()
    _check_against(sd, hidden, codes, rh, rc, rl.tolist(), "bf16x3 vs fp32 mode")


def test_bf16x3_long_clips_vs_reference_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "s3_long_golden.npz"))
    tok = _small(g)
    lens = [int(v) for v in g["mel_len"]]
    mel = torch.zeros(len(lens), int(g["cfg"][0]), max(lens))
    for i, n in enumerate(lens):
        mel[i, :, :n] = synth.s3_mel(40 + i, n)[0]
    codes, code_len = tok.quantize(mel.to(DEV), torch.tensor(lens))
    assert codes.dtype == torch.long and code_len.tolist() == g["code_len"].tolist()
    ref = torch.from_numpy(g["codes"])
    same = int((codes.cpu() == ref).sum())
    print(f"bf16x3 long clips: {same} of {ref.numel()} entries identical")
    assert same >= ref.numel() - 2


def _alone(tok, mel, lens):
    out = []
    for b, n in enumerate(lens):
        c, l, h = tok.quantize(mel[b:b + 1, :, :n].contiguous(), torch.tensor([n]), return_hidden=True)
        out.append((c[0], int(l[0]), h[0]))
    return out


def _assert_bitwise(codes, code_len, hidden, alone):
    for b, (c, n, h) in enumerate(alone):
        assert int(code_len[b]) == n
        assert torch.equal(codes[b, :n], c[:n]), f"clip {b}: tokens differ from the call with the clip alone"
        assert torch.equal(hidden[b, :n], h[:n]), f"clip {b}: hidden differs from the call with the clip alone"


def test_bf16x3_batch_invariance():
    tok = _full("bf16x3")
    lens = [1203, 400, 2999, 77, 650]
    mel = _batch(lens, first=60).to(DEV)
    alone = _alone(tok, mel, lens)
    for pad in (0.0, 1e4, float("nan")):
        m = mel.clone()
        for b, n in enumerate(lens):
            m[b, :, n:] = pad
        codes, code_len, hidden = tok.quantize(m, torch.tensor(lens), return_hidden=True)
        _assert_bitwise(codes, code_len, hidden, alone)
        assert torch.isfinite(hidden).all()
    # a handle whose workspace a larger batch left stale
    big = _batch([3000] * 12, first=80).to(DEV)
    big[:, :, 2000:] = float("nan")
    tok.quantize(big, torch.tensor([2000] * 12))
    codes, code_len, hidden = tok.quantize(mel, torch.tensor(lens), return_hidden=True)
    _assert_bitwise(codes, code_len, hidden, alone)


@pytest.mark.parametrize("lens,T", [([1, 2, 3, 4], 4), ([1, 2, 3, 4], 9), ([203, 150, 96], 203), ([3000] * 4, 3000),
                                    ([777], 777)])
def test_bf16x3_edges(lens, T):
    """mel_len 1..4, odd T, every clip at 3000 frames, B = 1: per-clip bitwise equality and agreement with fp32 mode."""
    fast, ref = _full("bf16x3"), _full("fp32")
    sd = {k: v.clone() for k, v in fast.state_dict().items()}
    mel = _batch(lens, first=200, T=T).to(DEV)
    ml = torch.tensor(lens)
    codes, code_len, hidden = fast.quantize(mel, ml, return_hidden=True)
    assert codes.shape == (len(lens), (((T - 1) // 2 + 1) - 1) // 2 + 1)
    _assert_bitwise(codes, code_len, hidden, _alone(fast, mel, lens))
    rc, rl, rh = ref.quantize(mel, ml, return_hidden=True)
    assert code_len.tolist() == rl.tolist()
    _check_against(sd, hidden, codes, rh, rc, rl.tolist(), f"edges {lens} T={T}")


def test_bf16x3_errors():
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "s3_golden.npz"))
    tok = _small(g)
    mel = synth.s3_mel(0, 96)
    with pytest.raises(RuntimeError):
        tok.quantize(mel, torch.tensor([96]))  # CPU tensors are rejected, not emulated
    with pytest.raises(ValueError, match="bf16x3"):
        _small(g, precision="bf16")
    with pytest.raises(ValueError):
        _small(g, precision="fp16")
    with pytest.raises(ValueError):
        _small(g, precision="tf32")
    tok.precision = "bf16"  # changed after construction: refused when the handle is (re)built
    with pytest.raises(ValueError):
        tok.quantize(mel.to(DEV), torch.tensor([96]))
    tok.precision = "fp32"  # and a valid change rebuilds the handle in the new precision
    c32, _ = tok.quantize(mel.to(DEV), torch.tensor([96]))
    assert tok.handle(DEV).precision == "fp32"
    tok.precision = "bf16x3"
    c3, _ = tok.quantize(mel.to(DEV), torch.tensor([96]))
    assert tok.handle(DEV).precision == "bf16x3" and c3.shape == c32.shape
