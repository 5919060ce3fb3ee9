"""CPU emulation: how far do rounded GEMM operands move the S3 tokenizer, and which tokens change?

Runs ``oracle.s3_encode`` / ``s3_quantize`` with every dense ``F.linear`` / ``F.conv1d`` (not the depthwise FSMN conv)
replaced by a rounded-operand form; attention, FSMN, LayerNorm and the residual stream stay fp32:
  bf16    linear(bf16(a), bf16(w))
  bf16x3  linear(a_hi, w_hi) + linear(a_lo, w_hi) + linear(a_hi, w_lo),  hi = bf16(x), lo = bf16(x - hi)
The products of bf16 operands are exact in fp32, so this is what the tensor cores compute up to the fp32 summation order.

    python -m profiles.emulate_s3_precision            # shipped width, 4 clips of 1000 / 1000 / 760 / 520 mel frames

Log: profiles/r04_emulate_s3_precision.log.
"""
import argparse
import contextlib
import os
import sys
import time

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import restatement as O  # noqa: E402


def _bf16(x):
    return x.to(torch.bfloat16).to(torch.float32)


def _split(x):
    hi = _bf16(x)
    return hi, _bf16(x - hi)


@contextlib.contextmanager
def rounded_operands(mode):
    """Within the block, F.linear and dense F.conv1d use `mode` operands ("fp32", "bf16" or "bf16x3")."""
    lin, conv = F.linear, F.conv1d
    if mode == "fp32":
        yield
        return

    def three(op, a, w, bias, **kw):
        if mode == "bf16":
            return op(_bf16(a), _bf16(w), bias, **kw)
        ah, al = _split(a)
        wh, wl = _split(w)
        return op(ah, wh, bias, **kw) + op(al, wh, None, **kw) + op(ah, wl, None, **kw)

    def linear(a, w, bias=None):
        return three(lin, a.float(), w.float(), bias)

    def conv1d(a, w, bias=None, stride=1, padding=0, dilation=1, groups=1):
        if groups != 1:  # the depthwise FSMN memory stays fp32
            return conv(a, w, bias, stride=stride, padding=padding, dilation=dilation, groups=groups)
        return three(conv, a.float(), w.float(), bias, stride=stride, padding=padding, dilation=dilation)

    F.linear, F.conv1d = linear, conv1d
    try:
        yield
    finally:
        F.linear, F.conv1d = lin, conv


def fsq_margin(sd, hidden):
    """Per frame: the smallest distance of any of the 8 FSQ decisions (tanh(project_down(h)) * 0.999) from a rounding
    boundary (+-0.5), for the fp32 hidden [B, T, D] -> [B, T]."""
    w, b = sd["quantizer._codebook.project_down.weight"], sd["quantizer._codebook.project_down.bias"]
    h = torch.tanh(F.linear(hidden.double(), w.double(), b.double())) * 0.999
    return (h.abs() - 0.5).abs().min(dim=-1).values


def emulate(sd, mel, mel_len, mode):
    """-> (hidden [B, T', D], code_len [B], codes [B, T']) with `mode` GEMM operands."""
    with torch.inference_mode(), rounded_operands(mode):
        hidden, code_len = O.s3_encode(sd, mel, mel_len)
        codes = O.fsq_encode(sd["quantizer._codebook.project_down.weight"], sd["quantizer._codebook.project_down.bias"], hidden)
    return hidden, code_len, codes


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seed", type=int, default=33)
    ap.add_argument("--frames", default="1000,1000,760,520")
    ap.add_argument("--threads", type=int, default=0)
    a = ap.parse_args()
    if a.threads:
        torch.set_num_threads(a.threads)
    import minimax_speech_b200.synth as synth
    from minimax_speech_b200.tokenizer import S3TokenizerV2
    sd = {k: v.clone() for k, v in S3TokenizerV2(weight_seed=a.seed).state_dict().items()}
    lens = [int(v) for v in a.frames.split(",")]
    mel = torch.zeros(len(lens), 128, max(lens))
    for i, n in enumerate(lens):
        mel[i, :, :n] = synth.s3_mel(10 + i, n)[0]
    mel_len = torch.tensor(lens)
    t0 = time.time()
    ref_h, ref_l, ref_c = emulate(sd, mel, mel_len, "fp32")
    total = int(ref_l.sum())
    margin = torch.cat([fsq_margin(sd, ref_h[b:b + 1, :n])[0] for b, n in enumerate(ref_l.tolist())])
    print(f"S3TokenizerV2(weight_seed={a.seed}), 1280 wide, 20 heads, 6 blocks; mel frames {lens} -> {total} tokens")
    print(f"fp32: frames with an FSQ decision within 1e-2 of a rounding boundary: {100.0 * float((margin < 1e-2).float().mean()):.1f} %")
    print("| operands of every linear / conv | encoder output rel-L2 vs fp32 | tokens identical |")
    print("|---|---|---|")
    for mode in ("bf16", "bf16x3"):
        h, l, c = emulate(sd, mel, mel_len, mode)
        assert l.tolist() == ref_l.tolist()
        num = sum(float((h[b, :n].double() - ref_h[b, :n].double()).pow(2).sum()) for b, n in enumerate(ref_l.tolist()))
        den = sum(float(ref_h[b, :n].double().pow(2).sum()) for b, n in enumerate(ref_l.tolist()))
        same = sum(int((c[b, :n] == ref_c[b, :n]).sum()) for b, n in enumerate(ref_l.tolist()))
        print(f"| {mode} | {(num / den) ** 0.5:.1e} | {same} of {total} ({100.0 * same / total:.1f} %) |")
    print(f"({time.time() - t0:.0f} s on the CPU)")


if __name__ == "__main__":
    main()
