"""CPU emulation of the S3 tokenizer's bf16x3 mode (profiles/emulate_s3_precision.py) on the reduced-width reference
golden: split bf16 operands with fp32 sums reproduce the reference's tokens and its encoder output within 5e-5."""
import os

import numpy as np
import torch

import minimax_speech_b200.synth as synth
from oracle import restatement as O
from profiles.emulate_s3_precision import emulate


def test_bf16x3_emulation_matches_reference_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "s3_golden.npz"))
    n_mels, n_state, n_head, n_layer = [int(v) for v in g["cfg"]]

    sd = synth.s3_tokenizer_state_dict(int(g["weights_seed"]), n_mels, n_state, n_head, n_layer)
    lens = [int(v) for v in g["mel_len"]]
    mel = torch.cat([synth.s3_mel(i, int(g["frames"])) for i in range(len(lens))], 0)
    hidden, code_len, codes = emulate(sd, mel, torch.tensor(lens), "bf16x3")
    assert code_len.tolist() == g["code_len"].tolist()
    ref_h, ref_c = torch.from_numpy(g["hidden"]), torch.from_numpy(g["codes"])
    for b, n in enumerate(code_len.tolist()):
        assert O.rel_l2(hidden[b, :n], ref_h[b, :n]) < 5e-5
        assert torch.equal(codes[b, :n], ref_c[b, :n])
