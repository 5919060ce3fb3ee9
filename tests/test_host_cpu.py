"""CPU-only checks: the C-ABI library builds/loads and exports every symbol of include/ls_b200.h, and the
drop-in modules expose exactly the reference's state_dict schema.  No compute calls (no GPU here)."""
import ctypes
import json
import os
import re

import pytest
import torch

import minimax_speech_b200.build as build
import minimax_speech_b200.synth as synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    src = open(os.path.join(ROOT, "include", "ls_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(ls_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    path = build.build()
    lib = ctypes.CDLL(path)
    syms = header_symbols()
    assert len(syms) >= 14
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in ls_b200.h but not exported"
    lib.ls_abi_version.restype = ctypes.c_int32
    assert lib.ls_abi_version() == 1


def test_binding_covers_header():
    import minimax_speech_b200.native as native
    assert sorted(native.EXPORTS) == header_symbols()


def test_create_fails_loudly_without_gpu_or_weights():
    import minimax_speech_b200.native as native
    lib = native.load()
    h = ctypes.c_void_p()
    arr, keep = native.tensor_table({"bogus": torch.zeros(3)})
    code = lib.ls_flow_create(arr, 1, 0, ctypes.byref(h))
    assert code != 0 and not h.value
    assert lib.ls_last_error()


def test_state_dict_schema_matches_reference(golden_dir):
    keys = json.load(open(os.path.join(golden_dir, "state_dict_keys.json")))
    from minimax_speech_b200.flow import CausalConditionalDecoder
    from minimax_speech_b200.dac import DACVAEDecoder
    est = CausalConditionalDecoder()
    assert {k: list(v.shape) for k, v in est.state_dict().items()} == keys["estimator"]
    dac = DACVAEDecoder()
    assert {k: list(v.shape) for k, v in dac.state_dict().items()} == keys["dac_decoder"]
    # reference checkpoints carry encoder keys too (ckpt['generator']); they are ignored, not rejected
    sd = dict(dac.state_dict())
    sd["encoder.block.0.weight_v"] = torch.zeros(1)
    dac.load_state_dict(sd)


def test_cpu_tensors_are_rejected_not_emulated():
    from minimax_speech_b200.flow import CausalConditionalCFM, CausalConditionalDecoder
    est = CausalConditionalDecoder(n_blocks=1, num_mid_blocks=1)
    cfm = CausalConditionalCFM(240, dict(t_scheduler="cosine", inference_cfg_rate=0.7), 1, 80, est)
    mu, mask, spks, cond = synth.batch_inputs([16])
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        cfm(mu, mask, 2, spks=spks, cond=cond)


def test_t_span_matches_oracle():
    from minimax_speech_b200.flow import CausalConditionalCFM
    from oracle import restatement as O
    cfm = CausalConditionalCFM(240, dict(t_scheduler="cosine", inference_cfg_rate=0.7), 1, 80, None)
    assert torch.equal(cfm._t_span(10), O.cosine_t_span(10))
    assert abs(float(cfm.rand_noise[0, 0, 0]) + 1.12584) < 1e-4


def test_non_prefix_mask_rejected():
    from minimax_speech_b200.flow import _check_prefix_mask
    m = torch.ones(1, 1, 8)
    _check_prefix_mask(m)
    m[0, 0, 3] = 0
    with pytest.raises(ValueError):
        _check_prefix_mask(m)


def test_latent_extraction_sharding_and_record_format(tmp_path):
    """pipeline.extract_latents: the reference tool's contiguous per-rank slices (extract_dac_latents.py:146-150) and its
    ``*_latent2x.pt`` record (:184-196), with a stand-in encoder (the real one needs a GPU)."""
    import torch
    from minimax_speech_b200 import pipeline

    for n, world in [(10, 4), (7, 8), (16, 2), (3, 1)]:
        covered = []
        for r in range(world):
            s, e = pipeline.shard_files(n, r, world)
            per = n // world
            assert (s, e) == (r * per, r * per + per if r < world - 1 else n)
            covered += list(range(s, e))
        assert covered == list(range(n))

    class FakeEncoder:
        hop_length, latent_dim, sample_rate = 480, 80, 24000

        def preprocess(self, a):
            return torch.nn.functional.pad(a, (0, (-a.shape[-1]) % self.hop_length))

        def encode(self, audio, noise):
            L = audio.shape[-1] // self.hop_length
            m = audio.reshape(1, 1, L, self.hop_length).mean(-1).expand(1, self.latent_dim, L).contiguous()
            logs = torch.zeros_like(m)
            return m + noise * torch.exp(logs), m, logs

    paths = []
    for i in range(5):
        p = tmp_path / f"clip{i}.pt"
        torch.save(torch.linspace(-2, 2, 1000 + 300 * i), p)
        paths.append(str(p))
    g = torch.Generator().manual_seed(0)
    recs = pipeline.extract_latents(paths, torch.load, FakeEncoder(), "cpu", rank=1, world_size=2, generator=g)
    assert [os.path.basename(p) for p, _ in recs] == ["clip2_latent2x.pt", "clip3_latent2x.pt", "clip4_latent2x.pt"]
    path, rec = recs[0]
    saved = torch.load(path)
    assert set(saved) == {"z", "mu", "logs", "sample_rate", "compression_ratio", "original_duration", "original_samples",
                          "latent_shape", "original_path"}
    assert saved["compression_ratio"] == 480 and saved["original_samples"] == 1600 and saved["latent_shape"] == [80, 4]
    assert saved["mu"].shape == (80, 4) and float(saved["mu"].abs().max()) <= 1.0  # clamped to [-1, 1] before encoding


def test_pipeline_state_dict_schema_matches_reference(golden_dir):
    """The CausalMaskedDiffWithXvec drop-in (front half + speaker encoder + CFM) exposes the unmodified reference module's
    state_dict keys and shapes, and loads such a checkpoint strictly."""
    keys = json.load(open(os.path.join(golden_dir, "pipeline_keys.json")))
    from minimax_speech_b200.flow import CausalConditionalCFM, CausalConditionalDecoder
    from minimax_speech_b200.front import CausalMaskedDiffWithXvec
    est = CausalConditionalDecoder(**synth.PIPE_EST)
    cfm = CausalConditionalCFM(240, dict(t_scheduler="cosine", inference_cfg_rate=0.7), 1, 80, est)
    m = CausalMaskedDiffWithXvec(use_speaker_encoder=True, decoder=cfm)
    assert {k: list(v.shape) for k, v in m.state_dict().items()} == keys
    fsd, esd, ssd = synth.pipeline_state_dicts()
    full = dict(fsd)
    full.update({"decoder.estimator." + k: v for k, v in esd.items()})
    full.update({"speaker_encoder." + k: v for k, v in ssd.items()})
    m.load_state_dict(full, strict=True)
    assert torch.equal(m.state_dict()["speaker_encoder.attn.3.qkv.weight"], ssd["attn.3.qkv.weight"])
    with pytest.raises(RuntimeError):
        m.inference(torch.zeros(1, 8, dtype=torch.int64), None, torch.zeros(1, 0, dtype=torch.int64), None,
                    torch.zeros(1, 0, 80), None, finalize=True)  # CPU tensors are rejected, not emulated


def test_header_is_plain_c(tmp_path):
    """The drop-in boundary is a C ABI: include/ls_b200.h must compile as C99 (no torch / C++ types in the signatures), and a
    C translation unit that only includes it must link against the library."""
    import shutil
    import subprocess
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("no gcc")
    hdr = os.path.join(ROOT, "include", "ls_b200.h")
    subprocess.run([gcc, "-std=c99", "-Wall", "-Werror", "-fsyntax-only", "-x", "c", hdr], check=True)
    src = tmp_path / "use.c"
    src.write_text('#include "ls_b200.h"\nint main(void) { return ls_abi_version() == LS_ABI_VERSION ? 0 : 1; }\n')
    lib = build.build()
    exe = tmp_path / "use"
    subprocess.run([gcc, "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), lib, "-o", str(exe),
                    "-Wl,-rpath," + os.path.dirname(lib)], check=True)
    assert subprocess.run([str(exe)]).returncode == 0


def test_bench_dump_outputs(tmp_path, monkeypatch):
    """bench.py --dump-outputs: float32 .npy per output, whole when it fits its share of the byte budget, else a seeded
    sample of the same positions on every run."""
    import numpy as np
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 800)
    small, large = torch.randn(2, 1, 10, dtype=torch.float64), torch.arange(1000.0).reshape(1, 1, 1000)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"small": small, "large": large})
    s = np.load(tmp_path / "a" / "small.npy")
    assert s.dtype == np.float32 and s.shape == (2, 1, 10) and np.array_equal(s, small.float().numpy())
    la, lb = np.load(tmp_path / "a" / "large.npy"), np.load(tmp_path / "b" / "large.npy")
    assert la.dtype == np.float32 and 0 < la.size <= 100 and np.array_equal(la, lb)
    assert np.all(np.diff(la) > 0) and np.all(la == np.round(la)) and la.max() < 1000  # distinct elements, in order


def test_tblock_wide_ring_protocol():
    """The table-driven weight ring of csrc/tblock.cu (TBLOCK_WIDE_FF): no producer warp can alias a parity wait, and a
    randomised simulation of the real wait conditions neither overwrites an unconsumed box nor deadlocks."""
    import profiles.ring_protocol_sim as sim
    for mode in ("head", "tail0", "tail1"):
        assert sim.static_invariant(mode) == 0
        for seed in range(4):
            assert sim.simulate(mode, tiles=3, seed=seed) == "ok"
