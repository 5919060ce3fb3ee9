"""ctypes binding of include/ls_b200.h.  There is no fallback: if the CUDA library cannot be loaded
(or built with nvcc) every entry point raises."""
import ctypes as C
import os
import threading

import numpy as np
import torch

from . import build as _build

LS_OK = 0
ACT_NONE, ACT_LRELU, ACT_GELU, ACT_LN_MISH, ACT_LRELU_TANH = range(5)
OUT_NONE, OUT_F32, OUT_BF16 = range(3)
OUT1_NONE, OUT1_LN, OUT1_COPY, OUT1_SNAKE = range(4)

EXPORTS = ["ls_abi_version", "ls_last_error", "ls_device_check", "ls_flow_create", "ls_flow_create_fp16", "ls_flow_create_fp32", "ls_dac_create_fp32", "ls_dac_create_fp16", "ls_dac_encode",
           "ls_dac_encode_lengths",
           "ls_front_create", "ls_front_create_fp32", "ls_front_destroy", "ls_front_encode", "ls_front_encode_sessions",
           "ls_speaker_create", "ls_speaker_create_fp32", "ls_speaker_destroy", "ls_speaker_encode",
           "ls_s3_create", "ls_s3_create_fp32", "ls_s3_destroy", "ls_s3_code_frames", "ls_s3_quantize", "ls_s3_log_mel",
           "ls_resampler_create", "ls_resampler_destroy", "ls_resample", "ls_resample_taps", "ls_latent_resize_linear",
           "ls_flow_destroy",
           "ls_flow_estimator_forward", "ls_flow_solve", "ls_dac_create", "ls_dac_destroy", "ls_dac_hop_length",
           "ls_dac_decode", "ls_synthesize_host", "ls_fsq_encode", "ls_mask_to_lengths", "ls_graph_create", "ls_graph_buffer",
           "ls_graph_launch", "ls_graph_kernel_count", "ls_graph_destroy", "ls_launch_count", "ls_debug_set_buffer", "ls_profile_begin", "ls_profile_end", "ls_test_conv_gemm", "ls_test_attention", "ls_test_tblock",
           "ls_test_groupnorm_mish"]


class LsTensor(C.Structure):
    _fields_ = [("name", C.c_char_p), ("data", C.c_void_p), ("ndim", C.c_int32), ("shape", C.c_int64 * 4)]


class ConvGemmDesc(C.Structure):
    _fields_ = [
        ("a0", C.c_void_p), ("a1", C.c_void_p), ("w", C.c_void_p),
        ("a0_C", C.c_int32), ("a1_C", C.c_int32), ("T_in", C.c_int32), ("K", C.c_int32),
        ("B", C.c_int32), ("M", C.c_int32), ("N", C.c_int32), ("block_n", C.c_int32),
        ("taps", C.c_int32), ("dil", C.c_int32), ("pad", C.c_int32),
        ("lengths", C.c_void_p),
        ("m_len_mul", C.c_int32), ("m_len_add", C.c_int32), ("skip_halo", C.c_int32),
        ("chan_mod", C.c_int32),
        ("bias", C.c_void_p),
        ("act", C.c_int32),
        ("ln_g", C.c_void_p), ("ln_b", C.c_void_p),
        ("temb", C.c_void_p), ("temb_bstride", C.c_int64),
        ("addend", C.c_void_p), ("addend_dtype", C.c_int32),
        ("out0", C.c_void_p), ("out0_dtype", C.c_int32),
        ("out1", C.c_void_p), ("out1_mode", C.c_int32),
        ("p1_a", C.c_void_p), ("p1_b", C.c_void_p),
        ("n_store", C.c_int32),
        ("out_ld", C.c_int64), ("out_shift", C.c_int64), ("out_bstride", C.c_int64), ("out_alloc", C.c_int64),
        ("out_valid_mul", C.c_int64),
        ("fp16", C.c_int32),  # 0 (the default of a fresh descriptor): bf16 operands; 1: fp16
        ("zero_skipped", C.c_int32),
        # fused residual GEMM (res_w set): a 1x1 convolution of res_a0 (| res_a1) added in the epilogue
        ("res_a0", C.c_void_p), ("res_a1", C.c_void_p), ("res_a0_C", C.c_int32), ("res_a1_C", C.c_int32),
        ("res_w", C.c_void_p), ("res_K", C.c_int32), ("res_bias", C.c_void_p),
    ]


class ProfileEntry(C.Structure):
    _fields_ = [("launches", C.c_int64), ("ms", C.c_double), ("flops", C.c_double), ("bytes", C.c_double)]


PROFILE_KINDS = ["conv_gemm_estimator", "attention", "conv_gemm_dac", "bandwidth", "tblock_estimator"]

_lib = None
_lock = threading.Lock()


def lib_path():
    return _build.LIB


def load():
    """Load the library, building it first when the .so is missing or was built from other sources (content hash of
    csrc/ + the header, see build.is_stale).  LS_NO_REBUILD=1 loads a stale library as is, with a warning."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        path = _build.LIB
        if _build.is_stale():
            if os.path.exists(path) and os.environ.get("LS_NO_REBUILD") == "1":
                import warnings
                warnings.warn(f"{path} was not built from the current csrc/ (LS_NO_REBUILD=1: loading it anyway)")
            else:
                _build.build()
        try:
            lib = C.CDLL(path)
        except OSError as e:
            raise RuntimeError(f"cannot load {path}: {e}.  The hot path has no CPU or PyTorch fallback; "
                               "build it with `python minimax-speech_b200/build.py`.") from e
        vp, i32, i64, f32 = C.c_void_p, C.c_int32, C.c_int64, C.c_float
        lib.ls_abi_version.restype = i32
        lib.ls_last_error.restype = C.c_char_p
        lib.ls_launch_count.restype = i64
        lib.ls_device_check.argtypes = [i32, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32)]
        lib.ls_flow_create.argtypes = [C.POINTER(LsTensor), i32, i32, C.POINTER(vp)]
        lib.ls_flow_create_fp32.argtypes = [C.POINTER(LsTensor), i32, i32, C.POINTER(vp)]
        lib.ls_flow_create_fp16.argtypes = [C.POINTER(LsTensor), i32, i32, C.POINTER(vp)]
        lib.ls_dac_create_fp32.argtypes = [C.POINTER(LsTensor), i32, i32, C.POINTER(vp)]
        lib.ls_dac_create_fp16.argtypes = [C.POINTER(LsTensor), i32, i32, C.POINTER(vp)]
        lib.ls_flow_destroy.argtypes = [vp]
        lib.ls_flow_destroy.restype = None
        lib.ls_flow_estimator_forward.argtypes = [vp] * 8 + [i32, i32, i32, vp]
        lib.ls_flow_solve.argtypes = [vp, vp, vp, vp, vp, vp, i64, vp, i32, f32, f32, i32, vp, i32, i32, vp]
        lib.ls_dac_create.argtypes = [C.POINTER(LsTensor), i32, i32, C.POINTER(vp)]
        lib.ls_dac_destroy.argtypes = [vp]
        lib.ls_dac_destroy.restype = None
        lib.ls_dac_hop_length.argtypes = [vp]
        lib.ls_dac_decode.argtypes = [vp, vp, vp, vp, i32, i32, vp]
        lib.ls_dac_encode.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, vp]
        lib.ls_dac_encode_lengths.argtypes = [vp, vp, vp, vp, vp, vp, vp, i32, i32, vp]
        lib.ls_front_create.argtypes = [C.POINTER(LsTensor), i32, i32, C.POINTER(vp)]
        lib.ls_front_create_fp32.argtypes = [C.POINTER(LsTensor), i32, i32, C.POINTER(vp)]
        lib.ls_front_destroy.argtypes = [vp]
        lib.ls_front_destroy.restype = None
        lib.ls_front_encode.argtypes = [vp, vp, vp, vp, vp, i32, i32, i32, i32, vp, vp]
        lib.ls_front_encode_sessions.argtypes = [vp, vp, vp, vp, vp, i32, i32, i32, vp, vp, i32, vp]
        lib.ls_speaker_create.argtypes = [C.POINTER(LsTensor), i32, i32, C.POINTER(vp)]
        lib.ls_speaker_create_fp32.argtypes = [C.POINTER(LsTensor), i32, i32, C.POINTER(vp)]
        lib.ls_speaker_destroy.argtypes = [vp]
        lib.ls_speaker_destroy.restype = None
        lib.ls_speaker_encode.argtypes = [vp, vp, vp, i32, i32, i32, vp]
        lib.ls_s3_create_fp32.argtypes = [C.POINTER(LsTensor), i32, i32, C.POINTER(vp)]
        lib.ls_s3_create.argtypes = [C.POINTER(LsTensor), i32, i32, C.POINTER(vp)]
        lib.ls_s3_destroy.argtypes = [vp]
        lib.ls_s3_destroy.restype = None
        lib.ls_s3_code_frames.argtypes = [i32]
        lib.ls_s3_quantize.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, vp]
        lib.ls_s3_log_mel.argtypes = [vp, vp, vp, i32, vp, vp, i32, i64, vp]
        pi32 = C.POINTER(i32)
        lib.ls_resampler_create.argtypes = [i32, i32, i32, C.POINTER(vp)]
        lib.ls_resampler_destroy.argtypes = [vp]
        lib.ls_resampler_destroy.restype = None
        lib.ls_resample.argtypes = [vp, vp, vp, vp, vp, i32, i64, i64, vp]
        lib.ls_resample_taps.argtypes = [i32, i32, pi32, pi32, pi32, pi32, vp, vp, vp]
        lib.ls_latent_resize_linear.argtypes = [vp, vp, vp, vp, i32, i32, i32, i32, vp]
        lib.ls_synthesize_host.argtypes =[vp, vp, vp, vp, vp, vp, vp, i64, vp, i32, f32, f32, vp, i32, i32, vp]
        lib.ls_mask_to_lengths.argtypes = [vp, vp, i32, i32, vp]
        lib.ls_fsq_encode.argtypes = [vp, vp, vp, vp, i64, i32, vp]
        lib.ls_graph_create.argtypes = [vp, vp, vp, i64, vp, i32, f32, f32, i32, i32, i32, vp, C.POINTER(vp)]
        lib.ls_graph_buffer.argtypes = [vp, i32]
        lib.ls_graph_buffer.restype = vp
        lib.ls_graph_launch.argtypes = [vp, vp]
        lib.ls_graph_kernel_count.argtypes = [vp]
        lib.ls_graph_kernel_count.restype = i64
        lib.ls_graph_destroy.argtypes = [vp]
        lib.ls_graph_destroy.restype = None
        lib.ls_debug_set_buffer.argtypes = [vp, i64]
        lib.ls_profile_end.argtypes = [C.POINTER(ProfileEntry), i32]
        lib.ls_test_tblock.argtypes = [vp] * 10 + [i32, i32, i32, i32, i32, i32, vp, vp]
        lib.ls_test_groupnorm_mish.argtypes = [vp, vp, vp, vp, vp, i64, vp, vp, vp, i32, i32, i32, i32, vp, i32, vp]
        lib.ls_test_conv_gemm.argtypes = [C.POINTER(ConvGemmDesc), i32, vp, vp]
        lib.ls_test_attention.argtypes = [vp, vp, vp, i32, i32, i32, i32, i32, vp, i64, i64, vp]
        for name in EXPORTS:
            fn = getattr(lib, name)
            if fn.restype is C.c_int:
                fn.restype = i32
        # the kernel test hooks' SM count and plan arguments (just before the stream) are optional for Python callers
        lib.ls_test_conv_gemm = _plan_args_optional(lib.ls_test_conv_gemm, 1)
        lib.ls_test_tblock = _tblock_args_optional(lib.ls_test_tblock)
        # ... and so are the attention hook's fp16 flag and bias arguments (bf16, no bias)
        lib.ls_test_attention = _attention_args_optional(lib.ls_test_attention)
        _lib = lib
        return lib


def _plan_args_optional(fn, n_fixed):
    """fn(fixed..., num_sms, plan_out, stream) also callable as fn(fixed..., stream): the device's SM count, no plan"""
    def call(*args):
        if len(args) == n_fixed + 1:
            args = args[:-1] + (0, None, args[-1])
        return fn(*args)
    call.__name__ = fn.__name__
    return call


def _tblock_args_optional(fn):
    """fn(13 fixed, fp16, no_skip, num_sms, plan_out, stream) also callable as fn(13 fixed, num_sms, plan_out, stream) and
    fn(13 fixed, stream): bf16 operands, padding-only tiles skipped (and the device's SM count, no plan)"""
    def call(*args):
        if len(args) == 14:
            args = args[:-1] + (0, None, args[-1])
        if len(args) == 16:
            args = args[:13] + (0, 0) + args[13:]
        return fn(*args)
    call.__name__ = fn.__name__
    return call


def _attention_args_optional(fn):
    """fn(qkv, out, lengths, B, T, H, chunk, fp16, bias, bias_ld, bias_bh, stream) also callable as
    fn(qkv, out, lengths, B, T, H, chunk, stream): bf16 operands, no bias"""
    def call(*args):
        if len(args) == 8:
            args = args[:-1] + (0, None, 0, 0, args[-1])
        return fn(*args)
    call.__name__ = fn.__name__
    return call


def check(code, what):
    if code != LS_OK:
        msg = load().ls_last_error()
        raise RuntimeError(f"{what} failed (code {code}): {msg.decode() if msg else ''}")


def profile_begin():
    check(load().ls_profile_begin(), "ls_profile_begin")


def profile_end():
    arr = (ProfileEntry * len(PROFILE_KINDS))()
    check(load().ls_profile_end(arr, len(PROFILE_KINDS)), "ls_profile_end")
    return {k: dict(launches=int(e.launches), ms=float(e.ms), flops=float(e.flops), bytes=float(e.bytes))
            for k, e in zip(PROFILE_KINDS, arr)}


def launch_count():
    return int(load().ls_launch_count())


def current_stream_ptr(device=None):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def tensor_table(state_dict):
    """state_dict (any device/dtype) -> (ctypes array of LsTensor, keep-alive list) over host fp32 copies."""
    keep, arr = [], (LsTensor * len(state_dict))()
    for i, (k, v) in enumerate(state_dict.items()):
        a = np.ascontiguousarray(v.detach().to("cpu", torch.float32).numpy())
        name = k.encode()
        keep.append((a, name))
        arr[i].name = name
        arr[i].data = a.ctypes.data
        arr[i].ndim = a.ndim
        if a.ndim > 4:
            raise ValueError(f"{k}: more than 4 dims")
        for d in range(a.ndim):
            arr[i].shape[d] = a.shape[d]
    return arr, keep


def check_precision(precision, fp16_ok=False):
    """"bf16": tensor-core path (bf16 operands, fp32 accumulation; latents within about 1e-2 of the fp32 reference);
    "fp16" (the flow estimator and the DAC-VAE decoder / encoder, callers pass fp16_ok=True): the same tensor-core path
    with fp16 operands -- the reference's own half-precision format -- with 3 more mantissa bits, at the speed of bf16
    for the flow estimator and 1-5 % slower for the DAC (DESIGN section 2);
    "fp32": validation mode, fp32 end to end on the CUDA cores (within 1e-4)."""
    if precision not in ("bf16", "fp16", "fp32"):
        raise ValueError(f"precision must be 'bf16', 'fp16' or 'fp32', not {precision!r}")
    if precision == "fp16" and not fp16_ok:
        raise ValueError("precision='fp16' (fp16 GEMM operands) is available for the flow estimator "
                         "(CausalConditionalDecoder) and the DAC-VAE decoder / encoder (DACVAEDecoder, DACVAEEncoder) only")
    return precision


class FlowHandle:
    """Owns an ls_flow*: the packed estimator weights + workspace on one device."""

    def __init__(self, state_dict, device, precision="bf16"):
        lib = load()
        self.device = torch.device(device)
        self.precision = check_precision(precision, fp16_ok=True)
        arr, keep = tensor_table(state_dict)
        h = C.c_void_p()
        create = {"bf16": lib.ls_flow_create, "fp16": lib.ls_flow_create_fp16, "fp32": lib.ls_flow_create_fp32}[precision]
        with torch.cuda.device(self.device):
            check(create(arr, len(state_dict), self.device.index or 0, C.byref(h)), "ls_flow_create")
        self._h = h
        from . import ops
        self.key = ops.register_handle(self)  # the handle argument of torch.ops.ls_b200.*

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h and _lib is not None:
            _lib.ls_flow_destroy(h)

    def estimator_forward(self, x, mask, mu, t, spks, cond, streaming=False, out=None):
        rows, _, T = x.shape
        out = torch.empty_like(x) if out is None else out
        check(load().ls_flow_estimator_forward(self._h, ptr(x), ptr(mask), ptr(mu), ptr(t), ptr(spks), ptr(cond),
                                               ptr(out), rows, T, int(bool(streaming)),
                                               current_stream_ptr(self.device)), "ls_flow_estimator_forward")
        return out

    def solve(self, mu, mask, spks, cond, noise, t_span, temperature, cfg_rate, streaming=False):
        B, F, T = mu.shape
        out = torch.empty(B, F, T, device=mu.device, dtype=torch.float32)
        ts = np.ascontiguousarray(t_span, dtype=np.float32)  # (a list of Python floats holding fp32 values round-trips)
        check(load().ls_flow_solve(self._h, ptr(mu), ptr(mask), ptr(spks), ptr(cond), ptr(noise),
                                   noise.stride(-2), C.c_void_p(ts.ctypes.data), len(ts) - 1, float(temperature),
                                   float(cfg_rate), int(bool(streaming)), ptr(out), B, T,
                                   current_stream_ptr(self.device)), "ls_flow_solve")
        return out


class FrontHandle:
    """Owns an ls_front*: the token -> mu front half (tensor-core path or fp32 mode)."""

    def __init__(self, state_dict, device, precision="bf16"):
        lib = load()
        self.device = torch.device(device)
        self.precision = check_precision(precision)
        arr, keep = tensor_table(state_dict)
        h = C.c_void_p()
        create = lib.ls_front_create_fp32 if self.precision == "fp32" else lib.ls_front_create
        with torch.cuda.device(self.device):
            check(create(arr, len(state_dict), self.device.index or 0, C.byref(h)), "ls_front_create")
        self._h = h
        self.out_dim = int(state_dict["encoder_proj.weight"].shape[0])

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h and _lib is not None:
            _lib.ls_front_destroy(h)

    def encode(self, tokens, embedding, n_context=0, streaming=False, token_len=None):
        B, T = tokens.shape
        mu = torch.empty(B, self.out_dim, 2 * (T - n_context), device=tokens.device, dtype=torch.float32)
        spks = torch.empty(B, self.out_dim, device=tokens.device, dtype=torch.float32)
        check(load().ls_front_encode(self._h, ptr(tokens), ptr(embedding), ptr(mu), ptr(spks), B, T, int(n_context),
                                     int(bool(streaming)), ptr(token_len) if token_len is not None else None,
                                     current_stream_ptr(self.device)), "ls_front_encode")
        return mu, spks

    def encode_sessions(self, tokens, embedding, T, token_len, n_context, streaming=False):
        """Session mode (ls_front_encode_sessions): token_len / n_context are int32 device tensors [B]; mu [B,80,2T]."""
        B, T_all = tokens.shape
        mu = torch.empty(B, self.out_dim, 2 * T, device=tokens.device, dtype=torch.float32)
        spks = torch.empty(B, self.out_dim, device=tokens.device, dtype=torch.float32)
        check(load().ls_front_encode_sessions(self._h, ptr(tokens), ptr(embedding), ptr(mu), ptr(spks), B, T_all, int(T),
                                              ptr(token_len), ptr(n_context), int(bool(streaming)),
                                              current_stream_ptr(self.device)), "ls_front_encode_sessions")
        return mu, spks


class SpeakerHandle:
    """Owns an ls_speaker*: LearnableSpeakerEncoder (tensor-core path or fp32 mode)."""

    def __init__(self, state_dict, device, precision="fp32"):
        lib = load()
        self.device = torch.device(device)
        self.precision = check_precision(precision)
        arr, keep = tensor_table(state_dict)
        h = C.c_void_p()
        create = lib.ls_speaker_create_fp32 if self.precision == "fp32" else lib.ls_speaker_create
        with torch.cuda.device(self.device):
            check(create(arr, len(state_dict), self.device.index or 0, C.byref(h)), "ls_speaker_create")
        self._h = h
        self.out_dim = int(state_dict["output_proj.weight"].shape[0])

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h and _lib is not None:
            _lib.ls_speaker_destroy(h)

    def encode(self, mel):
        """mel [n_refs, B, 80, T] (contiguous) -> [B, out_dim]"""
        n_refs, B, _, T = mel.shape
        emb = torch.empty(B, self.out_dim, device=mel.device, dtype=torch.float32)
        check(load().ls_speaker_encode(self._h, ptr(mel), ptr(emb), B, T, n_refs, current_stream_ptr(self.device)),
              "ls_speaker_encode")
        return emb


S3_PRECISIONS = ("fp32", "bf16x3")


def check_s3_precision(precision):
    """The S3 tokenizer's precisions: "fp32" (CUDA cores) or "bf16x3" (tensor cores, every GEMM operand split into a bf16
    high and low part: fp32-level error).  A token is a rounding decision, so plain 16-bit operands are refused."""
    if precision in ("bf16", "fp16"):
        raise ValueError(f"precision={precision!r} is not offered for the S3 tokenizer: 16-bit GEMM operands move the "
                         "encoder output by about 5e-3 (rel-L2), and about 2 % of tokens change (801 of 820 identical "
                         "with bf16 operands); use 'bf16x3' (tensor cores, fp32-level error) or 'fp32'")
    if precision not in S3_PRECISIONS:
        raise ValueError(f"precision must be 'fp32' or 'bf16x3', not {precision!r}")
    return precision


class S3Handle:
    """Owns an ls_s3*: S3TokenizerV2, fp32 mode or the bf16x3 tensor-core mode."""

    def __init__(self, state_dict, device, precision="fp32"):
        lib = load()
        self.device = torch.device(device)
        self.precision = check_s3_precision(precision)
        arr, keep = tensor_table(state_dict)
        h = C.c_void_p()
        create, name = (lib.ls_s3_create, "ls_s3_create") if precision == "bf16x3" else (lib.ls_s3_create_fp32, "ls_s3_create_fp32")
        with torch.cuda.device(self.device):
            check(create(arr, len(state_dict), self.device.index or 0, C.byref(h)), name)
        self._h = h
        self.n_state = int(state_dict["encoder.conv1.weight"].shape[0])

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h and _lib is not None:
            _lib.ls_s3_destroy(h)

    def quantize(self, mel, mel_len, want_hidden=False):
        """mel [B, n_mels, T] fp32, mel_len [B] int32 (both on the handle's device) -> codes [B, T2] int32, code_len [B] int32
        (and the encoder output [B, T2, n_state] when asked for)"""
        B, _, T = mel.shape
        T2 = int(load().ls_s3_code_frames(T))
        codes = torch.empty(B, T2, device=mel.device, dtype=torch.int32)
        code_len = torch.empty(B, device=mel.device, dtype=torch.int32)
        hidden = torch.empty(B, T2, self.n_state, device=mel.device, dtype=torch.float32) if want_hidden else None
        check(load().ls_s3_quantize(self._h, ptr(mel), ptr(mel_len), ptr(codes), ptr(code_len),
                                    ptr(hidden) if hidden is not None else None, B, T, current_stream_ptr(self.device)),
              "ls_s3_quantize")
        return (codes, code_len, hidden) if want_hidden else (codes, code_len)


class DacHandle:
    def __init__(self, state_dict, device, precision="bf16"):
        lib = load()
        self.device = torch.device(device)
        self.precision = check_precision(precision, fp16_ok=True)
        arr, keep = tensor_table(state_dict)
        h = C.c_void_p()
        create, name = {"bf16": (lib.ls_dac_create, "ls_dac_create"), "fp16": (lib.ls_dac_create_fp16, "ls_dac_create_fp16"),
                        "fp32": (lib.ls_dac_create_fp32, "ls_dac_create_fp32")}[precision]
        with torch.cuda.device(self.device):
            check(create(arr, len(state_dict), self.device.index or 0, C.byref(h)), name)
        self._h = h
        from . import ops
        self.key = ops.register_handle(self)
        self.hop_length = int(lib.ls_dac_hop_length(h))
        self.latent_dim = 80
        for k, v in state_dict.items():
            if k in ("en_conv_post.0.weight_v", "de_conv_pre.0.weight_v"):
                self.latent_dim = int(v.shape[1])

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h and _lib is not None:
            _lib.ls_dac_destroy(h)

    def encode(self, audio, noise=None, lengths=None):
        """``lengths`` (optional device int32 [B]): valid latent frames per clip of a right-padded batch."""
        B, _, S = audio.shape
        latent, L = self.latent_dim, S // self.hop_length
        z, m, logs = (torch.empty(B, latent, L, device=audio.device, dtype=torch.float32) for _ in range(3))
        check(load().ls_dac_encode_lengths(self._h, ptr(audio), ptr(lengths), ptr(noise), ptr(z), ptr(m), ptr(logs), B, S,
                                           current_stream_ptr(self.device)), "ls_dac_encode_lengths")
        return z, m, logs

    def decode(self, z, lengths=None):
        B, _, L = z.shape
        wav = torch.empty(B, 1, L * self.hop_length, device=z.device, dtype=torch.float32)
        check(load().ls_dac_decode(self._h, ptr(z), ptr(lengths), ptr(wav), B, L,
                                   current_stream_ptr(self.device)), "ls_dac_decode")
        return wav


def s3_log_mel(audio, audio_len, filters):
    """audio [B, S] float32, audio_len [B] int32, filters [n_mels, 201] float32 (all on one device, contiguous) ->
    mel [B, n_mels, S // 160] float32 (zeros past each clip's frames), mel_len [B] int32 (ls_s3_log_mel)."""
    B, S = audio.shape
    n_mels = filters.shape[0]
    mel = torch.empty(B, n_mels, S // 160, device=audio.device, dtype=torch.float32)
    mel_len = torch.empty(B, device=audio.device, dtype=torch.int32)
    check(load().ls_s3_log_mel(ptr(audio), ptr(audio_len), ptr(filters), n_mels, ptr(mel), ptr(mel_len), B, S,
                               current_stream_ptr(audio.device)), "ls_s3_log_mel")
    return mel, mel_len


def resample_taps(orig_freq, new_freq):
    """The tap table ls_resample uses for orig_freq -> new_freq (host only, no device needed): dict with the reduced
    ratio ``O`` / ``N``, torchaudio's ``width``, ``max_taps``, and numpy ``first`` [N], ``count`` [N] (int32) and ``taps``
    [N, max_taps] (float32, zero-padded).  Raises for a table over 96 KiB (``ls_resample_taps``)."""
    lib = load()
    O, N, W, M = (C.c_int32() for _ in range(4))
    check(lib.ls_resample_taps(int(orig_freq), int(new_freq), C.byref(O), C.byref(N), C.byref(W), C.byref(M), None, None, None),
          "ls_resample_taps")
    first, count = np.zeros(N.value, np.int32), np.zeros(N.value, np.int32)
    taps = np.zeros((N.value, M.value), np.float32)
    check(lib.ls_resample_taps(int(orig_freq), int(new_freq), None, None, None, None, C.c_void_p(first.ctypes.data),
                               C.c_void_p(count.ctypes.data), C.c_void_p(taps.ctypes.data)), "ls_resample_taps")
    return dict(O=O.value, N=N.value, width=W.value, max_taps=M.value, first=first, count=count, taps=taps)


class ResamplerHandle:
    """Owns an ls_resampler*: the tap table of one (orig_freq, new_freq) pair on one device."""

    def __init__(self, orig_freq, new_freq, device):
        lib = load()
        self.device = torch.device(device)
        self.orig_freq, self.new_freq = int(orig_freq), int(new_freq)
        h = C.c_void_p()
        with torch.cuda.device(self.device):
            check(lib.ls_resampler_create(self.orig_freq, self.new_freq, self.device.index or 0, C.byref(h)),
                  "ls_resampler_create")
        self._h = h

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h and _lib is not None:
            _lib.ls_resampler_destroy(h)

    def resample(self, audio, audio_len, S_out):
        """audio [B, S_in] float32, audio_len [B] int32 (device, contiguous) -> out [B, S_out], out_len [B] int32."""
        B, S_in = audio.shape
        out = torch.empty(B, S_out, device=audio.device, dtype=torch.float32)
        out_len = torch.empty(B, device=audio.device, dtype=torch.int32)
        check(load().ls_resample(self._h, ptr(audio), ptr(audio_len), ptr(out), ptr(out_len), B, S_in, int(S_out),
                                 current_stream_ptr(audio.device)), "ls_resample")
        return out, out_len


def latent_resize_linear(z, len_in, len_out, L_out):
    """z [B, C, L_in] float32, len_in / len_out [B] int32 (device) -> [B, C, L_out] (ls_latent_resize_linear)."""
    B, Cz, L_in = z.shape
    out = torch.empty(B, Cz, L_out, device=z.device, dtype=torch.float32)
    check(load().ls_latent_resize_linear(ptr(z), ptr(len_in), ptr(len_out), ptr(out), B, Cz, L_in, int(L_out),
                                         current_stream_ptr(z.device)), "ls_latent_resize_linear")
    return out


def mask_to_lengths(mask):
    """mask [B,1,T] float32 (device) -> int32 [B]: valid frames per utterance."""
    B, _, T = mask.shape
    out = torch.empty(B, device=mask.device, dtype=torch.int32)
    check(load().ls_mask_to_lengths(ptr(mask), ptr(out), B, T, current_stream_ptr(mask.device)), "ls_mask_to_lengths")
    return out


def fsq_encode(hidden, weight, bias):
    """hidden [B, T, D] float32 (device) -> int32 tokens [B, T] (FSQCodebook.encode)."""
    B, T, D = hidden.shape
    out = torch.empty(B, T, device=hidden.device, dtype=torch.int32)
    check(load().ls_fsq_encode(ptr(hidden), ptr(weight), ptr(bias), ptr(out), B * T, D, current_stream_ptr(hidden.device)),
          "ls_fsq_encode")
    return out


def _host_f32(name, t, shape):
    """Host buffers cross the C ABI as raw pointers: they must be CPU, float32, contiguous and of the expected shape
    (anything else would be copied as raw bytes)."""
    if not isinstance(t, torch.Tensor) or t.device.type != "cpu":
        raise ValueError(f"{name} must be a CPU tensor (host buffer), got {getattr(t, 'device', type(t))}")
    if tuple(t.shape) != tuple(shape):
        raise ValueError(f"{name} must have shape {tuple(shape)}, got {tuple(t.shape)}")
    if t.dtype != torch.float32 or not t.is_contiguous():
        t = t.to(torch.float32).contiguous()
    return t


def synthesize_host(flow, dac, mu, mask, spks, cond, noise_dev, t_span, temperature, cfg_rate, wav_out):
    """End-to-end call on HOST tensors (pinned preferred): copies, solve, decode and read-back inside."""
    if mu.dim() != 3:
        raise ValueError(f"mu must be [B, F, T], got {tuple(mu.shape)}")
    B, F, T = mu.shape
    mu = _host_f32("mu", mu, (B, F, T))
    mask = _host_f32("mask", mask, (B, 1, T))
    spks = _host_f32("spks", spks, (B, F))
    cond = _host_f32("cond", cond, (B, F, T))
    if not isinstance(wav_out, torch.Tensor) or wav_out.device.type != "cpu" or wav_out.dtype != torch.float32 or \
            not wav_out.is_contiguous() or tuple(wav_out.shape) != (B, 1, T * dac.hop_length):
        raise ValueError(f"wav_out must be a contiguous float32 CPU tensor [{B}, 1, {T * dac.hop_length}]")
    if noise_dev.device.type != "cuda" or noise_dev.dtype != torch.float32 or noise_dev.stride(-1) != 1:
        raise ValueError("noise must be a float32 CUDA tensor with a contiguous last dim")
    ts = np.ascontiguousarray(t_span, dtype=np.float32)
    check(load().ls_synthesize_host(flow._h, dac._h, ptr(mu), ptr(mask), ptr(spks), ptr(cond), ptr(noise_dev),
                                    noise_dev.stride(-2), C.c_void_p(ts.ctypes.data), len(ts) - 1,
                                    float(temperature), float(cfg_rate), ptr(wav_out), B, T,
                                    current_stream_ptr(flow.device)), "ls_synthesize_host")
    return wav_out


class GraphHandle:
    """Owns an ls_graph*: one (B, T, n_timesteps) solve (+ decode) captured as a CUDA graph over static buffers."""

    def __init__(self, flow, dac, noise_dev, t_span, temperature, cfg_rate, streaming, B, T):
        lib = load()
        self.flow, self.dac, self.noise = flow, dac, noise_dev  # keep the handles and the noise buffer alive
        self.device = flow.device
        ts = np.ascontiguousarray(t_span, dtype=np.float32)
        h = C.c_void_p()
        with torch.cuda.device(self.device):
            check(lib.ls_graph_create(flow._h, dac._h if dac is not None else None, ptr(noise_dev), noise_dev.stride(-2),
                                      C.c_void_p(ts.ctypes.data), len(ts) - 1, float(temperature), float(cfg_rate),
                                      int(bool(streaming)), B, T, current_stream_ptr(self.device), C.byref(h)),
                  "ls_graph_create")
        self._h = h
        F = 80
        hop = dac.hop_length if dac is not None else 0
        shapes = [(B, F, T), (B, 1, T), (B, F), (B, F, T), (B, F, T), (B, 1, T * hop)]
        self.buffers = []
        for i, shp in enumerate(shapes):
            p = lib.ls_graph_buffer(h, i)
            self.buffers.append(_wrap_device_f32(p, shp, self.device) if p else None)
        self.kernels = int(lib.ls_graph_kernel_count(h))

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h and _lib is not None:
            _lib.ls_graph_destroy(h)

    def launch(self):
        check(load().ls_graph_launch(self._h, current_stream_ptr(self.device)), "ls_graph_launch")


class _CudaArray:
    """__cuda_array_interface__ view of library-owned device memory (no copy, no ownership)."""

    def __init__(self, p, shape):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": "<f4", "data": (int(p), False), "version": 3,
                                         "strides": None}


def _wrap_device_f32(p, shape, device):
    with torch.cuda.device(device):
        return torch.as_tensor(_CudaArray(p, shape), device=device)
