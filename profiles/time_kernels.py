"""Micro-timing of single kernels through the C-ABI test hooks (CUDA events, after warm-up).  Development aid:
prints per-launch microseconds and algorithmic TFLOP/s; not a bench value."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import minimax_speech_b200.native as native

DEV = torch.device("cuda:0")


def timeit(fn, iters=20, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1000.0 / iters


def tblock(R, tail_mode=0):
    g = torch.Generator().manual_seed(0)
    rn = lambda *s, scale=1.0: (torch.randn(*s, generator=g) * scale).to(DEV)
    att = rn(R, 512).bfloat16()
    u = rn(R, 256)
    wo, w1 = rn(256, 512, scale=0.04).bfloat16(), rn(1024, 256, scale=0.06).bfloat16()
    w2, wq = rn(256, 1024, scale=0.03).bfloat16(), rn(1536, 256, scale=0.06).bfloat16()
    vec = rn(2560, scale=0.1)
    qkv = torch.empty(R, 1536, device=DEV, dtype=torch.bfloat16)
    tail = torch.empty(R, 256, device=DEV, dtype=torch.bfloat16)
    lib = native.load()
    s = native.current_stream_ptr(DEV)

    def fn():
        native.check(lib.ls_test_tblock(native.ptr(att), native.ptr(u), native.ptr(wo), native.ptr(w1), native.ptr(w2),
                                        native.ptr(wq), native.ptr(vec), native.ptr(qkv), native.ptr(tail), None, R, R,
                                        tail_mode, 0, None, s), "tblock")
    us = timeit(fn)
    macs = (0 if tail_mode == 2 else 512 * 256 + 2 * 256 * 1024) + (256 * 1536 if tail_mode != 1 else 0)
    print(f"tblock R={R} tail={tail_mode}: {us:8.1f} us  {2.0 * R * macs / us / 1e6:7.1f} TFLOP/s")


def attention(B, T, H=8):
    qkv = torch.randn(B, T, 3 * H * 64, device=DEV).bfloat16()
    out = torch.empty(B, T, H * 64, device=DEV, dtype=torch.bfloat16)
    lib = native.load()
    s = native.current_stream_ptr(DEV)

    def fn():
        native.check(lib.ls_test_attention(native.ptr(qkv), native.ptr(out), None, B, T, H, 0, s), "attention")
    us = timeit(fn)
    print(f"attention B={B} T={T}: {us:8.1f} us  {4.0 * B * H * T * T * 64 / us / 1e6:7.1f} TFLOP/s")


if __name__ == "__main__":
    for R in (16000, 96000):
        for tm in (0, 1, 2):
            tblock(R, tm)
    attention(32, 500)
    attention(64, 1500)
