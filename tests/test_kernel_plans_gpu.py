"""Launch plans of the persistent tensor-core kernels, at a chosen SM count.

conv_gemm and the fused transformer-block kernel (tblock) are persistent: CTA c walks tiles c, c + grid, ...  How many
tiles a CTA gets decides the plan `launch_conv_gemm` picks (streamed or resident weights, one or two MMA-issuing warps),
and from its second tile on a CTA runs code its first tile never reaches (the second TMEM accumulator, the LayerNorm
statistics area of the other parity, the wrap of every mbarrier ring, dual-issue pairs formed across skipped tiles).
The test hooks take the SM count the launch plans for, so small shapes reach the plans full-size launches take, and
report the plan that ran; every case asserts it.

Checks, for every case at every SM count:
  * against a float64 reference on the same 16-bit operands, PER TILE (item, 128-row tile, N tile), so that one wrong
    tile cannot hide in a whole-tensor norm;
  * bit patterns identical across SM counts (no kernel's summation order depends on the grid, DESIGN §2);
  * outputs start as NaN (or the in-place input): regions a launch must not write keep their initial bits, padding
    rows inside processed tiles are exactly zero.
"""
import ctypes as C
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

if not torch.cuda.is_available():
    pytest.skip("needs a CUDA device", allow_module_level=True)

import minimax_speech_b200.native as native  # noqa: E402

DEV = torch.device("cuda:0")
SMS = torch.cuda.get_device_properties(DEV).multi_processor_count
OUT_F16 = 3  # IEEE-half out0 / addend (kernels.h OutDtype)
PLAN_FIELDS = ("grid", "tiles_per_cta", "dual", "b_resident", "a_stages", "b_stages", "tma_out", "halo_mode")
HALO_MODE = 2  # the default activation staging (one halo box per K block)

# Bars on the per-tile error.  fp32 outputs of the GEMM: rel-L2 1e-5.  16-bit outputs that round the accumulator:
# 1 ulp of the rounded reference.  Outputs after a LayerNorm, Snake or the block kernel's bf16 intermediates: the
# worst tile measured on a B200, times 2 to 3.5 (DESIGN §2).
F32_BAR = 1e-5
BARS = {
    "ln_mish_f32": 1e-6,    # LayerNorm + Mish in fp32 (measured 2.9e-7)
    "ln_bf16": 4e-3,        # bf16 of a LayerNorm output (measured 1.7e-3: the bf16 rounding itself)
    "mish_bf16": 4e-3,      # bf16 of a LayerNorm + Mish output (measured 1.7e-3)
    "snake_bf16": 4e-3,     # bf16 of a Snake output (measured 1.7e-3)
    "tanh_f32": F32_BAR,    # tanh of the fp32 accumulator, fp32 output (measured 2.3e-7)
    "tblock_u": 3e-4,       # u'' = u + out-proj + FF2 in fp32; the reference rounds n3 and h to bf16 where the kernel
                            # does, and a last-bit difference in the fp32 statistics flips single roundings (measured 9.9e-5)
    "tblock_qkv": 4e-3,     # QKV of bf16(LayerNorm(u'')), bf16 output (measured 1.8e-3)
    "tblock_tail": 4e-3,    # bf16 copy of u'' (measured 1.7e-3)
    # the same outputs with fp16 operands (fp32 outputs keep the bars above)
    "ln_f16": 6e-4,         # fp16 of a LayerNorm output (measured 2.1e-4: the fp16 rounding itself)
    "mish_f16": 6e-4,       # fp16 of a LayerNorm + Mish output (measured 2.1e-4)
    "tblock_u_f16": 7.5e-5, # u'' with the reference's fp16 roundings of n3 and h (measured 3.2e-5)
    "tblock_qkv_f16": 6e-4, # QKV of fp16(LayerNorm(u'')), fp16 output (measured 2.4e-4)
    "tblock_tail_f16": 6e-4,  # fp16 copy of u'' (measured 2.1e-4)
}

_measured = {}  # bar name -> worst per-tile error seen (printed at the end of the module)


def _note(name, v):
    _measured[name] = max(_measured.get(name, 0.0), v)


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    print("\nworst per-tile error per bar:")
    for k, v in sorted(_measured.items()):
        print(f"  {k:14s} {v:.3e}  (bar {BARS[k]:.1e})" if k in BARS else f"  {k:14s} {v}")


def bf16(t):
    return t.to(torch.bfloat16)


# the 16-bit operand format of a launch: dtype, rounding, the fp16 flag of the hooks, the suffix of its bar names
H16 = {"bf16": (torch.bfloat16, bf16, 0, ""), "fp16": (torch.float16, lambda t: t.half(), 1, "_f16")}


def bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t.view(torch.int16)


def plan_dict(plan):
    return dict(zip(PLAN_FIELDS, list(plan)))


# ------------------------------------------------------------------------------------------------ conv_gemm
def conv_gemm(a0, w, num_sms, *, M=None, block_n=None, dil=1, pad=0, lengths=None, m_len_mul=1, m_len_add=0,
              skip_halo=0, chan_mod=None, bias=None, act=0, ln=None, temb=None, addend=None, out0=None, out1=None,
              out1_mode=0, p1=None, n_store=None, out_ld=None, out_shift=0, out_bstride=None, out_alloc=None,
              out_valid_mul=None, a1=None, res=None, zero_skipped=0, fp16=0):
    """a0 [B,T,C0] (+ a1 [B,T,C1], the K split) bf16, w [taps,N,K] bf16 (fp16 = 1: both fp16); res = (res_a0,
    res_a1 or None, res_w [N][res_K], res_bias or None): the fused residual GEMM.  Returns the plan the launch used."""
    B, T_in, C0 = a0.shape
    taps, N, K = w.shape
    d = native.ConvGemmDesc()
    d.a0, d.a0_C, d.T_in = native.ptr(a0), C0, T_in
    d.a1, d.a1_C = native.ptr(a1), (a1.shape[2] if a1 is not None else 0)
    d.w, d.K = native.ptr(w), K
    d.B, d.M, d.N = B, M or T_in, N
    d.block_n = block_n or N
    d.taps, d.dil, d.pad = taps, dil, pad
    d.lengths = native.ptr(lengths)
    d.m_len_mul, d.m_len_add, d.skip_halo = m_len_mul, m_len_add, skip_halo
    d.chan_mod = chan_mod or N
    d.bias = native.ptr(bias)
    d.act = act
    d.ln_g, d.ln_b = (native.ptr(ln[0]), native.ptr(ln[1])) if ln else (C.c_void_p(0), C.c_void_p(0))
    d.temb, d.temb_bstride = native.ptr(temb), (N if temb is not None else 0)
    d.addend = native.ptr(addend)
    kind = lambda t: 0 if t is None else {torch.float32: 1, torch.bfloat16: 2, torch.float16: OUT_F16}[t.dtype]
    d.addend_dtype = kind(addend)
    d.out0, d.out0_dtype = native.ptr(out0), kind(out0)
    d.out1, d.out1_mode = native.ptr(out1), out1_mode
    d.p1_a, d.p1_b = (native.ptr(p1[0]), native.ptr(p1[1])) if p1 else (C.c_void_p(0), C.c_void_p(0))
    d.n_store = n_store or N
    d.out_ld = out_ld or N
    d.out_shift = out_shift
    d.out_bstride = out_bstride if out_bstride is not None else d.M * d.out_ld
    d.out_alloc = out_alloc if out_alloc is not None else d.M * d.out_ld
    d.out_valid_mul = out_valid_mul if out_valid_mul is not None else d.out_ld
    d.zero_skipped = zero_skipped
    if fp16:  # (a descriptor may already come with fp16 = 1)
        d.fp16 = 1
    if res is not None:
        ra0, ra1, rw, rbias = res
        d.res_a0, d.res_a0_C = native.ptr(ra0), (ra0.shape[2] if ra0 is not None else 0)
        d.res_a1, d.res_a1_C = native.ptr(ra1), (ra1.shape[2] if ra1 is not None else 0)
        d.res_w, d.res_K, d.res_bias = native.ptr(rw), rw.shape[1], native.ptr(rbias)
    plan = (C.c_int32 * 8)()
    native.check(native.load().ls_test_conv_gemm(C.byref(d), num_sms, plan, native.current_stream_ptr(DEV)),
                 "ls_test_conv_gemm")
    torch.cuda.synchronize()
    return plan_dict(plan)


def conv64(a, w, dil, pad):
    """float64 conv: a [B,T,C], w [taps,N,K] -> [B,T,N]; tap k reads row t + k*dil - pad, rows outside [0,T) are 0."""
    T = a.shape[1]
    taps = w.shape[0]
    x = F.pad(a.double().transpose(1, 2), (pad, max(0, (taps - 1) * dil - pad)))
    y = F.conv1d(x, w.double().permute(1, 2, 0).contiguous(), dilation=dil)
    return y[:, :, :T].transpose(1, 2).contiguous()


def lrelu(x):
    return torch.where(x > 0, x, 0.1 * x)


def snake(x, alpha, ialpha):
    return x + ialpha.double() * torch.sin(alpha.double() * x) ** 2


def mish(x):
    return x * torch.tanh(F.softplus(x))


class Geometry:
    """Where every element of one output of a conv_gemm launch comes from.  Output element f (flat index inside a
    batch item) is GEMM element (q, n) with q * out_ld + n + out_shift = f; its tile is (b, q // 128, n // block_n).
    state: 2 = stored value, 1 = zero (padding inside a processed tile, or every stored position of a skipped tile when
    the launch has zero_skipped = 1), 0 = never written (keeps its initial bits)."""

    def __init__(self, shape, B, M, N, block_n, lengths, m_len_mul=1, m_len_add=0, skip_halo=0, n_store=None,
                 out_ld=None, out_shift=0, out_valid_mul=None, zero_skipped=0):
        out_ld = out_ld or N
        n_store = n_store or N
        out_valid_mul = out_valid_mul if out_valid_mul is not None else out_ld
        per_item = math.prod(shape[1:])
        f = torch.arange(per_item, dtype=torch.int64)
        q = torch.div(f - out_shift, out_ld, rounding_mode="floor")
        n = (f - out_shift) - q * out_ld
        produced = (q >= 0) & (q < M) & (n < n_store)
        self.m_tiles = (M + 127) // 128
        self.n_tiles = N // block_n
        lens = lengths.cpu().long() if lengths is not None else torch.full((B,), 1 << 40, dtype=torch.int64)
        mt = torch.div(q, 128, rounding_mode="floor").clamp(0, self.m_tiles - 1)
        nt = torch.div(n, block_n, rounding_mode="floor").clamp(0, self.n_tiles - 1)
        tile = (torch.arange(B)[:, None] * self.m_tiles + mt[None]) * self.n_tiles + nt[None]
        skipped = (mt[None] * 128) >= (lens[:, None] * m_len_mul + m_len_add + skip_halo)
        valid = f[None] < (lens[:, None] * out_valid_mul)
        state = torch.where(valid, 2, 1)
        state = torch.where(skipped, 1 if zero_skipped else 0, state)
        state = torch.where(~produced[None], 0, state)
        self.shape = shape
        self.tile = tile.view(shape)
        self.state = state.view(shape).to(torch.int8)
        self.n_all = B * self.m_tiles * self.n_tiles
        # tiles that are not all padding (the kernel's tile_skipped)
        tb = torch.arange(self.n_all) // (self.m_tiles * self.n_tiles)
        tm = (torch.arange(self.n_all) // self.n_tiles) % self.m_tiles
        self.tile_real = (tm * 128) < (lens[tb] * m_len_mul + m_len_add + skip_halo)

    def real_tiles_per_cta(self, grid):
        return [int(self.tile_real[c::grid].sum()) for c in range(grid)]


def per_tile_rel(out, ref, geo):
    """max over tiles of ||out - ref|| / ||ref|| on the stored elements of each tile"""
    m = (geo.state == 2).to(DEV)
    t = geo.tile.to(DEV)[m]
    d = (out.double()[m] - ref[m]) ** 2
    r = ref[m] ** 2
    num = torch.zeros(geo.n_all, dtype=torch.float64, device=DEV).index_add_(0, t, d)
    den = torch.zeros(geo.n_all, dtype=torch.float64, device=DEV).index_add_(0, t, r)
    has = torch.zeros(geo.n_all, dtype=torch.bool, device=DEV).index_fill_(0, t.unique(), True)
    e = (num / den.clamp_min(1e-300)).sqrt()
    return float(e[has].max()) if bool(has.any()) else 0.0


def ulp_check(out16, ref, mag, geo):
    """16-bit outputs that round the fp32 accumulator: at most 1 ulp from the rounded float64 reference.  Where the
    exact value cancels to far below the magnitude of its terms (mag = sum of |terms|), the fp32 accumulation error
    (<= 2^-20 * mag here) is larger than a 16-bit ulp of the result: there the bound is that accumulation error."""
    m = (geo.state == 2).to(DEV)
    r16 = ref[m].float().to(out16.dtype)
    o = out16[m]
    order = lambda v: torch.where(v < 0, -(v & 0x7FFF), v)
    ul = (order(bits(o).int()) - order(bits(r16).int())).abs()
    near = (o.double() - ref[m]).abs() <= mag[m] * 2.0 ** -20
    bad = int(((ul > 1) & ~near).sum())
    return int(ul.max()) if ul.numel() else 0, int((ul > 1).sum()), bad


def check_masks(name, out, init_bits, geo):
    st = geo.state.to(DEV)
    b = bits(out)
    assert torch.equal(b[st == 0], init_bits[st == 0]), f"{name}: a region the launch must not write was written"
    assert bool((b[st == 1] == 0).all()), f"{name}: padding rows inside processed tiles are not exactly zero"


def run_conv_case(case, sm_counts, expect):
    """case() -> dict(launch=kwargs without outputs, outputs={name: (init tensor, geo, kind, ref, mag)}).
    Runs the launch at every SM count, checks the plan (expect(num_sms, plan_geometry) -> dict of fields), the
    numbers, the masks and bitwise identity across the SM counts; returns the plans."""
    c = case()
    first = {}
    plans = []
    for sms in sm_counts:
        outs = {k: v[0].clone() for k, v in c["outputs"].items()}
        kw = dict(c["launch"])
        for k, t in outs.items():
            kw[k] = t
        if c.get("inplace"):  # the residual is read from and written to out0
            kw["addend"] = outs["out0"]
        plan = conv_gemm(**kw, num_sms=sms)
        geo0 = next(iter(c["outputs"].values()))[1]
        want = expect(sms if sms else SMS, geo0)
        want.setdefault("halo_mode", HALO_MODE)
        grid = min(geo0.n_all, sms if sms else SMS)
        want.setdefault("grid", grid)
        want.setdefault("tiles_per_cta", -(-geo0.n_all // grid))
        got = {k: plan[k] for k in want}
        reals = geo0.real_tiles_per_cta(plan["grid"]) if plan["grid"] else []
        print(f"  {c['name']:28s} sms={sms if sms else SMS:3d} " + " ".join(f"{k}={plan[k]}" for k in PLAN_FIELDS) +
              f"  real tiles per CTA: min {min(reals)} max {max(reals)}")
        assert got == want, (c["name"], sms, plan, want)
        plans.append((sms, plan, reals))
        for k, (init, geo, kind, ref, mag) in c["outputs"].items():
            out = outs[k]
            check_masks(f"{c['name']}/{k} sms={sms}", out, bits(init), geo)
            if kind == "ulp":
                mx, n1, bad = ulp_check(out, ref, mag, geo)
                _note("ulp16 max", mx)
                _note("ulp16 >1 (cancellation)", n1)
                assert bad == 0, (c["name"], k, sms, f"{bad} elements beyond 1 ulp ({n1} > 1 ulp in all)")
            else:
                e = per_tile_rel(out, ref, geo)
                _note(kind, e)
                assert e <= BARS.get(kind, F32_BAR), (c["name"], k, sms, e)
            if k in first:
                assert torch.equal(bits(out), first[k]), f"{c['name']}/{k}: sms={sms} differs bitwise from sms={sm_counts[0]}"
            else:
                first[k] = bits(out).clone()
    return plans


def _gen(seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return lambda *s, scale=1.0: (torch.randn(*s, generator=g) * scale).to(DEV)


def _nan(*shape, dtype=torch.float32):
    return torch.full(shape, float("nan"), device=DEV, dtype=dtype)


def _lens(v):
    return torch.tensor(v, dtype=torch.int32, device=DEV)


# The DAC-style length pattern: with skip_halo = 64 and M = 1000 (8 row tiles per item, the last one partial), the
# real (not all-padding) tiles are {0}, {8, 9, 10}, {16}, {24 .. 28}: at 1, 2, 5, 7 and 8 SMs the CTAs hold even and odd
# numbers of real tiles, exactly one, and (8 SMs) none; pairs of the dual mode form across skipped tiles.
DAC_B, DAC_M, DAC_LENS, DAC_SMS = 4, 1000, [0, 300, 0, 500], [0, 1, 2, 5, 7, 8]


def _dac_conv7_case(Cc, dil, seed):
    def case():
        rn = _gen(seed)
        a = bf16(rn(DAC_B, DAC_M, Cc))
        w = bf16(rn(7, Cc, Cc, scale=(7 * Cc) ** -0.5))
        bias, alpha = rn(Cc, scale=0.1), rn(Cc, scale=0.5) + 1.0
        ialpha = 1.0 / (alpha + 1e-9)
        lengths = _lens(DAC_LENS)
        pad = 3 * dil
        y = lrelu(conv64(a, w, dil, pad) + bias.double())
        geo = Geometry((DAC_B, DAC_M, Cc), DAC_B, DAC_M, Cc, Cc, lengths, skip_halo=64)
        return dict(name=f"dac conv7 C={Cc} dil={dil}",
                    launch=dict(a0=a, w=w, dil=dil, pad=pad, lengths=lengths, skip_halo=64, bias=bias,
                                act=native.ACT_LRELU, out1_mode=native.OUT1_SNAKE, p1=(alpha, ialpha)),
                    outputs={"out1": (_nan(DAC_B, DAC_M, Cc, dtype=torch.bfloat16), geo, "snake_bf16",
                                      snake(y, alpha, ialpha), None)})
    return case


def _check_edges(plans, field):
    """the SM counts of a case must give CTAs with an even and an odd number (>= 3) of real tiles, one with exactly one
    and one with none, in the plan under test (plan[field] == 1)"""
    reals = [r for sms, plan, rr in plans if plan[field] == 1 for r in rr]
    assert any(r >= 2 and r % 2 == 0 for r in reals), "no CTA with an even number of real tiles"
    assert any(r >= 3 and r % 2 == 1 for r in reals), "no CTA with an odd number (>= 3) of real tiles"
    assert 1 in reals, "no CTA with exactly one real tile"
    assert 0 in reals, "no CTA whose tiles are all skipped"


@pytest.mark.parametrize("Cc,dil", [(48, 1), (48, 3)])
def test_resident_weights_conv7_snake(Cc, dil):
    """Thin DAC conv7 (C = 48): weights resident in shared memory from 3 tiles per CTA on, the activation loads shared
    by every producer warp."""
    def expect(sms, geo):
        tpc = -(-geo.n_all // min(geo.n_all, sms))
        if tpc >= 3:
            return dict(dual=0, b_resident=1, b_stages=7, a_stages=6, tma_out=1)
        return dict(dual=0, b_resident=0, tma_out=1)
    plans = run_conv_case(_dac_conv7_case(Cc, dil, 100 + dil), DAC_SMS, expect)
    assert any(p["b_resident"] for _, p, _ in plans) and any(not p["b_resident"] for _, p, _ in plans)
    _check_edges(plans, "b_resident")


@pytest.mark.parametrize("Cc,dil,b_stages", [(96, 9, 6), (192, 3, 3)])
def test_dual_issue_conv7_snake(Cc, dil, b_stages):
    """DAC conv7 at C = 96 / 192: two MMA warps on alternating tiles from 4 tiles per CTA on (streamed weights, every
    weight box released by both warps, a lone last tile released twice)."""
    def expect(sms, geo):
        tpc = -(-geo.n_all // min(geo.n_all, sms))
        if tpc >= 4:
            return dict(dual=1, b_resident=0, a_stages=4, b_stages=b_stages, tma_out=1)
        return dict(dual=0, b_resident=0, tma_out=1)
    plans = run_conv_case(_dac_conv7_case(Cc, dil, 200 + Cc), DAC_SMS, expect)
    assert any(p["dual"] for _, p, _ in plans) and any(not p["dual"] for _, p, _ in plans)
    _check_edges(plans, "dual")


def test_resident_conv1_inplace_f16_residual_snake():
    """DAC 1x1 conv1 (C = 96): LeakyReLU + the fp16 residual stream read and written in place, Snake of the result."""
    Cc = 96

    def case():
        rn = _gen(300)
        a = bf16(rn(DAC_B, DAC_M, Cc))
        w = bf16(rn(1, Cc, Cc, scale=Cc ** -0.5))
        bias, alpha = rn(Cc, scale=0.1), rn(Cc, scale=0.5) + 1.0
        ialpha = 1.0 / (alpha + 1e-9)
        x = (rn(DAC_B, DAC_M, Cc, scale=2.0)).half()
        lengths = _lens(DAC_LENS)
        y = lrelu(conv64(a, w, 1, 0) + bias.double()) + x.double()
        mag = lrelu(conv64(a.abs(), w.abs(), 1, 0) + bias.double().abs()) + x.double().abs()
        geo = Geometry((DAC_B, DAC_M, Cc), DAC_B, DAC_M, Cc, Cc, lengths, skip_halo=64)
        return dict(name="dac conv1 C=96 in-place x", inplace=True,
                    launch=dict(a0=a, w=w, lengths=lengths, skip_halo=64, bias=bias, act=native.ACT_LRELU,
                                out1_mode=native.OUT1_SNAKE, p1=(alpha, ialpha)),
                    outputs={"out0": (x, geo, "ulp", y, mag),
                             "out1": (_nan(DAC_B, DAC_M, Cc, dtype=torch.bfloat16), geo, "snake_bf16",
                                      snake(y, alpha, ialpha), None)})

    def expect(sms, geo):
        tpc = -(-geo.n_all // min(geo.n_all, sms))
        return dict(dual=0, b_resident=1, a_stages=6, b_stages=2, tma_out=1) if tpc >= 3 else dict(dual=0, b_resident=0,
                                                                                                   tma_out=1)
    plans = run_conv_case(case, DAC_SMS, expect)
    assert any(p["b_resident"] for _, p, _ in plans)
    _check_edges(plans, "b_resident")


def test_streamed_qkv_linear_several_n_tiles():
    """QKV-style linear K 256 -> N 1536 in 256-wide tiles (512 TMEM columns): streamed weights, one issuer, several N
    tiles and several tiles per CTA; out1 = 16-bit copy of the accumulator (1 ulp), with bf16 and with fp16 operands."""
    B, M, K, N = 3, 300, 256, 1536

    def make_case(precision):
        dt, r16, fp16, _ = H16[precision]

        def case():
            rn = _gen(400)
            a = r16(rn(B, M, K))
            w = r16(rn(1, N, K, scale=K ** -0.5))
            lengths = _lens([300, 0, 77])
            geo = Geometry((B, M, N), B, M, N, 256, lengths)
            return dict(name=f"qkv linear 256->1536 {precision}",
                        launch=dict(a0=a, w=w, block_n=256, lengths=lengths, out1_mode=native.OUT1_COPY, fp16=fp16),
                        outputs={"out1": (_nan(B, M, N, dtype=dt), geo, "ulp", conv64(a, w, 1, 0),
                                          conv64(a.abs(), w.abs(), 1, 0))})
        return case

    def expect(sms, geo):
        return dict(dual=0, b_resident=0, a_stages=3, b_stages=3, tma_out=1)
    for precision in ("bf16", "fp16"):
        plans = run_conv_case(make_case(precision), [0, 1, 2, 5, 7], expect)
        assert max(p["tiles_per_cta"] for _, p, _ in plans) >= 2


@pytest.mark.parametrize("variant,precision", [("temb_copy", "bf16"), ("addend_ln", "bf16"), ("temb_copy", "fp16"),
                                               ("addend_ln", "fp16")],
                         ids=["temb_copy", "addend_ln", "temb_copy-fp16", "addend_ln-fp16"])
def test_layernorm_epilogues_multi_tile(variant, precision):
    """Flow-estimator resnet conv (k = 3, pad 2) with the LayerNorm + Mish epilogue over several tiles per CTA: the
    statistics area alternates with the tile parity.  temb_copy: + time embedding -> 16-bit copy; addend_ln: + fp32
    residual -> fp32 out0 and 16-bit LayerNorm of it.  bf16 or fp16 operands and 16-bit outputs."""
    B, M, K, N = 3, 333, 320, 256
    dt, r16, fp16, sfx = H16[precision]

    def case():
        rn = _gen(500 + len(variant))
        a = r16(rn(B, M, K))
        w = r16(rn(3, N, K, scale=(3 * K) ** -0.5))
        bias = rn(N, scale=0.1)
        lg, lb = 1 + rn(N, scale=0.1), rn(N, scale=0.1)
        lengths = _lens([333, 0, 200])
        geo = Geometry((B, M, N), B, M, N, N, lengths)
        y = mish(F.layer_norm(conv64(a, w, 1, 2) + bias.double(), (N,), lg.double(), lb.double(), 1e-5))
        kw = dict(a0=a, w=w, pad=2, lengths=lengths, bias=bias, act=native.ACT_LN_MISH, ln=(lg, lb), fp16=fp16)
        if variant == "temb_copy":
            temb = rn(B, N)
            y = y + temb.double()[:, None, :]
            kw.update(temb=temb, out1_mode=native.OUT1_COPY)
            outputs = {"out1": (_nan(B, M, N, dtype=dt), geo, "mish_bf16" if not fp16 else "mish_f16", y, None)}
        else:
            addend = rn(B, M, N)
            g2, b2 = 1 + rn(N, scale=0.1), rn(N, scale=0.1)
            y = y + addend.double()
            y1 = F.layer_norm(y, (N,), g2.double(), b2.double(), 1e-5)
            kw.update(addend=addend, out1_mode=native.OUT1_LN, p1=(g2, b2))
            outputs = {"out0": (_nan(B, M, N), geo, "ln_mish_f32", y, None),
                       "out1": (_nan(B, M, N, dtype=dt), geo, "ln_bf16" if not fp16 else "ln_f16", y1, None)}
        return dict(name=f"resnet conv3 LN+Mish {variant} {precision}", launch=kw, outputs=outputs)

    def expect(sms, geo):
        return dict(dual=0, b_resident=0, a_stages=2, b_stages=3, tma_out=1)
    plans = run_conv_case(case, [0, 1, 2, 3, 5], expect)
    assert max(r for _, _, rr in plans for r in rr) >= 3  # both parities of the statistics area, and a wrap


@pytest.mark.parametrize("cin,cout,s,L,lens,sm_counts", [
    (96, 48, 2, 500, [0, 150, 0, 260], [0, 1, 3, 5, 8]),
    (384, 192, 4, 300, [300, 0, 90], [0, 1, 4, 7]),
])
def test_polyphase_transposed_conv_multi_tile(cin, cout, s, L, lens, sm_counts):
    """DAC up-sampling ConvTranspose1d as a two-tap GEMM over q in [0, L] (m_len_add = 1), output row q*s + phi - pad
    (negative out_shift: the stores go through the LSU path): fp16 residual stream + bf16 Snake of it."""
    B = len(lens)
    N = s * cout
    block_n = max(b for b in range(16, 257, 16) if N % b == 0)
    padT = (s + 1) // 2
    rows = L * s

    def case():
        rn = _gen(600 + s)
        x = bf16(rn(B, L, cin))
        wt = bf16(rn(cin, cout, 2 * s, scale=cin ** -0.5))  # ConvTranspose1d layout
        bias, alpha = rn(cout, scale=0.1), rn(cout, scale=0.5) + 1.0
        ialpha = 1.0 / (alpha + 1e-9)
        w = torch.zeros(2, N, cin, device=DEV, dtype=torch.bfloat16)  # polyphase packing (dac_engine.cu)
        for phi in range(s):
            w[1, phi * cout:(phi + 1) * cout] = wt[:, :, phi].t()
            w[0, phi * cout:(phi + 1) * cout] = wt[:, :, phi + s].t()
        lengths = _lens(lens)
        ct = lambda xx, ww, bb: F.conv_transpose1d(xx.double().transpose(1, 2), ww.double(), bb, stride=s, padding=padT,
                                                   output_padding=s % 2).transpose(1, 2)
        y = ct(x, wt, bias.double())
        mag = ct(x.abs(), wt.abs(), bias.double().abs())
        chan = lambda v: v.repeat(s)  # per-channel vectors indexed with n % chan_mod
        geo = Geometry((B, rows, cout), B, L + 1, N, block_n, lengths, m_len_add=1, skip_halo=64, out_shift=-padT * cout,
                       out_valid_mul=s * cout)
        return dict(name=f"transposed conv s={s}",
                    launch=dict(a0=x, w=w, M=L + 1, block_n=block_n, pad=1, lengths=lengths, m_len_add=1, skip_halo=64,
                                chan_mod=cout, bias=bias, out1_mode=native.OUT1_SNAKE, p1=(alpha, ialpha),
                                out_ld=N, out_shift=-padT * cout, out_bstride=rows * cout, out_alloc=rows * cout,
                                out_valid_mul=s * cout),
                    outputs={"out0": (_nan(B, rows, cout, dtype=torch.float16), geo, "ulp", y, mag),
                             "out1": (_nan(B, rows, cout, dtype=torch.bfloat16), geo, "snake_bf16",
                                      snake(y, alpha, ialpha), None)})

    def expect(sms, geo):
        tpc = -(-geo.n_all // min(geo.n_all, sms))
        if N == block_n and tpc >= 3:
            return dict(dual=0, b_resident=1, tma_out=0)
        return dict(dual=0, b_resident=0, tma_out=0)
    plans = run_conv_case(case, sm_counts, expect)
    assert max(p["tiles_per_cta"] for _, p, _ in plans) >= 4


def test_final_conv_tanh_mono_multi_tile():
    """DAC final conv7 (C = 48 -> 1, padded to one 16-wide tile): LeakyReLU + tanh, only column 0 stored."""
    B, T, Cc = 3, 1000, 48

    def case():
        rn = _gen(700)
        a = bf16(rn(B, T, Cc))
        w = torch.zeros(7, 16, Cc, device=DEV, dtype=torch.bfloat16)
        w[:, :1] = bf16(rn(7, 1, Cc, scale=(7 * Cc) ** -0.5))
        bias = torch.zeros(16, device=DEV)
        bias[0] = 0.05
        lengths = _lens([1000, 0, 400])
        ref = torch.tanh(lrelu(conv64(a, w[:, :1], 1, 3)[..., 0] + 0.05))
        geo = Geometry((B, T), B, T, 16, 16, lengths, skip_halo=64, n_store=1, out_ld=1, out_valid_mul=1)
        return dict(name="final conv tanh mono",
                    launch=dict(a0=a, w=w, block_n=16, pad=3, lengths=lengths, skip_halo=64, chan_mod=16, bias=bias,
                                act=native.ACT_LRELU_TANH, n_store=1, out_ld=1, out_bstride=T, out_alloc=T,
                                out_valid_mul=1),
                    outputs={"out0": (_nan(B, T), geo, "tanh_f32", ref, None)})

    def expect(sms, geo):
        tpc = -(-geo.n_all // min(geo.n_all, sms))
        return dict(dual=0, b_resident=int(tpc >= 3), tma_out=0)
    plans = run_conv_case(case, [0, 1, 3, 5], expect)
    assert max(p["tiles_per_cta"] for _, p, _ in plans) >= 3


def test_dual_issue_production_grid():
    """The dual plan at the device's own SM count: B = 4 utterances of about 15 k rows (DAC C = 96, dil 9), so every
    CTA gets 3 or 4 tiles; the same launch on a smaller grid must give the same bits."""
    B, Cc, dil = 4, 96, 9
    m_tiles = -(-int(3.25 * SMS) // B)
    M = m_tiles * 128 - 37

    def case():
        rn = _gen(800)
        a = bf16(rn(B, M, Cc))
        w = bf16(rn(7, Cc, Cc, scale=(7 * Cc) ** -0.5))
        bias, alpha = rn(Cc, scale=0.1), rn(Cc, scale=0.5) + 1.0
        ialpha = 1.0 / (alpha + 1e-9)
        lengths = _lens([M, M - 3000, 0, M // 2])
        y = lrelu(conv64(a, w, dil, 3 * dil) + bias.double())
        geo = Geometry((B, M, Cc), B, M, Cc, Cc, lengths, skip_halo=64)
        return dict(name="dual, production grid",
                    launch=dict(a0=a, w=w, dil=dil, pad=3 * dil, lengths=lengths, skip_halo=64, bias=bias,
                                act=native.ACT_LRELU, out1_mode=native.OUT1_SNAKE, p1=(alpha, ialpha)),
                    outputs={"out1": (_nan(B, M, Cc, dtype=torch.bfloat16), geo, "snake_bf16",
                                      snake(y, alpha, ialpha), None)})

    def expect(sms, geo):
        return dict(dual=1, b_resident=0, a_stages=4, b_stages=6, tma_out=1)
    plans = run_conv_case(case, [0, SMS // 2 + 3], expect)
    assert plans[0][1]["grid"] == SMS and plans[0][1]["tiles_per_cta"] >= 4


def test_conv_hook_refuses_sm_counts_outside_the_device():
    a = bf16(torch.randn(1, 128, 64, device=DEV))
    w = bf16(torch.randn(1, 64, 64, device=DEV))
    out = _nan(1, 128, 64)
    for bad in (-1, SMS + 1):
        with pytest.raises(RuntimeError, match="num_sms"):
            conv_gemm(a, w, bad, out0=out)
    assert bool(out.isnan().all())


# ------------------------------------------------------------------------------------------ fused transformer block
def _tblock_operands(R, seed, r16=bf16):
    rn = _gen(seed)
    att = r16(rn(R, 512))
    u = rn(R, 256, scale=2.0) + 0.5
    wo = r16(rn(256, 512, scale=512 ** -0.5))
    w1 = r16(rn(1024, 256, scale=256 ** -0.5))
    w2 = r16(rn(256, 1024, scale=1024 ** -0.5))
    wqkv = r16(rn(1536, 256, scale=256 ** -0.5))
    vec = torch.cat([rn(256, scale=0.1), 1 + rn(256, scale=0.1), rn(256, scale=0.1), rn(1024, scale=0.2),
                     rn(256, scale=0.1), 1 + rn(256, scale=0.1), rn(256, scale=0.1)]).contiguous()
    return att, u, wo, w1, w2, wqkv, vec


def _tblock_ref64(att, u, wo, w1, w2, wqkv, vec, head, r16=bf16):
    """float64, with the kernel's 16-bit roundings (r16: bf16 or fp16) of the FF input, the GELU output and the QKV
    input"""
    d = lambda t: t.double()
    rnd = r16
    r16 = lambda t: rnd(t.float()).double()
    bo, g3, be3, b1, b2, g1n, be1n = [d(v) for v in torch.split(vec, [256, 256, 256, 1024, 256, 256, 256])]
    if head:
        u2 = d(u)
    else:
        u1 = d(att) @ d(wo).T + bo + d(u)
        n3 = r16(F.layer_norm(u1, (256,), g3, be3, 1e-5))
        h = r16(F.gelu(n3 @ d(w1).T + b1))
        u2 = u1 + h @ d(w2).T + b2
    n1 = r16(F.layer_norm(u2, (256,), g1n, be1n, 1e-5))
    return u2, n1 @ d(wqkv).T


def _tblock_launch(ops, u, tail_mode, lengths, T, num_sms, fp16=0, no_skip=0):
    att, _, wo, w1, w2, wqkv, vec = ops
    R = att.shape[0]
    qkv = _nan(R, 1536, dtype=att.dtype) if tail_mode != 1 else None
    tail = _nan(R, 256, dtype=att.dtype) if tail_mode == 1 else None
    plan = (C.c_int32 * 2)()
    native.check(native.load().ls_test_tblock(native.ptr(att), native.ptr(u), native.ptr(wo), native.ptr(w1),
                                              native.ptr(w2), native.ptr(wqkv), native.ptr(vec), native.ptr(qkv),
                                              native.ptr(tail), native.ptr(lengths), R, T, tail_mode, fp16, no_skip,
                                              num_sms, plan, native.current_stream_ptr(DEV)), "ls_test_tblock")
    torch.cuda.synchronize()
    return qkv, tail, (plan[0], plan[1])


def _tile_rel(out, ref, rows_mask, col_block):
    """max over (128-row tile, col_block-wide column block) of rel-L2 on the rows in rows_mask"""
    R, Ncol = out.shape
    worst = 0.0
    for r0 in range(0, R, 128):
        m = rows_mask[r0:r0 + 128]
        if not bool(m.any()):
            continue
        for c0 in range(0, Ncol, col_block):
            o = out[r0:r0 + 128, c0:c0 + col_block][m].double()
            rf = ref[r0:r0 + 128, c0:c0 + col_block][m]
            worst = max(worst, float((o - rf).norm() / rf.norm().clamp_min(1e-300)))
    return worst


# T = 700 rows per item, lengths [700, 0, 130, 450, 690]: R = 3500 = 27 full tiles + a partial one (valid rows and
# padding); tiles 6 .. 9, 12 .. 15 and 20 hold only padding and lie between real tiles of the same CTA.  At 14 SMs one
# CTA has only skipped tiles and another exactly one real tile.
TB_T, TB_LENS, TB_SMS = 700, [700, 0, 130, 450, 690], [0, 1, 3, 5, 7, 14]


def tblock_plans(tail_mode, precision="bf16", no_skip=0):
    """Every SM count of TB_SMS: the plan, the initial bits of what a launch must not write, per-tile errors against
    float64 (bars tblock_* with the precision's suffix) and bitwise identity across the SM counts.  no_skip = 1: every
    tile is processed, padding rows included (row-local reference there, a zero tail).  Returns the outputs of the
    first launch (u, qkv, tail) and the row masks (valid, in_real)."""
    dt, r16, fp16, sfx = H16[precision]
    R = TB_T * len(TB_LENS)
    n_tiles = -(-R // 128)
    ops = _tblock_operands(R, 900 + tail_mode, r16)
    lengths = _lens(TB_LENS)
    u_ref, qkv_ref = _tblock_ref64(*ops, head=tail_mode == 2, r16=r16)
    row = torch.arange(R, device=DEV)
    valid = (row % TB_T) < lengths.long()[row // TB_T]
    tile_real = torch.stack([valid[t * 128:(t + 1) * 128].any() for t in range(n_tiles)])
    assert not bool(tile_real.all()) and bool(tile_real[-1])
    if no_skip:
        tile_real = torch.ones_like(tile_real)
    in_real = tile_real[row // 128]  # rows of tiles that are processed
    first = None
    all_reals = []
    for sms in TB_SMS:
        u = ops[1].clone()
        qkv, tail, (grid, tpc) = _tblock_launch(ops, u, tail_mode, lengths, TB_T, sms, fp16, no_skip)
        n = sms if sms else SMS
        reals = [int(tile_real[c::grid].sum()) for c in range(grid)]
        all_reals += reals if tpc >= 2 else []
        print(f"  tblock tail_mode={tail_mode} {precision} no_skip={no_skip} sms={n:3d} grid={grid} tiles_per_cta={tpc}"
              f"  real tiles per CTA: min {min(reals)} max {max(reals)}")
        assert (grid, tpc) == (min(n_tiles, n), -(-n_tiles // min(n_tiles, n)))
        # rows of skipped tiles keep their initial bits; u is only written in tail_mode 0
        if tail_mode == 0:
            assert torch.equal(bits(u)[~in_real], bits(ops[1])[~in_real])
            e = _tile_rel(u, u_ref, in_real, 256)
            _note("tblock_u" + sfx, e)
            assert e <= BARS["tblock_u" + sfx], (sms, e)
        else:
            assert torch.equal(bits(u), bits(ops[1]))
        if tail_mode != 1:
            assert bool(qkv[~in_real].isnan().all()) and not bool(qkv[in_real].isnan().any())
            e = _tile_rel(qkv, qkv_ref, in_real, 128)
            _note("tblock_qkv" + sfx, e)
            assert e <= BARS["tblock_qkv" + sfx], (sms, e)
            res = [bits(qkv)] + ([bits(u)] if tail_mode == 0 else [])
        else:
            assert bool(tail[~in_real].isnan().all()) and not bool(tail[in_real].isnan().any())
            assert bool((bits(tail)[in_real & ~valid] == 0).all())  # padding rows of processed tiles: zero
            e = _tile_rel(tail, u_ref, valid, 256)
            _note("tblock_tail" + sfx, e)
            assert e <= BARS["tblock_tail" + sfx], (sms, e)
            res = [bits(tail)]
        if first is None:
            first = [r.clone() for r in res]
            outs = (u, qkv, tail)
        else:
            for a_, b_ in zip(res, first):
                assert torch.equal(a_, b_), f"tblock tail_mode={tail_mode} {precision}: sms={n} differs bitwise"
    if not no_skip:
        assert 0 in all_reals and 1 in all_reals and any(r >= 3 for r in all_reals)
    return outs, valid, in_real


@pytest.mark.parametrize("tail_mode", [0, 1, 2])
def test_tblock_plans_bitwise_and_per_tile(tail_mode):
    tblock_plans(tail_mode)


def test_tblock_grid_follows_num_sms_on_every_call():
    """The grid follows the SM count of every call, not of the first one."""
    R = 128 * 20
    ops = _tblock_operands(R, 950)
    grids = []
    for sms in (3, 7, 0, 2):
        u = ops[1].clone()
        _, _, (grid, _) = _tblock_launch(ops, u, 2, None, R, sms)
        grids.append(grid)
    assert grids == [3, 7, min(20, SMS), 2]
    with pytest.raises(RuntimeError, match="num_sms"):
        _tblock_launch(ops, ops[1].clone(), 2, None, R, SMS + 1)
