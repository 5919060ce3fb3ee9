"""Kernel-level tests of the launch forms the flow estimator uses and the DAC shapes do not: the resnet's res_conv fused
into the conv2 launch (a second GEMM into the second TMEM accumulator), the zero-filled skipped tiles and symmetric
(pad 1) convolutions of the non-causal estimator, the fused block kernel's fp16 build and its no-skip mode, and the
GroupNorm + Mish kernels of the non-causal estimator's blocks.

Every case checks the plan the hook reports, outputs that start as NaN (by bit pattern), the error against a float64
reference on the same 16-bit operands per tile (or per GroupNorm group), and bitwise identity across its SM counts.
The launch-plan machinery (geometry, references, plan checks) is test_kernel_plans_gpu's."""
import types

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

if not torch.cuda.is_available():
    pytest.skip("needs a CUDA device", allow_module_level=True)

import minimax_speech_b200.native as native  # noqa: E402
import test_kernel_plans_gpu as KP  # noqa: E402  (the launch-plan test machinery)

DEV = KP.DEV
SMS = KP.SMS
bits = KP.bits

# GroupNorm + Mish in fp32, per (batch row, group) rel-L2 (measured 7.6e-6 on a B200; a one-pass fp32 variance is off
# by about 2e-3 on the item with the DC offset)
GN_BAR = 2e-5


@pytest.fixture(scope="module", autouse=True)
def _report():
    """the worst error per bar of this module's cases"""
    saved = dict(KP._measured)
    KP._measured.clear()
    yield
    print("\nworst per-tile error per bar:")
    bars = dict(KP.BARS, gn_mish_f32=GN_BAR, f32=KP.F32_BAR)
    for k, v in sorted(KP._measured.items()):
        print(f"  {k:18s} {v:.3e}  (bar {bars[k]:.1e})" if k in bars else f"  {k:18s} {v}")
    for k, v in saved.items():
        KP._note(k, v)


# ------------------------------------------------------------------------------------ A. fused residual GEMM
# The causal resnet's conv2 (3 taps, pad 2, 256 -> 256, LayerNorm + Mish, u in fp32) with res_conv riding in the same
# launch.  M = 333 gives 3 row tiles per item; lengths: a multiple of 128 (its third tile is skipped), 0, a partial last
# tile, and an item whose only real tile is its first.  12 tiles: the launch needs one CTA per tile.
RES_B, RES_T, RES_LENS = 4, 333, [256, 0, 333, 77]


def _res_operands(sources, precision, B, T, seed):
    """conv2 input h [B,T,256], w [3,256,256], bias, LayerNorm affine; residual sources (the down block's x: 320
    channels; the up block's [x | skip]: 256 + 256), res_w [256][res_K], res_bias"""
    _, r16, _, _ = KP.H16[precision]
    rn = KP._gen(seed)
    N = 256
    h = r16(rn(B, T, N))
    w = r16(rn(3, N, N, scale=(3 * N) ** -0.5))
    bias, lg, lb = rn(N, scale=0.1), 1 + rn(N, scale=0.1), rn(N, scale=0.1)
    if sources == 1:
        ra0, ra1 = r16(rn(B, T, 320)), None
    else:
        ra0, ra1 = r16(rn(B, T, 256)), r16(rn(B, T, 256))
    rk = ra0.shape[2] + (ra1.shape[2] if ra1 is not None else 0)
    rw = r16(rn(N, rk, scale=rk ** -0.5))
    rbias = rn(N, scale=0.1)
    g2, b2 = 1 + rn(N, scale=0.1), rn(N, scale=0.1)
    return h, w, bias, (lg, lb), (ra0, ra1, rw, rbias), (g2, b2)


def _res_case(sources, out1, precision, B, T, lens, seed):
    dt, _, fp16, sfx = KP.H16[precision]
    N = 256
    h, w, bias, ln, res, p1 = _res_operands(sources, precision, B, T, seed)
    ra0, ra1, rw, rbias = res
    lengths = KP._lens(lens)
    xin = ra0 if ra1 is None else torch.cat([ra0, ra1], 2)
    r = KP.conv64(xin, rw[None], 1, 0) + rbias.double()
    y = KP.mish(F.layer_norm(KP.conv64(h, w, 1, 2) + bias.double(), (N,), ln[0].double(), ln[1].double(), 1e-5)) + r
    geo = KP.Geometry((B, T, N), B, T, N, N, lengths)
    kw = dict(a0=h, w=w, pad=2, lengths=lengths, bias=bias, act=native.ACT_LN_MISH, ln=ln, fp16=fp16)
    outputs = {"out0": (KP._nan(B, T, N), geo, "ln_mish_f32", y, None)}
    if out1:
        y1 = F.layer_norm(y, (N,), p1[0].double(), p1[1].double(), 1e-5)
        kw.update(out1_mode=native.OUT1_LN, p1=p1)
        outputs["out1"] = (KP._nan(B, T, N, dtype=dt), geo, "ln_bf16" if not fp16 else "ln" + sfx, y1, None)
    name = f"res_conv fused {sources} src {'OUT1_LN' if out1 else 'OUT1_NONE'} {precision}"
    return dict(name=name, launch=dict(kw, res=res), outputs=outputs), kw, res


def _unfused(kw, res, outputs):
    """the engine's two-launch form: res_conv (1x1, bias, fp32 out0), then conv2 with it as an fp32 addend"""
    ra0, ra1, rw, rbias = res
    B, T, _ = kw["a0"].shape
    r = KP._nan(B, T, rw.shape[0])
    KP.conv_gemm(ra0, rw[None], 0, a1=ra1, lengths=kw["lengths"], bias=rbias, out0=r, fp16=kw["fp16"])
    outs = {k: v[0].clone() for k, v in outputs.items()}
    KP.conv_gemm(num_sms=0, addend=r, **kw, **outs)
    return outs


def _fused(launch, outputs, num_sms):
    outs = {k: v[0].clone() for k, v in outputs.items()}
    plan = KP.conv_gemm(num_sms=num_sms, **launch, **outs)
    return outs, plan


def _expect_single_tile(sms, geo):
    return dict(tiles_per_cta=1, dual=0, b_resident=0)


@pytest.mark.parametrize("precision", ["bf16", "fp16"])
@pytest.mark.parametrize("out1", [0, 1], ids=["out1_none", "out1_ln"])
@pytest.mark.parametrize("sources", [1, 2], ids=["down_320", "up_256_256"])
def test_fused_res_conv(sources, out1, precision):
    """conv2 + res_conv in one launch at exactly the tile count, 5 more SMs and the device's count; bitwise equal to the
    unfused two-launch form; the launch refuses fewer SMs than tiles, N != block_n and a missing res_bias, and then
    writes nothing."""
    seed = 1000 + 10 * sources + out1 + (5 if precision == "fp16" else 0)
    c, kw, res = _res_case(sources, out1, precision, RES_B, RES_T, RES_LENS, seed)
    geo = c["outputs"]["out0"][1]
    tiles = geo.n_all
    assert tiles == 12 and tiles + 5 <= SMS
    KP.run_conv_case(lambda: c, [tiles, tiles + 5, 0], _expect_single_tile)

    fused, _ = _fused(c["launch"], c["outputs"], 0)
    unfused = _unfused(kw, res, c["outputs"])
    for k in fused:
        assert torch.equal(bits(fused[k]), bits(unfused[k])), f"{c['name']}/{k}: fused and unfused forms differ"

    ra0, ra1, rw, _ = res
    refusals = [dict(num_sms=tiles - 1),
                dict(num_sms=0, block_n=128, act=native.ACT_NONE, ln=None, out1_mode=native.OUT1_NONE, p1=None),
                dict(num_sms=0, res=(ra0, ra1, rw, None))]
    for over in refusals:
        outs = {k: v[0].clone() for k, v in c["outputs"].items()}
        launch = dict(c["launch"], **over)
        if launch.get("out1_mode", native.OUT1_NONE) == native.OUT1_NONE:
            outs_passed = {"out0": outs["out0"]}
        else:
            outs_passed = outs
        with pytest.raises(RuntimeError, match="ls_test_conv_gemm"):
            KP.conv_gemm(**launch, **outs_passed)
        torch.cuda.synchronize()
        for k, o in outs.items():
            assert bool(o.isnan().all()), (c["name"], over, k)


@pytest.mark.parametrize("precision", ["bf16", "fp16"])
def test_fused_res_conv_headline_grid(precision):
    """The headline geometry (B2 = 32, T = 500: 128 tiles, between 120 and the device's SM count) at the device's
    count, one source, OUT1_NONE (the production form)."""
    B, T = 32, 500
    lens = [T - 13 * i for i in range(B)]
    assert B * -(-T // 128) <= SMS
    c, kw, res = _res_case(1, 0, precision, B, T, lens, 1100 + (5 if precision == "fp16" else 0))
    KP.run_conv_case(lambda: c, [0], _expect_single_tile)
    fused, plan = _fused(c["launch"], c["outputs"], 0)
    assert plan["grid"] == 128
    unfused = _unfused(kw, res, c["outputs"])
    assert torch.equal(bits(fused["out0"]), bits(unfused["out0"]))


def test_fused_res_conv_hook_refuses_bad_descriptors():
    """The hook itself refuses what would build a bad tensor map, before any launch."""
    c, kw, res = _res_case(2, 0, "bf16", RES_B, RES_T, RES_LENS, 1200)
    ra0, ra1, rw, rbias = res
    out = KP._nan(RES_B, RES_T, 256)
    bad = [dict(res=(None, ra1, rw, rbias)),  # no res_a0
           dict(res=(ra0, None, rw, rbias)),  # res_K != res_a0_C + res_a1_C
           dict(res=(ra0[..., :200].contiguous(), torch.cat([ra1, ra0[..., :56]], 2), rw, rbias)),  # 200 + 312: split off a K block
           dict(res=res, addend=out)]         # both a residual GEMM and an addend
    for over in bad:
        o = KP._nan(RES_B, RES_T, 256)
        with pytest.raises(RuntimeError, match="residual GEMM"):
            KP.conv_gemm(num_sms=0, **dict(c["launch"], **over), out0=o)
        assert bool(o.isnan().all())


# --------------------------------------------------- B. zero-filled skipped tiles, symmetric (pad 1) convolutions
# The non-causal estimator's convolutions.  4 row tiles per item; lengths: 256 (row `len` starts a skipped tile), 0,
# 130, 383.  Real tiles {0, 1}, {8, 9}, {12, 13, 14} of 16: at 8 SMs CTAs 2 and 3 hold only skipped tiles.
ZS_B, ZS_T, ZS_LENS, ZS_SMS = 4, 400, [256, 0, 130, 383], [0, 1, 3, 5, 8]


@pytest.mark.parametrize("precision", ["bf16", "fp16"])
@pytest.mark.parametrize("layer", ["resnet_conv3", "down_up_conv", "final_proj"])
def test_zero_skipped_noncausal_convs(layer, precision):
    """zero_skipped = 1: every stored position of a skipped tile is exactly zero (row `len` included when it starts a
    skipped tile), valid rows are bitwise those of the same launch with zero_skipped = 0.  The activation's padding rows
    hold random data: the pad-1 conv reads row `len` as stored, and the reference does too."""
    dt, r16, fp16, _ = KP.H16[precision]
    B, T = ZS_B, ZS_T
    K, N, taps, pad = {"resnet_conv3": (320, 256, 3, 1), "down_up_conv": (256, 256, 3, 1),
                       "final_proj": (256, 80, 1, 0)}[layer]
    rn = KP._gen(1300 + len(layer) + (5 if fp16 else 0))
    a = r16(rn(B, T, K))  # random on padding rows too
    w = r16(rn(taps, N, K, scale=(taps * K) ** -0.5))
    bias = rn(N, scale=0.1)
    lengths = KP._lens(ZS_LENS)
    y = KP.conv64(a, w, 1, pad) + bias.double()
    mag = KP.conv64(a.abs(), w.abs(), 1, pad) + bias.double().abs()
    geo = KP.Geometry((B, T, N), B, T, N, N, lengths, zero_skipped=1)
    geo0 = KP.Geometry((B, T, N), B, T, N, N, lengths)
    if taps > 1:  # the reference of valid rows depends on row `len` as stored
        row = torch.arange(T, device=DEV)
        am = torch.where((row[None, :, None] < lengths.long()[:, None, None]), a, torch.zeros_like(a))
        ym = KP.conv64(am, w, 1, pad) + bias.double()
        assert KP.per_tile_rel(ym, y, geo0) > 1e-3
    launch = dict(a0=a, w=w, pad=pad, lengths=lengths, bias=bias, fp16=fp16)
    if layer == "down_up_conv":
        launch.update(out1_mode=native.OUT1_COPY)
        outputs = {"out1": (KP._nan(B, T, N, dtype=dt), geo, "ulp", y, mag)}
    else:
        outputs = {"out0": (KP._nan(B, T, N), geo, "f32", y, None)}
    case = dict(name=f"zero_skipped {layer} {precision}", launch=dict(launch, zero_skipped=1), outputs=outputs)
    plans = KP.run_conv_case(lambda: case, ZS_SMS, lambda sms, g: {})
    assert any(0 in rr for _, p, rr in plans if p["tiles_per_cta"] >= 2), "no CTA holding only skipped tiles"

    (k, (init, _, _, _, _)), = outputs.items()
    o1, o0 = init.clone(), init.clone()
    KP.conv_gemm(num_sms=0, **dict(launch, zero_skipped=1), **{k: o1})
    KP.conv_gemm(num_sms=0, **dict(launch, zero_skipped=0), **{k: o0})
    KP.check_masks(f"{case['name']} zero_skipped=0", o0, bits(init), geo0)
    valid = (geo.state == 2).to(DEV)
    assert torch.equal(bits(o1)[valid], bits(o0)[valid])
    # row `len` of item 0 starts its skipped tile 2: zero with zero_skipped = 1, untouched without
    assert bool((bits(o1)[0, ZS_LENS[0]] == 0).all()) and bool(o0[0, ZS_LENS[0]].isnan().all())


# ------------------------------------------------------------------- D. fused block kernel: fp16 build, no_skip
@pytest.mark.parametrize("tail_mode", [0, 1, 2])
def test_tblock_fp16(tail_mode):
    """The fp16 build: fp16 operands and outputs, the reference rounds n3, h and n1 to fp16.  Its errors must be far
    below the bf16 bars (a hook or dispatch that ran the bf16 build would not be)."""
    KP.tblock_plans(tail_mode, "fp16")
    for name in {0: ("tblock_u", "tblock_qkv"), 1: ("tblock_tail",), 2: ("tblock_qkv",)}[tail_mode]:
        assert KP._measured[name + "_f16"] < 0.25 * KP.BARS[name], (name, KP._measured[name + "_f16"])


@pytest.mark.parametrize("precision", ["bf16", "fp16"])
@pytest.mark.parametrize("tail_mode", [0, 1, 2])
def test_tblock_no_skip(tail_mode, precision):
    """no_skip = 1 (the non-causal estimator): padding-only tiles are processed -- no NaN is left, the tail is zero on
    every padding row, u'' and QKV of padding rows follow the row-local reference -- and valid rows are bitwise those
    of the launch that skips."""
    (u1, qkv1, tail1), valid, _ = KP.tblock_plans(tail_mode, precision, no_skip=1)
    (u0, qkv0, tail0), _, _ = KP.tblock_plans(tail_mode, precision, no_skip=0)
    for t in (u1, qkv1, tail1):
        if t is not None:
            assert not bool(t.isnan().any())
    if tail1 is not None:
        assert bool((bits(tail1)[~valid] == 0).all())
    for t1, t0 in ((u1, u0), (qkv1, qkv0), (tail1, tail0)):
        if t1 is not None:
            assert torch.equal(bits(t1)[valid], bits(t0)[valid])


# ------------------------------------------------------------------------------------------ E. GroupNorm + Mish
GN_B, GN_C, GN_G, GN_T, GN_LENS = 5, 256, 8, 3000, [3000, 0, 1, 1037, 3500]  # 3500 > T counts as T


def gn_mish_ref64(x, gamma, beta, lengths, G, temb=None, addend=None):
    """float64 GroupNorm(G) over (C/G channels x the valid frames) of each batch row (biased variance, eps 1e-5), affine,
    Mish, + temb[b] + addend on valid frames, 0 on padding frames.  Returns (y, mag, valid): mag bounds the magnitude of
    the terms the kernel's fp32 result is made of."""
    B, T, Cc = x.shape
    xd = x.double()
    lens = lengths.long().clamp(max=T)
    valid = torch.arange(T, device=x.device)[None, :] < lens[:, None]
    m = valid[:, :, None, None].double()
    xg = xd.view(B, T, G, Cc // G)
    cnt = (lens.double() * (Cc // G)).clamp(min=1)[:, None]
    mean = (xg * m).sum((1, 3)) / cnt
    var = (((xg - mean[:, None, :, None]) ** 2) * m).sum((1, 3)) / cnt
    rstd = 1.0 / torch.sqrt(var + 1e-5)
    z = (xg - mean[:, None, :, None]) * rstd[:, None, :, None]
    z = z.view(B, T, Cc) * gamma.double() + beta.double()
    spread = ((xg.abs() + mean.abs()[:, None, :, None]) * rstd[:, None, :, None]).view(B, T, Cc)
    y = KP.mish(z)
    mag = spread * gamma.double().abs() + beta.double().abs()
    if temb is not None:
        y = y + temb.double()[:, None, :]
        mag = mag + temb.double().abs()[:, None, :]
    if addend is not None:
        y = y + addend.double()
        mag = mag + addend.double().abs()
    vm = valid[:, :, None]
    return torch.where(vm, y, 0.0), torch.where(vm, mag, 0.0), valid


def groupnorm_mish(x, gamma, beta, lengths, G, temb=None, temb_bstride=0, addend=None, out_f32=None, out_h=None,
                   fp16=0):
    B, T, Cc = x.shape
    stats = torch.empty(B * G * 2, device=DEV)
    native.check(native.load().ls_test_groupnorm_mish(
        native.ptr(x), native.ptr(stats), native.ptr(gamma), native.ptr(beta), native.ptr(temb), temb_bstride,
        native.ptr(addend), native.ptr(out_f32), native.ptr(out_h), B, Cc, T, G, native.ptr(lengths), fp16,
        native.current_stream_ptr(DEV)), "ls_test_groupnorm_mish")
    torch.cuda.synchronize()


@pytest.mark.parametrize("precision", ["bf16", "fp16"])
@pytest.mark.parametrize("outs", ["f32", "h", "both"])
@pytest.mark.parametrize("extras", ["none", "temb", "addend", "temb_addend"])
def test_groupnorm_mish(extras, outs, precision):
    """Per-row statistics over the valid frames (a length above T counts as T), one item with a DC offset of 100 (a
    one-pass E[x^2] - E[x]^2 variance in fp32 loses it), optional temb and fp32 addend, fp32 and / or 16-bit outputs;
    padding frames are exactly zero, without temb or addend."""
    dt, _, fp16, _ = KP.H16[precision]
    B, Cc, G, T = GN_B, GN_C, GN_G, GN_T
    rn = KP._gen(1400 + len(extras) + 10 * len(outs))
    x = rn(B, T, Cc)
    x[3] += 100.0
    gamma, beta = 1 + rn(Cc, scale=0.2), rn(Cc, scale=0.2)
    temb = rn(B, 2 * Cc) if "temb" in extras else None  # row stride 2C: rows b*temb_bstride
    addend = rn(B, T, Cc) if "addend" in extras else None
    lengths = KP._lens(GN_LENS)
    y, mag, valid = gn_mish_ref64(x, gamma, beta, lengths, G, temb[:, :Cc] if temb is not None else None, addend)
    of = KP._nan(B, T, Cc) if outs != "h" else None
    oh = KP._nan(B, T, Cc, dtype=dt) if outs != "f32" else None
    groupnorm_mish(x, gamma, beta, lengths, G, temb, 2 * Cc, addend, of, oh, fp16)
    pad = ~valid
    if of is not None:
        assert bool((bits(of)[pad] == 0).all()), "padding frames of the fp32 output are not exactly zero"
        d = ((of.double() - y) ** 2).view(B, T, G, Cc // G).sum((1, 3))
        r = (y ** 2).view(B, T, G, Cc // G).sum((1, 3))
        has = valid.any(1)
        e = float((d[has] / r[has]).sqrt().max())
        KP._note("gn_mish_f32", e)
        assert e <= GN_BAR, e
    if oh is not None:
        assert bool((bits(oh)[pad] == 0).all()), "padding frames of the 16-bit output are not exactly zero"
        st = types.SimpleNamespace(state=torch.where(valid[:, :, None], 2, 0).expand(B, T, Cc).cpu())
        mx, n1, bad = KP.ulp_check(oh, y, mag * 8.0, st)
        KP._note("ulp16 max", mx)
        KP._note("ulp16 >1 (cancellation)", n1)
        assert bad == 0, f"{bad} elements beyond 1 ulp ({n1} > 1 ulp in all)"
    if of is not None and oh is not None:  # one value, two formats
        assert torch.equal(bits(of.to(dt))[valid], bits(oh)[valid])


def test_groupnorm_mish_refusals():
    """Group sizes the kernel cannot serve (C/G not a multiple of 32, C not a multiple of 4G) are refused; nothing is
    written."""
    for Cc, G in ((256, 16), (96, 8)):
        x = torch.randn(2, 64, Cc, device=DEV)
        gamma, beta = torch.ones(Cc, device=DEV), torch.zeros(Cc, device=DEV)
        of, oh = KP._nan(2, 64, Cc), KP._nan(2, 64, Cc, dtype=torch.bfloat16)
        with pytest.raises(RuntimeError, match="ls_test_groupnorm_mish"):
            groupnorm_mish(x, gamma, beta, None, G, out_f32=of, out_h=oh)
        assert bool(of.isnan().all()) and bool(oh.isnan().all())
