"""Flash-attention kernel (attention.cu, both the bf16 and the fp16-operand build) against a float64 reference, element
by element.

The reference takes the same 16-bit Q / K / V and fp32 bias: score (q.k + bias) * 0.125, the key-length mask, the
block-causal mask j < (i // chunk + 1) * chunk, softmax.  The kernel rounds P to the 16-bit type before P.V (the row
sum l stays fp32) and rounds the output, so every element must satisfy

    |o - ref| <= u |ref| + K_BOUND u (sum_j p_j |v_j|) / (sum_j p_j) + tiny

with u = 2^-8 (bf16) or 2^-11 (fp16).  The fp16 build also flushes P below fp16's subnormal range: at most 2^-25 per
key against l >= 1 (the key that set the running maximum contributes 1), a further 2^-25 sum_j |v_j| over the visible
keys.  Channel 0 of V is 1.0 in every head, so that output channel is 1 within u whatever the other channels do: it
pins the normalisation by l on its own.

Every launch also checks what the kernel writes: the output starts as NaN with guard rows after B*T; rows of query
tiles (128 rows) that hold a valid row are finite and match the reference (rows past the length are attention over the
valid keys), rows of padding-only query tiles and the guard keep their NaN bits.  Each batch item is bitwise equal to
a launch of that item alone, and a second identical launch is bitwise equal to the first.

The kernel keeps a lazy running maximum per row: it moves only when a key tile's maximum exceeds it by more than 2^8
(log2 units), and then O is reloaded from tensor memory and scaled by alpha under a warp-uniform branch.  Random Q / K
never get there after the first key tile, so the rescale cases build their scores from Q channel 0 (a per-row alpha)
times K channel 0 (a per-key level), both exact in either 16-bit type, plus small noise; each case asserts that its
scores take the branches it is meant to take (`lazy_max_trace` follows the kernel's decisions).
"""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

if not torch.cuda.is_available():
    pytest.skip("needs a CUDA device", allow_module_level=True)

import minimax_speech_b200.native as native  # noqa: E402

DEV = torch.device("cuda:0")
KV_TILE, Q_TILE, WARP = 64, 128, 32  # keys per key tile (ATTN_KV), query rows per CTA, rows per softmax warp
SCALE = 0.125
C_LOG2 = SCALE / math.log(2.0)       # score -> log2 units
THRESHOLD = 8.0                      # kRescaleThreshold: log2 units the row maximum must grow by before it moves
GUARD = 64                           # output rows after B*T that no launch may touch
DTYPES = {"bf16": (torch.bfloat16, 2.0 ** -8), "fp16": (torch.float16, 2.0 ** -11)}
K_BOUND = 2.0                        # worst error / bound measured with it: 0.59 (B200, 1000 W power limit)
TINY = 2.0 ** -24                    # output rounding of fp16 subnormals

_worst = {}  # category -> worst error / bound ratio


def _note(cat, v):
    _worst[cat] = max(_worst.get(cat, 0.0), v)


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    print("\nworst error-to-bound ratio per category (bound: u|ref| + %.1f u mean_p|v| + subnormal terms; "
          "ones: |o - 1| / u):" % K_BOUND)
    for k, v in sorted(_worst.items()):
        print(f"  {k:16s} {v:.3f}")


def bits(t):
    return t.view(torch.int16)


def _lens(v):
    return None if v is None else torch.tensor(v, dtype=torch.int32, device=DEV)


def _gen(seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return lambda *s, scale=1.0: (torch.randn(*s, generator=g) * scale).to(DEV)


def random_qkv(B, T, H, dtype, seed, scale=1.5):
    """[B][T][3*H*64] with Q, K ~ N(0, scale^2), V ~ N(0, 1) and V channel 0 = 1 in every head"""
    x = _gen(seed)(B, T, 3, H, 64, scale=scale)
    x[:, :, 2] /= scale
    x[:, :, 2, :, 0] = 1.0
    return x.to(dtype).view(B, T, 3 * H * 64)


def launch(qkv, lengths, chunk, bias=None):
    """the kernel through the test hook; returns out [B*T + GUARD][H*64] (NaN where nothing was written)"""
    B, T, C3 = qkv.shape
    H = C3 // 192
    out = torch.full((B * T + GUARD, H * 64), float("nan"), device=DEV, dtype=qkv.dtype)
    ld = bias.shape[-1] if bias is not None else 0
    native.check(native.load().ls_test_attention(native.ptr(qkv), native.ptr(out), native.ptr(lengths), B, T, H,
                                                 chunk, int(qkv.dtype == torch.float16), native.ptr(bias), ld, T * ld,
                                                 native.current_stream_ptr(DEV)), "ls_test_attention")
    torch.cuda.synchronize()
    return out


def visible(T, n, chunk):
    """[T, T] bool: key j visible to query i"""
    pos = torch.arange(T, device=DEV)
    vis = (pos < n)[None, :].expand(T, T)
    if chunk:
        vis = vis & (pos[None, :] < ((pos // chunk + 1) * chunk)[:, None])
    return vis


def scores(qkv, b, bias=None):
    """float64 [H, T, T] (q.k + bias) * 0.125 of batch item b"""
    B, T, C3 = qkv.shape
    H = C3 // 192
    q, k, _ = qkv[b].double().view(T, 3, H, 64).permute(1, 2, 0, 3)
    s = q @ k.transpose(-1, -2)
    if bias is not None:  # score(i, j) += bias[b, h, i, T-1-i+j]
        pos = torch.arange(T, device=DEV)
        idx = (T - 1 - pos[:, None] + pos[None, :]).expand(H, T, T)
        s = s + torch.gather(bias[b].double(), 2, idx)
    return s * SCALE


def reference(qkv, b, n, chunk, bias=None):
    """float64 reference of item b with n valid keys: ref, mean_p |v| and sum over the visible keys of |v|, each
    [T][H*64]"""
    B, T, C3 = qkv.shape
    H = C3 // 192
    v = qkv[b].double().view(T, 3, H, 64)[:, 2].transpose(0, 1)  # [H, T, 64]
    vis = visible(T, n, chunk)
    s = scores(qkv, b, bias).masked_fill(~vis, float("-inf"))
    p = torch.exp(s - s.amax(-1, keepdim=True))
    l = p.sum(-1, keepdim=True)
    ref, mag = (p @ v) / l, (p @ v.abs()) / l
    sub = vis.double() @ v.abs()
    flat = lambda t: t.transpose(0, 1).reshape(T, H * 64)
    return flat(ref), flat(mag), flat(sub)


def written_rows(T, n):
    """rows of item b the kernel writes: those of query tiles that start below the length"""
    return 0 if n <= 0 else min(T, -(-n // Q_TILE) * Q_TILE)


def check_launch(cat, qkv, lengths, chunk, bias=None, alone=None):
    """one launch against the reference, the written region, determinism and batch independence (items `alone`,
    default all).  Returns the output."""
    B, T, C3 = qkv.shape
    H = C3 // 192
    dtype = qkv.dtype
    u = DTYPES["fp16" if dtype == torch.float16 else "bf16"][1]
    sub_unit = 2.0 ** -25 if dtype == torch.float16 else 0.0
    out = launch(qkv, lengths, chunk, bias)
    nan_bits = bits(torch.full((1,), float("nan"), dtype=dtype, device=DEV))
    ob = bits(out)
    assert bool((ob[B * T:] == nan_bits).all()), f"{cat}: guard rows after B*T were written"
    o = out[:B * T].view(B, T, H * 64)
    lens = [T] * B if lengths is None else [min(int(x), T) for x in lengths.tolist()]
    for b, n in enumerate(lens):
        w = written_rows(T, n)
        assert bool((bits(o[b, w:]) == nan_bits).all()), f"{cat}: item {b} (len {n}) wrote rows of padding-only tiles"
        if w == 0:
            continue
        ob64 = o[b, :w].double()
        assert bool(torch.isfinite(ob64).all()), f"{cat}: item {b} (len {n}) non-finite output in rows < {w}"
        ref, mag, sub = (t[:w] for t in reference(qkv, b, n, chunk, bias))
        bound = u * ref.abs() + K_BOUND * u * mag + sub_unit * sub + TINY
        ratio = (ob64 - ref).abs() / bound
        worst = float(ratio.max())
        _note(cat, worst)
        if worst > 1.0:
            r, c = divmod(int(ratio.argmax()), H * 64)
            raise AssertionError(f"{cat}: item {b} (len {n}, chunk {chunk}) row {r} head {c // 64} channel {c % 64}: "
                                 f"out {float(ob64[r, c]):.6g} ref {float(ref[r, c]):.6g} bound {float(bound[r, c]):.3g}"
                                 f" (error / bound {worst:.3g})")
        ones = float((ob64[:, 0::64] - 1.0).abs().max()) / u
        _note("ones " + cat.split()[-1], ones)
        assert ones <= 1.0, f"{cat}: item {b}: the ones channel is off by {ones:.3g} u"
    again = launch(qkv, lengths, chunk, bias)
    assert torch.equal(bits(again), ob), f"{cat}: two identical launches differ"
    if B == 1:
        return out
    for b in range(B) if alone is None else alone:
        one = launch(qkv[b:b + 1], None if lengths is None else lengths[b:b + 1], chunk,
                     None if bias is None else bias[b:b + 1])
        assert torch.equal(bits(one[:T]), bits(o[b])), f"{cat}: item {b} differs from a launch of that item alone"
    return out


# ------------------------------------------------------------------------------------------------ shapes and masks
# T around the 64-key and 128-query tiles, lengths 0 / 1 / tile edges / T, chunks unaligned to both tiles and >= T.
SHAPES = [
    # T, lengths, chunk, H
    (1, None, 0, 8),
    (1, [1, 0], 1, 8),
    (17, [17, 1, 0], 0, 8),
    (17, None, 25, 8),
    (63, [63, 1], 50, 8),
    (64, [64, 63, 0], 0, 8),
    (65, [65, 64, 1], 25, 8),
    (127, [127, 65, 64], 64, 8),
    (128, [128, 127, 0, 1], 100, 8),
    (129, [129, 128, 127, 0], 128, 8),
    (129, None, 1, 8),
    (300, [300, 100], 0, 2),
    (300, [300, 250], 600, 8),
    (500, [500, 129, 128, 127, 65, 64, 63, 1, 0], 0, 8),
    (500, [500, 377, 129, 0], 50, 8),
    (500, None, 25, 8),
    (1500, [1500, 1000, 129], 0, 8),
    (1500, [1500, 700], 50, 8),
    (2999, [2999, 2000], 50, 8),  # the token encoder's up level for a long utterance
]


@pytest.mark.parametrize("dt", ["bf16", "fp16"])
@pytest.mark.parametrize("T,lens,chunk,H", SHAPES)
def test_shapes_and_masks(T, lens, chunk, H, dt):
    B = 1 if lens is None else len(lens)
    qkv = random_qkv(B, T, H, DTYPES[dt][0], seed=1000 + T + chunk + H)
    check_launch(f"shapes {dt}", qkv, _lens(lens), chunk)


def test_speaker_encoder_many_rows():
    """The speaker encoder's launch: hundreds of batch rows, no lengths."""
    B, T = 300, 200
    qkv = random_qkv(B, T, 8, torch.bfloat16, seed=7)
    check_launch("speaker bf16", qkv, None, 0, alone=[0, 1, 149, 299])


# ------------------------------------------------------------------------------------------------ running-max rescale
def lazy_max_trace(t, vis):
    """The kernel's running-maximum decisions: t [R, T] scores in log2 units, vis [R, T].  Returns, per row and key
    tile, the growth of the tile's maximum over the running maximum and whether O is rescaled there, and per row the
    largest log2 P written (P <= 2^THRESHOLD keeps fp16 in range)."""
    R, T = t.shape
    nt = -(-T // KV_TILE)
    tt = torch.full((R, nt * KV_TILE), float("-inf"), dtype=t.dtype, device=t.device)
    tt[:, :T] = t.masked_fill(~vis, float("-inf"))
    mx = tt.view(R, nt, KV_TILE).amax(-1)
    m = torch.full((R,), float("-inf"), dtype=t.dtype, device=t.device)
    growth = torch.full((R, nt), float("nan"), dtype=t.dtype, device=t.device)
    resc = torch.zeros(R, nt, dtype=torch.bool, device=t.device)
    pmax = torch.full((R,), float("-inf"), dtype=t.dtype, device=t.device)
    for k in range(nt):
        growth[:, k] = mx[:, k] - m
        grow = mx[:, k] > m + THRESHOLD
        resc[:, k] = grow & torch.isfinite(m)
        m = torch.where(grow, mx[:, k], m)
        pmax = torch.maximum(pmax, mx[:, k] - m)
    return growth, resc, pmax


def _row_pattern(warps):
    """per query row (i % 128): warp w takes its values from warps[w] cyclically over its lanes"""
    return torch.tensor([warps[(i % Q_TILE) // WARP][i % WARP % len(warps[(i % Q_TILE) // WARP])]
                         for i in range(Q_TILE)], dtype=torch.float64)


# alpha (Q channel 0) per row, by softmax warp: with K channel 0 stepping by 1 per key tile, a row's maximum grows by
# alpha * 0.125 / ln 2 log2 units per tile: 52 -> 9.38 (a rescale every tile; would pass a threshold of 16 to 20
# unrescaled, past fp16's range), 56 -> 10.1, 224 -> 40.4 (earlier tiles underflow), 28 -> 5.05 (every second tile),
# 0 -> none.  Warps 1 and 3 mix rows that rescale with rows that do not.
GROW_ALPHA = _row_pattern([[52.0], [56.0, 0.0], [224.0], [28.0, 52.0, 0.0, 224.0]])
# 43.75 -> 7.89 log2 units at tile 1 (no rescale, P up to 2^7.89), 45 -> 8.12 (one rescale)
EDGE_ALPHA = _row_pattern([[43.75, 45.0], [43.75], [45.0], [43.75, 45.0, 0.0, -45.0]])
DOM_ALPHA = _row_pattern([[56.0], [56.0, 0.0], [-56.0], [224.0, 0.0, 56.0, 28.0]])


def designed_qkv(alpha, kappa, H, dtype, seed):
    """alpha [T] per row (Q channel 0), kappa [B, T] per key (K channel 0); channel 1 adds 8 * omega with omega in
    {-1, -7/8, .., 0} per key (0 at the first key of every tile, so a tile's maximum is alpha * kappa); the other Q / K
    channels are noise of sigma 1/16.  All designed values are exact in bf16 and fp16.  Heads see the row pattern
    shifted by 5 rows each."""
    B, T = kappa.shape
    rn = _gen(seed)
    x = rn(B, T, 3, H, 64, scale=1.0 / 16)
    x[:, :, 2] = rn(B, T, H, 64)
    x[:, :, 2, :, 0] = 1.0
    g = torch.Generator(device="cpu").manual_seed(seed + 1)
    omega = -torch.randint(0, 9, (B, T), generator=g).double() / 8
    omega[:, ::KV_TILE] = 0.0
    for h in range(H):
        x[:, :, 0, h, 0] = alpha.roll(5 * h).to(DEV).float()[None, :]
        x[:, :, 1, h, 0] = kappa.to(DEV).float()
        x[:, :, 0, h, 1] = 8.0
        x[:, :, 1, h, 1] = omega.to(DEV).float()
    return x.to(dtype).view(B, T, 3 * H * 64)


def _rows(pattern, T):
    return pattern.repeat(-(-T // Q_TILE))[:T]


def _trace(qkv, lengths, chunk):
    """lazy_max_trace over every (item, head) of a launch"""
    B, T, C3 = qkv.shape
    out = []
    for b in range(B):
        n = T if lengths is None else min(int(lengths[b]), T)
        vis = visible(T, n, chunk)
        t = scores(qkv, b) / math.log(2.0)
        for h in range(C3 // 192):
            out.append(lazy_max_trace(t[h], vis))
    return out


def _mixed_warp(resc):
    """some softmax warp (32 consecutive rows) has rows that rescale and rows that do not at the same key tile"""
    for r0 in range(0, resc.shape[0], WARP):
        w = resc[r0:r0 + WARP]
        if bool((w.any(0) & ~w.all(0)).any()):
            return True
    return False


RESCALE_MASKS = [(0, None), (50, "lens")]


@pytest.mark.parametrize("dt", ["bf16", "fp16"])
@pytest.mark.parametrize("chunk,lens", RESCALE_MASKS)
@pytest.mark.parametrize("design", ["grow", "edge", "dominant", "decreasing"])
def test_running_max_rescale(design, chunk, lens, dt):
    """grow: every key tile raises the maximum by about 10 log2 units (or 40, or 5 for every second tile);
    edge: growth 7.89 (no rescale, P near 2^8) against 8.12 (a rescale) at tile 1;
    dominant: one key 20 log2 units above the rest in a partial last tile, followed by masked keys that would dominate
    even more (key `len` among them);
    decreasing: the maximum falls by 10 log2 units per tile (later P underflow; rows with negative alpha rise)."""
    T = {"grow": 500, "edge": 200, "dominant": 200, "decreasing": 500}[design]
    B = 3
    tile = (torch.arange(T) // KV_TILE).double()
    if design == "grow":
        alpha, kappa = _rows(GROW_ALPHA, T), tile.expand(B, T).clone()
        lengths = [T, 437, 200]
    elif design == "edge":
        alpha, kappa = _rows(EDGE_ALPHA, T), tile.clamp(max=1).expand(B, T).clone()
        lengths = [T, 130, 100]
    elif design == "decreasing":
        alpha, kappa = _rows(DOM_ALPHA, T), (-tile).expand(B, T).clone()
        lengths = [T, 437, 200]
    else:
        alpha = _rows(DOM_ALPHA, T)
        lengths = [197, T, 130]
        kappa = torch.zeros(B, T, dtype=torch.float64)
        for b, (n, dom) in enumerate(zip(lengths, [195, 199, 129])):
            kappa[b, dom] = 2.0
            kappa[b, n:] = 4.0
    lengths = _lens(lengths) if lens else None
    qkv = designed_qkv(alpha, kappa, 8, DTYPES[dt][0], seed=2000 + len(design) + chunk)

    traces = _trace(qkv, lengths, chunk)
    growth = torch.cat([g for g, _, _ in traces])
    resc = torch.cat([r for _, r, _ in traces])
    pmax = torch.cat([p for _, _, p in traces])
    nt = resc.shape[1]
    assert float(pmax.max()) <= THRESHOLD
    if design == "grow":
        assert bool(resc[:, 1:].all(1).any()), "no row rescales at every key tile"
        assert any(_mixed_warp(r) for _, r, _ in traces), "no warp mixes rows that rescale and rows that do not"
        assert float(growth[resc].max()) > 40.0  # a rescale by 2^-40
    elif design == "edge":
        g1 = growth[:, 1]
        no, yes = (g1 > 7.85) & (g1 < 7.95), (g1 > 8.05) & (g1 < 8.15)
        assert bool(no.any()) and bool(yes.any()), "tile 1 does not grow by both 7.9 and 8.1"
        assert not bool(resc[no].any()) and bool(resc[yes, 1].all())
        assert float(pmax[no].min()) > 7.8  # P close to 2^8 without a rescale
        assert any(_mixed_warp(r) for _, r, _ in traces)
    elif design == "dominant":
        assert bool(resc[:, nt - 1].any()), "the dominant key in the last tile never moves the maximum"
        assert float(growth[:, nt - 1][resc[:, nt - 1]].max()) > 19.0
    else:
        assert bool(resc.any()) and float(growth[:, 1:].nan_to_num(0.0).min()) < -9.0
    check_launch(f"rescale {dt}", qkv, lengths, chunk)


# ------------------------------------------------------------------------------------------------ relative-position bias
def skewed_bias(B, H, T, seed, ld=None):
    """[B][H][T][ld] fp32 in the token encoder's layout (ld = Ppad = 2T-1 rounded up to 128): distinct random values on
    the band the kernel reads (columns [T-1-i, 2T-2-i] of row i), NaN everywhere else"""
    ld = ld or -(-(2 * T - 1) // 128) * 128
    bias = torch.full((B, H, T, ld), float("nan"), device=DEV)
    band = _gen(seed)(B, H, T, T, scale=6.0)
    pos = torch.arange(T, device=DEV)
    idx = (T - 1 - pos[:, None] + pos[None, :]).expand(B, H, T, T)
    bias.scatter_(3, idx, band)
    return bias


BIAS_CASES = [
    # T, lengths, chunk, dtype, row pitch: the token encoder's level 0 (T) and up level (2T), T not a multiple of 64
    (150, [150, 127, 61], 0, "bf16", None),
    (150, [150, 127, 61], 25, "bf16", None),
    (150, [150, 100, 1], 50, "bf16", None),
    (300, [300, 254, 122], 0, "bf16", None),
    (300, [300, 254, 122], 25, "bf16", None),
    (300, [300, 200, 129], 50, "bf16", None),
    (150, [150, 149, 64], 50, "bf16", 299),  # the tightest layout the hook accepts: rows of exactly 2T-1 entries
    (150, [150, 127, 61], 25, "fp16", None),
]


@pytest.mark.parametrize("T,lens,chunk,dt,ld", BIAS_CASES)
def test_relative_position_bias(T, lens, chunk, dt, ld):
    B, H = len(lens), 8
    qkv = random_qkv(B, T, H, DTYPES[dt][0], seed=3000 + T + chunk)
    bias = skewed_bias(B, H, T, seed=3100 + T + chunk, ld=ld)
    check_launch(f"bias {dt}", qkv, _lens(lens), chunk, bias)


# ------------------------------------------------------------------------------------------------ the hook itself
def test_hook_refuses_bad_arguments():
    """A bad call returns an error and launches nothing."""
    T, H = 100, 8
    qkv = random_qkv(1, T, H, torch.bfloat16, seed=5)
    out = torch.full((T, H * 64), float("nan"), device=DEV, dtype=torch.bfloat16)
    bias = skewed_bias(1, H, T, seed=6)
    ld = bias.shape[-1]
    lib = native.load()
    s = native.current_stream_ptr(DEV)
    P = native.ptr
    bad = {
        "null qkv": (None, out, None, 1, T, H, 0, 0, None, 0, 0),
        "null out": (qkv, None, None, 1, T, H, 0, 0, None, 0, 0),
        "B = 0": (qkv, out, None, 0, T, H, 0, 0, None, 0, 0),
        "B > 65535": (qkv, out, None, 65536, T, H, 0, 0, None, 0, 0),
        "T = 0": (qkv, out, None, 1, 0, H, 0, 0, None, 0, 0),
        "H = 0": (qkv, out, None, 1, T, 0, 0, 0, None, 0, 0),
        "chunk < 0": (qkv, out, None, 1, T, H, -1, 0, None, 0, 0),
        "fp16 = 2": (qkv, out, None, 1, T, H, 0, 2, None, 0, 0),
        "bias_ld < 2T-1": (qkv, out, None, 1, T, H, 0, 0, bias, 2 * T - 2, T * ld),
        "bias_bh < T*bias_ld": (qkv, out, None, 1, T, H, 0, 0, bias, ld, T * ld - 1),
    }
    for what, (q, o, ln, B, T_, H_, chunk, fp16, bi, bld, bbh) in bad.items():
        code = lib.ls_test_attention(P(q), P(o), P(ln), B, T_, H_, chunk, fp16, P(bi), bld, bbh, s)
        assert code == -1, f"{what}: returned {code}"  # LS_ERR_INVALID
    torch.cuda.synchronize()
    assert bool(out.isnan().all())
