"""The ReLU-net training kernels (csrc/relu_mlp.cu) launch by launch, and the autograd node layer by layer, against
float64 on the kernels' own operand images.

Every launch reads and writes fp16 operand images (tc.cuh): a [rows x 64] plane holds chunk(r, c) -- 8 fp16 values of
row r, samples 8c..8c+7 -- at byte c*rows*16 + (r/8)*128 + (r%8)*16, and a tile is `hi | lo` (`hi` only in the fp16
variant).  `encode` below is the kernels' split2 bit for bit and `decode` its inverse, so a test can feed a launch exact,
known operands and read back exactly what it wrote.  The node keeps its activation images on the autograd ctx
(`out.grad_fn.acts`) until backward runs: a float64 chain that takes each layer's input from the kernel's decoded
activations, and its ReLU mask from `decoded > 0`, takes exactly the kernel's branches, so EVERY row and every parameter
is bounded -- no "all but a few samples".

Bound, per element of a product W x (+ b):
    |err| <= tau * (sum_j |W_ij x_j| + |b_i|) + 2^-24 * sum_j (|W_ij| + |x_j|)
The second term is the absolute floor of a lo plane that falls into fp16 subnormals; an output stored as an image
adds its own, 2^-25.  Gradients summed over samples (fp32
TMEM accumulation per CTA, fp32 atomics across CTAs) are bounded the same way with sum_s |a| |zb| as the condition
number.  Backward chains carry the bound of their cotangent down through |W|^T.  Cotangents enter scaled by one
launch-wide power of two (max -> [1, 2)), so the floor of a backward product is relative to the launch maximum: that is
the stated contract of the scale, and rows far below the maximum are only that accurate.

TAU = 2^-19 (fp16 variant: 2^-9).  Measured on an NVIDIA B200 (1000 W power limit; `pytest -s` prints the worst
err / bound of every check at the end of the module): where the tau term dominates -- O(1) operands -- the worst element
of any launch or node check used 0.28 of its bound (fwd_hidden 0.12, gW 0.12-0.23, gb_prev 0.27), i.e. an effective tau
of about 2^-21; the checks that reach 0.98-0.99 (bwd_head_zb, the 2^-10 weight sweep) are values below 2^-14 whose
image store rounds to the 2^-24 grid of fp16 subnormals, which the 2^-25 store term bounds exactly.  The fp16 variant
used at most 0.45 of its 2^-9.

The bound is operand-aware: below input scale ~2^-3 or weight scale ~2^-4 the split is not fp32-class relative to the
OUTPUT (the lo planes lose bits to fp16 subnormals), and test_operand_scale_sweep states where the plain "3e-6 of the
output scale" holds.
"""
import ctypes

import pytest
import torch

from rise_sdf_b200 import _lib as L
from rise_sdf_b200 import relu_mlp
from rise_sdf_b200.fused_mlp import PackedMLP, pack_weight, pad16
from rise_sdf_b200.network_utils import VanillaMLP

pytestmark = pytest.mark.gpu

NS, HID = 64, 128
TAU = 2.0 ** -19            # fp32-class path (hi|lo operands, three products, fp32 accumulation); B200: <= 0.28 of it
TAU16 = 2.0 ** -9           # fp16 variant (one plane, one product)
FLOOR = 2.0 ** -24
STORE = 2.0 ** -25          # an image output's own split: hi and lo both fp16 subnormal below 2^-14 * 2^-11
F16_MAX = 65504.0
# 1, partial groups of 16, exact tiles, partial tiles, one tile per CTA, and 7 tiles on some CTAs: the 2-deep mbarrier
# ring's parity wraps back to 0 at the 3rd, 5th and 7th tile of a CTA.
SIZES = (1, 15, 16, 17, 63, 64, 65, 148 * 64, 148 * 64 * 6 + 33)
N_INS = (1, 16, 17, 127, 128)
DIM_OUTS = (1, 15, 16)
SEGS = {1: [1], 16: [5, 11], 17: [3, 7, 7], 127: [61, 3, 63], 67: [48, 16, 3], 84: [45, 35, 4], 73: [61, 9, 3],
        76: [65, 5, 6], 128: [45, 45, 38]}
SCALES, SHIFTS = [1.0, 2.0, 0.5], [0.0, -1.0, 0.25]       # powers of two: fmaf(x, s, t) == fl(x * s + t)
WORST = {}


@pytest.fixture(params=["fp32", "fp16"])
def prec(request):
    VanillaMLP.mlp_precision = request.param
    yield 1 if request.param == "fp16" else 0
    VanillaMLP.mlp_precision = "fp32"


@pytest.fixture(scope="module", autouse=True)
def report_worst():
    yield
    print("\nworst err / bound per check:")
    for k in sorted(WORST):
        print(f"  {k:28s} {WORST[k]:.3g}")


def tau_of(fp16):
    return TAU16 if fp16 else TAU


# ---------------------------------------------------------------------------------------------------------------------
# operand-image codec
# ---------------------------------------------------------------------------------------------------------------------
def split(x, fp16):
    """tc.cuh split2: hi = fp16(x) (round to nearest even, saturating), lo = fp16(x - hi) (exact fp32 subtraction)."""
    hi = x.clamp(-F16_MAX, F16_MAX).half()
    lo = None if fp16 else (x - hi.float()).clamp(-F16_MAX, F16_MAX).half()
    return hi, lo


def encode(x, rows, fp16):
    """[S, n <= rows] fp32 -> image stream [n_tiles, planes * rows * 128] uint8; rows >= n and samples >= S are 0."""
    S, n = x.shape
    n_tiles = (S + NS - 1) // NS
    full = torch.zeros(n_tiles * NS, rows, dtype=torch.float32, device=x.device)
    full[:S, :n] = x
    hi, lo = split(full, fp16)
    planes = torch.stack([hi] if fp16 else [hi, lo])                        # [P, samples, rows]
    t = planes.view(len(planes), n_tiles, 8, 8, rows // 8, 8)              # P, tile, c, j, r/8, r%8
    return t.permute(1, 0, 2, 4, 5, 3).contiguous().view(torch.uint8).view(n_tiles, -1)


def decode(stream, rows, fp16):
    """image stream -> (hi, lo) fp16 [n_tiles * 64, rows] (lo None in the fp16 variant)."""
    planes = 1 if fp16 else 2
    t = stream.view(torch.float16).view(-1, planes, 8, rows // 8, 8, 8)     # tile, P, c, r/8, r%8, j
    t = t.permute(1, 0, 2, 5, 3, 4).reshape(planes, -1, rows)
    return t[0], (None if fp16 else t[1])


def value(stream, rows, fp16, S):
    """what a launch reads from an image stream, as float64 [S, rows] (hi + lo is exact)."""
    hi, lo = decode(stream, rows, fp16)
    v = hi.double() if fp16 else hi.double() + lo.double()
    return v[:S]


def assert_canonical(stream, rows, fp16):
    """every (hi, lo) pair is one split2 can make: hi is a nearest fp16 of hi + lo, i.e. |lo| <= ulp(hi) / 2.  (Re-
    splitting hi + lo does not always give the same bits: a residual that rounds to exactly half an ulp makes a tie,
    and one that underflows to -0 comes back as +0.)"""
    if fp16:
        return
    hi, lo = decode(stream, rows, fp16)
    h, l = hi.float(), lo.float()
    ulp = torch.exp2(torch.floor(torch.log2(h.abs().clamp_min(2.0 ** -14))) - 10)
    ok = (l.abs() <= 0.5 * ulp) | (h.abs() == F16_MAX)                     # saturated hi: lo keeps what it can
    assert bool(torch.isfinite(h).all()) and bool(ok.all()), "non-canonical hi|lo pair"


def new_stream(S, rows, fp16, dev="cuda"):
    """pre-filled with 0x7E bytes (fp16 NaN), so an unwritten byte shows"""
    return torch.full(((S + NS - 1) // NS, (1 if fp16 else 2) * rows * 128), 0x7E, dtype=torch.uint8, device=dev)


# ---------------------------------------------------------------------------------------------------------------------
# bounds
# ---------------------------------------------------------------------------------------------------------------------
def bound(W, x, tau, bias=None):
    """bound of x @ W^T (+ b) [S, r] for W [r, k], x [S, k] (float64)."""
    Wa, xa = W.abs(), x.abs()
    cond = xa @ Wa.T
    if bias is not None:
        cond = cond + bias.abs()
    return tau * cond + FLOOR * (Wa.sum(1)[None, :] + xa.sum(1)[:, None])


def prefill_bound(P, S):
    """rounding of the fp32 atomics onto a pre-filled buffer: <= 8 adds per element and CTA, each within 2^-24 of
    the running value"""
    return 8 * min((S + NS - 1) // NS, 148) * FLOOR * P.abs()


def bound_sum(zb, a, tau, ginv, prefill):
    """bound of prefill + ginv * zb^T a [r, k] for scaled cotangents zb [S, r] and activations a [S, k]."""
    return (tau * ginv * (zb.abs().T @ a.abs()) + prefill_bound(prefill, zb.shape[0])
            + FLOOR * ginv * (zb.abs().sum(0)[:, None] + a.abs().sum(0)[None, :]))


def check(name, got, want, bnd):
    got = got.double()
    assert got.shape == want.shape, (name, got.shape, want.shape)
    assert torch.isfinite(got).all(), (name, "non-finite or unwritten output")
    err = (got - want).abs()
    r = torch.where(bnd > 0, err / bnd.clamp_min(1e-300), torch.where(err > 0, float("inf"), 0.0))
    worst = float(r.max()) if r.numel() else 0.0
    WORST[name] = max(WORST.get(name, 0.0), worst)
    if worst > 1:
        i = int(r.argmax())
        raise AssertionError(f"{name}: err/bound {worst:.3g} at flat index {i} (shape {tuple(r.shape)}): "
                             f"got {float(got.flatten()[i])!r}, want {float(want.flatten()[i])!r}, "
                             f"bound {float(bnd.flatten()[i]):.3g}")


def check_relu(name, got_stream, z, bnd, fp16, S):
    """a hidden activation image against relu(z64): values, canonical pairs, and every differing ReLU branch."""
    assert_canonical(got_stream, HID, fp16)
    got = value(got_stream, HID, fp16, S)
    bnd = bnd + STORE
    check(name, got, z.clamp_min(0.0), bnd)
    flips = (got > 0) != (z > 0)
    assert bool((z[flips].abs() <= bnd[flips]).all()), (name, "ReLU branch off by more than the bound")


def scales_of(amax_bits):
    """(2^K, 2^-K) the launches take from the launch-wide cotangent maximum."""
    e = (amax_bits >> 23) & 0xFF
    return (2.0 ** (127 - e), 2.0 ** (e - 127)) if 0 < e < 254 else (1.0, 1.0)


def amax_tensor(m):
    bits = int(torch.tensor([m], dtype=torch.float32).view(torch.int32))
    return torch.tensor([bits], dtype=torch.int32, device="cuda"), bits


# ---------------------------------------------------------------------------------------------------------------------
# operands
# ---------------------------------------------------------------------------------------------------------------------
def gen(seed):
    return torch.Generator().manual_seed(seed)


def randn(g, *shape, scale=1.0):
    return (torch.randn(*shape, generator=g) * scale).cuda()


def activations(g, S, k=HID):
    """post-ReLU-like operand: about half exact zeros, the rest O(1)"""
    return randn(g, S, k).clamp_min(0.0)


def cotangents(g, S, r):
    """scaled cotangents (max in [1, 2)) with exact zeros, as a backward launch receives them"""
    z = randn(g, S, r, scale=0.5).clamp(-1.9, 1.9) * (torch.rand(S, r, generator=g) > 0.3).cuda()
    if S:
        z[0, 0] = 1.75
    return z


def weights(g, r, k, scale=1.0):
    return randn(g, r, k, scale=scale / k ** 0.5), randn(g, r, scale=0.05)


# ---------------------------------------------------------------------------------------------------------------------
# direct launches
# ---------------------------------------------------------------------------------------------------------------------
def launch_fwd(W, b, S, fp16, *, segs=None, a_in=None, head=False):
    """one rsdf_relu_layer_fwd: rows mode (segs = [(x, scale, shift)]) or image mode (a_in); hidden -> image, head ->
    rows.  Returns (a0_save stream or None, output)."""
    r_real, k = W.shape
    r_pad = 16 if head else HID
    k_pad = pad16(k) if segs is not None else HID
    blob = pack_weight(W, r_pad, k_pad)
    p = L.ReluFwdC()
    p.w, p.bias = blob.data_ptr(), b.data_ptr()
    p.r_pad, p.r_real, p.k_pad, p.n_samples, p.fp16 = r_pad, r_real, k_pad, S, fp16
    a0 = None
    if segs is not None:
        for g, (x, sc, sh) in enumerate(segs):
            p.inp[g], p.in_w[g], p.in_scale[g], p.in_shift[g] = x.data_ptr(), x.shape[1], sc, sh
        p.n_in = k
        a0 = new_stream(S, k_pad, fp16)
        p.a0_save = a0.data_ptr()
    else:
        p.a_in = a_in.data_ptr()
    if head:
        out = torch.full((S, r_real), float("nan"), device="cuda")
        p.rows_out = out.data_ptr()
    else:
        out = new_stream(S, HID, fp16)
        p.a_out = out.data_ptr()
    L.call("rsdf_relu_layer_fwd", ctypes.byref(p), L.stream())
    torch.cuda.synchronize()
    return a0, out


def launch_bwd(W, S, fp16, amax, a_in, k_pad, *, zb_in=None, g_rows=None, gW, gb_prev=None, gb_self=None,
               segs=None):
    """one rsdf_relu_layer_bwd.  segs = [(out tensor or None, width, scale)] selects the first-layer mode (segment rows
    out); otherwise a zb_out image stream is returned."""
    r_real, k_real = W.shape
    r_pad = 16 if g_rows is not None else HID
    blob = pack_weight(W, r_pad, k_pad)
    p = L.ReluBwdC()
    p.w = blob.data_ptr()
    p.r_pad, p.r_real, p.k_pad, p.k_real, p.n_samples, p.fp16 = r_pad, r_real, k_pad, k_real, S, fp16
    p.amax, p.a_in, p.gW = amax.data_ptr(), a_in.data_ptr(), gW.data_ptr()
    if g_rows is not None:
        p.g_rows = g_rows.data_ptr()
    else:
        p.zb_in = zb_in.data_ptr()
    if gb_self is not None:
        p.gb_self = gb_self.data_ptr()
    zb_out = None
    if segs is not None:
        p.first_layer = 1
        for g, (o, w, sc) in enumerate(segs):
            p.seg_w[g], p.seg_scale[g] = w, sc
            p.rows_out[g] = None if o is None else o.data_ptr()
    else:
        zb_out = new_stream(S, HID, fp16)
        p.zb_out = zb_out.data_ptr()
        if gb_prev is not None:
            p.gb_prev = gb_prev.data_ptr()
    L.call("rsdf_relu_layer_bwd", ctypes.byref(p), L.stream())
    torch.cuda.synchronize()
    return zb_out


def prefilled(g, *shape):
    """non-zero start values for a gradient buffer (the launches accumulate with +=)"""
    return randn(g, *shape)


# ---------------------------------------------------------------------------------------------------------------------
# 1. forward, each role
# ---------------------------------------------------------------------------------------------------------------------
def make_segs(g, S, n_in):
    xs = [randn(g, S, w) for w in SEGS[n_in]]
    return [(x, SCALES[i], SHIFTS[i]) for i, x in enumerate(xs)]


@pytest.mark.parametrize("S", SIZES)
@pytest.mark.parametrize("n_in", N_INS)
def test_fwd_first_layer_rows(prec, n_in, S):
    """rows -> a0 image (bit exact) and the first hidden image."""
    g = gen(1000 * n_in + S)
    segs = make_segs(g, S, n_in)
    W, b = weights(g, HID, n_in)
    a0, a1 = launch_fwd(W, b, S, prec, segs=segs)
    x = torch.cat([xx * sc + sh for xx, sc, sh in segs], -1)
    want = encode(x, pad16(n_in), prec)
    assert torch.equal(a0, want), "a0 stream is not encode(x * scale + shift) with zero padding"
    xd = value(a0, pad16(n_in), prec, S)[:, :n_in]
    Wd, bd = W.double(), b.double()
    check_relu(f"fwd_first_{'fp16' if prec else 'fp32'}", a1, xd @ Wd.T + bd, bound(Wd, xd, tau_of(prec), bd), prec, S)


@pytest.mark.parametrize("S", SIZES)
def test_fwd_hidden_image(prec, S):
    g = gen(S)
    a = activations(g, S)
    a_in = encode(a, HID, prec)
    W, b = weights(g, HID, HID)
    _, out = launch_fwd(W, b, S, prec, a_in=a_in)
    ad = value(a_in, HID, prec, S)
    Wd, bd = W.double(), b.double()
    check_relu(f"fwd_hidden_{'fp16' if prec else 'fp32'}", out, ad @ Wd.T + bd, bound(Wd, ad, tau_of(prec), bd), prec, S)


@pytest.mark.parametrize("S", SIZES)
@pytest.mark.parametrize("dim_out", DIM_OUTS)
def test_fwd_head_rows(prec, dim_out, S):
    """image -> rows: every row written (the output is pre-filled with NaN), within the bound."""
    g = gen(7 * S + dim_out)
    a_in = encode(activations(g, S), HID, prec)
    W, b = weights(g, dim_out, HID)
    _, out = launch_fwd(W, b, S, prec, a_in=a_in, head=True)
    ad = value(a_in, HID, prec, S)
    Wd, bd = W.double(), b.double()
    check(f"fwd_head_{'fp16' if prec else 'fp32'}", out, ad @ Wd.T + bd, bound(Wd, ad, tau_of(prec), bd))


# ---------------------------------------------------------------------------------------------------------------------
# 2. backward, each role
# ---------------------------------------------------------------------------------------------------------------------
def check_zb_out(name, zb_out, y, ybnd, mask, fp16, S):
    """zb_out = (W^T zb) . [a > 0], carrying the launch's 2^K: exact zeros where masked, the bound elsewhere."""
    assert_canonical(zb_out, HID, fp16)
    got = value(zb_out, HID, fp16, S)
    assert bool((got[~mask] == 0).all()), (name, "masked cotangent not zero")
    check(name, got, y * mask, (ybnd + STORE) * mask)


@pytest.mark.parametrize("S", SIZES)
@pytest.mark.parametrize("dim_out", DIM_OUTS)
def test_bwd_head_rows(prec, dim_out, S):
    """rows cotangent -> zb image of the last hidden layer, gW and gb of the head, gb of the layer below."""
    tag = "fp16" if prec else "fp32"
    g = gen(11 * S + dim_out)
    a = activations(g, S)
    a_in = encode(a, HID, prec)
    W, _ = weights(g, dim_out, HID)
    gr = randn(g, S, dim_out, scale=3e-3) * (torch.rand(S, dim_out, generator=g) > 0.2).cuda()
    m = float(gr.abs().max()) if S else 0.0
    amax, bits = amax_tensor(m)
    gsc, ginv = scales_of(bits)
    P_W, P_bs, P_bp = prefilled(g, dim_out, HID), prefilled(g, dim_out), prefilled(g, HID)
    gW, gb_self, gb_prev = P_W.clone(), P_bs.clone(), P_bp.clone()
    zb_out = launch_bwd(W, S, prec, amax, a_in, HID, g_rows=gr, gW=gW, gb_prev=gb_prev, gb_self=gb_self)
    tau = tau_of(prec)
    ad, Wd, zs = value(a_in, HID, prec, S), W.double(), gr.double() * gsc          # zs: the staged, scaled cotangent
    mask = ad > 0
    y = zs @ Wd
    ybnd = bound(Wd.T, zs, tau)
    check_zb_out(f"bwd_head_zb_{tag}", zb_out, y, ybnd, mask, prec, S)
    check(f"bwd_head_gW_{tag}", gW, P_W.double() + ginv * zs.T @ ad, bound_sum(zs, ad, tau, ginv, P_W.double()))
    grd = gr.double()
    check(f"bwd_head_gb_self_{tag}", gb_self, P_bs.double() + grd.sum(0),
          tau * grd.abs().sum(0) + prefill_bound(P_bs.double(), S))
    # bprev sums the masked fp32 values before their split: the zb bound summed, plus the summation
    check(f"bwd_head_gb_prev_{tag}", gb_prev, P_bp.double() + ginv * (y * mask).sum(0),
          ginv * (ybnd * mask).sum(0) + tau * ginv * ((zs.abs() @ Wd.abs()) * mask).sum(0) + prefill_bound(P_bp.double(), S))


@pytest.mark.parametrize("S", SIZES)
def test_bwd_hidden(prec, S):
    tag = "fp16" if prec else "fp32"
    g = gen(13 * S)
    a = activations(g, S)
    a_in = encode(a, HID, prec)
    zb_in = encode(cotangents(g, S, HID), HID, prec)
    W, _ = weights(g, HID, HID)
    amax, bits = amax_tensor(1.75 * 2.0 ** -9)
    _, ginv = scales_of(bits)
    assert ginv == 2.0 ** -9
    P_W, P_bp = prefilled(g, HID, HID), prefilled(g, HID)
    gW, gb_prev = P_W.clone(), P_bp.clone()
    zb_out = launch_bwd(W, S, prec, amax, a_in, HID, zb_in=zb_in, gW=gW, gb_prev=gb_prev)
    tau = tau_of(prec)
    ad, zs, Wd = value(a_in, HID, prec, S), value(zb_in, HID, prec, S), W.double()
    mask = ad > 0
    y = zs @ Wd
    ybnd = bound(Wd.T, zs, tau)
    check_zb_out(f"bwd_hidden_zb_{tag}", zb_out, y, ybnd, mask, prec, S)
    check(f"bwd_hidden_gW_{tag}", gW, P_W.double() + ginv * zs.T @ ad, bound_sum(zs, ad, tau, ginv, P_W.double()))
    check(f"bwd_hidden_gb_prev_{tag}", gb_prev, P_bp.double() + ginv * (y * mask).sum(0),
          ginv * (ybnd * mask).sum(0) + tau * ginv * ((zs.abs() @ Wd.abs()) * mask).sum(0) + prefill_bound(P_bp.double(), S))


@pytest.mark.parametrize("S", SIZES)
@pytest.mark.parametrize("n_in", N_INS)
def test_bwd_first_layer_segments(prec, n_in, S):
    """zb image -> per-segment input-gradient rows (x seg_scale x 2^-K), a NULL segment untouched, gW of layer 1."""
    tag = "fp16" if prec else "fp32"
    g = gen(17 * S + n_in)
    widths = SEGS[n_in]
    k_pad = pad16(n_in)
    x = randn(g, S, n_in)
    a_in = encode(x, k_pad, prec)
    zb_in = encode(cotangents(g, S, HID), HID, prec)
    W, _ = weights(g, HID, n_in)
    amax, bits = amax_tensor(1.5 * 2.0 ** -12)
    _, ginv = scales_of(bits)
    seg_scales = [2.0, -0.375, 1.5][:len(widths)]
    null = 1 if len(widths) > 1 else None
    outs = [torch.full((S, w), -7.0 if i == null else float("nan"), device="cuda") for i, w in enumerate(widths)]
    P_W = prefilled(g, HID, n_in)
    gW = P_W.clone()
    launch_bwd(W, S, prec, amax, a_in, k_pad, zb_in=zb_in, gW=gW,
               segs=[(None if i == null else o, w, sc) for i, (o, w, sc) in enumerate(zip(outs, widths, seg_scales))])
    tau = tau_of(prec)
    ad, zs, Wd = value(a_in, k_pad, prec, S)[:, :n_in], value(zb_in, HID, prec, S), W.double()
    y, ybnd = zs @ Wd, bound(Wd.T, zs, tau)
    f0 = 0
    for i, (o, w, sc) in enumerate(zip(outs, widths, seg_scales)):
        if i == null:
            assert bool((o == -7.0).all()), "a NULL segment's buffer was written"
        else:
            check(f"bwd_first_rows_{tag}", o, y[:, f0:f0 + w] * ginv * sc, ybnd[:, f0:f0 + w] * ginv * abs(sc))
        f0 += w
    check(f"bwd_first_gW_{tag}", gW, P_W.double() + ginv * zs.T @ ad, bound_sum(zs, ad, tau, ginv, P_W.double()))


# ---------------------------------------------------------------------------------------------------------------------
# 4. the node against the exact-mask float64 chain
# ---------------------------------------------------------------------------------------------------------------------
def make(dim_in, dim_out, hidden, seed=0, w_scale=1.0, in_scale=1.0):
    torch.manual_seed(seed)
    m = VanillaMLP(dim_in, dim_out, {"n_neurons": 128, "n_hidden_layers": hidden, "sphere_init": False,
                                     "weight_norm": False, "output_activation": "none"}).cuda()
    with torch.no_grad():
        for l, lin in enumerate(m.linears()):
            lin.bias.normal_(0.0, 0.05)
            lin.weight.mul_(w_scale)
            lin.bias.mul_(in_scale * w_scale ** (l + 1))        # keeps every layer's bias beside its W x
    return m


def node_inputs(g, S, dim_in, in_scale=1.0):
    widths = SEGS.get(dim_in, [dim_in])
    segs = [randn(g, S, w, scale=in_scale).requires_grad_(i != 1) for i, w in enumerate(widths)]
    return segs, SCALES[:len(widths)], SHIFTS[:len(widths)]


def run_node(m, segs, scales, shifts, c):
    """forward + backward through relu_mlp; returns (out, decoded activations [a0, a1, ...], input grads, param grads)"""
    fp16 = 1 if VanillaMLP.mlp_precision == "fp16" else 0
    out = relu_mlp.relu_mlp(m, segs, scales, shifts)
    k0 = pad16(sum(s.shape[1] for s in segs))
    acts = [a.clone() for a in out.grad_fn.acts]                 # the ctx drops them in backward
    S = out.shape[0]
    dec = [value(a, k0 if i == 0 else HID, fp16, S) for i, a in enumerate(acts)]
    wrt = [s for s in segs if s.requires_grad]
    grads = torch.autograd.grad((out * c).sum(), wrt + list(m.parameters()))
    torch.cuda.synchronize()
    return out.detach(), acts, dec, grads[:len(wrt)], grads[len(wrt):]


def node_check(m, segs, scales, shifts, c, tag):
    """every output, activation, input-gradient row and parameter gradient of the node within the propagated bound"""
    fp16 = 1 if VanillaMLP.mlp_precision == "fp16" else 0
    tau = tau_of(fp16)
    tag = f"{tag}_{'fp16' if fp16 else 'fp32'}"
    out, acts, dec, g_in, g_par = run_node(m, segs, scales, shifts, c)
    S, n_in = out.shape[0], sum(s.shape[1] for s in segs)
    x = torch.cat([s.detach() * sc + sh for s, sc, sh in zip(segs, scales, shifts)], -1)
    assert torch.equal(acts[0], encode(x, pad16(n_in), fp16))
    ws = [(W.detach().double(), b.detach().double()) for W, b in m.effective_weights()]
    ins = [dec[0][:, :n_in]] + dec[1:]
    for l, (W, b) in enumerate(ws):
        z, zb = ins[l] @ W.T + b, bound(W, ins[l], tau, b)
        if l + 1 < len(ws):
            check_relu(f"node_fwd_hidden_{tag}", acts[l + 1], z, zb, fp16, S)
        else:
            check(f"node_fwd_out_{tag}", out, z, zb)
    # backward, in the launches' scaled units: zs = 2^K * cotangent, E = its error bound
    m_abs = float(c.abs().max()) if S else 0.0
    gsc, ginv = scales_of(int(torch.tensor([m_abs], dtype=torch.float32).view(torch.int32)))
    zs = c.double() * gsc
    E = torch.zeros_like(zs)
    g_W, g_b = [None] * len(ws), [None] * len(ws)
    for l in range(len(ws) - 1, -1, -1):
        W, a = ws[l][0], ins[l]
        g_W[l] = (ginv * zs.T @ a, ginv * E.T @ a.abs() + bound_sum(zs, a, tau, ginv, torch.zeros_like(W)))
        g_b[l] = (ginv * zs.sum(0), ginv * (E.sum(0) + tau * zs.abs().sum(0)))
        y = zs @ W
        ybnd = E @ W.abs() + bound(W.T, zs, tau)
        if l:
            mask = a > 0
            zs, E = y * mask, (ybnd + STORE) * mask
    f0, gi = 0, 0
    for s, sc in zip(segs, scales):
        w = s.shape[1]
        if s.requires_grad:
            check(f"node_grad_in_{tag}", g_in[gi], y[:, f0:f0 + w] * ginv * sc, ybnd[:, f0:f0 + w] * ginv * abs(sc))
            gi += 1
        f0 += w
    for l in range(len(ws)):
        check(f"node_grad_W_{tag}", g_par[2 * l], *g_W[l])
        check(f"node_grad_b_{tag}", g_par[2 * l + 1], *g_b[l])
    return out, g_in, g_par


SHAPES = [
    (67, 3, 4, 5000),                   # neus radiance
    (84, 6, 4, 1000),                   # split albedo
    (84, 1, 2, 777),                    # split roughness
    (73, 3, 4, 64 * 148 * 2 + 5),       # split env
    (76, 3, 4, 63),                     # split secondary
    (16, 2, 1, 300),
    (1, 16, 7, 65),
    (17, 15, 2, 148 * 64 * 6 + 33),
    (127, 1, 1, 17),
    (128, 16, 4, 1),
    (128, 15, 7, 148 * 64),
]


@pytest.mark.parametrize("dim_in,dim_out,hidden,S", SHAPES)
def test_node_exact_mask_chain(prec, dim_in, dim_out, hidden, S):
    m = make(dim_in, dim_out, hidden, seed=S)
    g = gen(S + dim_in)
    segs, scales, shifts = node_inputs(g, S, dim_in)
    c = randn(g, S, dim_out, scale=1.0 / S)
    node_check(m, segs, scales, shifts, c, "shapes")


# ---------------------------------------------------------------------------------------------------------------------
# 5. cotangent range
# ---------------------------------------------------------------------------------------------------------------------
def test_zero_cotangent(prec):
    """amax = 0 takes the unscaled branch: every gradient exactly zero"""
    m = make(67, 3, 4, seed=1)
    segs, scales, shifts = node_inputs(gen(1), 3000, 67)
    _, _, _, g_in, g_par = run_node(m, segs, scales, shifts, torch.zeros(3000, 3, device="cuda"))
    for t in list(g_in) + list(g_par):
        assert bool((t == 0).all())


def test_cotangent_decades(prec):
    """cotangent rows spanning 1e-12 .. 1: each row within the bound relative to the launch maximum"""
    S = 148 * 64 + 77
    m = make(67, 3, 4, seed=2)
    g = gen(2)
    segs, scales, shifts = node_inputs(g, S, 67)
    c = randn(g, S, 3) * (10.0 ** (-12.0 * torch.rand(S, 1, generator=g))).cuda()
    node_check(m, segs, scales, shifts, c, "decades")


@pytest.mark.parametrize("e", [40, -40])
def test_loss_scaling(prec, e):
    """loss x 2^e: the scaled cotangent images are the same bits, so input gradients are x 2^e bit for bit; weight
    gradients (atomics in any order) scale within the bound."""
    S = 5000
    m = make(67, 3, 4, seed=3)
    g = gen(3)
    segs, scales, shifts = node_inputs(g, S, 67)
    c = randn(g, S, 3, scale=1e-3)
    _, g1, p1 = node_check(m, segs, scales, shifts, c, "loss_scale")
    _, g2, p2 = node_check(m, segs, scales, shifts, c * 2.0 ** e, "loss_scale")
    for a, b in zip(g1, g2):
        assert torch.equal(a * 2.0 ** e, b)
    for a, b in zip(p1, p2):
        assert torch.isfinite(b).all()


# ---------------------------------------------------------------------------------------------------------------------
# 6. determinism and batch invariance
# ---------------------------------------------------------------------------------------------------------------------
def test_deterministic(prec):
    S = 148 * 64 * 3 + 9
    m = make(67, 3, 4, seed=4)
    g = gen(4)
    segs, scales, shifts = node_inputs(g, S, 67)
    c = randn(g, S, 3, scale=1.0 / S)
    o1, a1, _, i1, _ = run_node(m, segs, scales, shifts, c)
    o2, a2, _, i2, _ = run_node(m, segs, scales, shifts, c)
    assert torch.equal(o1, o2)
    assert all(torch.equal(x, y) for x, y in zip(a1, a2))
    assert all(torch.equal(x, y) for x, y in zip(i1, i2))


def test_batch_invariant(prec):
    S = 148 * 64 * 2 + 41
    m = make(67, 3, 4, seed=5)
    segs, scales, shifts = node_inputs(gen(5), S, 67)
    segs = [s.detach() for s in segs]
    with torch.no_grad():
        full = relu_mlp.relu_mlp(m, segs, scales, shifts)
        for n in (1, 16, 63, 65, 148 * 64 + 1):
            part = relu_mlp.relu_mlp(m, [s[:n] for s in segs], scales, shifts)
            assert torch.equal(part, full[:n]), n


# ---------------------------------------------------------------------------------------------------------------------
# 7. non-finite inputs
# ---------------------------------------------------------------------------------------------------------------------
def test_nan_input_row(prec):
    """one NaN feature makes its sample's output row all NaN, as torch.relu does; every other row is bit-identical"""
    S = 1000
    m = make(67, 3, 4, seed=6)
    x = randn(gen(6), S, 67)
    xn = x.clone()
    rows = [5, 300, S - 1]
    for i, r in enumerate(rows):
        xn[r, [0, 40, 66][i]] = float("nan")
    keep = torch.ones(S, dtype=torch.bool)
    keep[rows] = False
    with torch.no_grad():
        for name, f in (("relu_mlp", lambda t: relu_mlp.relu_mlp(m, t)), ("PackedMLP", PackedMLP(m))):
            clean, dirty = f(x), f(xn)
            assert bool(dirty[rows].isnan().all()), (name, dirty[rows])
            assert torch.equal(dirty[keep.cuda()], clean[keep.cuda()]), name
            assert bool(torch.isfinite(clean).all())


# ---------------------------------------------------------------------------------------------------------------------
# 8. operand scale
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("in_log2", [-12, -8, -3, 0, 4, 8])
@pytest.mark.parametrize("w_log2", [-10, -4, -1, 0])
def test_operand_scale_sweep(in_log2, w_log2):
    """The operand-aware bound holds at every scale; the plain 'outputs within 3e-6 of the output scale' only for inputs
    >= 2^-3 and weights >= 2^-4 (max-abs).  Below that the lo planes lose bits to fp16 subnormals: emulating the split
    gives 1.7e-5 of the output at input scale 1e-3 and 3.5e-5 at weight scale 9e-4.  The package's nets see O(1)
    features, SH values and normals."""
    S = 4096 + 17
    sx, sw = 2.0 ** in_log2, 2.0 ** w_log2
    m = make(32, 3, 2, seed=in_log2 * 100 + w_log2, w_scale=sw, in_scale=sx)
    g = gen(8)
    x = (randn(g, S, 32) * sx).requires_grad_(True)
    c = randn(g, S, 3, scale=1.0 / S)
    out, _, _ = node_check(m, [x], [1.0], [0.0], c, "sweep")
    if float(x.detach().abs().max()) >= 2.0 ** -3 and max(float(W.detach().abs().max()) for W, _ in m.effective_weights()) >= 2.0 ** -4:
        h = x.detach().double()
        ws = [(W.detach().double(), b.detach().double()) for W, b in m.effective_weights()]
        for i, (W, b) in enumerate(ws):
            h = h @ W.T + b
            if i + 1 < len(ws):
                h = h.clamp_min(0.0)
        e = float((out.double() - h).abs().max() / h.abs().max())
        WORST["sweep_rel_out_fp32"] = max(WORST.get("sweep_rel_out_fp32", 0.0), e / 3e-6)
        assert e <= 3e-6, e
