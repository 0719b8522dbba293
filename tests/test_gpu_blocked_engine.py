"""The blocked-GEMM engine (`spade_const_kernel`, csrc/synth.cu), the blocked weight gradients (csrc/synth_bwd.cu) and the
small training-path kernels around them, one entry point at a time, against plain fp64 torch statements of each kernel's
contract (include/hg3d.h), evaluated on the device so that real sizes stay affordable.

The shapes are the ones where such kernels go wrong: one partial tile, HW = 1 (mod 128), more than two tiles per CTA with the
walk crossing sample boundaries (B*T > 2*148, T not dividing 148), B = 1, and the C2 training renderer's 96*96*32 points per
sample.  Every tile-blocked input carries NaN in its padding rows and every output starts as a sentinel, so each case also
checks that padding never leaks into valid outputs, sums or statistics, and which padding rows a kernel writes.

The CPU tests at the end (no `gpu` mark) are the negative controls: on the same data they show that the fp64 reference under
each plausible kernel mistake differs from the correct reference by at least 100x the GPU tolerance, so the GPU tests can
fail.  No edited kernel is ever run."""
import importlib

import pytest
import torch
import torch.nn.functional as F

gpu = pytest.mark.gpu

C = 256
TOL = 2e-5            # fp32x3 (bf16x3 split) rel-L2 bound; elementwise: 50 * TOL * max|ref| (tests/test_gpu_linear.py)
TOL_BF16 = 1e-2       # passes=1 (plain bf16 operands)
SENT = 1234.5         # initial value of every output buffer: padding rows a kernel does not write keep it
NUM_SMS = 148         # B200

# (B, Hg, Wg)
SHAPES = {
    "a_one_partial_tile": (2, 7, 11),          # HW = 77 < 128
    "b_hw_1_mod_128": (2, 3, 43),              # HW = 129: a second tile with one pixel
    "c_multi_tile": (3, 2, 10009),             # HW = 20018, T = 157: 471 tiles, 3-4 per CTA, walks cross samples
    "d_b1": (1, 20, 50),                       # HW = 1000
}
C2_RENDER = (2, 1, 96 * 96 * 32)               # modules/render_train.py calls the engine with Hg = 1, Wg = N


def _abi():
    return importlib.import_module("3dhumangan_b200.abi")


# ================================================================================================================
# fp64 references (device-agnostic)
# ================================================================================================================
def to_blocked(x, fill=0.0):
    """[B,C,HW] -> tile-blocked [B,T,C,128]; the padding rows past HW hold `fill`."""
    B, Cc, HW = x.shape
    T = (HW + 127) // 128
    pad = torch.full((B, Cc, T * 128), fill, dtype=x.dtype, device=x.device)
    pad[:, :, :HW] = x
    return pad.reshape(B, Cc, T, 128).permute(0, 2, 1, 3).contiguous()


def from_blocked(t, HW):
    """[B,T,C,128] -> [B,C,HW] (valid pixels only)."""
    B, T, Cc, _ = t.shape
    return t.permute(0, 2, 1, 3).reshape(B, Cc, T * 128)[:, :, :HW]


def padding_of(t, HW):
    """The padding rows of a tile-blocked tensor, [B,C,T*128-HW]."""
    B, T, Cc, _ = t.shape
    return t.permute(0, 2, 1, 3).reshape(B, Cc, T * 128)[:, :, HW:]


def f32_affine(x, g1, g0):
    """x*g1 + g0 rounded once to fp32, as the kernels' FFMA computes it, returned in fp64 (the sine of a large argument is
    only defined up to that rounding, so the references take the kernel's argument and test the sine itself)."""
    return (x.double() * g1.double() + g0.double()).float().double()


def act_ref(pre, act, slope=0.2):
    """act 0: LeakyReLU(slope), 1: sine, 2: identity."""
    if act == 0:
        return torch.where(pre > 0, pre, slope * pre)
    if act == 1:
        return torch.sin(pre)
    return pre


def fwd_ref(x, W, bias, *, mod=None, act=2, slope=0.2, x2=None, mod2=None, skip=None, rgb_w=None, rgb_b=None, rgb_in=None):
    """Forward engine: out = W [act(x*g1+g0); act(x2*g1'+g0')] + bias (+ skip), all [B,C,HW];  g' = mod2, or mod when mod2
    is None; no table = identity.  ToRGB: rgb = rgb_in + rgb_w . out + rgb_b.  Statistics: (sum, sumsq) of out per channel
    over the valid pixels of the whole batch."""
    def y_of(src, m):
        if m is None:
            return act_ref(src.double(), act, slope)
        g1, g0 = m[:, 0, :, None], m[:, 1, :, None]
        return act_ref(f32_affine(src, g1, g0), act, slope)
    ys = [y_of(x, mod)]
    if x2 is not None:
        ys.append(y_of(x2, mod2 if mod2 is not None else mod))
    y = torch.cat(ys, 1)
    out = torch.einsum("ok,bkp->bop", W.double(), y) + bias.double()[None, :, None]
    if skip is not None:
        out = out + skip.double()
    rgb = None
    if rgb_w is not None:
        rgb = torch.einsum("jc,bcp->bjp", rgb_w.double(), out) + rgb_b.double()[None, :, None]
        if rgb_in is not None:
            rgb = rgb + rgb_in.double()
    stats = torch.stack([out.sum((0, 2)), (out * out).sum((0, 2))])
    return out, rgb, stats


def bwd_ref(g, M, aux, *, cout=256, mod=None, act=0, slope=0.2, ascale=None, g2=None, rk_w=None, rk_v=None):
    """Data-gradient engine: acc = M [g*ascale; g2] (M = the packed [256 x K] image, W^T in the callers; only its first
    `cout` rows are used) + sum_j rk_w[j] rk_v[:, j]; out = acc * mask(aux*g1+g0) with mask = cos (act 1) or 1 / slope
    (act 0); sums [B,2,cout] = (sum_p out, sum_p out*aux)."""
    op = g.double()
    if ascale is not None:
        op = op * ascale.double()[:, :, None]
    if g2 is not None:
        op = torch.cat([op, g2.double()], 1)
    acc = torch.einsum("ok,bkp->bop", M[:cout].double(), op)
    if rk_v is not None:
        n = rk_v.shape[1]
        acc = acc + torch.einsum("jc,bjp->bcp", rk_w[:n, :cout].double(), rk_v.double())
    if mod is None:
        pre = aux.double()
    else:
        pre = f32_affine(aux, mod[:, 0, :, None], mod[:, 1, :, None])
    mask = torch.cos(pre) if act == 1 else torch.where(pre > 0, 1.0, slope).double()
    out = acc * mask
    sums = torch.stack([out.sum(2), (out * aux.double()).sum(2)], 1)
    return out, sums


def wgrad_ref(dout, x, *, mod=None, act=0, pscale=None):
    """dW [256,Cx] = sum_{b,p} (dout*pscale) (x) act(x*g1+g0) (act 0 LeakyReLU 0.2, 1 sine, 2 identity); dbias = sum dout*pscale.
    x [B or 1,Cx,HW] (1 = shared by the batch); mod [B,2,256] (rows past Cx unused) or None."""
    d = dout.double()
    if pscale is not None:
        d = d * pscale.double()[:, :, None]
    Cx = x.shape[1]
    xb = x.expand(d.shape[0], -1, -1)
    if mod is None:
        y = act_ref(xb.double(), act)
    else:
        y = act_ref(f32_affine(xb, mod[:, 0, :Cx, None], mod[:, 1, :Cx, None]), act)
    return torch.einsum("bop,bcp->oc", d, y), d.sum((0, 2))


def composite_ref(port, sig, z, noise, rgbp, feat, *, R, S, noise_std, white_back, softplus, last_back=False, mask=None):
    """ray_out [B,R,260] = feat | sigmoid(rgb) | depth through oracle.port.ray_integration (volume_rendering.py:12-56).
    `mask` replaces the ReLU of sigma by the clamp mask the kernel differentiates through."""
    B = sig.shape[0]
    feats = torch.cat([feat, torch.sigmoid(rgbp)], 1).permute(0, 2, 1).reshape(B, R, S, 259)
    out = torch.cat([feats, sig.reshape(B, R, S, 1)], -1)
    nz = (noise if noise is not None else torch.zeros_like(sig)).reshape(B, R, S, 1)
    relu = port.F.relu
    if mask is not None:
        port.F.relu = lambda v: v * mask.reshape(B, R, S, 1)
    try:
        rgbf, depth, w = port.ray_integration(out, z.reshape(B, R, S, 1), nz, noise_std, white_back, last_back,
                                              "softplus" if softplus else "relu")
    finally:
        port.F.relu = relu
    return torch.cat([rgbf, depth], -1), w.reshape(B, R * S)


# ---------------------------------------------------------------------------------------------------------------
# data
# ---------------------------------------------------------------------------------------------------------------
def gen(device, seed):
    return torch.Generator(device=device).manual_seed(seed)


def randn(g, *shape, scale=1.0):
    return torch.randn(*shape, generator=g, device=g.device) * scale


def rand_mod(g, B, n=C, sine=False):
    """Per-sample (g1, g0) tables [B,2,n] that differ strongly between samples: g1's sign alternates and its size grows with
    b; g0 is offset by b.  sine: FiLM frequencies around 15*N(0,1)+30 (modulated.py:43) and phases."""
    s = torch.arange(B, device=g.device, dtype=torch.float32)[:, None]
    if sine:
        g1 = 30.0 + 15.0 * torch.randn(B, n, generator=g, device=g.device) * (1 + 0.5 * s)
        g0 = torch.randn(B, n, generator=g, device=g.device) + s
    else:
        g1 = (0.5 + torch.rand(B, n, generator=g, device=g.device)) * (1 + s) * torch.where(s % 2 == 0, 1.0, -1.0)
        g0 = 0.5 * torch.randn(B, n, generator=g, device=g.device) + (s - (B - 1) / 2)
    return torch.stack([g1, g0], 1).contiguous()


def away_from_zero(x, mod):
    """Shift x so that |x*g1+g0| >= 0.04: the LeakyReLU / ReLU mask of the backward is discontinuous at 0 and a
    pre-activation within rounding distance of it may legitimately pick either side."""
    g1, g0 = (1.0, 0.0) if mod is None else (mod[:, 0, :, None], mod[:, 1, :, None])
    pre = x * g1 + g0
    bad = pre.abs() < 0.04
    return torch.where(bad, x + 0.1 / g1 * torch.where(pre >= 0, 1.0, -1.0), x)


def rel_l2(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm())


def assert_close(got, ref, tol=TOL, what=""):
    got, ref = got.double(), ref.double()
    assert torch.isfinite(got).all(), f"{what}: non-finite values"
    err = rel_l2(got, ref)
    assert err <= tol, f"{what}: rel-L2 {err:.3e} > {tol:.1e}"
    mx = float((got - ref).abs().max())
    assert mx <= 50 * tol * float(ref.abs().max()), f"{what}: max-abs {mx:.3e} vs max|ref| {float(ref.abs().max()):.3e}"


def assert_padding_untouched(t, HW, what=""):
    pad = padding_of(t, HW)
    assert bool((pad == SENT).all()), f"{what}: the kernel wrote padding rows"


def out_blocked(B, Cc, HW, device="cuda"):
    T = (HW + 127) // 128
    return torch.full((B, T, Cc, 128), SENT, dtype=torch.float32, device=device)


def pack(M):
    return _abi().pack_weight(M.float().contiguous(), Nb=256)[0]


def tol_of(passes):
    return TOL if passes == 3 else TOL_BF16


# ================================================================================================================
# forward engine: hg_conv1x1_blocked, hg_act_conv1x1_blocked, hg_blocked_conv_wide
# ================================================================================================================
@gpu
@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("Cin", [64, 128, 256])
def test_conv1x1_blocked(shape, Cin):
    """out = W x + bias; Cin 64 is one K chunk per tile (nkc = 1)."""
    abi = _abi()
    B, Hg, Wg = SHAPES[shape]
    HW = Hg * Wg
    g = gen("cuda", 100 + Cin)
    x, W, bias = randn(g, B, Cin, HW), randn(g, C, Cin, scale=Cin ** -0.5), randn(g, C)
    out = out_blocked(B, C, HW)
    abi.conv1x1_blocked(to_blocked(x, float("nan")), Cin, pack(W), bias, out, B=B, Hg=Hg, Wg=Wg, passes=3)
    ref, _, _ = fwd_ref(x, W, bias)
    assert_close(from_blocked(out, HW), ref, what=f"conv1x1_blocked Cin={Cin}")
    assert_padding_untouched(out, HW, "conv1x1_blocked")


@gpu
def test_conv1x1_blocked_bf16():
    abi = _abi()
    B, Hg, Wg = SHAPES["c_multi_tile"]
    HW = Hg * Wg
    g = gen("cuda", 7)
    x, W, bias = randn(g, B, 128, HW), randn(g, C, 128, scale=128 ** -0.5), randn(g, C)
    out = out_blocked(B, C, HW)
    abi.conv1x1_blocked(to_blocked(x, float("nan")), 128, pack(W), bias, out, B=B, Hg=Hg, Wg=Wg, passes=1)
    assert_close(from_blocked(out, HW), fwd_ref(x, W, bias)[0], tol=TOL_BF16, what="conv1x1_blocked bf16")


def _act_conv_case(g, B, HW, act, with_x2, big_args=False):
    sine = act == 1
    x = randn(g, B, C, HW, scale=30.0 if big_args else 1.0)
    x2 = randn(g, B, C, HW) if with_x2 else None
    mod = rand_mod(g, B, sine=sine)
    if big_args:      # |x*g1+g0| up to ~4000, the range reduce_2pi is written for
        mod[:, 0] = mod[:, 0].abs().clamp(20, 40)
        x = x.clamp(-100, 100)
    K = 512 if with_x2 else 256
    W, bias = randn(g, C, K, scale=K ** -0.5), randn(g, C)
    return x, x2, mod, W, bias


@gpu
@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("act", [0, 1])
@pytest.mark.parametrize("with_x2", [False, True])
def test_act_conv1x1_blocked(shape, act, with_x2):
    """out = W [act(x*g1+g0); act(x2*g1+g0)] + bias with per-sample tables that differ strongly between samples."""
    abi = _abi()
    B, Hg, Wg = SHAPES[shape]
    HW = Hg * Wg
    x, x2, mod, W, bias = _act_conv_case(gen("cuda", 200 + act + 2 * with_x2), B, HW, act, with_x2)
    out = out_blocked(B, C, HW)
    abi.act_conv1x1_blocked(to_blocked(x, float("nan")), mod, pack(W), bias, out, B=B, Hg=Hg, Wg=Wg,
                            x2=to_blocked(x2, float("nan")) if with_x2 else None, act=act, passes=3)
    ref, _, _ = fwd_ref(x, W, bias, mod=mod, act=act, x2=x2)
    assert_close(from_blocked(out, HW), ref, what=f"act_conv1x1_blocked act={act} x2={with_x2}")
    assert_padding_untouched(out, HW, "act_conv1x1_blocked")


@gpu
def test_act_conv1x1_blocked_sine_large_arguments():
    """sin of arguments up to ~4000.  reduce_2pi + __sinf claim ~2^-21 absolute error per element (the reference takes the
    kernel's fp32-rounded argument); through a K = 256 product of O(1/16) weights that is ~1e-6 relative, well inside TOL."""
    abi = _abi()
    B, Hg, Wg = SHAPES["c_multi_tile"]
    HW = Hg * Wg
    x, _, mod, W, bias = _act_conv_case(gen("cuda", 250), B, HW, 1, False, big_args=True)
    pre = f32_affine(x, mod[:, 0, :, None], mod[:, 1, :, None])
    assert float(pre.abs().max()) > 2500
    out = out_blocked(B, C, HW)
    abi.act_conv1x1_blocked(to_blocked(x, float("nan")), mod, pack(W), bias, out, B=B, Hg=Hg, Wg=Wg, act=1, passes=3)
    assert_close(from_blocked(out, HW), fwd_ref(x, W, bias, mod=mod, act=1)[0], what="sine, large arguments")


@gpu
def test_act_conv1x1_blocked_c2_render_size():
    """The renderer's first FiLM layer at C2 training size: K = 512 (coordinate and geometry halves), one table."""
    abi = _abi()
    B, Hg, Wg = C2_RENDER
    HW = Hg * Wg
    g = gen("cuda", 260)
    x, x2, mod, W, bias = _act_conv_case(g, B, HW, 1, True)
    out = torch.empty(B, HW // 128, C, 128, device="cuda")
    abi.act_conv1x1_blocked(to_blocked(x), mod, pack(W), bias, out, B=B, Hg=Hg, Wg=Wg, x2=to_blocked(x2), act=1, passes=3)
    assert_close(from_blocked(out, HW), fwd_ref(x, W, bias, mod=mod, act=1, x2=x2)[0], what="C2 render size")


@gpu
def test_act_conv1x1_blocked_bf16():
    abi = _abi()
    B, Hg, Wg = SHAPES["b_hw_1_mod_128"]
    HW = Hg * Wg
    x, x2, mod, W, bias = _act_conv_case(gen("cuda", 270), B, HW, 1, True)
    out = out_blocked(B, C, HW)
    abi.act_conv1x1_blocked(to_blocked(x), mod, pack(W), bias, out, B=B, Hg=Hg, Wg=Wg, x2=to_blocked(x2), act=1, passes=1)
    assert_close(from_blocked(out, HW), fwd_ref(x, W, bias, mod=mod, act=1, x2=x2)[0], tol=TOL_BF16, what="bf16")


def wide(x, x2, mod, mod2, act, slope, wimg, bias, skip, out, stats, rgb_w, rgb_b, rgb_in, rgb_out, *, B, Hg, Wg, passes=3):
    """hg_blocked_conv_wide has no typed wrapper (modules/wide_ops.py calls it through abi.call)."""
    abi = _abi()
    with torch.cuda.device_of(out):
        abi.call("hg_blocked_conv_wide", abi.ptr(x), abi.ptr(x2), abi.ptr(mod), abi.ptr(mod2), int(act), float(slope),
                 abi.ptr(wimg), abi.ptr(bias), abi.ptr(skip), abi.ptr(out), abi.ptr(stats), abi.ptr(rgb_w), abi.ptr(rgb_b),
                 abi.ptr(rgb_in), abi.ptr(rgb_out), B, Hg, Wg, passes, abi.stream())


def _run_wide(shape, *, skip, rgb, stats, act=0, slope=0.2, with_x2=True, with_mod2=True, passes=3, seed=300):
    B, Hg, Wg = shape
    HW = Hg * Wg
    g = gen("cuda", seed)
    x, x2, mod, W, bias = _act_conv_case(g, B, HW, act, with_x2)
    mod2 = rand_mod(g, B, sine=act == 1) if with_mod2 else None
    sk = randn(g, B, C, HW) if skip else None
    rw, rb, rin = (randn(g, 3, C, scale=C ** -0.5), randn(g, 3), randn(g, B, 3, HW)) if rgb else (None, None, None)
    out = out_blocked(B, C, HW)
    st = torch.zeros(2, C, dtype=torch.float64, device="cuda") if stats else None
    rout = torch.full((B, 3, HW), SENT, device="cuda") if rgb else None
    wide(to_blocked(x, float("nan")), to_blocked(x2, float("nan")) if with_x2 else None, mod, mod2, act, slope, pack(W), bias,
         to_blocked(sk, float("nan")) if skip else None, out, st, rw, rb, rin, rout, B=B, Hg=Hg, Wg=Wg, passes=passes)
    ref, rref, sref = fwd_ref(x, W, bias, mod=mod, act=act, slope=slope, x2=x2, mod2=mod2, skip=sk, rgb_w=rw, rgb_b=rb, rgb_in=rin)
    return out, rout, st, ref, rref, sref, HW


@gpu
@pytest.mark.parametrize("skip", [False, True], ids=["noskip", "skip"])
@pytest.mark.parametrize("rgb", [False, True], ids=["norgb", "rgb"])
@pytest.mark.parametrize("stats", [False, True], ids=["nostats", "stats"])
def test_blocked_conv_wide_epilogue_variants(skip, rgb, stats):
    """The 8 compiled forward epilogues (skip x ToRGB x statistics) at the multi-tile shape with a partial last tile."""
    out, rout, st, ref, rref, sref, HW = _run_wide(SHAPES["c_multi_tile"], skip=skip, rgb=rgb, stats=stats)
    assert_close(from_blocked(out, HW), ref, what="out")
    assert_padding_untouched(out, HW, "wide")
    if rgb:
        assert_close(rout, rref, what="rgb_out")
    if stats:
        assert_close(st[0], sref[0], what="sum")
        assert_close(st[1], sref[1], what="sumsq")


@gpu
@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("act,slope", [(0, 0.2), (0, 0.05), (1, 0.2)], ids=["lrelu0.2", "lrelu0.05", "sine"])
@pytest.mark.parametrize("with_mod2", [False, True], ids=["mod", "mod2"])
def test_blocked_conv_wide_modes(shape, act, slope, with_mod2):
    out, rout, st, ref, rref, sref, HW = _run_wide(SHAPES[shape], skip=True, rgb=True, stats=True, act=act, slope=slope,
                                                   with_mod2=with_mod2, seed=310 + act)
    assert_close(from_blocked(out, HW), ref, what="out")
    assert_close(rout, rref, what="rgb_out")
    assert_close(st, sref, what="stats")


@gpu
def test_blocked_conv_wide_k256_no_table():
    """One source, no modulation table: out = W LeakyReLU(x) + bias."""
    out, rout, st, ref, rref, sref, HW = _run_wide(SHAPES["b_hw_1_mod_128"], skip=False, rgb=False, stats=True, with_x2=False,
                                                   with_mod2=False, seed=320)
    assert_close(from_blocked(out, HW), ref, what="out")
    assert_close(st, sref, what="stats")


@gpu
def test_blocked_conv_wide_bf16():
    out, rout, st, ref, rref, sref, HW = _run_wide(SHAPES["c_multi_tile"], skip=True, rgb=True, stats=True, passes=1, seed=330)
    assert_close(from_blocked(out, HW), ref, tol=TOL_BF16, what="out")
    assert_close(rout, rref, tol=TOL_BF16, what="rgb_out")


# ================================================================================================================
# pixel-style half-block (hg_spade_conv with p_lr)
# ================================================================================================================
def _bilinear_up(p_lr, B, Rh, Rw, Hg, Wg):
    """[B,Rh*Rw,>=128] -> [B,128,Hg*Wg], fp64 F.interpolate(align_corners=False)."""
    p = p_lr[:, :, :128].double().reshape(B, Rh, Rw, 128).permute(0, 3, 1, 2)
    return F.interpolate(p, (Hg, Wg), mode="bilinear", align_corners=False).reshape(B, 128, Hg * Wg)


PIXEL_SHAPES = {"partial": (2, 20, 37, 7, 9), "multi_tile": (3, 100, 201, 13, 17), "b1_24x18": (1, 128, 96, 24, 18)}


@gpu
@pytest.mark.parametrize("shape", list(PIXEL_SHAPES))
@pytest.mark.parametrize("with_pbias", [False, True], ids=["nopbias", "pbias"])
def test_spade_conv_pixel_style(shape, with_pbias):
    """out = W lrelu((x*sc+sh)*gam + bet) + bias (+ skip, ToRGB, statistics) with gam|bet = Wgb relu(up(p_lr) + p_bias) + bgb:
    p_lr rows have stride 160 > 128 and NaN past column 128; Rh x Rw does not divide Hg x Wg."""
    abi = _abi()
    so = importlib.import_module("3dhumangan_b200.modules.synthesis_ops")
    B, Hg, Wg, Rh, Rw = PIXEL_SHAPES[shape]
    HW = Hg * Wg
    g = gen("cuda", 400)
    x = randn(g, B, C, HW)
    p_stride = 160
    p_lr = torch.full((B, Rh * Rw, p_stride), float("nan"), device="cuda")
    p_lr[:, :, :128] = randn(g, B, Rh * Rw, 128)
    p_bias = randn(g, B, 128, scale=0.5) if with_pbias else None
    wg_, bg_, wb_, bb_ = randn(g, C, 128, scale=0.1), randn(g, C, scale=0.1), randn(g, C, 128, scale=0.1), randn(g, C, scale=0.1)
    wgb, bgb = so._gamma_beta_interleaved(wg_, bg_, wb_, bb_)
    scsh = torch.stack([1 + 0.3 * randn(g, C), 0.3 * randn(g, C)]).contiguous()
    W, bias, skip = randn(g, C, C, scale=1 / 16), randn(g, C), randn(g, B, C, HW)
    rw, rb, rin = randn(g, 3, C, scale=1 / 16), randn(g, 3), randn(g, B, 3, HW)
    out = out_blocked(B, C, HW)
    st = torch.zeros(2, C, dtype=torch.float64, device="cuda")
    rout = torch.full((B, 3, HW), SENT, device="cuda")
    abi.spade_conv(to_blocked(x, float("nan")), (HW + 127) // 128 * C * 128, pack(W), bias, out, B=B, Hg=Hg, Wg=Wg,
                   scsh=scsh, p_lr=p_lr, p_stride=p_stride, p_bias=p_bias, wgb=pack(wgb), bgb=bgb,
                   skip=to_blocked(skip, float("nan")), stats=st, rgb_w=rw, rgb_b=rb, rgb_in=rin, rgb_out=rout, Rh=Rh, Rw=Rw)
    up = _bilinear_up(p_lr, B, Rh, Rw, Hg, Wg)
    a1 = torch.relu(up + (p_bias.double()[:, :, None] if with_pbias else 0.0))
    gam = torch.einsum("ok,bkp->bop", wg_.double(), a1) + bg_.double()[None, :, None] + 1
    bet = torch.einsum("ok,bkp->bop", wb_.double(), a1) + bb_.double()[None, :, None]
    pre = (x.double() * scsh[0, :, None].double() + scsh[1, :, None].double()) * gam + bet
    ref, rref, sref = fwd_ref(pre, W, bias, act=0, skip=skip, rgb_w=rw, rgb_b=rb, rgb_in=rin)
    assert_close(from_blocked(out, HW), ref, what="pixel-style out")
    assert_padding_untouched(out, HW, "pixel-style")
    assert_close(rout, rref, what="rgb_out")
    assert_close(st, sref, what="stats")


# ================================================================================================================
# data-gradient engine: hg_conv1x1_blocked_bwd
# ================================================================================================================
def _bwd_case(g, B, HW, *, cout=256, act=0, with_mod=True, ascale=False, with_g2=False, rk_n=0):
    sine = act == 1
    mod = rand_mod(g, B, cout, sine=sine) if with_mod else None
    aux = randn(g, B, cout, HW)
    if not sine:
        aux = away_from_zero(aux, mod)
    gg = randn(g, B, C, HW)
    g2 = randn(g, B, C, HW) if with_g2 else None
    K = 512 if with_g2 else 256
    M = randn(g, C, K, scale=K ** -0.5)          # rows >= cout carry data the kernel must ignore
    asc = (1.0 + torch.rand(B, C, generator=g, device=g.device)) * (1 + torch.arange(B, device=g.device)[:, None]) if ascale else None
    rk_w = randn(g, 3, C) if rk_n else None
    rk_v = randn(g, B, rk_n, HW) if rk_n else None
    return gg, g2, aux, mod, M, asc, rk_w, rk_v


def _run_bwd(shape, *, cout=256, act=0, slope=0.2, pixel_major=False, with_mod=True, ascale=False, with_g2=False, rk_n=0,
             passes=3, seed=500):
    abi = _abi()
    B, Hg, Wg = shape
    HW = Hg * Wg
    gg, g2, aux, mod, M, asc, rk_w, rk_v = _bwd_case(gen("cuda", seed), B, HW, cout=cout, act=act, with_mod=with_mod, ascale=ascale,
                                                       with_g2=with_g2, rk_n=rk_n)
    out = torch.full((B, HW, cout), SENT, device="cuda") if pixel_major else out_blocked(B, cout, HW)
    sums = torch.zeros(B, 2, cout, dtype=torch.float64, device="cuda")
    abi.conv1x1_blocked_bwd(to_blocked(gg, float("nan")), to_blocked(aux, float("nan")), pack(M), out, sums, B=B, Hg=Hg, Wg=Wg,
                            g2=to_blocked(g2, float("nan")) if with_g2 else None, mod=mod, Cout=cout, slope=slope,
                            pixel_major=pixel_major, passes=passes, act=act, ascale=asc, rk_w=rk_w, rk_v=rk_v)
    ref, sref = bwd_ref(gg, M, aux, cout=cout, mod=mod, act=act, slope=slope, ascale=asc, g2=g2, rk_w=rk_w, rk_v=rk_v)
    got = out.permute(0, 2, 1) if pixel_major else from_blocked(out, HW)
    if not pixel_major:
        assert_padding_untouched(out, HW, "conv1x1_blocked_bwd")
    return got, sums, ref, sref


# the 4 compiled backward epilogues
BWD_EPILOGUES = {
    "lrelu_tile_blocked": dict(act=0),
    "lrelu_pixel_major_cout128": dict(act=0, cout=128, pixel_major=True, slope=0.0, with_g2=True, with_mod=False),
    "sine": dict(act=1, ascale=True),
    "sine_rank_k": dict(act=1, rk_n=3),
}


@gpu
@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("variant", list(BWD_EPILOGUES))
def test_conv1x1_blocked_bwd_epilogues(shape, variant):
    got, sums, ref, sref = _run_bwd(SHAPES[shape], **BWD_EPILOGUES[variant])
    assert_close(got, ref, what=f"{variant} out")
    assert_close(sums, sref, what=f"{variant} S1/S2")


@gpu
@pytest.mark.parametrize("case", [
    dict(act=0, slope=0.0),                                        # ReLU mask
    dict(act=0, slope=0.2, with_mod=False),                        # mod None: g1 = 1, g0 = 0
    dict(act=0, slope=0.2, ascale=True),
    dict(act=0, slope=0.2, with_g2=True),                          # K = 512
    dict(act=0, cout=128, slope=0.2),                              # Cout 128, tile-blocked
    dict(act=0, cout=128, slope=0.0, with_g2=True, with_mod=False, pixel_major=True),   # synthesis_train.py's gamma/beta MLP
    dict(act=0, cout=128, slope=0.2, pixel_major=True, ascale=True),
    dict(act=1, ascale=False),
    dict(act=1, with_g2=True),
    dict(act=1, rk_n=1),
    dict(act=1, rk_n=2),
    dict(act=1, rk_n=3, ascale=True),
    dict(act=1, rk_n=2, with_mod=False),
], ids=lambda c: "-".join(f"{k}{v}" for k, v in c.items()))
def test_conv1x1_blocked_bwd_options(case):
    got, sums, ref, sref = _run_bwd(SHAPES["c_multi_tile"], seed=510, **case)
    assert_close(got, ref, what="out")
    assert_close(sums, sref, what="S1/S2")


@gpu
def test_conv1x1_blocked_bwd_c2_render_size():
    """The renderer's colour layer at C2 training size: sine mask, operand scale and the sigma head's rank-1 term."""
    got, sums, ref, sref = _run_bwd(C2_RENDER, act=1, ascale=True, rk_n=1, seed=520)
    assert_close(got, ref, what="out")
    assert_close(sums, sref, what="S1/S2")


@gpu
def test_conv1x1_blocked_bwd_bf16():
    got, sums, ref, sref = _run_bwd(SHAPES["c_multi_tile"], act=1, rk_n=3, passes=1, seed=530)
    assert_close(got, ref, tol=TOL_BF16, what="out")


# ================================================================================================================
# weight gradients: hg_wgrad_blocked, hg_act_wgrad_blocked
# ================================================================================================================
def _run_wgrad(shape, *, act=0, pscale=False, Cx=256, shared=False, with_mod=True, want_bias=True, via_act=True, passes=3, seed=600):
    abi = _abi()
    B, Hg, Wg = shape
    HW = Hg * Wg
    g = gen("cuda", seed)
    dout = randn(g, B, C, HW)
    x = randn(g, 1 if shared else B, Cx, HW)
    mod = rand_mod(g, B, C, sine=act == 1) if with_mod else None
    ps = (0.5 + torch.rand(B, C, generator=g, device="cuda")) * (1 + torch.arange(B, device="cuda")[:, None]) if pscale else None
    xb = to_blocked(x, float("nan"))
    xstride = 0 if shared else xb.shape[1] * Cx * 128
    if shared:
        xb = xb[0]
    db_ = to_blocked(dout, float("nan"))
    if via_act:
        dw, db = abi.act_wgrad_blocked(db_, xb, xstride, mod, B=B, Hg=Hg, Wg=Wg, act=act, pscale=ps, Cx=Cx, passes=passes)
    else:
        assert act == 0 and not pscale
        dw, db = abi.spade_bwd_wgrad(db_, xb, xstride, mod, B=B, Hg=Hg, Wg=Wg, passes=passes, want_bias=want_bias, Cx=Cx)
    dw_ref, db_ref = wgrad_ref(dout, x, mod=mod, act=act, pscale=ps)
    return dw, db, dw_ref, db_ref, (db_, xb, xstride, mod, ps)


@gpu
@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("act", [0, 1, 2])
def test_act_wgrad_blocked(shape, act):
    dw, db, dw_ref, db_ref, _ = _run_wgrad(SHAPES[shape], act=act, pscale=True, seed=600 + act)
    assert_close(dw, dw_ref, what=f"dW act={act}")
    assert_close(db, db_ref, what="dbias")


@gpu
@pytest.mark.parametrize("case", [
    dict(act=0, pscale=False),
    dict(act=1, pscale=False, Cx=128, with_mod=False),
    dict(act=2, pscale=True, Cx=128, with_mod=False),                 # the renderer's first layers (render_train.py:180)
    dict(act=0, Cx=128, with_mod=True),                               # mod [B,2,256]: rows past Cx unused
    dict(act=0, shared=True),                                         # x_bstride = 0 (the synthesis input)
    dict(act=1, shared=True, Cx=128, pscale=True),
], ids=lambda c: "-".join(f"{k}{v}" for k, v in c.items()))
def test_act_wgrad_blocked_options(case):
    dw, db, dw_ref, db_ref, _ = _run_wgrad(SHAPES["c_multi_tile"], seed=610, **case)
    assert_close(dw, dw_ref, what="dW")
    assert_close(db, db_ref, what="dbias")


@gpu
@pytest.mark.parametrize("Cx,with_mod,want_bias", [(256, True, True), (128, False, False), (256, False, False)])
def test_wgrad_blocked(Cx, with_mod, want_bias):
    dw, db, dw_ref, db_ref, _ = _run_wgrad(SHAPES["c_multi_tile"], Cx=Cx, with_mod=with_mod, want_bias=want_bias, via_act=False,
                                           seed=620)
    assert_close(dw, dw_ref, what="dW")
    if want_bias:
        assert_close(db, db_ref, what="dbias")
    else:
        assert db is None


@gpu
def test_act_wgrad_blocked_c2_render_size():
    dw, db, dw_ref, db_ref, _ = _run_wgrad(C2_RENDER, act=1, pscale=True, seed=630)
    assert_close(dw, dw_ref, what="dW")
    assert_close(db, db_ref, what="dbias")


@gpu
def test_act_wgrad_blocked_bf16():
    dw, db, dw_ref, db_ref, _ = _run_wgrad(SHAPES["c_multi_tile"], act=1, pscale=True, passes=1, seed=640)
    assert_close(dw, dw_ref, tol=TOL_BF16, what="dW")


@gpu
@pytest.mark.parametrize("act", [0, 1])
def test_wgrad_deterministic(act):
    """Per-CTA partials reduced in a fixed order in fp64 (DESIGN.md): two runs are bit-identical."""
    abi = _abi()
    shape = SHAPES["c_multi_tile"]
    B, Hg, Wg = shape
    dw, db, _, _, (d, xb, xs, mod, ps) = _run_wgrad(shape, act=act, pscale=True, seed=650)
    dw2, db2 = abi.act_wgrad_blocked(d, xb, xs, mod, B=B, Hg=Hg, Wg=Wg, act=act, pscale=ps, Cx=C)
    assert torch.equal(dw, dw2) and torch.equal(db, db2)


# ================================================================================================================
# renderer training kernels: hg_render_heads(_bwd), hg_render_composite(_bwd)
# ================================================================================================================
def _heads_case(g, B, N):
    out3, linc = randn(g, B, C, N), randn(g, B, C, N)
    mod3 = rand_mod(g, B, sine=True)
    w_sigma, w_rgb, hb = randn(g, C, scale=1 / 16), randn(g, 3, C, scale=1 / 16), randn(g, 4)
    return out3, linc, mod3, w_sigma, w_rgb, hb


@gpu
@pytest.mark.parametrize("B,N", [(2, 128), (3, 157 * 128), (1, 1024), C2_RENDER[::2]])
def test_render_heads(B, N):
    """sig = w_sigma . sin(f*out3+phi) + b0;  rgbp = W_rgb . sin(f*linc+phi) + b1..3; and the fp64 weight / bias sums of
    the backward."""
    abi = _abi()
    g = gen("cuda", 700)
    out3, linc, mod3, w_sigma, w_rgb, hb = _heads_case(g, B, N)
    sig, rgbp = abi.render_heads(to_blocked(out3), to_blocked(linc), mod3, w_sigma, w_rgb, hb, B=B, N=N)
    f, ph = mod3[:, 0, :, None], mod3[:, 1, :, None]
    h4, cc = torch.sin(f32_affine(out3, f, ph)), torch.sin(f32_affine(linc, f, ph))
    sig_ref = torch.einsum("c,bcp->bp", w_sigma.double(), h4) + hb[0].double()
    rgb_ref = torch.einsum("jc,bcp->bjp", w_rgb.double(), cc) + hb[1:].double()[None, :, None]
    assert_close(sig, sig_ref, what="sigma")
    assert_close(rgbp, rgb_ref, what="rgb")
    dsig, drgbp = randn(g, B, N), randn(g, B, 3, N)
    acc = abi.render_heads_bwd(to_blocked(out3), to_blocked(linc), mod3, dsig, drgbp, B=B, N=N)
    acc_ref = torch.cat([torch.einsum("bp,bcp->c", dsig.double(), h4), torch.einsum("bjp,bcp->jc", drgbp.double(), cc).reshape(-1),
                         dsig.double().sum().reshape(1), drgbp.double().sum((0, 2))])
    assert_close(acc, acc_ref, what="heads backward")


def _composite_case(g, B, R, S, *, softplus, saturate):
    N = R * S
    z = (torch.rand(B, R, S, generator=g, device="cuda") * 0.02 + 0.03).cumsum(-1) + 8.0
    sig = randn(g, B, R, S, scale=30.0)
    sig[:, : R // 4] = -50.0 - torch.rand(B, R // 4, S, generator=g, device="cuda")       # fully transparent rays
    if saturate:
        sig[:, R // 4: R // 2, : S // 4] = 1e3                                               # rays that saturate early
    noise = randn(g, B, R, S)
    rgbp, feat = randn(g, B, 3, N), randn(g, B, C, N)
    return sig.reshape(B, N).contiguous(), z.reshape(B, N).contiguous(), noise.reshape(B, N).contiguous(), rgbp, feat


@gpu
@pytest.mark.parametrize("S", [8, 16, 32, 64, 128])
@pytest.mark.parametrize("softplus", [False, True], ids=["relu", "softplus"])
@pytest.mark.parametrize("white_back,noise_std", [(True, 0.0), (False, 0.5)], ids=["white", "noise"])
def test_render_composite(port, S, softplus, white_back, noise_std):
    abi = _abi()
    B, R = 2, 25 * 128 // S                      # 25 tiles per sample: CTAs past the first, ray counts not a power of 2
    N = R * S
    g = gen("cuda", 800 + S)
    sig, z, noise, rgbp, feat = _composite_case(g, B, R, S, softplus=softplus, saturate=True)
    if noise_std > 0:
        pre = (sig.double() + noise.double() * noise_std)
        noise = torch.where(pre.abs() < 1e-2, noise + 0.1, noise)      # keep the ReLU clamp decision away from 0
    pre32 = (sig.double() + noise.double() * noise_std).float().double()
    mask = (pre32 > 0).double()
    assert 0.1 < float(mask.mean()) < 0.9
    nz = noise if noise_std > 0 else None
    kw = dict(B=B, R=R, S=S, noise_std=noise_std, white_back=white_back, softplus=softplus)
    ray_out, w = abi.render_composite(sig, z, nz, rgbp, to_blocked(feat), **kw)
    ref, w_ref = composite_ref(port, sig.double(), z.double(), nz.double() if nz is not None else None, rgbp.double(), feat.double(),
                               R=R, S=S, noise_std=noise_std, white_back=white_back, softplus=softplus)
    assert_close(ray_out, ref, what="ray_out")
    assert_close(w, w_ref, what="weights")
    # backward: fp64 autograd through the oracle on the kernel's clamp mask
    dray = randn(g, B, R, 260)
    dfeat, drgbp, dsig = abi.render_composite_bwd(sig, z, nz, rgbp, to_blocked(feat), dray, **kw)
    leaves = [t.double().requires_grad_(True) for t in (sig, rgbp, feat)]
    ref, _ = composite_ref(port, leaves[0], z.double(), nz.double() if nz is not None else None, leaves[1], leaves[2], R=R, S=S,
                           noise_std=noise_std, white_back=white_back, softplus=softplus, mask=None if softplus else mask)
    (ref[..., :259] * dray[..., :259].double()).sum().backward()
    assert_close(from_blocked(dfeat, N), leaves[2].grad, what="dfeat")
    assert_close(drgbp, leaves[1].grad, what="drgbp")
    assert_close(dsig, leaves[0].grad, what="dsigma")


@gpu
def test_render_composite_last_back(port):
    """last_back (forward only): the last sample absorbs the remaining transmittance."""
    abi = _abi()
    B, R, S = 1, 64, 32
    g = gen("cuda", 850)
    sig, z, noise, rgbp, feat = _composite_case(g, B, R, S, softplus=False, saturate=False)
    kw = dict(B=B, R=R, S=S, noise_std=0.0, white_back=False, softplus=False)
    ray_out, w = abi.render_composite(sig, z, None, rgbp, to_blocked(feat), last_back=True, **kw)
    ref, _ = composite_ref(port, sig.double(), z.double(), None, rgbp.double(), feat.double(), R=R, S=S, noise_std=0.0,
                           white_back=False, softplus=False, last_back=True)
    assert_close(ray_out, ref, what="ray_out last_back")


@gpu
def test_render_composite_c2_render_size(port):
    abi = _abi()
    B, _, N = C2_RENDER
    S = 32
    R = N // S
    g = gen("cuda", 860)
    sig, z, noise, rgbp, feat = _composite_case(g, B, R, S, softplus=False, saturate=True)
    kw = dict(B=B, R=R, S=S, noise_std=0.0, white_back=True, softplus=False)
    ray_out, w = abi.render_composite(sig, z, None, rgbp, to_blocked(feat), **kw)
    ref, w_ref = composite_ref(port, sig.double(), z.double(), None, rgbp.double(), feat.double(), R=R, S=S, noise_std=0.0,
                               white_back=True, softplus=False)
    assert_close(ray_out, ref, what="ray_out")


# ================================================================================================================
# pixel-style training pieces: hg_spade_a1, hg_spade_pixel_pre, hg_spade_pixel_mod_bwd, hg_bilinear_adjoint
# ================================================================================================================
ADJ_SHAPES = {"24x18_to_128x96": (2, 128, 96, 24, 18), "1to1": (2, 20, 30, 20, 30), "ragged": (3, 37, 41, 7, 9)}


@gpu
@pytest.mark.parametrize("shape", list(ADJ_SHAPES))
def test_spade_a1_and_bilinear_adjoint(shape):
    """A1 = relu(up(p_lr) + p_bias) against fp64 F.interpolate; its adjoint against autograd of that interpolation and by
    <A p, q> = <p, A^T q> with both kernels."""
    abi = _abi()
    B, Hg, Wg, Rh, Rw = ADJ_SHAPES[shape]
    HW = Hg * Wg
    g = gen("cuda", 900)
    stride = 136
    p_lr = torch.full((B, Rh * Rw, stride), float("nan"), device="cuda")
    p_lr[:, :, :128] = randn(g, B, Rh * Rw, 128)
    p_bias = randn(g, B, 128, scale=0.3)
    a1 = out_blocked(B, 128, HW)
    abi.spade_a1(p_lr, stride, p_bias, a1, B=B, Hg=Hg, Wg=Wg, Rh=Rh, Rw=Rw)
    up = _bilinear_up(p_lr, B, Rh, Rw, Hg, Wg)
    assert_close(from_blocked(a1, HW), torch.relu(up + p_bias.double()[:, :, None]), what="A1")
    assert bool((padding_of(a1, HW) == 0).all())               # the gather writes zeros into the padding rows
    # adjoint vs autograd of the fp64 interpolation
    da1 = randn(g, B, HW, 128)
    dp = torch.full((B * Rh * Rw, stride), SENT, device="cuda")
    abi.bilinear_adjoint(da1, dp, stride, B=B, Hg=Hg, Wg=Wg, Rh=Rh, Rw=Rw)
    pl = p_lr[:, :, :128].double().clone().requires_grad_(True)
    (_bilinear_up(pl, B, Rh, Rw, Hg, Wg) * da1.double().permute(0, 2, 1)).sum().backward()
    assert_close(dp[:, :128].reshape(B, Rh * Rw, 128), pl.grad, what="bilinear adjoint")
    assert bool((dp[:, 128:] == SENT).all())
    # <A p, q> = <p, A^T q> with both kernels (p >= 0 and no bias: the ReLU of spade_a1 is the identity)
    p = torch.rand(B, Rh * Rw, 128, generator=g, device="cuda")
    ap = torch.empty(B, (HW + 127) // 128, 128, 128, device="cuda")
    abi.spade_a1(p, 128, None, ap, B=B, Hg=Hg, Wg=Wg, Rh=Rh, Rw=Rw)
    atq = torch.empty(B * Rh * Rw, 128, device="cuda")
    abi.bilinear_adjoint(da1, atq, 128, B=B, Hg=Hg, Wg=Wg, Rh=Rh, Rw=Rw)
    lhs = (from_blocked(ap, HW).double() * da1.double().permute(0, 2, 1)).sum()
    rhs = (p.double().reshape(-1, 128) * atq.double()).sum()
    assert abs(float(lhs - rhs)) <= 1e-5 * float((from_blocked(ap, HW).double().abs() * da1.double().permute(0, 2, 1).abs()).sum())


@gpu
@pytest.mark.parametrize("shape", list(SHAPES))
def test_spade_pixel_pre_and_mod_bwd(shape):
    """pre = (x*sc+sh)*gam + bet;  backward: dxn = dpre*gam, dgam = dpre*(x*sc+sh), sums (sum dxn*x, sum dxn, sum dgam) over
    the valid pixels only, with NaN in every input's padding rows."""
    abi = _abi()
    B, Hg, Wg = SHAPES[shape]
    HW = Hg * Wg
    T = (HW + 127) // 128
    g = gen("cuda", 950)
    x, gam, bet, dpre = randn(g, B, C, HW), randn(g, B, C, HW), randn(g, B, C, HW), randn(g, B, C, HW)
    scsh = torch.stack([1 + 0.3 * randn(g, C), 0.3 * randn(g, C)]).contiguous()
    xb = to_blocked(x, float("nan"))
    pre = to_blocked(bet, float("nan"))
    abi.spade_pixel_pre(xb, T * C * 128, scsh, to_blocked(gam, float("nan")), pre, B=B, Hg=Hg, Wg=Wg)
    xn = x.double() * scsh[0, :, None].double() + scsh[1, :, None].double()
    assert_close(from_blocked(pre, HW), xn * gam.double() + bet.double(), what="pixel_pre")
    gd = to_blocked(gam, float("nan"))
    dxn = out_blocked(B, C, HW)
    sums = torch.zeros(3, C, dtype=torch.float64, device="cuda")
    abi.spade_pixel_mod_bwd(to_blocked(dpre, float("nan")), xb, T * C * 128, scsh, gd, dxn, sums, B=B, Hg=Hg, Wg=Wg)
    dxn_ref, dgam_ref = dpre.double() * gam.double(), dpre.double() * xn
    assert_close(from_blocked(dxn, HW), dxn_ref, what="dxn")
    assert_close(from_blocked(gd, HW), dgam_ref, what="dgam")
    assert_close(sums, torch.stack([(dxn_ref * x.double()).sum((0, 2)), dxn_ref.sum((0, 2)), dgam_ref.sum((0, 2))]), what="sums")
    assert bool((padding_of(dxn, HW) == 0).all()) and bool((padding_of(gd, HW) == 0).all())


@gpu
@pytest.mark.parametrize("B,Hg,Wg", [(2, 4, 25), (3, 4, 5005), (1, 20, 50)])      # drgb needs H*W a multiple of 4
def test_spade_bwd_combine_padding(B, Hg, Wg):
    """dx = dpre*g1 + a + k*x + dskip + rgb_w^T drgb and dW_rgb with NaN in every input's padding rows: the padding rows of
    dx are written as zeros and nothing reaches the valid pixels or dW_rgb."""
    abi = _abi()
    HW = Hg * Wg
    g = gen("cuda", 960)
    x, dpre, dskip, drgb = randn(g, B, C, HW), randn(g, B, C, HW), randn(g, B, C, HW), randn(g, B, 3, HW)
    rgb_w, g1, ak = randn(g, 3, C), randn(g, B, 2, C), randn(g, 2, C)
    ref = (dpre.double() * g1[:, 0, :, None].double() + ak[0, None, :, None].double() + ak[1, None, :, None].double() * x.double()
           + dskip.double() + torch.einsum("jc,bjp->bcp", rgb_w.double(), drgb.double()))
    dw_ref = torch.einsum("bjp,bcp->jc", drgb.double(), x.double())
    xb = to_blocked(x, float("nan"))
    dx = out_blocked(B, C, HW)
    dwrgb = torch.zeros(3, C, dtype=torch.float64, device="cuda")
    abi.spade_bwd_combine(dx, B=B, Hg=Hg, Wg=Wg, dpre=to_blocked(dpre, float("nan")), x=xb, x_bstride=xb.shape[1] * C * 128, g1=g1,
                          ak=ak, dskip=to_blocked(dskip, float("nan")), drgb=drgb, rgb_w=rgb_w, dwrgb=dwrgb)
    assert_close(from_blocked(dx, HW), ref, what="dx")
    assert bool((padding_of(dx, HW) == 0).all())
    assert_close(dwrgb, dw_ref, what="dW_rgb")


# ================================================================================================================
# hg_synth_input / _bwd, hg_bn_finalize
# ================================================================================================================
@gpu
@pytest.mark.parametrize("Hg,Wg,B", [(7, 11, 2), (3, 43, 1), (128, 96, 8)])
def test_synth_input_and_bwd(Hg, Wg, B):
    abi = _abi()
    HW = Hg * Wg
    T = (HW + 127) // 128
    g = gen("cuda", 1000)
    w, b = randn(g, C, 2), randn(g, C)
    ic, jc = torch.linspace(-1, 1, Hg, device="cuda"), torch.linspace(-1, 1, Wg, device="cuda")
    x0 = torch.full((T, C, 128), SENT, device="cuda")
    stats = torch.zeros(2, C, dtype=torch.float64, device="cuda")
    abi.synth_input(w, b, ic, jc, x0, stats, B)
    arg = (w[:, 0, None, None].double() * ic.double()[None, :, None] + w[:, 1, None, None].double() * jc.double()[None, None, :]
           + b.double()[:, None, None]).reshape(C, HW)
    ref = torch.sin(arg)
    assert_close(from_blocked(x0[None], HW)[0], ref, what="x0")
    assert bool((padding_of(x0[None], HW) == SENT).all())
    assert_close(stats, B * torch.stack([ref.sum(1), (ref * ref).sum(1)]), what="stats")
    dx = randn(g, B, C, HW)
    dw, db = abi.synth_input_bwd(to_blocked(dx, float("nan")), w, b, ic, jc, B)
    darg = torch.cos(arg) * dx.double().sum(0)
    ii = ic.double()[:, None].expand(Hg, Wg).reshape(-1)
    jj = jc.double()[None, :].expand(Hg, Wg).reshape(-1)
    assert_close(dw, torch.stack([(darg * ii).sum(1), (darg * jj).sum(1)], 1), tol=1e-5, what="dw")
    assert_close(db, darg.sum(1), tol=1e-5, what="db")


@gpu
@pytest.mark.parametrize("mode", ["count", "count_dev", "eval"])
@pytest.mark.parametrize("with_gb", [False, True], ids=["scsh", "gb"])
def test_bn_finalize(mode, with_gb):
    """nn.SyncBatchNorm semantics: biased variance to normalise, running_var with torch's unbiased n/(n-1), momentum."""
    abi = _abi()
    g = gen("cuda", 1100)
    B, n, momentum, eps = 3, 777.0, 0.3, 1e-5
    xs = randn(g, C, int(n), scale=2.0) + randn(g, C, 1)
    stats = torch.stack([xs.double().sum(1), (xs.double() ** 2).sum(1)]).contiguous()
    weight, bias = randn(g, C), randn(g, C)
    rm0, rv0 = randn(g, C), 0.5 + torch.rand(C, generator=g, device="cuda")
    rm, rv = rm0.clone(), rv0.clone()
    gb = torch.stack([1 + randn(g, B, C, scale=0.3), randn(g, B, C)], 1).contiguous() if with_gb else None
    scsh = torch.full((2, C), SENT, device="cuda")
    mod = torch.full((B, 2, C), SENT, device="cuda") if with_gb else None
    training = mode != "eval"
    cnt_dev = torch.tensor([n], dtype=torch.float64, device="cuda") if mode == "count_dev" else None
    abi.bn_finalize(stats if training else None, weight, bias, rm, rv, training, count=n if mode == "count" else 0.0,
                    count_dev=cnt_dev, gb=gb, B=B if with_gb else 0, scsh=scsh, mod=mod, eps=eps, momentum=momentum)
    if training:
        mean, var = xs.double().mean(1), xs.double().var(1, unbiased=False)
        assert_close(rm, (1 - momentum) * rm0.double() + momentum * mean, tol=1e-6, what="running_mean")
        assert_close(rv, (1 - momentum) * rv0.double() + momentum * xs.double().var(1, unbiased=True), tol=1e-6, what="running_var")
    else:
        mean, var = rm0.double(), rv0.double()
        assert torch.equal(rm, rm0) and torch.equal(rv, rv0)
    sc = weight.double() / torch.sqrt(var + eps)
    sh = bias.double() - mean * sc
    assert_close(scsh, torch.stack([sc, sh]), tol=1e-6, what="scale/shift")
    if with_gb:
        assert_close(mod, torch.stack([sc * gb[:, 0].double(), sh * gb[:, 0].double() + gb[:, 1].double()], 1), tol=1e-6, what="mod")


# ================================================================================================================
# batch independence: each output element's K-sum happens inside one tile in a fixed order
# ================================================================================================================
@gpu
@pytest.mark.parametrize("kind", ["forward", "backward_lrelu", "backward_sine_rk"])
def test_batch_independence(kind):
    """At B = 3 (303 tiles: CTAs take 2-3 tiles and walk across samples) every per-pixel output is bit-identical to running
    each sample alone at B = 1; the atomically accumulated sums agree within tolerance."""
    abi = _abi()
    B, Hg, Wg = 3, 1, 100 * 128 + 77
    HW = Hg * Wg
    T = (HW + 127) // 128
    g = gen("cuda", 1200)
    if kind == "forward":
        x, x2, mod, W, bias = _act_conv_case(g, B, HW, 0, True)
        mod2, skip = rand_mod(g, B), randn(g, B, C, HW)
        rw, rb, rin = randn(g, 3, C, scale=1 / 16), randn(g, 3), randn(g, B, 3, HW)
        wimg = pack(W)
        xb, x2b, skb = to_blocked(x), to_blocked(x2), to_blocked(skip)

        def run(sl, n):
            out, st = out_blocked(n, C, HW), torch.zeros(2, C, dtype=torch.float64, device="cuda")
            rout = torch.empty(n, 3, HW, device="cuda")
            wide(xb[sl].contiguous(), x2b[sl].contiguous(), mod[sl].contiguous(), mod2[sl].contiguous(), 0, 0.2, wimg, bias,
                 skb[sl].contiguous(), out, st, rw, rb, rin[sl].contiguous(), rout, B=n, Hg=Hg, Wg=Wg)
            return out, rout, st
    else:
        sine = kind == "backward_sine_rk"
        gg, g2, aux, mod, M, asc, rk_w, rk_v = _bwd_case(g, B, HW, act=int(sine), ascale=True, rk_n=3 if sine else 0)
        wimg = pack(M)
        gb_, auxb = to_blocked(gg), to_blocked(aux)

        def run(sl, n):
            out = out_blocked(n, C, HW)
            sums = torch.zeros(n, 2, C, dtype=torch.float64, device="cuda")
            abi.conv1x1_blocked_bwd(gb_[sl].contiguous(), auxb[sl].contiguous(), wimg, out, sums, B=n, Hg=Hg, Wg=Wg,
                                    mod=mod[sl].contiguous(), act=int(sine), ascale=asc[sl].contiguous(),
                                    rk_w=rk_w, rk_v=rk_v[sl].contiguous() if sine else None)
            return out, None, sums
    full = run(slice(0, B), B)
    singles = [run(slice(b, b + 1), 1) for b in range(B)]
    for b in range(B):
        assert torch.equal(full[0][b], singles[b][0][0]), f"sample {b}: per-pixel output differs"
        if full[1] is not None:
            assert torch.equal(full[1][b], singles[b][1][0])
    if kind == "forward":
        assert_close(full[2], sum(s[2] for s in singles), what="statistics")
    else:
        assert_close(full[2], torch.cat([s[2] for s in singles]), what="S1/S2")


# ================================================================================================================
# ABI refusals: RuntimeError before anything is launched (outputs keep their sentinel)
# ================================================================================================================
@gpu
def test_abi_refusals():
    abi = _abi()
    B, Hg, Wg = 2, 1, 256
    HW = Hg * Wg
    g = gen("cuda", 1300)
    gg = to_blocked(randn(g, B, C, HW))
    aux = to_blocked(randn(g, B, C, HW))
    aux128 = to_blocked(randn(g, B, 128, HW))
    wimg = pack(randn(g, C, C, scale=1 / 16))
    wimg512 = pack(randn(g, C, 512, scale=1 / 32))
    mod = rand_mod(g, B)
    asc = torch.ones(B, C, device="cuda")
    rk_w, rk_v = randn(g, 3, C), randn(g, B, 1, HW)

    def refused(fn, *outs):
        torch.cuda.synchronize()
        before = [o.clone() for o in outs]
        with pytest.raises(RuntimeError):
            fn()
        torch.cuda.synchronize()
        for o, b in zip(outs, before):
            assert torch.equal(o, b), "a refused call wrote its output"

    out, sums = out_blocked(B, C, HW), torch.zeros(B, 2, C, dtype=torch.float64, device="cuda")
    out_pm = torch.full((B, HW, C), SENT, device="cuda")
    kw = dict(B=B, Hg=Hg, Wg=Wg)
    refused(lambda: abi.conv1x1_blocked_bwd(gg, aux, wimg, out_pm, sums, pixel_major=True, Cout=256, **kw), out_pm, sums)
    refused(lambda: abi.conv1x1_blocked_bwd(gg, aux, wimg512, out, sums, g2=gg, ascale=asc, **kw), out, sums)
    refused(lambda: abi.conv1x1_blocked_bwd(gg, aux, wimg, out, sums, act=0, rk_w=rk_w, rk_v=rk_v, **kw), out, sums)
    refused(lambda: abi.conv1x1_blocked_bwd(gg, aux128, wimg, out, sums, act=1, Cout=128, rk_w=rk_w, rk_v=rk_v, **kw), out, sums)
    refused(lambda: wide(gg, None, mod, mod, 0, 0.2, wimg, torch.zeros(C, device="cuda"), None, out, None, None, None, None, None,
                         **kw), out)
    refused(lambda: wide(gg, gg, mod, None, 0, 1.5, wimg512, torch.zeros(C, device="cuda"), None, out, None, None, None, None, None,
                         **kw), out)       # LeakyReLU slope outside [0, 1]
    refused(lambda: abi.conv1x1_blocked(to_blocked(randn(g, B, 96, HW)), 96, wimg, torch.zeros(C, device="cuda"), out, **kw), out)
    sig = torch.zeros(B, 384, device="cuda")
    feat = torch.zeros(B, 3, C, 128, device="cuda")
    rgbp = torch.zeros(B, 3, 384, device="cuda")
    with pytest.raises(RuntimeError):
        abi.render_composite(sig, sig, None, rgbp, feat, B=B, R=32, S=12, noise_std=0.0, white_back=False, softplus=False)
    with pytest.raises(RuntimeError):
        abi.render_composite(sig[:, :136], sig[:, :136], None, rgbp[:, :, :136], feat, B=B, R=17, S=8, noise_std=0.0,
                             white_back=False, softplus=False)
    with pytest.raises(RuntimeError):
        abi.render_composite_bwd(sig, sig, None, rgbp, feat, torch.zeros(B, 32, 260, device="cuda"), B=B, R=32, S=12, noise_std=0.0,
                                 white_back=False, softplus=False)
    torch.cuda.synchronize()


# ================================================================================================================
# negative controls (CPU): the references under plausible kernel mistakes differ by >= 100x the GPU tolerance
# ================================================================================================================
NEG_SHAPES = {k: SHAPES[k] for k in ("a_one_partial_tile", "b_hw_1_mod_128")}


def _differs(a, b, tol=TOL):
    assert torch.isfinite(a).all() and torch.isfinite(b).all()
    d = rel_l2(a, b)
    assert d >= 100 * tol, f"the data cannot tell the mistake apart: rel-L2 {d:.2e}"


@pytest.mark.parametrize("shape", list(NEG_SHAPES))
def test_negative_wrong_sample_table(shape):
    B, Hg, Wg = NEG_SHAPES[shape]
    HW = Hg * Wg
    g = gen("cpu", 10)
    for act in (0, 1):
        x, x2, mod, W, bias = _act_conv_case(g, B, HW, act, True)
        wrong = mod.roll(1, 0)
        _differs(fwd_ref(x, W, bias, mod=mod, act=act, x2=x2)[0], fwd_ref(x, W, bias, mod=wrong, act=act, x2=x2)[0])
        gg, _, aux, modb, M, asc, rk_w, rk_v = _bwd_case(g, B, HW, act=act, ascale=True)
        ok = bwd_ref(gg, M, aux, mod=modb, act=act, ascale=asc)
        _differs(ok[0], bwd_ref(gg, M, aux, mod=modb.roll(1, 0), act=act, ascale=asc)[0])
        _differs(ok[0], bwd_ref(gg, M, aux, mod=modb, act=act, ascale=asc.roll(1, 0))[0])
        _differs(ok[1], bwd_ref(gg, M, aux, mod=modb.roll(1, 0), act=act, ascale=asc)[1])
        dout = randn(g, B, C, HW)
        _differs(wgrad_ref(dout, x, mod=mod, act=act)[0], wgrad_ref(dout, x, mod=wrong, act=act)[0])


@pytest.mark.parametrize("shape", list(NEG_SHAPES))
def test_negative_padding_not_zeroed(shape):
    """Padding rows taken into the statistics, S1/S2, dW: their data (here finite noise, NaN on the GPU) changes the sums."""
    B, Hg, Wg = NEG_SHAPES[shape]
    HW = Hg * Wg
    T = (HW + 127) // 128
    g = gen("cpu", 11)
    x, _, mod, W, bias = _act_conv_case(g, B, T * 128, 0, False)        # full tiles: the last T*128 - HW pixels are padding
    cut = lambda t: t[..., :HW]
    _differs(fwd_ref(cut(x), W, bias, mod=mod, act=0)[2], fwd_ref(x, W, bias, mod=mod, act=0)[2])
    gg, _, aux, modb, M, *_ = _bwd_case(g, B, T * 128)
    _differs(bwd_ref(cut(gg), M, cut(aux), mod=modb)[1], bwd_ref(gg, M, aux, mod=modb)[1])
    dout = randn(g, B, C, T * 128)
    _differs(wgrad_ref(cut(dout), cut(x), mod=mod)[0], wgrad_ref(dout, x, mod=mod)[0])
    _differs(wgrad_ref(cut(dout), cut(x), mod=mod)[1], wgrad_ref(dout, x, mod=mod)[1])


@pytest.mark.parametrize("shape", list(NEG_SHAPES))
def test_negative_bwd_epilogue_mistakes(shape):
    B, Hg, Wg = NEG_SHAPES[shape]
    HW = Hg * Wg
    g = gen("cpu", 12)
    gg, _, aux, mod, M, asc, _, _ = _bwd_case(g, B, HW, ascale=True)
    _differs(bwd_ref(gg, M, aux, mod=mod, slope=0.0)[0], bwd_ref(gg, M, aux, mod=mod, slope=0.2)[0])     # slope 0.2 for 0
    _differs(bwd_ref(gg, M, aux, mod=mod, ascale=asc)[0], bwd_ref(gg, M, aux, mod=mod)[0])                # ascale dropped
    gg, _, aux, mod, M, _, rk_w, rk_v = _bwd_case(g, B, HW, act=1, rk_n=3)
    ok = bwd_ref(gg, M, aux, mod=mod, act=1, rk_w=rk_w, rk_v=rk_v)[0]
    _differs(ok, bwd_ref(gg, M, aux, mod=mod, act=1)[0])                                                  # rank-k dropped
    _differs(ok, bwd_ref(gg, M, aux, mod=mod, act=1, rk_w=rk_w, rk_v=rk_v[:, :1])[0])                     # first row only
    _differs(bwd_ref(gg, M, aux, mod=mod, act=1, rk_w=rk_w, rk_v=rk_v[:, :2])[0],
             bwd_ref(gg, M, aux, mod=mod, act=1, rk_w=rk_w, rk_v=rk_v[:, :1])[0])                         # rk_n = 2 vs 1


@pytest.mark.parametrize("shape", list(NEG_SHAPES))
def test_negative_mod2_ignored(shape):
    B, Hg, Wg = NEG_SHAPES[shape]
    HW = Hg * Wg
    g = gen("cpu", 13)
    for act in (0, 1):
        x, x2, mod, W, bias = _act_conv_case(g, B, HW, act, True)
        mod2 = rand_mod(g, B, sine=act == 1)
        _differs(fwd_ref(x, W, bias, mod=mod, mod2=mod2, act=act, x2=x2)[0], fwd_ref(x, W, bias, mod=mod, act=act, x2=x2)[0])


def test_negative_tmem_halves_swapped():
    """Two consecutive tiles' outputs exchanged (the accumulator half of tile t read for tile t+1)."""
    B, Hg, Wg = SHAPES["b_hw_1_mod_128"]
    HW = Hg * Wg
    g = gen("cpu", 14)
    x, _, mod, W, bias = _act_conv_case(g, B, HW, 0, False)
    ok = to_blocked(fwd_ref(x, W, bias, mod=mod, act=0)[0])
    swapped = ok.clone()
    swapped[:, 0], swapped[:, 1] = ok[:, 1], ok[:, 0]
    _differs(from_blocked(ok, HW), from_blocked(swapped, HW))
    gg, _, aux, modb, M, *_ = _bwd_case(g, B, HW)
    ok_b = to_blocked(bwd_ref(gg, M, aux, mod=modb)[0])
    sw_b = ok_b.clone()
    sw_b[:, 0], sw_b[:, 1] = ok_b[:, 1], ok_b[:, 0]
    _differs(from_blocked(ok_b, HW), from_blocked(sw_b, HW))


def test_negative_last_back_dropped(port):
    B, R, S = 1, 64, 32
    g = gen("cpu", 15)
    z = (torch.rand(B, R, S, generator=g) * 0.02 + 0.03).cumsum(-1) + 8.0
    sig = torch.randn(B, R, S, generator=g) * 30.0
    sig[:, : R // 4] = -50.0
    rgbp, feat = torch.randn(B, 3, R * S, generator=g), torch.randn(B, C, R * S, generator=g)
    kw = dict(R=R, S=S, noise_std=0.0, white_back=False, softplus=False)
    a, _ = composite_ref(port, sig.reshape(B, -1).double(), z.reshape(B, -1).double(), None, rgbp.double(), feat.double(), last_back=True, **kw)
    b, _ = composite_ref(port, sig.reshape(B, -1).double(), z.reshape(B, -1).double(), None, rgbp.double(), feat.double(), last_back=False, **kw)
    _differs(a, b)


def test_reference_helpers_roundtrip():
    """to_blocked / from_blocked are inverse on the valid pixels and put `fill` in the padding rows only."""
    g = gen("cpu", 16)
    x = torch.randn(2, 5, 300, generator=g)
    xb = to_blocked(x, float("nan"))
    assert xb.shape == (2, 3, 5, 128)
    assert torch.equal(from_blocked(xb, 300), x)
    assert bool(padding_of(xb, 300).isnan().all()) and padding_of(xb, 300).shape == (2, 5, 84)
    assert float(xb[1, 2, 3, 7]) == float(x[1, 3, 2 * 128 + 7])
