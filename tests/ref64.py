"""fp64 references of the tensor-core convolution, the fused ResBlock pair and the AdaIN family, each with a bound
per output element on what the fp32 kernels may legitimately differ by.

Written from the contracts in include/artspeech_b200.h, in plain torch float64 on the CPU (independent of
tests/sim_backend.py).  Every function returns ``(ref, bound)``: a kernel output ``out`` is right when
``|out - ref| <= bound`` holds element by element (``check``).  Rows a contract masks are exact zeros with a bound of 0.

Rounding units: ``U32`` = 2^-24 (fp32), ``U16`` = 2^-11 (fp16) / 2^-8 (bf16).  The bounds are worst-case
(deterministic) error analyses of the kernels' fp32 arithmetic, not fitted tolerances; their derivations are next to
the code.  tests/test_ref64_cpu.py checks that fp32 models fall inside them and that small injected faults do not.
"""
from __future__ import annotations

import math

import torch

from artspeech_b200 import ops

U32 = 2.0 ** -24
EPS32 = 2.0 ** -23
U16 = {torch.float16: 2.0 ** -11, torch.bfloat16: 2.0 ** -8}
TINY = {torch.float16: 2.0 ** -24, torch.bfloat16: 2.0 ** -133, torch.float32: 2.0 ** -149}
D = torch.float64


def _d(t):
    return None if t is None else t.detach().to("cpu", D)


def _row_mask(B, T, lens, extra_dims=1):
    if lens is None:
        return torch.ones(B, T, *([1] * extra_dims), dtype=torch.bool)
    m = torch.arange(T)[None, :] < lens.cpu().long()[:, None]
    return m.reshape(B, T, *([1] * extra_dims))


# ------------------------------------------------------------------------------------------------------------------
# activations: value, Lipschitz constant, rounding of the fp32 evaluation
# ------------------------------------------------------------------------------------------------------------------
def _act(v, act, slope):
    if act == ops.ACT_NONE:
        return v, 1.0, torch.zeros_like(v)
    if act == ops.ACT_LRELU:          # max(v, v * slope): one rounded product
        return torch.where(v > 0, v, v * slope), max(1.0, abs(slope)), 2 * U32 * v.abs() * abs(slope)
    if act == ops.ACT_RELU:
        return v.clamp(min=0), 1.0, torch.zeros_like(v)
    if act == ops.ACT_ABS:
        return v.abs(), 1.0, torch.zeros_like(v)
    if act == ops.ACT_TANH:
        r = torch.tanh(v)
        return r, 1.0, 8 * EPS32 * r.abs() + 1e-7
    if act == ops.ACT_SWISH:          # |d/dv v*sigmoid(v)| <= 1.1
        r = v * torch.sigmoid(v)
        return r, 1.1, 8 * EPS32 * r.abs() + 1e-7
    raise ValueError(act)


def _to_out(ref, bound, dtype):
    """Rounding of the fp32 result into the output dtype: half an ulp of the value the kernel held (|ref| + bound)."""
    if dtype in U16:
        bound = bound + U16[dtype] * (ref.abs() + bound) + TINY[dtype]
    return ref, bound


# ------------------------------------------------------------------------------------------------------------------
# implicit-GEMM convolution (as_conv_igemm)
# ------------------------------------------------------------------------------------------------------------------
def _gather_taps(x4, taps, To, Fo):
    """Per tap, x[b, to + dt, fo + df, :] with zeros outside the input (the TMA out-of-bounds fill)."""
    B, T, F, _ = x4.shape
    for dt, df in taps:
        ti, fi = torch.arange(To) + dt, torch.arange(Fo) + df
        tv, fv = (ti >= 0) & (ti < T), (fi >= 0) & (fi < F)
        g = x4[:, ti.clamp(0, T - 1)][:, :, fi.clamp(0, F - 1)]
        yield g * (tv[None, :, None, None] & fv[None, None, :, None])


def _contract(x4, w, taps, To, Fo):
    """acc = sum_j x_j @ w_j^T and S = sum_j |x_j| @ |w_j|^T."""
    B = x4.shape[0]
    acc = torch.zeros(B, To, Fo, w.shape[1], dtype=D)
    S = torch.zeros_like(acc)
    for j, g in enumerate(_gather_taps(x4, taps, To, Fo)):
        acc += g @ w[j].t()
        S += g.abs() @ w[j].abs().t()
    return acc, S


def conv_v(x, w, taps, *, bias=None, res1=None, res2=None, scale=1.0, lens=None, out_shape=None):
    """Pre-activation value v of as_conv_igemm and its bound, before any output rounding.

    ``x`` 16-bit [B,T,C] or [B,T,F,C]; ``w`` [ntaps, Cout, Cin] holding the 16-bit weight values (any float dtype).
    Products of 16-bit operands are exact in fp32; the tensor-core accumulation over K = ntaps * CinP terms is bounded
    by (K + 2) * 2^-23 * sum |x * w| (each partial sum rounded or truncated once).  The epilogue adds bias, res1 and
    res2 (three fp32 roundings, each at most U32 * (sum |x w| + |bias| + |res1| + |res2|): 2^-23 covers the first on
    the products, 3 * U32 the rest) and multiplies by out_scale (U32 * |v|, counted twice for the output store).
    Returns ``(v, bound, valid)`` in fp64, shaped like the output; ``valid`` marks the rows t < lens[b]."""
    squeeze = x.dim() == 3
    x4 = _d(x.unsqueeze(2) if squeeze else x)
    B, T, F, Cin = x4.shape
    To, Fo = (T, F) if out_shape is None else out_shape
    w = _d(w)
    ntaps, Cout, _ = w.shape
    bk = 64 if Cin >= 64 else 32
    K = ntaps * ((Cin + bk - 1) // bk * bk)
    acc, S = _contract(x4, w, taps, To, Fo)
    extra = torch.zeros_like(acc)
    v = acc
    if bias is not None:
        b = _d(bias)[:Cout]
        v = v + b
        extra = extra + b.abs()
    for r in (res1, res2):
        if r is not None:
            r = _d(r).reshape(B, To, Fo, Cout)
            v = v + r
            extra = extra + r.abs()
    s = float(scale)
    v = v * s
    bound = abs(s) * ((K + 2) * EPS32 * S + 3 * U32 * extra) + 2 * U32 * v.abs()
    valid = _row_mask(B, To, lens, 2).expand(B, To, Fo, Cout)
    v = torch.where(valid, v, torch.zeros((), dtype=D))
    bound = torch.where(valid, bound, torch.zeros((), dtype=D))
    if squeeze:
        v, bound, valid = v.squeeze(2), bound.squeeze(2), valid.squeeze(2)
    return v, bound, valid


def conv_out(vb, act=ops.ACT_NONE, slope=0.0, dtype=torch.float32):
    """One output of the convolution from ``conv_v``: act(v) in ``dtype``."""
    v, bv, valid = vb
    r, L, rnd = _act(v, act, slope)
    ref, bound = _to_out(r, L * bv + rnd, dtype)
    zero = torch.zeros((), dtype=D)
    return torch.where(valid, ref, zero), torch.where(valid, bound, zero)


def conv(x, w, taps, *, bias=None, res1=None, res2=None, scale=1.0, lens=None, out_shape=None, act=ops.ACT_NONE,
         slope=0.0, dtype=torch.float32):
    """as_conv_igemm: ``(ref, bound)`` of the output act(v) stored as ``dtype`` (raw output: act = ACT_NONE)."""
    return conv_out(conv_v(x, w, taps, bias=bias, res1=res1, res2=res2, scale=scale, lens=lens, out_shape=out_shape),
                    act, slope, dtype)


# ------------------------------------------------------------------------------------------------------------------
# fused HiFi-GAN ResBlock pair (as_hifigan_resblock_pair)
# ------------------------------------------------------------------------------------------------------------------
def resblock_pair(xa, w1, b1, w2, b2, k, dil, *, slope, res2=None, res3=None, scale=1.0, out_act=ops.ACT_NONE,
                  out_slope=1.0, lens=None, dtype=None):
    """Contract of as_hifigan_resblock_pair.  ``w1`` / ``w2`` [k, C, C] (tap, cout, cin) holding 16-bit values.

    t is computed in fp64 and rounded to the 16-bit type, as the kernel rounds it.  The kernel's fp32 value of t
    before that rounding lies within the conv1 bound b1 of the fp64 one, so its 16-bit t equals the reference's
    wherever [t - b1, t + b1] holds no rounding midpoint; elsewhere it may land one ulp away.  conv2 therefore sees
    an operand error of at most round(t + b1) - round(t - b1) per element, carried by |w2|.  ``dtype`` is the output
    type (default: the activation dtype, as the kernel stores); torch.float32 gives the bound before that rounding."""
    dt = xa.dtype
    dtype = dt if dtype is None else dtype
    B, L, C = xa.shape
    a = _d(xa)
    x_raw = torch.where(a < 0, a / slope, a)
    xraw_err = torch.where(a < 0, 2 * U32 * x_raw.abs(), torch.zeros((), dtype=D))     # a * fl(1 / slope)
    valid = _row_mask(B, L, lens, 1)
    zero = torch.zeros((), dtype=D)
    v1, bv1, _ = conv_v(xa, w1, ops.taps_1d(k, dil), bias=b1)
    t_pre, _, rnd = _act(v1, ops.ACT_LRELU, slope)
    bt_pre = bv1 + rnd
    t_pre = torch.where(valid, t_pre, zero)
    bt_pre = torch.where(valid, bt_pre, zero)
    t16 = t_pre.to(dt)
    lo, hi = (t_pre - bt_pre).to(dt).to(D), (t_pre + bt_pre).to(dt).to(D)
    bt = hi - lo                                   # 0 unless a rounding midpoint lies within the conv1 bound
    t = t16.to(D)
    w2d = _d(w2)
    taps2 = ops.taps_1d(k, 1)
    acc, S = _contract(t.unsqueeze(2), w2d, taps2, L, 1)
    Sb, _ = _contract(bt.unsqueeze(2), w2d.abs(), taps2, L, 1)
    acc, S, Sb = acc.squeeze(2), S.squeeze(2), Sb.squeeze(2)
    v = acc + _d(b2) + x_raw
    extra = _d(b2).abs() + x_raw.abs()
    for r in (res2, res3):
        if r is not None:
            v = v + _d(r)
            extra = extra + _d(r).abs()
    s = float(scale)
    v = v * s
    K = k * C
    bound = abs(s) * ((K + 2) * EPS32 * (S + Sb) + Sb + 4 * U32 * extra + xraw_err) + 2 * U32 * v.abs()
    r, Lc, rnd = _act(v, out_act, out_slope)
    ref, bound = _to_out(r, Lc * bound + rnd, dtype)
    return torch.where(valid, ref, zero), torch.where(valid, bound, zero)


# ------------------------------------------------------------------------------------------------------------------
# instance-norm statistics and AdaIN (as_instnorm_stats, as_adain_apply, as_adain_norm_apply)
# ------------------------------------------------------------------------------------------------------------------
def _depth(n):
    """Longest chain of dependent fp32 additions in the kernels' reductions over n frames: at least 8 lanes, warps or
    CTAs share the frames of a channel (n / 8), then warp shuffles and cross-warp / cross-CTA folds (< 32)."""
    return math.ceil(n / 8) + 32


def _stats64(x, lens, eps):
    """fp64 mean / biased variance / rstd over valid frames, with bounds on the kernels' fp32 mean and rstd.

    Mean: a sum of depth-d chains has error <= d * U32 * sum |x - p| for the shift p the kernel sums about (0 for the
    plain two-pass kernels, a frame of the row for the ring kernel), so dm <= d U32 max(mean|x|, 2M) + 2 U32 |mean|,
    M = max |x - mean|.  Variance (two-pass around the fp32 mean, or shifted one-pass sum of squares): relative
    (d + 4) U32 on terms <= var + 2 M^2, plus the mean error's own 2 dm M + dm^2.  rstd = rsqrt(var + eps) over
    that interval, plus 4 U32 for rsqrtf."""
    B, T, C = x.shape
    xd = _d(x)
    lens_l = [T] * B if lens is None else [min(int(v), T) for v in lens.cpu()]
    mean = torch.zeros(B, C, dtype=D)
    var = torch.zeros(B, C, dtype=D)
    dm = torch.full((B, C), math.inf, dtype=D)
    dvar = torch.full((B, C), math.inf, dtype=D)
    for b, n in enumerate(lens_l):
        if n == 0:
            continue
        xb = xd[b, :n]
        m = xb.mean(0)
        dev = xb - m
        v = (dev * dev).mean(0)
        M = dev.abs().amax(0)
        d = _depth(n)
        dm_b = d * U32 * torch.maximum(xb.abs().mean(0), 2 * M) + 2 * U32 * m.abs()
        mean[b], var[b], dm[b] = m, v, dm_b
        dvar[b] = (d + 4) * U32 * (v + 2 * M * M) + 2 * dm_b * M + dm_b * dm_b
    rstd = (var + eps).rsqrt()
    r_lo = (var + eps + dvar).rsqrt()
    r_hi = torch.clamp(var + eps - dvar, min=1e-300).rsqrt()
    dr = torch.maximum(rstd - r_lo, r_hi - rstd) + 4 * U32 * r_hi
    return mean, rstd, dm, dr


def instnorm_stats(x, lens, eps=1e-5):
    """as_instnorm_stats: ``(ref, bound)`` of stats [B, C, 2] = {mean, rstd}; items with no valid frame get an
    infinite bound (the contract leaves their statistics open)."""
    mean, rstd, dm, dr = _stats64(x, lens, eps)
    return torch.stack([mean, rstd], -1), torch.stack([dm, dr], -1)


def _apply64(x, mean, rstd, dm, dr, gb, slope, lens, up_w, up_b, dtype):
    """a = lrelu((x - mean) * rstd * (1 + g) + beta) and the optional k3 s2 pool, with the mean / rstd errors
    (dm, dr) carried through and the fp32 evaluation's own roundings: x - mean, 1 + g, two products, + beta
    (5 U32 on the product chain, 2 U32 on |a| + |beta|); the pool's two products and two sums (4 U32)."""
    B, T, C = x.shape
    zero = torch.zeros((), dtype=D)
    xd = _d(x)
    g1 = 1 + _d(gb[:, :C])[:, None, :]
    be = _d(gb[:, C:2 * C])[:, None, :]
    m, r = mean[:, None, :], rstd[:, None, :]
    dev = xd - m
    a = dev * r * g1 + be
    dm_, dr_ = dm[:, None, :], dr[:, None, :]
    ba = g1.abs() * (dm_ * (r + dr_) + dev.abs() * dr_ + 5 * U32 * (dev.abs() + dm_) * (r + dr_)) + \
        2 * U32 * (a.abs() + be.abs())
    a, Lc, rnd = _act(a, ops.ACT_LRELU, slope)
    ba = Lc * ba + rnd
    valid = _row_mask(B, T, lens, 1)
    a = torch.where(valid, a, zero)
    ba = torch.where(valid, ba, zero)
    if up_w is not None:
        w = _d(up_w).reshape(C, 3)
        ub = _d(up_b)
        an = torch.cat([a[:, 1:], torch.zeros(B, 1, C, dtype=D)], 1)
        bn = torch.cat([ba[:, 1:], torch.zeros(B, 1, C, dtype=D)], 1)
        even = a * w[:, 1] + ub
        odd = a * w[:, 2] + an * w[:, 0] + ub
        be_ = w[:, 1].abs() * ba + 3 * U32 * ((a * w[:, 1]).abs() + ub.abs())
        bo_ = w[:, 2].abs() * ba + w[:, 0].abs() * bn + 4 * U32 * ((a * w[:, 2]).abs() + (an * w[:, 0]).abs() + ub.abs())
        a = torch.stack([even, odd], 2).reshape(B, 2 * T, C)
        ba = torch.stack([be_, bo_], 2).reshape(B, 2 * T, C)
        valid = _row_mask(B, 2 * T, None if lens is None else 2 * lens.cpu().long(), 1)
        a = torch.where(valid, a, zero)
        ba = torch.where(valid, ba, zero)
    ref, bound = _to_out(a, ba, dtype)
    return torch.where(valid, ref, zero), torch.where(valid, bound, zero)


def adain_apply(x, stats, gb, slope, lens, dtype, up_w=None, up_b=None):
    """as_adain_apply with the statistics taken as given (exact fp32 inputs)."""
    st = _d(stats)
    z = torch.zeros_like(st[..., 0])
    return _apply64(x, st[..., 0], st[..., 1], z, z, gb, slope, lens, up_w, up_b, dtype)


def adain_norm(x, gb, slope, lens, dtype, up_w=None, up_b=None, eps=1e-5):
    """as_adain_norm_apply: statistics in fp64 (their fp32 errors bounded by ``_stats64``), then ``adain_apply``."""
    mean, rstd, dm, dr = _stats64(x, lens, eps)
    dm = torch.where(torch.isfinite(dm), dm, torch.zeros((), dtype=D))    # items with no valid frame are all zeros
    dr = torch.where(torch.isfinite(dr), dr, torch.zeros((), dtype=D))
    return _apply64(x, mean, rstd, dm, dr, gb, slope, lens, up_w, up_b, dtype)


# ------------------------------------------------------------------------------------------------------------------
def check(out, ref, bound, what, rows_per_tile=128, cols_per_tile=None):
    """Assert |out - ref| <= bound element by element.  On failure, name the worst element by err / bound: its index
    (b, t, [f,] c), the tile it belongs to (item, row tile t // rows_per_tile, column tile c // cols_per_tile), the
    number of offending elements and the values involved."""
    o = out.detach().to("cpu", D)
    assert o.shape == ref.shape, f"{what}: shape {tuple(o.shape)} != {tuple(ref.shape)}"
    err = (o - ref).abs()
    bad = ~(err <= bound)                               # NaN counts as a failure
    if not bool(bad.any()):
        return
    ratio = torch.where(bad, err / bound.clamp(min=1e-300), torch.zeros((), dtype=D))
    ratio = torch.where(torch.isnan(ratio), torch.full((), math.inf, dtype=D), ratio)
    flat = int(torch.argmax(ratio))
    idx = tuple(int(i) for i in torch.unravel_index(torch.tensor(flat), ref.shape))
    b, t, c = idx[0], idx[1], idx[-1]
    tile = (b, t // rows_per_tile, c // cols_per_tile if cols_per_tile else 0)
    raise AssertionError(
        f"{what}: {int(bad.sum())} of {bad.numel()} elements outside the bound; worst at index {idx} "
        f"(tile item {tile[0]}, row tile {tile[1]}, column tile {tile[2]}): out {float(o[idx]):.9g} ref "
        f"{float(ref[idx]):.9g} err {float(err[idx]):.3e} bound {float(bound[idx]):.3e} ratio {float(ratio[idx]):.3g}")
