"""fp64 references of the memory-bound kernels (csrc/elementwise.cu) and of the single-output-channel convolution
(csrc/conv_cout1.cu), each with a bound per output element.

Written from the contracts in include/artspeech_b200.h, in plain torch float64 on the CPU (independent of
tests/sim_backend.py); checked with ``ref64.check``.  Every function returns ``(ref, bound)``; rows a contract masks are
exact zeros with a bound of 0.  Rounding units and the output rounding are those of tests/ref64.py.

Library calls: ``build.py`` passes no fast-math flag, so ``expf`` / ``tanhf`` / ``rsqrtf`` are within 2 ulp, ``logf``
within 1 ulp, and ``sqrtf`` and division are correctly rounded.  ``__expf`` (the GLU and ``ACT_SWISH``) is modelled as
in tests/ref64_seq.py: 2^-22 relative plus the rounding of its argument, 2^-24 |x|.  FMA contraction only removes
roundings, so every bound below counts one rounding per operation.

Pure copies (``repeat_rows``, ``length_regulate``, ``expand_tokens``, ``embed`` at scale 1 and an un-affine
``transpose_cast``) are bit-exact: their reference is the input rounded to the output dtype (round to nearest even, as
``__float2half_rn`` / ``__float2bfloat16_rn``) and their bound is 0.

The accumulating kernels (``conv_small*``, ``conv_cout1*``, ``dwconv*``) start their fp32 chain from the bias.  Each
of the chain's n additions rounds a partial sum that holds the bias, so the bias is charged n * U32 * |bias| on top of
``ref64.conv_v``'s bound (which charges it 3 U32 |bias|, right for the tensor-core epilogue that adds it once).
"""
from __future__ import annotations

import numpy as np
import torch

from artspeech_b200 import ops
from tests import audio_ref
from tests.ref64 import U32, _act, _d, _row_mask, _stats64, _to_out, conv_v
from tests.ref64_seq import EXP_REL

D = torch.float64
ZERO = torch.zeros((), dtype=D)


def _mask(ref, bound, valid):
    return torch.where(valid, ref, ZERO), torch.where(valid, bound, ZERO)


def _exact(v, dtype):
    """Bit-exact copy of fp32 values ``v`` into ``dtype``: the reference is the rounded value, the bound 0."""
    ref = v.to(torch.float32).to(dtype).to(D)
    return ref, torch.zeros_like(ref)


def _sig_fast(g):
    """sigmoid(g) and the relative error of the kernels' fp32 ``1 / (1 + __expf(-g))`` form (value / (1 + e)): the exp
    error moves 1 + e by (1 - s) of itself; the add and the divide round once each."""
    s = torch.sigmoid(g)
    return s, (1 - s) * (EXP_REL + U32 * g.abs()) + 3 * U32


def _act_mem(v, act, slope):
    """``ref64._act`` with ACT_SWISH as the kernels compute it: v / (1 + __expf(-v))."""
    if act != ops.ACT_SWISH:
        return _act(v, act, slope)
    s, rel = _sig_fast(v)
    r = v * s
    return r, 1.1, rel * r.abs() + 2.0 ** -126


def _out(v, bv, act, slope, dtype):
    r, L, rnd = _act_mem(v, act, slope)
    return _to_out(r, L * bv + rnd, dtype)


# ------------------------------------------------------------------------------------------------------------------
# embedding, LayerNorm
# ------------------------------------------------------------------------------------------------------------------
def embed(tokens, table, scale, lens, dtype):
    """as_embed: table[id] * scale, id outside [0, n_vocab) read as 0; one rounded product by the fp32 scale."""
    ids = tokens.cpu().long()
    ids = torch.where((ids >= 0) & (ids < table.shape[0]), ids, torch.zeros((), dtype=torch.long))
    B, T = ids.shape
    s32 = float(torch.tensor(float(scale), dtype=torch.float32))
    ref = _d(table)[ids] * s32
    if s32 == 1.0:
        ref, bound = _exact(ref, dtype)
    else:
        ref, bound = _to_out(ref, U32 * ref.abs(), dtype)
    return _mask(ref, bound, _row_mask(B, T, lens, 1))


def layernorm(x, gamma, beta, eps, act, slope, lens, dtype):
    """as_layernorm: y = act((x - mean) * rstd * gamma + beta) per row of C channels.

    The statistics are ``ref64._stats64`` over a [rows, C, 1] view: a lane sums ceil(C / 32) channels serially, then
    5 shuffles, a chain that ``_depth(C)`` covers; the variance is two-pass around the fp32 mean.  The affine part
    carries the mean / rstd errors (dm, dr) and rounds x - mean, two products and + beta (as ``ref64._apply64``)."""
    B, T, C = x.shape
    rows = B * T
    mean, rstd, dm, dr = _stats64(x.reshape(rows, C, 1), None, eps)          # [rows, 1] each
    xd = _d(x).reshape(rows, C)
    g, be = _d(gamma)[None, :], _d(beta)[None, :]
    dev = xd - mean
    a = dev * rstd * g + be
    ba = g.abs() * (dm * (rstd + dr) + dev.abs() * dr + 5 * U32 * (dev.abs() + dm) * (rstd + dr)) + \
        2 * U32 * (a.abs() + be.abs())
    ref, bound = _out(a, ba, act, slope, dtype)
    ref, bound = ref.reshape(B, T, C), bound.reshape(B, T, C)
    return _mask(ref, bound, _row_mask(B, T, lens, 1))


# ------------------------------------------------------------------------------------------------------------------
# copies: nearest upsample, length regulation, token expansion, layout change
# ------------------------------------------------------------------------------------------------------------------
def repeat_rows(x, rep, lens, dtype):
    """as_repeat_rows: out[b, r] = x[b, r / rep] for r < rep * min(lens[b], T), else 0."""
    B, T, C = x.shape
    xr = x.float().repeat_interleave(rep, 1)
    valid = _row_mask(B, T * rep, None if lens is None else lens.cpu().long().clamp(max=T) * rep, 1)
    return _mask(*_exact(torch.where(valid, xr, torch.zeros(())), dtype), valid)


def length_regulate(x, dur, lens_t, rep, To, dtype):
    """as_length_regulate: ``(ref, bound, out_lens)``.  Token j of item b covers frames [rep cum[j], rep cum[j + 1])
    with cum the exclusive prefix sum of max(dur, 0) over the first min(lens_t[b], Tt) tokens; durations past lens_t
    are never read; out_lens[b] = min(rep * sum, To)."""
    B, Tt, C = x.shape
    ref = torch.zeros(B, To, C, dtype=D)
    olens = torch.zeros(B, dtype=torch.int32)
    for b in range(B):
        nt = Tt if lens_t is None else max(0, min(int(lens_t[b]), Tt))
        d = dur[b, :nt].cpu().long().clamp(min=0)
        idx = torch.repeat_interleave(torch.arange(nt), d * rep)[:To]
        ref[b, :len(idx)] = _exact(x[b].float()[idx], dtype)[0]
        olens[b] = min(int(d.sum()) * rep, To)
    return ref, torch.zeros_like(ref), olens


def expand_tokens(x, tok):
    """as_expand_tokens: out[b, c, y] = x[b, c, tok[b, y]], 0 where tok is outside [0, Tx)."""
    B, C, Tx = x.shape
    t = tok.cpu().long()
    ok = (t >= 0) & (t < Tx)
    g = torch.gather(_d(x), 2, t.clamp(0, Tx - 1)[:, None, :].expand(B, C, -1))
    ref = torch.where(ok[:, None, :], g, ZERO)
    return ref, torch.zeros_like(ref)


def transpose_cast(src, to_cl, sub, mul, lens, dtype):
    """as_transpose_cast: dst[b, t, c] = src[b, c, t] (to_cl) or the inverse, y = (x - sub[c]) * mul[c] when given,
    frames t >= lens[b] zero.  Two fp32 roundings with the affine part, a bit-exact copy without."""
    s = _d(src)
    cf = s if to_cl else s.transpose(1, 2)                           # [B, C, T]
    B, C, T = cf.shape
    if sub is None:
        ref, bound = _exact(cf, dtype)
    else:
        y = (cf - _d(sub)[None, :, None]) * _d(mul)[None, :, None]
        ref, bound = _to_out(y, 3 * U32 * y.abs(), dtype)
    valid = _row_mask(B, T, lens, 0)[:, None, :]
    ref, bound = _mask(ref, bound, valid)
    if to_cl:
        ref, bound = ref.transpose(1, 2), bound.transpose(1, 2)
    return ref.contiguous(), bound.contiguous()


# ------------------------------------------------------------------------------------------------------------------
# pools and reductions
# ------------------------------------------------------------------------------------------------------------------
def _x4(x):
    return _d(x.unsqueeze(2) if x.dim() == 3 else x)


def avgpool(x, pt, pf, dtype):
    """as_avgpool: mean over pt x pf windows (stride = window), the last T row replicated when T % pt != 0, trailing F
    columns that fill no window dropped.  n - 1 additions (U32 sum |x| in all), 1 / (pt pf) and the product (2 U32)."""
    x4 = _x4(x)
    B, T, F, C = x4.shape
    To, Fo = -(-T // pt), F // pf
    ti = (torch.arange(To * pt)).clamp(max=T - 1)
    xp = x4[:, ti, :Fo * pf].reshape(B, To, pt, Fo, pf, C)
    ref = xp.mean((2, 4))
    bound = U32 * xp.abs().sum((2, 4)) + 2 * U32 * ref.abs()
    if x.dim() == 3:
        ref, bound = ref.squeeze(2), bound.squeeze(2)
    return _to_out(ref, bound, dtype)


def affine_act_maxpool(x, scale, shift, slope, pf, dtype):
    """as_affine_act_maxpool: max over pf consecutive F of lrelu(x * scale[c] + shift[c]).  Each candidate within 2 U32
    (|x scale| + |shift|), times the LeakyReLU's Lipschitz constant, plus its own rounding; max is 1-Lipschitz in the
    largest candidate error."""
    x4 = _d(x)
    B, T, F, C = x4.shape
    Fo = F // pf
    v = x4[:, :, :Fo * pf] * _d(scale) + _d(shift)
    bv = 2 * U32 * ((x4[:, :, :Fo * pf] * _d(scale)).abs() + _d(shift).abs())
    a, L, rnd = _act(v, ops.ACT_LRELU, slope)
    ba = L * bv + rnd
    ref = a.reshape(B, T, Fo, pf, C).amax(3)
    bound = ba.reshape(B, T, Fo, pf, C).amax(3)
    return _to_out(ref, bound, dtype)


def global_avgpool(x, slope, t_stride, dtype):
    """as_global_avgpool: mean of lrelu(x) over t = 0, ts, 2 ts, .. < T and every f.  One serial chain of n additions
    (n U32 sum |a|), the LeakyReLU products (U32 each) and the divide."""
    x4 = _x4(x)[:, ::t_stride]
    B, Tn, F, C = x4.shape
    n = Tn * F
    a = torch.where(x4 > 0, x4, x4 * slope)
    ref = a.mean((1, 2))
    bound = (n + 1) * U32 * a.abs().sum((1, 2)) / n + U32 * ref.abs()
    return _to_out(ref, bound, dtype)


def log_norm(mel):
    """as_log_norm: log(||exp(4 mel - 4)||_2) over the mel axis, an absolute bound (the value crosses 0).
    e = expf(4m - 4): 2 ulp (4 U32) plus the argument's rounding (U32 |4m - 4|) relative; e * e doubles that and rounds;
    the sum of M positive terms adds (M + 1) U32 relative; sqrtf halves the relative error and rounds (U32); logf turns a
    relative error into an absolute one and adds 1 ulp (2 U32 |out|)."""
    m = _d(mel)
    B, M, T = m.shape
    arg = 4 * m - 4
    e2 = torch.exp(2 * arg)
    s = e2.sum(1)
    de = 4 * U32 + U32 * arg.abs()
    ds = ((2 * de + U32) * e2).sum(1) / s + (M + 1) * U32
    ref = 0.5 * torch.log(s)
    bound = ds / 2 + U32 + 2 * U32 * ref.abs() + 1e-30
    return ref, bound


# ------------------------------------------------------------------------------------------------------------------
# convolutions that accumulate from the bias
# ------------------------------------------------------------------------------------------------------------------
def _bias_chain(bv, bias, n, Cout, scale=1.0):
    """Add the rounding of a chain of n additions that starts from the bias (see the module docstring)."""
    if bias is None:
        return bv
    return bv + abs(float(scale)) * n * U32 * _d(bias)[:Cout].abs()


def conv_small(x, w, bias, taps, lens, act, slope, dtype):
    """as_conv_small: ``ref64.conv_v`` (fp32 weights, any x dtype; ntaps * Cin fma steps inside its (K + 2) 2^-23 bound)
    plus the bias chain of ntaps * Cin additions.  Rows t >= lens[b] are zeros in both outputs."""
    vb = conv_v(x, w, taps, bias=bias, lens=lens)
    v, bv, valid = vb
    ntaps, Cout, Cin = w.shape
    bv = _bias_chain(bv, bias, ntaps * Cin, Cout)
    ref, bound = _out(v, bv, act, slope, dtype)
    return _mask(ref, bound, valid)


def conv_cout1(x, w, bias, taps, lens, scale, act, slope, dtype, path):
    """as_conv_igemm with Cout = 1 on conv_cout1_mma_kernel (``path`` "mma": ntaps fp32 additions of tensor-core
    partials) or conv_cout1_kernel ("fp32": ntaps * Cin / 8 additions of 8-product groups).  ``dtype`` torch.int16 is
    the AS_PCM16 epilogue: the codes ``audio_ref.encode`` accepts, as the midpoint of the two with half their distance
    as the bound."""
    v, bv, valid = conv_v(x, w, taps, bias=bias, lens=lens, scale=scale)
    ntaps, _, Cin = w.shape
    n = ntaps if path == "mma" else ntaps * -(-Cin // 8)
    bv = _bias_chain(bv, bias, n, 1, scale)
    if dtype != torch.int16:
        ref, bound = _out(v, bv, act, slope, dtype)
        return _mask(ref, bound, valid)
    r, L, rnd = _act_mem(v, act, slope)
    want, alt = audio_ref.encode(r.numpy(), (L * bv + rnd).numpy(), "pcm16")
    want, alt = torch.from_numpy(want.astype(np.float64)), torch.from_numpy(alt.astype(np.float64))
    return _mask((want + alt) / 2, (want - alt).abs() / 2, valid)


def dwconv(x, w, bias, k, stride, pad, glu, act, slope, lens_in, lens_out, dtype):
    """as_dwconv: depthwise conv over (T, F), input rows t >= lens_in[b] read as zero, output rows to >= lens_out[b]
    zero.  With GLU the input has 2C channels and the value is x[c] * sigmoid(x[C + c]) in the __expf form.  The chain
    starts from the bias and adds kt * kf products (fma): (n + 1) U32 (|bias| + sum |v w|), plus the GLU's relative error
    carried by |w|."""
    x4 = _x4(x)
    B, T, F, Cx = x4.shape
    (kt, kf), (st, sf), (pt, pf) = k, stride, pad
    if glu:
        C = Cx // 2
        s, rel = _sig_fast(x4[..., C:])
        val = x4[..., :C] * s
        verr = rel * val.abs()
    else:
        C = Cx
        val, verr = x4, torch.zeros_like(x4)
    vm = _row_mask(B, T, lens_in, 2)
    val = torch.where(vm, val, ZERO)                  # also clears NaN poison past lens_in
    verr = torch.where(vm, verr, ZERO)
    To = (T + 2 * pt - kt) // st + 1
    Fo = (F + 2 * pf - kf) // sf + 1
    wd = _d(w).reshape(kt, kf, C)
    acc = torch.zeros(B, To, Fo, C, dtype=D)
    S = torch.zeros_like(acc)
    E = torch.zeros_like(acc)
    for jt in range(kt):
        ti = torch.arange(To) * st + jt - pt
        tv = (ti >= 0) & (ti < T)
        for jf in range(kf):
            fi = torch.arange(Fo) * sf + jf - pf
            fv = (fi >= 0) & (fi < F)
            m = (tv[:, None] & fv[None, :])[None, :, :, None]
            g = val[:, ti.clamp(0, T - 1)][:, :, fi.clamp(0, F - 1)]
            ge = verr[:, ti.clamp(0, T - 1)][:, :, fi.clamp(0, F - 1)]
            g, ge = torch.where(m, g, ZERO), torch.where(m, ge, ZERO)
            acc += g * wd[jt, jf]
            S += (g * wd[jt, jf]).abs()
            E += ge * wd[jt, jf].abs()
    bb = torch.zeros(C, dtype=D) if bias is None else _d(bias)
    v = acc + bb
    bv = (kt * kf + 1) * U32 * (bb.abs() + S) + E
    ref, bound = _out(v, bv, act, slope, dtype)
    ref, bound = _mask(ref, bound, _row_mask(B, To, lens_out, 2))
    if x.dim() == 3:
        ref, bound = ref.squeeze(2), bound.squeeze(2)
    return ref, bound
