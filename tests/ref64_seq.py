"""fp64 references of the attention and LSTM kernels, each with a bound per output element.

Written from the contracts in include/artspeech_b200.h, in plain torch float64 on the CPU (independent of
tests/sim_backend.py); checked with ``ref64.check``.  Every function returns ``(ref, bound)``; rows a contract masks
are exact zeros with a bound of 0.

The tensor-core kernels round some operands to fp16 before they multiply: q, k, v, E_k, ``fl32(q + u)`` and
``fl32(q + v)``, the positions, and W_hh for H in {128, 256}.  That rounding is a function of the inputs alone, so the
references apply it themselves (``_h``) and the bounds cover only what is left:
  * fp32 accumulation: ``(n + 2) * 2^-23`` times the sum of |terms| for a length-n dot product in an unknown order
    (as ``ref64.conv_v``: every partial sum rounded or truncated once);
  * ``expf`` / ``__expf`` / MUFU ``ex2.approx`` / ``rcp.approx``: 2^-22 relative on the result plus the rounding of the
    argument (2^-24 |x| relative on exp(x)), and IEEE roundings of the few fp32 operations around them;
  * the fp16 rounding of the softmax weights P before P.V (u16 p_j per key, plus 2^-25 per key for fp16 subnormals,
    relative to the running maximum) -- ``l_run`` sums the unrounded fp32 p, so the rounding reaches the numerator only;
  * the output-dtype rounding (``ref64._to_out``).

Softmax.  A relative error e_j on each unnormalised weight p_j (score error d_j gives e_j = d_j to first order; exp
and the online rescaling add theirs) changes the output by at most
    sum_j P_j e_j |w_j| + (sum_k P_k e_k) * sum_j P_j |w_j|
where w_j is what key j contributes (v_j, plus E_v[j - i + w] inside the band).  Products of the small e terms are
below 2^-40 and are not carried.
"""
from __future__ import annotations

import math

import torch

from tests.ref64 import EPS32, U16, U32, _to_out

D = torch.float64
U16H = U16[torch.float16]
SUB16 = 2.0 ** -25                # half the smallest fp16 subnormal
EXP_REL = 4 * U32                 # ex2.approx / expf: 2^-22 relative
LSTM_CAP = 1e-3                   # bilstm: elements are checked against the derived bound while it is below this


def _h(t):
    """fp32 -> fp16 round-to-nearest, as __floats2half2_rn, then exact in fp64."""
    return t.float().half().double()


def _f(t):
    return t.float().double()


def _lens_list(B, T, lens):
    return [T] * B if lens is None else [max(0, min(int(v), T)) for v in lens.cpu()]


def _softmax_out(s, E, eps, v):
    """Shared part of the attention references for one item: scores ``s`` [H, L, L] with a per-key absolute bound
    ``E`` and per-key relative error ``eps`` of the exp.  Returns P, the row sums l of exp(s - max), P.v, the
    score-error terms of the bound for v, sum_j P_j |v_j|, the per-key relative errors e and A = sum_k P_k e_k."""
    m = s.amax(-1, keepdim=True)
    p = torch.exp(s - m)
    l = p.sum(-1, keepdim=True)
    P = p / l
    e = E + eps
    pv_abs = P @ v.abs()
    A = (P * e).sum(-1, keepdim=True)
    return P, l, P @ v, (P * e) @ v.abs() + A * pv_abs, pv_abs, e, A


# ------------------------------------------------------------------------------------------------------------------
# windowed relative-position attention (as_relpos_attention)
# ------------------------------------------------------------------------------------------------------------------
RM_KT = 64                        # keys per tile of relpos_attention_mma_kernel (online-softmax rescales per tile)


def relpos_attention(qkv, ek, ev, window, H, lens, out_dtype, path):
    """as_relpos_attention: ``(ref, bound)`` [B, T, H*D].  ``path`` = "mma" (fp16 operands, fp32 accumulation, online
    softmax over 64-key tiles, P rounded to fp16 before P.V) or "fp32" (fp32 throughout, softmax in shared memory).

    Scores s_ij = (q_i.k_j + [|j-i| <= w] q_i.Ek[j-i+w]) * rsqrt(D).  Their error: the two dot products
    ((D + 2) 2^-23 sum |q||k|, sum |q||Ek|), the add (U32), the product by rsqrtf(D) (2 ulp) and its rounding: 6 U32 |s|.
    Per-key relative error of p_j: exp (4 U32), its argument s_j - m (3 U32 |s_j - m|); for the mma kernel also the
    rescale factors alpha = exp(m_old - m_new), one per tile (4 U32 each plus 2 U32 |m_old - m_new|, summing to at most
    2 U32 (max_j s - min_j s)).  Accumulation: P.V and the row sum l over L keys ((L + 2) 2^-23 each, the output and
    1/l), the per-tile rescales (2 U32 each) and the epilogue (normalise, 2w + 1 band FMAs: (2w + 4) U32)."""
    mma = path == "mma"
    rnd = _h if mma else _f
    B, T, C3 = qkv.shape
    HD = C3 // 3
    Dh = HD // H
    nrel = 2 * window + 1
    ekd = rnd(ek.reshape(-1, Dh)[:nrel])
    evd = _f(ev.reshape(-1, Dh)[:nrel])
    scale = 1.0 / math.sqrt(Dh)
    ref = torch.zeros(B, T, HD, dtype=D)
    bound = torch.zeros(B, T, HD, dtype=D)
    for b, L in enumerate(_lens_list(B, T, lens)):
        if L == 0:
            continue
        x = qkv[b, :L].float()
        q, k, v = [rnd(x[:, i * HD:(i + 1) * HD]).reshape(L, H, Dh).transpose(0, 1) for i in range(3)]
        s = q @ k.transpose(1, 2)
        S = q.abs() @ k.abs().transpose(1, 2)
        qe, QE = q @ ekd.t(), q.abs() @ ekd.abs().t()                     # [H, L, nrel]
        rel = torch.arange(L)[None, :] - torch.arange(L)[:, None]         # j - i
        inb = rel.abs() <= window
        ridx = (rel + window).clamp(0, nrel - 1).expand(H, L, L)
        s = s + torch.where(inb, torch.gather(qe, 2, ridx), torch.zeros((), dtype=D))
        S = S + torch.where(inb, torch.gather(QE, 2, ridx), torch.zeros((), dtype=D))
        raw = s
        s = s * scale
        E = scale * ((Dh + 2) * EPS32 * S + U32 * raw.abs()) + 6 * U32 * s.abs()
        m = s.amax(-1, keepdim=True)
        nt = -(-L // RM_KT) if mma else 0
        eps = EXP_REL + 3 * U32 * (s - m).abs()
        if mma:
            eps = eps + 2 * U32 * (m - s.amin(-1, keepdim=True)) + 4 * U32 * nt
        P, l, out, bnd, pv_abs, e, A = _softmax_out(s, E, eps, v)
        # rel-value term: sum_r P_{i,i+r} Ev[r] (fp32 scores and E_v in both kernels)
        Pb = torch.zeros(H, L, nrel, dtype=D)
        eb = torch.zeros(H, L, nrel, dtype=D)
        ii = torch.arange(L)
        for r in range(nrel):
            j = ii + r - window
            ok = (j >= 0) & (j < L)
            jc = j.clamp(0, L - 1)
            Pb[:, :, r] = torch.where(ok, P[:, ii, jc], torch.zeros((), dtype=D))
            eb[:, :, r] = torch.where(ok, e[:, ii, jc], torch.zeros((), dtype=D))
        out = out + Pb @ evd
        pe_abs = Pb @ evd.abs()
        bnd = bnd + (Pb * eb) @ evd.abs() + A * pe_abs
        acc = 2 * (L + 2) * EPS32 + (2 * nt + 2 * window + 4) * U32
        bnd = bnd + acc * (pv_abs + pe_abs)
        if mma:   # P rounded to fp16 (relative to the running max, which the rescales only shrink) before P.V
            bnd = bnd + U16H * pv_abs + SUB16 / l * v.abs().sum(1, keepdim=True)
        ref[b, :L] = out.transpose(0, 1).reshape(L, HD)
        bound[b, :L] = bnd.transpose(0, 1).reshape(L, HD)
    return _to_out(ref, bound, out_dtype)


# ------------------------------------------------------------------------------------------------------------------
# conformer (Transformer-XL) attention (as_conformer_attention)
# ------------------------------------------------------------------------------------------------------------------
CM_KT = 64                        # keys per tile of conformer_attention_mma_kernel


def shift_index(L):
    """The reference's view-based relative shift on an item's own [L x L] position scores M (attention.py:105-113):
    out[a][j] = M[i2][jj - 1] with (i2, jj) = divmod((a + 1) L + j, L + 1), 0 where jj == 0.  Returns (row, col, live)
    index tensors [L, L]; row may be L (the padded row a + 1 = L, which carries the bias v only)."""
    a = torch.arange(L)[:, None]
    j = torch.arange(L)[None, :]
    f = (a + 1) * L + j
    i2, jj = f // (L + 1), f % (L + 1)
    return i2, (jj - 1).clamp(min=0), jj != 0


def conformer_attention(q, k, v, pos, u_bias, v_bias, H, lens, out_dtype, path, shift_len=None):
    """as_conformer_attention: ``(ref, bound)`` [B, T, H*D].  ``path`` = "mma" (fp16 operands including
    fp16(fl32(q + u)) / fp16(fl32(q + v)), online softmax over 64-key tiles, fp16 P) or "fp32" (the tiled and the
    per-query kernels: fl32(q + u) / fl32(q + v), fp32 throughout).  Queries at or beyond the item's length are
    zeros; the row a + 1 = L of the position scores is (0 + v) . pos.

    Score error: the content and position dot products ((D + 2) 2^-23 sum |.||.| each), their sum (U32), the product by
    rsqrt(H D) (exact for H D = 256; 2 U32 |s| allowed).  Softmax, accumulation and P rounding as relpos_attention.
    ``shift_len`` (tests only) takes the shift over a different length than the item's own."""
    mma = path == "mma"
    rnd = _h if mma else _f
    B, T, HD = q.shape
    Dh = HD // H
    ub, vb = u_bias.reshape(HD).float(), v_bias.reshape(HD).float()
    scale = 1.0 / math.sqrt(HD)
    ref = torch.zeros(B, T, HD, dtype=D)
    bound = torch.zeros(B, T, HD, dtype=D)
    for b, L in enumerate(_lens_list(B, T, lens)):
        if L == 0:
            continue
        qf = q[b, :L].float()
        qpad = torch.cat([qf, torch.zeros(1, HD)], 0)                        # row L: bias only
        qu = rnd(qf + ub).reshape(L, H, Dh).transpose(0, 1)                 # the fp32 sum, then (mma) fp16
        qv = rnd(qpad + vb).reshape(L + 1, H, Dh).transpose(0, 1)
        kk = rnd(k[b, :L]).reshape(L, H, Dh).transpose(0, 1)
        vv = rnd(v[b, :L]).reshape(L, H, Dh).transpose(0, 1)
        pp = rnd(pos[:L]).reshape(L, H, Dh).transpose(0, 1)
        c, C = qu @ kk.transpose(1, 2), qu.abs() @ kk.abs().transpose(1, 2)
        M, MA = qv @ pp.transpose(1, 2), qv.abs() @ pp.abs().transpose(1, 2)   # [H, L + 1, L]
        Ls = L if shift_len is None else shift_len
        row, col, live = shift_index(Ls)
        row, col, live = row[:L, :L].clamp(max=L), col[:L, :L].clamp(max=L - 1), live[:L, :L]
        z = torch.zeros((), dtype=D)
        sh = torch.where(live, M[:, row, col], z)
        SH = torch.where(live, MA[:, row, col], z)
        raw = c + sh
        s = raw * scale
        E = scale * ((Dh + 2) * EPS32 * (C + SH) + U32 * raw.abs()) + 2 * U32 * s.abs()
        m = s.amax(-1, keepdim=True)
        nt = -(-L // CM_KT) if mma else 0
        eps = EXP_REL + 3 * U32 * (s - m).abs()
        if mma:
            eps = eps + 2 * U32 * (m - s.amin(-1, keepdim=True)) + 4 * U32 * nt
        P, l, out, bnd, pv_abs, _, _ = _softmax_out(s, E, eps, vv)
        bnd = bnd + (2 * (L + 2) * EPS32 + (2 * nt + 4) * U32) * pv_abs
        if mma:
            bnd = bnd + U16H * pv_abs + SUB16 / l * vv.abs().sum(1, keepdim=True)
        ref[b, :L] = out.transpose(0, 1).reshape(L, HD)
        bound[b, :L] = bnd.transpose(0, 1).reshape(L, HD)
    return _to_out(ref, bound, out_dtype)


# ------------------------------------------------------------------------------------------------------------------
# LSTM cell arithmetic
# ------------------------------------------------------------------------------------------------------------------
def _dsig_max(x, dx):
    """sup of sigmoid' over [x - dx, x + dx] (attained at the point nearest 0)."""
    y = torch.sigmoid(torch.clamp(torch.zeros_like(x), x - dx, x + dx))
    return y * (1 - y)


def _dtanh_max(x, dx):
    y = torch.tanh(torch.clamp(torch.zeros_like(x), x - dx, x + dx))
    return 1 - y * y


def _sig_err(x, s):
    """Error of the fp32 sigmoid forms 1 / (1 + exp(-x)) (expf, IEEE divide) and rcp.approx(1 + ex2.approx(-x log2e))
    (gsigm): exp relative 4 U32 + U32 |x| on its argument moves s by s (1 - s) times that; 1 + e and the reciprocal
    add 2 U32 s relative each (rcp.approx: 1 ulp)."""
    return s * (1 - s) * (EXP_REL + U32 * x.abs()) + 4 * U32 * s + 2.0 ** -126


def _tanh_err(x, t, mufu):
    """tanhf: 2 ulp (4 U32 |t|).  gtanh = 1 - 2 rcp(1 + ex2(2 x log2e)): the reciprocal r = (1 - t) / 2 carries the
    sigmoid-form error at argument 2x, doubled, plus the final fma's rounding."""
    if not mufu:
        return 4 * U32 * t.abs() + 2.0 ** -126
    r = (1 - t) / 2
    return 2 * (r * (1 - r) * (EXP_REL + 2 * U32 * x.abs()) + 4 * U32 * r) + U32


def _cell(g, c, dg, dc, H, mufu):
    """One cell update from gate pre-activations g [.., 4H] (order i, f, g, o) with bounds dg; returns h, c and their
    bounds (first order in the interval derivative bounds, plus the products of the input errors)."""
    gi, gf, gg, go = g.split(H, -1)
    di_, df_, dgg_, do_ = dg.split(H, -1)
    i, f, o = torch.sigmoid(gi), torch.sigmoid(gf), torch.sigmoid(go)
    t = torch.tanh(gg)
    di = _dsig_max(gi, di_) * di_ + _sig_err(gi, i)
    df = _dsig_max(gf, df_) * df_ + _sig_err(gf, f)
    do = _dsig_max(go, do_) * do_ + _sig_err(go, o)
    dt = _dtanh_max(gg, dgg_) * dgg_ + _tanh_err(gg, t, mufu)
    c2 = f * c + i * t
    dc2 = (f + df) * dc + c.abs() * df + (i + di) * dt + t.abs() * di + 2 * U32 * ((i * t).abs() + c2.abs())
    tc = torch.tanh(c2)
    dtc = _dtanh_max(c2, dc2) * dc2 + _tanh_err(c2, tc, mufu)
    h = o * tc
    dh = (o + do) * dtc + tc.abs() * do + U32 * h.abs()
    return h, c2, dh, dc2


def lstm_onestep(xproj, H, out_dtype):
    """as_lstm_onestep: one step from zero state per row and direction, fp32 expf / tanhf.  ``(ref, bound)``
    [rows.., 2H]."""
    x = _f(xproj)
    hs, bs = [], []
    for d in range(2):
        g = x[..., d * 4 * H:(d + 1) * 4 * H]
        z = torch.zeros(g.shape[:-1] + (H,), dtype=D)
        h, _, dh, _ = _cell(g, z, torch.zeros_like(g), z, H, mufu=False)
        hs.append(h)
        bs.append(dh)
    return _to_out(torch.cat(hs, -1), torch.cat(bs, -1), out_dtype)


# ------------------------------------------------------------------------------------------------------------------
# bidirectional LSTM recurrence (as_bilstm)
# ------------------------------------------------------------------------------------------------------------------
def bilstm(xproj, whh_t, H, lens, out_dtype, reverse_at_T=False):
    """as_bilstm, packed-sequence semantics, the reverse direction from lens[b] - 1.  Returns ``(ref, bound)``
    [B, T, 2H] with bound = inf where the derived bound has passed ``LSTM_CAP``.

    H in {128, 256}: W_hh and the h operand are fp16 (tensor cores), c and h fp32, MUFU gsigm / gtanh; the reference
    rounds W_hh and its own h to fp16 as the kernel does.  H = 64: fp32 W_hh and h, expf / tanhf.

    The bound is propagated with the recurrence: the kernel's h (within dh of the reference's) becomes the operand
    fp16(h_kernel), which differs from fp16(h_ref) by at most the width of fp16([h - dh, h + dh]) -- zero unless a
    rounding midpoint lies within dh (H = 64: dh itself).  Gates: sum_k |W_kr| times that, plus the accumulation of
    x + W^T h over H + 1 terms ((H + 3) 2^-23 of the sum of |terms|).  The cell update is ``_cell``.  A worst-case
    bound like this grows step by step; elements are given an infinite bound once their item and direction has passed
    ``LSTM_CAP``; tests check the rest against a fitted tolerance.

    ``reverse_at_T`` (tests only): start the reverse direction at T - 1 instead of lens[b] - 1."""
    B, T, _ = xproj.shape
    q16 = H in (128, 256)
    lens_l = _lens_list(B, T, lens)
    ref = torch.zeros(B, T, 2 * H, dtype=D)
    bound = torch.zeros(B, T, 2 * H, dtype=D)
    x = _f(xproj)
    for d in range(2):
        W = _h(whh_t[d]) if q16 else _f(whh_t[d])                            # [H, 4H]
        Wa = W.abs()
        h = torch.zeros(B, H, dtype=D)
        c = torch.zeros(B, H, dtype=D)
        dh = torch.zeros(B, H, dtype=D)
        dc = torch.zeros(B, H, dtype=D)
        capped = torch.zeros(B, dtype=torch.bool)
        run = [T if L else 0 for L in lens_l] if (d == 1 and reverse_at_T) else lens_l
        for s in range(max(run, default=0)):
            live = torch.tensor([s < L for L in run])
            t = torch.tensor([s if d == 0 else L - 1 - s for L in run]).clamp(0, T - 1)
            xs = x[torch.arange(B), t, d * 4 * H:(d + 1) * 4 * H]
            xs = torch.where(live[:, None] & torch.isfinite(xs), xs, torch.zeros((), dtype=D))
            if q16:
                ho = _h(h)
                dop = torch.maximum((_h(h + dh) - ho).abs(), (ho - _h(h - dh)).abs())
            else:
                ho, dop = h, dh
            g = xs + ho @ W
            dg = dop @ Wa + (H + 3) * EPS32 * (xs.abs() + ho.abs() @ Wa)
            h2, c2, dh2, dc2 = _cell(g, c, dg, dc, H, mufu=q16)
            m = live[:, None]
            h, c = torch.where(m, h2, h), torch.where(m, c2, c)
            dh, dc = torch.where(m, dh2, dh), torch.where(m, dc2, dc)
            capped |= live & ~(dh.amax(1) <= LSTM_CAP)
            for b in range(B):
                if live[b] and int(t[b]) < lens_l[b]:
                    ref[b, int(t[b]), d * H:(d + 1) * H] = h[b]
                    bound[b, int(t[b]), d * H:(d + 1) * H] = math.inf if capped[b] else dh[b]
    return _to_out(ref, bound, out_dtype)


def bounded_steps(bound, lens, H):
    """Per direction, how many steps from its start every item was checked under the derived bound: the first capped
    step over the items whose bound passed ``LSTM_CAP``, or the longest length when none did (whole sequences)."""
    B, T, _ = bound.shape
    out = []
    for d in range(2):
        n, longest = [], 0
        for b, L in enumerate(_lens_list(B, T, lens)):
            longest = max(longest, L)
            fin = torch.isfinite(bound[b, :L, d * H:(d + 1) * H]).all(1)
            steps = fin if d == 0 else fin.flip(0)
            if not bool(steps.all()):
                n.append(int(torch.argmin(steps.int())))
        out.append(min(n) if n else longest)
    return out
