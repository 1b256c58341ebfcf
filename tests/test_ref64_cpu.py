"""The fp64 references of tests/ref64.py are right (fp32 models of the same operations fall inside their bounds) and
sharp (small injected faults of the kind a tile schedule or a pipeline produces fall outside them)."""
import numpy as np
import pytest
import torch

from artspeech_b200 import ops
from tests import ref64
from tests import sim_backend as sim


def _raises(out, ref, bound, what):
    with pytest.raises(AssertionError, match="outside the bound"):
        ref64.check(out, ref, bound, what)


def _conv_case(dt, B=2, T=300, Cin=64, Cout=64, k=3, dil=1, seed=0):
    g = torch.Generator().manual_seed(seed)
    x = (torch.randn(B, T, Cin, generator=g) * 0.5).to(dt)
    w = (torch.randn(k, Cout, Cin, generator=g) / (Cin * k) ** 0.5).to(dt)
    bias = torch.randn(Cout, generator=g)
    r1 = torch.randn(B, T, Cout, generator=g).to(dt)
    r2 = torch.randn(B, T, Cout, generator=g)
    lens = torch.tensor([T, T // 2 + 7][:B], dtype=torch.int32)
    return x, w, bias, r1, r2, lens, ops.taps_1d(k, dil)


@pytest.mark.parametrize("dt", [torch.float16, torch.bfloat16])
def test_sim_conv_within_bounds(dt):
    x, w, bias, r1, r2, lens, taps = _conv_case(dt, k=5, dil=2)
    pw = ops.pack_conv(w.float(), bias, taps, dt, "cpu")
    raw, act = sim.conv(x, pw, res1=r1, res2=r2, scale=0.7, raw=torch.float32, act_out=dt, act=ops.ACT_LRELU,
                        slope=0.1, lens=lens)
    vb = ref64.conv_v(x, w, taps, bias=bias, res1=r1, res2=r2, scale=0.7, lens=lens)
    ref64.check(raw, *ref64.conv_out(vb), "raw")
    ref64.check(act, *ref64.conv_out(vb, ops.ACT_LRELU, 0.1, dt), "act")
    for a in (ops.ACT_TANH, ops.ACT_SWISH):
        _, y = sim.conv(x, pw, raw=None, act_out=torch.float32, act=a, lens=lens)
        ref64.check(y, *ref64.conv(x, w, taps, bias=bias, lens=lens, act=a), f"act {a}")
    # 2-D 3 x 3, 'same' padding, Cin outside the 16-channel granularity of one K chunk
    x2 = (torch.randn(2, 9, 20, 48) * 0.5).to(dt)
    w2 = (torch.randn(9, 40, 48) / 20).to(dt)
    taps2 = ops.taps_2d(3, 3, 1, 1)
    y2, _ = sim.conv(x2, ops.pack_conv(w2.float(), None, taps2, dt, "cpu"), raw=torch.float32)
    ref64.check(y2, *ref64.conv(x2, w2, taps2), "2-D")


@pytest.mark.parametrize("variant", ["mid", "stage_end"])
@pytest.mark.parametrize("dt", [torch.float16, torch.bfloat16])
def test_sim_resblock_pair_within_bounds(dt, variant):
    B, L, C, k, dil = 2, 260, 32, 5, 3
    g = torch.Generator().manual_seed(1)
    lens = torch.tensor([L, 131], dtype=torch.int32)
    x_raw = torch.randn(B, L, C, generator=g) * (torch.arange(L)[None, :] < lens[:, None])[:, :, None]
    xa = torch.where(x_raw > 0, x_raw, 0.1 * x_raw).to(dt)
    w1 = (torch.randn(k, C, C, generator=g) / (C * k) ** 0.5).to(dt)
    w2 = (torch.randn(k, C, C, generator=g) / (C * k) ** 0.5).to(dt)
    b1, b2 = torch.randn(C, generator=g) * 0.1, torch.randn(C, generator=g) * 0.1
    kw = dict(slope=0.1, out_act=ops.ACT_LRELU, out_slope=0.1)
    if variant == "stage_end":
        kw.update(res2=torch.randn(B, L, C, generator=g).to(dt), res3=torch.randn(B, L, C, generator=g).to(dt),
                  scale=1.0 / 3, out_slope=0.01)
    c1 = ops.pack_conv(w1.float(), b1, ops.taps_1d(k, dil), dt, "cpu")
    c2 = ops.pack_conv(w2.float(), b2, ops.taps_1d(k, 1), dt, "cpu")
    out = sim.resblock_pair(xa, c1, c2, k, dil, lens=lens, **kw)
    ref64.check(out, *ref64.resblock_pair(xa, w1, b1, w2, b2, k, dil, lens=lens, **kw), f"pair {variant}")


@pytest.mark.parametrize("up", [False, True])
@pytest.mark.parametrize("dt", [torch.float32, torch.bfloat16])
def test_sim_adain_within_bounds(dt, up):
    B, T, C = 3, 180, 48
    g = torch.Generator().manual_seed(2)
    # bias-dominated channels: |mean| / std = 40
    x = (torch.randn(B, T, C, generator=g) * 0.5 + 20.0 * torch.sign(torch.randn(C, generator=g))).to(dt)
    gb = torch.randn(B, 2 * C, generator=g) * 0.3
    lens = torch.tensor([T, 77, 1], dtype=torch.int32)
    up_w = torch.randn(C, 3, generator=g) if up else None
    up_b = torch.randn(C, generator=g) if up else None
    st = sim.instnorm_stats(x, lens)
    ref64.check(st, *ref64.instnorm_stats(x, lens), "stats")
    out = sim.adain_norm(x, gb, 0.2, lens, torch.float32, up_w, up_b)
    ref64.check(out, *ref64.adain_norm(x, gb, 0.2, lens, torch.float32, up_w, up_b), "adain_norm")
    out = sim.adain_apply(x, st, gb, -0.3, lens, torch.float16, up_w, up_b)
    ref64.check(out, *ref64.adain_apply(x, st, gb, -0.3, lens, torch.float16, up_w, up_b), "adain_apply")


# ---------------------------------------------------------------------------------------------------------------
# fault injection: each mutated fp32 result must leave the bound
# ---------------------------------------------------------------------------------------------------------------
def _conv32(x, w, taps, bias, chans=slice(None)):
    """fp32 convolution of 16-bit operands (what the tensor cores compute), optionally over some input channels."""
    B, T, _ = x.shape
    acc = torch.zeros(B, T, w.shape[1])
    xf, wf = x.float(), w.float()
    for j, (d, _) in enumerate(taps):
        ti = torch.arange(T) + d
        g_ = xf[:, ti.clamp(0, T - 1)] * ((ti >= 0) & (ti < T))[None, :, None]
        acc += g_[..., chans] @ wf[j][:, chans].t()
    return acc + (bias if bias is not None else 0)


@pytest.mark.parametrize("dt", [torch.float16, torch.bfloat16])
def test_conv_bound_catches_schedule_faults(dt):
    x, w, bias, _, _, _, taps = _conv_case(dt, T=400)
    ref, bound = ref64.conv(x, w, taps, bias=bias)
    good = _conv32(x, w, taps, bias)
    ref64.check(good, ref, bound, "unmutated")
    # one tap dropped on one output row
    bad = good.clone()
    xf, wf = x.float(), w.float()
    bad[0, 137] -= xf[0, 137 + taps[0][0]] @ wf[0].t()
    _raises(bad, ref, bound, "dropped tap")
    # one 16-channel K slice dropped on one tile (rows 128..255 of item 1)
    bad = good.clone()
    part = _conv32(x, w, taps, None, chans=slice(16, 32))
    bad[1, 128:256] -= part[1, 128:256]
    _raises(bad, ref, bound, "dropped K slice")
    # one tile's rows shifted by one frame
    bad = good.clone()
    bad[1, 256:384] = good[1, 257:385]
    _raises(bad, ref, bound, "shifted tile")
    # bias missing on one tile
    bad = good.clone()
    bad[0, 0:128] -= bias
    _raises(bad, ref, bound, "bias missing")


def _pair32(xa, w1, b1, w2, b2, k, dil, slope, round_t=True):
    """fp32 model of the pair before its output rounding; ``round_t=False`` feeds conv2 the fp32 t."""
    v1 = _conv32(xa, w1, ops.taps_1d(k, dil), b1)
    t = torch.where(v1 > 0, v1, v1 * slope)
    a = xa.float()
    return _conv32(t.to(xa.dtype) if round_t else t, w2, ops.taps_1d(k, 1), b2) + torch.where(a < 0, a / slope, a)


@pytest.mark.parametrize("dt", [torch.float16, torch.bfloat16])
def test_pair_bound_catches_unrounded_operand(dt):
    """The ResBlock pair rounds t = lrelu(conv1(a) + b1) to 16 bits before conv2.  The bound allows conv2 an operand
    one ulp away only where conv1's bound straddles a rounding midpoint.  Where t sits 0.4 ulp above a 16-bit value
    (an all-ones input, weights 2^-7, a bias of 0.4 ulp) and w2 > 0, the fp32 t of a kernel that skipped the rounding
    moves every output by 0.4 ulp * sum w2, far outside it.  Checked on the fp32 value before the output rounding."""
    B, L, C, k, dil, slope = 1, 300, 32, 3, 1, 0.1
    g = torch.Generator().manual_seed(3)
    xr = torch.randn(B, L, C, generator=g)
    xa = torch.where(xr > 0, xr, slope * xr).to(dt)
    w1 = (torch.randn(k, C, C, generator=g) / (C * k) ** 0.5).to(dt)
    w2 = (torch.randn(k, C, C, generator=g) / (C * k) ** 0.5).to(dt)
    b1, b2 = torch.randn(C, generator=g) * 0.1, torch.randn(C, generator=g) * 0.1
    ref, bound = ref64.resblock_pair(xa, w1, b1, w2, b2, k, dil, slope=slope, dtype=torch.float32)
    ref64.check(_pair32(xa, w1, b1, w2, b2, k, dil, slope), ref, bound, "random, rounded t")
    ulp = 2.0 ** -11 if dt == torch.float16 else 2.0 ** -8            # at t in [0.5, 1)
    xa = torch.ones(B, L, C).to(dt)
    w1 = torch.full((k, C, C), 2.0 ** -7).to(dt)                      # t = 0.75 inside, 0.5 at the two edge rows
    b1 = torch.full((C,), 0.4 * ulp)
    w2 = w2.abs()
    ref, bound = ref64.resblock_pair(xa, w1, b1, w2, b2, k, dil, slope=slope, dtype=torch.float32)
    ref64.check(_pair32(xa, w1, b1, w2, b2, k, dil, slope), ref, bound, "coherent, rounded t")
    _raises(_pair32(xa, w1, b1, w2, b2, k, dil, slope, round_t=False), ref, bound, "unrounded t")


@pytest.mark.parametrize("n", [64, 256])
def test_adain_bound_catches_one_pass_variance(n):
    """|mean| / std = 40: the two-pass statistics stay inside the bound, E[x^2] - mean^2 in fp32 does not."""
    C = 16
    g = torch.Generator().manual_seed(4)
    x = torch.randn(1, n, C, generator=g) * 0.5 + 20.0
    gb = torch.randn(1, 2 * C, generator=g) * 0.3
    ref, bound = ref64.adain_norm(x, gb, 0.2, None, torch.float32)
    xs = x[0].numpy().astype(np.float32)

    def apply(mean, var):
        rstd = (1.0 / np.sqrt(var.astype(np.float64) + 1e-5)).astype(np.float32)
        a = (xs - mean) * (rstd * (1 + gb[0, :C].numpy())) + gb[0, C:].numpy()
        return torch.from_numpy(np.where(a > 0, a, np.float32(0.2) * a))[None]

    s = np.cumsum(xs, 0, dtype=np.float32)[-1]          # sequential fp32 sums, as one thread would
    mean = (s / np.float32(n)).astype(np.float32)
    d = xs - mean
    var2 = (np.cumsum(d * d, 0, dtype=np.float32)[-1] / np.float32(n)).astype(np.float32)
    ref64.check(apply(mean, var2), ref, bound, "two-pass")
    var1 = (np.cumsum(xs * xs, 0, dtype=np.float32)[-1] / np.float32(n) - mean * mean).astype(np.float32)
    _raises(apply(mean, var1), ref, bound, "one-pass")
