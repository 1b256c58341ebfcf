"""The fp64 references of tests/ref64_mem.py are right (the fp32 models of tests/sim_backend.py and fp32 emulations of
the kernels' accumulation order fall inside their bounds) and sharp (small injected faults fall outside them)."""
import numpy as np
import pytest
import torch

from artspeech_b200 import ops
from tests import ref64, ref64_mem
from tests import sim_backend as sim

DTS = [torch.float32, torch.float16, torch.bfloat16]


def _raises(out, ref, bound, what):
    with pytest.raises(AssertionError, match="outside the bound"):
        ref64.check(out, ref, bound, what)


def _gen(seed):
    return torch.Generator().manual_seed(seed)


# ---------------------------------------------------------------------------------------------------------------
# the fp32 models fall inside the bounds
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dt", DTS)
def test_sim_embed_layernorm_within_bounds(dt):
    g = _gen(0)
    tok = torch.randint(0, 50, (3, 37), generator=g)
    table = torch.randn(50, 192, generator=g)
    lens = torch.tensor([37, 0, 20], dtype=torch.int32)
    for scale in (1.0, 192 ** 0.5):
        o32, o16 = sim.embed(tok, table, scale, lens, out32=True, out16=dt)
        ref64.check(o32, *ref64_mem.embed(tok, table, scale, lens, torch.float32), "embed fp32")
        ref64.check(o16, *ref64_mem.embed(tok, table, scale, lens, dt), "embed out16")
    for C in (1, 33, 192, 1000):
        x = torch.randn(2, 41, C, generator=g) * 2 + 3
        gam, bet = torch.randn(C, generator=g), torch.randn(C, generator=g)
        for act in (ops.ACT_NONE, ops.ACT_LRELU, ops.ACT_SWISH):
            a, b = sim.layernorm(x.to(dt), gam, bet, 1e-5, act=act, slope=0.2, lens=lens[:2], out_a=torch.float32,
                                 out_b=dt)
            ref, bound = ref64_mem.layernorm(x.to(dt), gam, bet, 1e-5, act, 0.2, lens[:2], torch.float32)
            ref64.check(a, ref, bound, f"layernorm C={C} act {act}")
            ref64.check(b, *ref64_mem.layernorm(x.to(dt), gam, bet, 1e-5, act, 0.2, lens[:2], dt), f"ln C={C} out_b")


@pytest.mark.parametrize("dt", DTS)
def test_sim_copies_within_bounds(dt):
    g = _gen(1)
    x = torch.randn(3, 29, 40, generator=g)
    lens = torch.tensor([29, 0, 7], dtype=torch.int32)
    ref64.check(sim.repeat_rows(x, 2, lens, dt), *ref64_mem.repeat_rows(x, 2, lens, dt), "repeat_rows")
    dur = torch.randint(-1, 4, (3, 29), generator=g, dtype=torch.int32)
    y, olens = sim.length_regulate(x, dur, lens, 2, 100, out_dtype=dt)
    ref, bound, rl = ref64_mem.length_regulate(x, dur, lens, 2, 100, dt)
    ref64.check(y, ref, bound, "length_regulate")
    assert torch.equal(olens, rl)
    sub, mul = torch.randn(40, generator=g), torch.rand(40, generator=g) + 0.5
    src = torch.randn(3, 40, 29, generator=g)
    for s, m in ((None, None), (sub, mul)):
        ref64.check(sim.to_channels_last(src, dt, lens, s, m), *ref64_mem.transpose_cast(src, True, s, m, lens, dt),
                    "to_channels_last")
        ref64.check(sim.to_channels_first(x, dt, lens, s, m), *ref64_mem.transpose_cast(x, False, s, m, lens, dt),
                    "to_channels_first")


@pytest.mark.parametrize("dt", DTS)
def test_sim_pools_within_bounds(dt):
    g = _gen(2)
    x = (torch.randn(2, 15, 22, 24, generator=g) * 3 + 1).to(dt)
    ref64.check(sim.avgpool(x, 2, 4, torch.float32), *ref64_mem.avgpool(x, 2, 4, torch.float32), "avgpool")
    ref64.check(sim.avgpool(x, 2, 4, dt), *ref64_mem.avgpool(x, 2, 4, dt), "avgpool out dt")
    sc, sh = torch.randn(24, generator=g), torch.randn(24, generator=g)
    ref64.check(sim.affine_act_maxpool(x, sc, sh, 0.01, 3, dt), *ref64_mem.affine_act_maxpool(x, sc, sh, 0.01, 3, dt),
                "affine_act_maxpool")
    for ts in (1, 2):
        ref64.check(sim.global_avgpool(x, 0.2, dt, ts), *ref64_mem.global_avgpool(x, 0.2, ts, dt), f"gap ts={ts}")
    mel = torch.randn(2, 80, 53, generator=g) - 1
    ref64.check(sim.log_norm(mel), *ref64_mem.log_norm(mel), "log_norm")


@pytest.mark.parametrize("dt", DTS)
def test_sim_convs_within_bounds(dt):
    g = _gen(3)
    lens = torch.tensor([30, 11], dtype=torch.int32)
    x = torch.randn(2, 30, 10, 3, generator=g).to(dt)
    w = torch.randn(9, 12, 3, generator=g) / 3
    b = torch.randn(12, generator=g)
    taps = ops.taps_2d(3, 3, 1, 1)
    sc = ops.pack_small_conv(w, b, taps, "cpu")
    r, a = sim.conv_small(x, sc, raw=torch.float32, act_out=dt, act=ops.ACT_LRELU, slope=0.1, lens=lens)
    ref64.check(r, *ref64_mem.conv_small(x, w, b, taps, lens, ops.ACT_NONE, 0.0, torch.float32), "conv_small raw")
    ref64.check(a, *ref64_mem.conv_small(x, w, b, taps, lens, ops.ACT_LRELU, 0.1, dt), "conv_small act")
    # depthwise: GLU, time-only k = 31, and a strided 2-D one
    xg = torch.randn(2, 30, 2 * 16, generator=g).to(dt)
    wd, bd = torch.randn(31, 16, generator=g) / 4, torch.randn(16, generator=g)
    y = sim.dwconv(xg, wd, bd, (31, 1), (1, 1), (15, 0), glu=True, act=ops.ACT_SWISH, out_dtype=torch.float32,
                   lens_in=lens, lens_out=lens)
    ref64.check(y, *ref64_mem.dwconv(xg, wd, bd, (31, 1), (1, 1), (15, 0), True, ops.ACT_SWISH, 0.0, lens, lens,
                                     torch.float32), "dwconv glu")
    x2 = torch.randn(2, 15, 9, 8, generator=g).to(dt)
    w2 = torch.randn(9, 8, generator=g)
    y = sim.dwconv(x2, w2, None, (3, 3), (2, 2), (1, 1), act=ops.ACT_LRELU, slope=0.2, out_dtype=dt)
    ref64.check(y, *ref64_mem.dwconv(x2, w2, None, (3, 3), (2, 2), (1, 1), False, ops.ACT_LRELU, 0.2, None, None, dt),
                "dwconv 2-D")
    if dt != torch.float32:      # Cout = 1 convolution of 16-bit operands
        x1 = torch.randn(2, 300, 32, generator=g).to(dt)
        w1 = (torch.randn(7, 1, 32, generator=g) / 8).to(dt)
        b1 = torch.randn(1, generator=g)
        taps1 = ops.taps_1d(7, 1)
        pw = ops.pack_conv(w1.float(), b1, taps1, dt, "cpu")
        raw, act = sim.conv(x1, pw, raw=torch.float32, act_out=torch.float32, act=ops.ACT_TANH, scale=0.5, lens=lens)
        for path in ("mma", "fp32"):
            ref64.check(raw, *ref64_mem.conv_cout1(x1, w1, b1, taps1, lens, 0.5, ops.ACT_NONE, 0.0, torch.float32,
                                                   path), f"cout1 raw {path}")
            ref64.check(act, *ref64_mem.conv_cout1(x1, w1, b1, taps1, lens, 0.5, ops.ACT_TANH, 0.0, torch.float32,
                                                   path), f"cout1 tanh {path}")
            pcm = torch.clamp(torch.round(act * 32767), -32768, 32767).to(torch.int16)
            ref64.check(pcm, *ref64_mem.conv_cout1(x1, w1, b1, taps1, lens, 0.5, ops.ACT_TANH, 0.0, torch.int16, path),
                        f"cout1 pcm16 {path}")


def _chain32(x, w, bias, taps, group):
    """fp32 emulation of the Cout = 1 kernels' order: acc = bias, then per tap (and per ``group`` channels) one rounded
    addition of that group's fp32 dot product."""
    B, T, Cin = x.shape
    xf, wf = x.float().numpy(), w.float().numpy()
    acc = np.full((B, T), np.float32(bias[0]), dtype=np.float32)
    for j, (d, _) in enumerate(taps):
        ti = np.arange(T) + d
        ok = (ti >= 0) & (ti < T)
        g = xf[:, np.clip(ti, 0, T - 1)] * ok[None, :, None]
        for c0 in range(0, Cin, group):
            part = (g[..., c0:c0 + group].astype(np.float64) @ wf[j, 0, c0:c0 + group].astype(np.float64))
            acc = (acc + part.astype(np.float32)).astype(np.float32)
    return torch.from_numpy(acc)[..., None]


@pytest.mark.parametrize("dt", [torch.float16, torch.bfloat16])
def test_bias_dominated_chain_within_bound(dt):
    """|bias| >> sum |x w|: every addition of the kernel's chain rounds at the bias's ulp.  The chain term of
    ``ref64_mem`` covers it for both Cout = 1 kernels and for conv_small's per-channel fma chain."""
    g = _gen(4)
    x = (torch.randn(2, 500, 32, generator=g) * 1e-3).to(dt)
    w = (torch.randn(7, 1, 32, generator=g) / 8).to(dt)
    bias = torch.tensor([1000.0 / 3])
    taps = ops.taps_1d(7, 1)
    for path, group in (("mma", 32), ("fp32", 8)):
        out = _chain32(x, w, bias, taps, group)
        ref64.check(out, *ref64_mem.conv_cout1(x, w, bias, taps, None, 1.0, ops.ACT_NONE, 0.0, torch.float32, path),
                    f"bias chain {path}")
    out = _chain32(x, w, bias, taps, 1)
    ref64.check(out, *ref64_mem.conv_small(x, w.float(), bias, taps, None, ops.ACT_NONE, 0.0, torch.float32),
                "bias chain conv_small")


# ---------------------------------------------------------------------------------------------------------------
# fault injection: each mutated result must leave the bound
# ---------------------------------------------------------------------------------------------------------------
def test_conv_small_dropped_tap():
    g = _gen(5)
    x = torch.randn(2, 20, 12, 1, generator=g)
    w = torch.randn(9, 16, 1, generator=g) / 3
    b = torch.randn(16, generator=g)
    taps = ops.taps_2d(3, 3, 1, 1)
    good, _ = sim.conv_small(x, ops.pack_small_conv(w, b, taps, "cpu"), raw=torch.float32)
    ref, bound = ref64_mem.conv_small(x, w, b, taps, None, ops.ACT_NONE, 0.0, torch.float32)
    ref64.check(good, ref, bound, "unmutated")
    bad = good.clone()
    bad[1, 7, 5] -= x[1, 7 + taps[4][0], 5 + taps[4][1], 0] * w[4, :, 0]        # the centre tap on one row
    _raises(bad, ref, bound, "dropped tap")


def test_dwconv_glu_halves_swapped():
    g = _gen(6)
    C = 16
    x = torch.randn(2, 40, 2 * C, generator=g)
    w, b = torch.randn(31, C, generator=g) / 4, torch.randn(C, generator=g)
    kw = dict(glu=True, out_dtype=torch.float32)
    ref, bound = ref64_mem.dwconv(x, w, b, (31, 1), (1, 1), (15, 0), True, ops.ACT_NONE, 0.0, None, None,
                                  torch.float32)
    ref64.check(sim.dwconv(x, w, b, (31, 1), (1, 1), (15, 0), **kw), ref, bound, "unmutated")
    swapped = torch.cat([x[..., C:], x[..., :C]], -1)
    _raises(sim.dwconv(swapped, w, b, (31, 1), (1, 1), (15, 0), **kw), ref, bound, "GLU halves swapped")


def test_dwconv_lens_mask_one_row_late():
    g = _gen(7)
    x, w = torch.randn(2, 40, 24, generator=g), torch.randn(5, 24, generator=g)
    lens = torch.tensor([40, 17], dtype=torch.int32)
    ref, bound = ref64_mem.dwconv(x, w, None, (5, 1), (1, 1), (2, 0), False, ops.ACT_NONE, 0.0, lens, lens,
                                  torch.float32)
    good = sim.dwconv(x, w, None, (5, 1), (1, 1), (2, 0), out_dtype=torch.float32, lens_in=lens, lens_out=lens)
    ref64.check(good, ref, bound, "unmutated")
    late = sim.dwconv(x, w, None, (5, 1), (1, 1), (2, 0), out_dtype=torch.float32, lens_in=lens, lens_out=lens + 1)
    _raises(late, ref, bound, "lens_out one row late")
    late_in = sim.dwconv(x, w, None, (5, 1), (1, 1), (2, 0), out_dtype=torch.float32, lens_in=lens + 1, lens_out=lens)
    _raises(late_in, ref, bound, "lens_in one row late")


def test_avgpool_zero_padding():
    g = _gen(8)
    x = torch.randn(2, 15, 8, 16, generator=g) + 2
    ref, bound = ref64_mem.avgpool(x, 2, 2, torch.float32)
    ref64.check(sim.avgpool(x, 2, 2), ref, bound, "unmutated")
    zp = torch.nn.functional.avg_pool2d(torch.cat([x, torch.zeros_like(x[:, :1])], 1).permute(0, 3, 1, 2),
                                        (2, 2)).permute(0, 2, 3, 1)
    _raises(zp, ref, bound, "zero padding")


@pytest.mark.parametrize("C", [192, 512])
def test_layernorm_one_pass_variance(C):
    """Rows with |mean| / std = 40: two-pass statistics in fp32 stay inside the bound, E[x^2] - mean^2 does not."""
    g = _gen(9)
    x = torch.randn(1, 8, C, generator=g) * 0.5 + 20.0
    gam, bet = torch.randn(C, generator=g), torch.randn(C, generator=g)
    ref, bound = ref64_mem.layernorm(x, gam, bet, 1e-5, ops.ACT_NONE, 0.0, None, torch.float32)
    xs = x[0].numpy()

    def apply(mean, var):
        rstd = (1.0 / np.sqrt(var.astype(np.float64) + 1e-5)).astype(np.float32)
        return torch.from_numpy((xs - mean) * rstd * gam.numpy() + bet.numpy())[None]

    mean = (np.cumsum(xs, 1, dtype=np.float32)[:, -1:] / np.float32(C)).astype(np.float32)
    d = xs - mean
    var2 = (np.cumsum(d * d, 1, dtype=np.float32)[:, -1:] / np.float32(C)).astype(np.float32)
    ref64.check(apply(mean, var2), ref, bound, "two-pass")
    var1 = (np.cumsum(xs * xs, 1, dtype=np.float32)[:, -1:] / np.float32(C) - mean * mean).astype(np.float32)
    _raises(apply(mean, var1), ref, bound, "one-pass")


def test_length_regulate_off_by_one_token():
    g = _gen(10)
    x = torch.randn(1, 12, 16, generator=g)
    dur = torch.tensor([[2, 0, 3, 1, 4, 2, 2, 1, 3, 1, 2, 2]], dtype=torch.int32)
    ref, bound, _ = ref64_mem.length_regulate(x, dur, None, 2, 60, torch.float32)
    good, _ = sim.length_regulate(x, dur, None, 2, 60)
    ref64.check(good, ref, bound, "unmutated")
    bad = good.clone()
    boundary = 2 * int(dur[0, :4].sum())          # first frame of token 4
    bad[0, boundary] = x[0, 3]                    # still the previous token
    _raises(bad, ref, bound, "token boundary one frame late")


def test_transpose_tile_shifted():
    g = _gen(11)
    src = torch.randn(2, 70, 100, generator=g)
    ref, bound = ref64_mem.transpose_cast(src, True, None, None, None, torch.float32)
    good = sim.to_channels_last(src, torch.float32)
    ref64.check(good, ref, bound, "unmutated")
    bad = good.clone()
    bad[1, 32:64, 32:64] = good[1, 33:65, 32:64]
    _raises(bad, ref, bound, "tile shifted by one frame")
