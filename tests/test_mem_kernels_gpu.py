"""The memory-bound kernels and the single-output-channel convolution on every dispatch path against the fp64
references of tests/ref64_mem.py.

Each case names the kernel that ran (torch.profiler, ``launches`` of tests/test_schedule_gpu.py) and checks every
output element against its bound.  Where a contract says a value is never read, the input holds NaN there (rows past
``lens_in`` for dwconv, past ``lens`` for repeat_rows, tokens past ``lens_t`` for length regulation) or an absurd value
(durations of 2^30 past ``lens_t``, token ids outside the table), and the masked outputs must be exact zeros.  Inputs of
conv_small and of the Cout = 1 convolution past ``lens`` are not poisoned: those kernels read them for valid rows near
the boundary, as the tensor-core convolution does.  ``WORST`` collects the largest err / bound per kernel; the last
test prints it.

Dispatch (artspeech_b200/csrc/elementwise.cu, conv_cout1.cu, conv_igemm.cu):
  * as_layernorm: layernorm_vec4_kernel<C / 128> for fp32 x with C in {256, 512, 1024} and 16-byte aligned x, gamma,
    beta and outputs (8-byte for 16-bit ones); layernorm_kernel otherwise.
  * as_length_regulate: one kernel with three copy modes chosen from the layout (``_lr_mode``): 1 = same dtype and
    16-byte rows, 2 = fp32 -> 16-bit with C % 8 == 0 and 16-byte rows, 0 = anything else.
  * as_conv_small: conv_small_vec_kernel<4> (F % 4 == 0) or <1> when Cout % 8 == 0 and the weights fit 40 KB of shared
    memory; conv_small_kernel otherwise.
  * as_dwconv: dwconv_time_tiled_kernel for F = 1, stride 1, 5 <= kt <= 32, To = T; dwconv_vec8_kernel for 16-bit
    in / out, C % 8 == 0, 16-byte aligned and no GLU; dwconv_kernel otherwise.
  * as_avgpool / as_affine_act_maxpool: the _vec8 kernel for 16-bit in / out with C % 8 == 0 and 16-byte alignment.
  * as_conv_igemm with Cout = 1, 1-D, 16-bit x with Cin % 8 == 0 and Cin <= 64, equally spaced taps (<= 16) spanning at
    most 64 rows: conv_cout1_mma_kernel for Cin % 16 == 0 and <= 8 taps, conv_cout1_kernel otherwise.  Other shapes go
    to the tensor-core convolution.  ASB_COUT1_NO_MMA / ASB_NO_COUT1 (read once per process) are tested in child processes
    by tests/test_zz_cout1_modes_gpu.py.
"""
import pytest
import torch

from artspeech_b200 import _lib, mas, ops
from tests import ref64, ref64_mem
from tests.test_schedule_gpu import launches

pytestmark = pytest.mark.gpu
DEV = "cuda"
F16, BF16, F32 = torch.float16, torch.bfloat16, torch.float32
NAN = float("nan")
MEM_KERNELS = ("embed_kernel", "layernorm_kernel", "layernorm_vec4_kernel", "repeat_rows_kernel", "expand_tokens_kernel",
               "length_regulate_kernel", "conv_small_kernel", "conv_small_vec_kernel", "dwconv_kernel",
               "dwconv_time_tiled_kernel", "dwconv_vec8_kernel", "avgpool_kernel", "avgpool_vec8_kernel",
               "affine_act_maxpool_kernel", "affine_act_maxpool_vec8_kernel", "global_avgpool_kernel", "log_norm_kernel",
               "transpose_cast_kernel", "conv_cout1_kernel", "conv_cout1_mma_kernel")
CONV_KERNELS = ("conv_igemm_kernel", "conv_igemm_2cta_kernel", "conv_halo_kernel", "conv_halo_sw_kernel")
WORST = {}


def _one_launch(fn, tmp_path, tag, kernel, families=MEM_KERNELS):
    """Run ``fn`` under the profiler and assert that the only kernel of ``families`` it launched is ``kernel``."""
    out, ks = launches(fn, tmp_path, tag)
    got = [k for k, _ in ks if k.split("<")[0] in families]
    assert got == [kernel], f"{tag}: launched {ks}, expected {kernel}"
    return out


def _check(kernel, out, ref, bound, what):
    ref64.check(out, ref, bound, what)
    o = out.detach().to("cpu", torch.float64)
    live = torch.isfinite(bound) & (bound > 0)
    if bool(live.any()):
        r = float(((o - ref).abs()[live] / bound[live]).max())
        WORST[kernel] = max(WORST.get(kernel, 0.0), r)
    else:
        WORST.setdefault(kernel, 0.0)


def _g(seed):
    return torch.Generator().manual_seed(seed)


def _nan_rows(x, lens):
    """Copy of ``x`` [B, T, ...] with the rows at or beyond each item's length set to NaN."""
    x = x.clone()
    for b, L in enumerate(lens.tolist()):
        x[b, max(0, L):] = NAN
    return x


def _offset_view(x):
    """``x`` on the device at one element's offset from an aligned allocation (same shape, dense): a 4-byte offset for
    fp32, an odd 2-byte one for 16-bit."""
    buf = torch.empty(x.numel() + 1, dtype=x.dtype, device=DEV)
    v = buf[1:].view(x.shape)
    v.copy_(x.to(DEV))
    return v


def _slice_out(shape, dtype, lead=1, extra=1):
    """A channel-slice view [.., C] of a [.., C + lead + extra] buffer: rows of C + lead + extra elements, base
    ``lead`` elements past an aligned allocation."""
    buf = torch.zeros(*shape[:-1], shape[-1] + lead + extra, dtype=dtype, device=DEV)
    return buf[..., lead:lead + shape[-1]]


# ------------------------------------------------------------------------------------------------------------------
# embedding
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("scale", [1.0, 192 ** 0.5])
def test_embed(scale, tmp_path):
    """Token ids -1, n_vocab and 10^6 read row 0; lens 0, 1, T and T + 13."""
    g = _g(1)
    B, T, C, V = 4, 37, 192, 50
    tok = torch.randint(0, V, (B, T), generator=g)
    tok[0, 3], tok[1, 5], tok[3, 36], tok[2, 0] = -1, V, 10 ** 6, V - 1
    table = torch.randn(V, C, generator=g)
    lens = torch.tensor([T, 0, 1, T + 13], dtype=torch.int32)
    tg, wg, lg = tok.to(DEV), table.to(DEV), lens.to(DEV)
    for i, dt in enumerate((F16, BF16)):
        fn = lambda: ops.embed(tg, wg, scale, lg, out32=True, out16=dt)
        o32, o16 = _one_launch(fn, tmp_path, "embed", "embed_kernel") if i == 0 else fn()
        _check("embed_kernel", o32, *ref64_mem.embed(tok, table, scale, lens, F32), f"embed fp32 scale {scale}")
        _check("embed_kernel", o16, *ref64_mem.embed(tok, table, scale, lens, dt), f"embed {dt} scale {scale}")


# ------------------------------------------------------------------------------------------------------------------
# LayerNorm
# ------------------------------------------------------------------------------------------------------------------
# name: (C, x dtype, layout, kernel); layout "offset" puts x one element past an aligned allocation, "odd_b" writes
# out_b into a 16-bit channel slice at an odd element offset
LN_CASES = {
    "vec4_256": (256, F32, "aligned", "layernorm_vec4_kernel<2>"),
    "vec4_512": (512, F32, "aligned", "layernorm_vec4_kernel<4>"),
    "vec4_1024": (1024, F32, "aligned", "layernorm_vec4_kernel<8>"),
    "f16_192": (192, F16, "aligned", "layernorm_kernel"),
    "bf16_512": (512, BF16, "aligned", "layernorm_kernel"),
    "C1": (1, F32, "aligned", "layernorm_kernel"),
    "C33": (33, F32, "aligned", "layernorm_kernel"),
    "C250": (250, F32, "aligned", "layernorm_kernel"),
    "C1000": (1000, F32, "aligned", "layernorm_kernel"),
    "C1024_offset": (1024, F32, "offset", "layernorm_kernel"),
    "C256_odd_out_b": (256, F32, "odd_b", "layernorm_kernel"),
}


@pytest.mark.parametrize("case", list(LN_CASES))
def test_layernorm(case, tmp_path):
    """lens T, 0, 1, T + 3; item 3 is bias-dominated (|mean| / std = 40); LeakyReLU and swish."""
    C, xdt, layout, kernel = LN_CASES[case]
    g = _g(C)
    B, T = 4, 45
    x = torch.randn(B, T, C, generator=g) * 2 + 1
    x[3] = torch.randn(T, C, generator=g) * 0.5 + 20
    x = x.to(xdt)
    gam, bet = torch.randn(C, generator=g), torch.randn(C, generator=g) * 0.5
    lens = torch.tensor([T, 0, 1, T + 3], dtype=torch.int32)
    xg = _offset_view(x) if layout == "offset" else x.to(DEV)
    gg, bg, lg = gam.to(DEV), bet.to(DEV), lens.to(DEV)
    for i, (act, slope, dtb) in enumerate(((ops.ACT_LRELU, 0.2, BF16), (ops.ACT_SWISH, 0.0, F16),
                                           (ops.ACT_NONE, 0.0, F32))):
        ob = _slice_out((B, T, C), dtb) if layout == "odd_b" else dtb

        def fn():
            return ops.layernorm(xg, gg, bg, 1e-5, act=act, slope=slope, lens=lg, out_a=F32, out_b=ob)
        oa, obt = _one_launch(fn, tmp_path, f"ln_{case}", kernel) if i == 0 else fn()
        for out, dt in ((oa, F32), (obt, dtb)):
            _check(kernel, out, *ref64_mem.layernorm(x, gam, bet, 1e-5, act, slope, lens, dt), f"ln {case} act {act} {dt}")


# ------------------------------------------------------------------------------------------------------------------
# copies
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("xdt", [F32, BF16])
def test_repeat_rows(xdt, tmp_path):
    """x is a channel slice (row stride C + 24), NaN past lens; lens T, 0, 1, T + 5, 20; C and T not multiples of 32."""
    g = _g(2)
    B, T, C, rep = 5, 33, 100, 2
    lens = torch.tensor([T, 0, 1, T + 5, 20], dtype=torch.int32)
    wide = _nan_rows(torch.randn(B, T, C + 24, generator=g), lens).to(xdt)
    x = wide[..., 8:8 + C]
    xg = wide.to(DEV)[..., 8:8 + C]
    lg = lens.to(DEV)
    for i, dt in enumerate((F32, F16, BF16)):
        fn = lambda: ops.repeat_rows(xg, rep, lg, out_dtype=dt)
        out = _one_launch(fn, tmp_path, "repeat", "repeat_rows_kernel") if i == 0 else fn()
        _check("repeat_rows_kernel", out, *ref64_mem.repeat_rows(x, rep, lens, dt), f"repeat_rows {xdt} -> {dt}")


def test_expand_tokens(tmp_path):
    """Frame -> token maps with -1 (past y_len), Tx (out of range) and repeated tokens; Ty not a multiple of 32."""
    g = _g(3)
    B, C, Tx, Ty = 3, 70, 41, 77
    x = torch.randn(B, C, Tx, generator=g)
    tok = torch.sort(torch.randint(0, Tx, (B, Ty), generator=g), 1).values.to(torch.int32)
    tok[0, 60:] = -1
    tok[1, -1] = Tx
    tok[2, :] = 0
    xg, tg = x.to(DEV), tok.to(DEV)
    out = _one_launch(lambda: mas.expand_tokens(xg, tg), tmp_path, "expand", "expand_tokens_kernel")
    _check("expand_tokens_kernel", out, *ref64_mem.expand_tokens(x, tok), "expand_tokens")


def _lr_mode(x, out, C):
    """The copy mode as_length_regulate picks from the layout (restated from the host code, to pin each case's)."""
    def al16(t):
        return t.data_ptr() % 16 == 0 and (t.stride(-2) * t.element_size()) % 16 == 0
    if al16(x) and al16(out):
        if x.dtype == out.dtype and (C * x.element_size()) % 16 == 0:
            return 1
        if x.dtype == F32 and out.dtype != F32 and C % 8 == 0:
            return 2
    return 0


# name: (C, x dtype, out dtype, x at an element offset, copy mode)
LR_CASES = {
    "vec1_f32": (64, F32, F32, False, 1),
    "vec1_bf16": (64, BF16, BF16, False, 1),
    "vec2_f16": (192, F32, F16, False, 2),
    "vec2_bf16": (192, F32, BF16, False, 2),
    "vec0_C250": (250, F32, F16, False, 0),
    "vec0_C250_f32": (250, F32, F32, False, 0),
    "vec0_offset": (64, F32, F32, True, 0),
}


@pytest.mark.parametrize("case", list(LR_CASES))
def test_length_regulate(case, tmp_path):
    """Durations 0, negative, and 2^30 past lens_t; lens_t 0, 1, Tt and > Tt; token rows past lens_t are NaN; To cuts
    the longest item and spans several 32-row CTAs; out_lens must be min(rep * sum, To)."""
    C, xdt, odt, offset, mode = LR_CASES[case]
    g = _g(4 + C)
    B, Tt, rep = 5, 40, 2
    lens_t = torch.tensor([Tt, 0, Tt + 60, 17, 1], dtype=torch.int32)
    dur = torch.randint(-2, 6, (B, Tt), generator=g, dtype=torch.int32)
    dur[2, :5] = 0
    for b, L in enumerate(lens_t.tolist()):
        dur[b, max(0, L):] = 2 ** 30
    x = _nan_rows(torch.randn(B, Tt, C, generator=g), lens_t).to(xdt)
    sums = [int(dur[b, :min(L, Tt)].clamp(min=0).sum()) for b, L in enumerate(lens_t.tolist())]
    To = rep * max(sums) - 7
    assert 32 < To < rep * max(sums)
    xg = _offset_view(x) if offset else x.to(DEV)
    dg, lg = dur.to(DEV), lens_t.to(DEV)
    out = torch.full((B, To, C), NAN, dtype=odt, device=DEV)
    assert _lr_mode(xg, out, C) == mode
    res, olens = _one_launch(lambda: ops.length_regulate(xg, dg, lg, rep, To, out=out), tmp_path, f"lr_{case}",
                             "length_regulate_kernel")
    ref, bound, rl = ref64_mem.length_regulate(x, dur, lens_t, rep, To, odt)
    _check("length_regulate_kernel", res, ref, bound, f"length_regulate {case}")
    assert torch.equal(olens.cpu(), rl), (olens.cpu(), rl)


def test_length_regulate_longest_token_sequence(tmp_path):
    """Tt = 12287 fills the kernel's 48 KB prefix-sum array ((Tt + 1) ints); 12288 is refused."""
    g = _g(5)
    B, Tt, C = 2, 12287, 8
    dur = torch.randint(0, 2, (B, Tt), generator=g, dtype=torch.int32)
    lens_t = torch.tensor([Tt, Tt - 1000], dtype=torch.int32)
    x = torch.randn(B, Tt, C, generator=g)
    To = 2 * int(dur[0].sum())
    xg, dg, lg = x.to(DEV), dur.to(DEV), lens_t.to(DEV)
    res, olens = _one_launch(lambda: ops.length_regulate(xg, dg, lg, 2, To, out_dtype=BF16), tmp_path, "lr_long",
                             "length_regulate_kernel")
    ref, bound, rl = ref64_mem.length_regulate(x, dur, lens_t, 2, To, BF16)
    _check("length_regulate_kernel", res, ref, bound, "length_regulate Tt=12287")
    assert torch.equal(olens.cpu(), rl)
    x2 = torch.zeros(1, Tt + 1, C, device=DEV)
    with pytest.raises(_lib.AsError, match="too large"):
        ops.length_regulate(x2, torch.ones(1, Tt + 1, dtype=torch.int32, device=DEV), None, 2, 64)


@pytest.mark.parametrize("sub", [False, True])
def test_transpose_cast(sub, tmp_path):
    """Both directions, into / out of channel slices (row stride C + 80 and C + 26), T and C not multiples of 32, lens
    0, T and 40, with and without the per-channel affine."""
    g = _g(6)
    B, C, T = 3, 70, 101
    lens = torch.tensor([T, 0, 40], dtype=torch.int32)
    sb, mb = (torch.randn(C, generator=g), torch.rand(C, generator=g) + 0.5) if sub else (None, None)
    sg, mg = (sb.to(DEV), mb.to(DEV)) if sub else (None, None)
    lg = lens.to(DEV)
    src = torch.randn(B, C, T, generator=g)
    out = _slice_out((B, T, C), BF16, lead=5, extra=75)
    sg_ = src.to(DEV)
    res = _one_launch(lambda: ops.to_channels_last(sg_, BF16, lg, sg, mg, out=out), tmp_path, "tcl",
                      "transpose_cast_kernel")
    _check("transpose_cast_kernel", res, *ref64_mem.transpose_cast(src, True, sb, mb, lens, BF16), f"to_cl sub={sub}")
    wide = torch.randn(B, T, C + 26, generator=g).to(F16)
    cl = wide[..., 3:3 + C]
    clg = wide.to(DEV)[..., 3:3 + C]
    for dt in (F32, F16):
        res = ops.to_channels_first(clg, dt, lg, sg, mg)
        _check("transpose_cast_kernel", res, *ref64_mem.transpose_cast(cl, False, sb, mb, lens, dt),
               f"to_cf sub={sub} {dt}")


# ------------------------------------------------------------------------------------------------------------------
# reductions and pools
# ------------------------------------------------------------------------------------------------------------------
def test_global_avgpool(tmp_path):
    """t_stride 2 with odd T (the last row counts), F = 5, C = 100; and a 1-D fp32 input with t_stride 1."""
    g = _g(7)
    x = (torch.randn(3, 15, 5, 100, generator=g) + 0.5).to(F16)
    xg = x.to(DEV)
    out = _one_launch(lambda: ops.global_avgpool(xg, 0.2, F32, t_stride=2), tmp_path, "gap", "global_avgpool_kernel")
    _check("global_avgpool_kernel", out, *ref64_mem.global_avgpool(x, 0.2, 2, F32), "gap ts=2")
    x1 = torch.randn(2, 301, 128, generator=g)
    out = ops.global_avgpool(x1.to(DEV), 0.01, BF16)
    _check("global_avgpool_kernel", out, *ref64_mem.global_avgpool(x1, 0.01, 1, BF16), "gap 1-D")


def test_log_norm(tmp_path):
    g = _g(8)
    mel = torch.randn(3, 80, 301, generator=g) * 1.5 - 1
    mel[1, :, :10] = -6                                   # all-quiet frames: the output is far below 0
    mg = mel.to(DEV)
    out = _one_launch(lambda: ops.log_norm(mg), tmp_path, "log_norm", "log_norm_kernel")
    _check("log_norm_kernel", out, *ref64_mem.log_norm(mel), "log_norm")


# name: (x dtype, out dtype, shape [B, T, F, C], pt, pf, kernel)
POOL_CASES = {
    "vec8": (F16, F16, (2, 15, 22, 64), 2, 4, "avgpool_vec8_kernel"),
    "vec8_bf16": (BF16, BF16, (2, 15, 10, 32), 2, 2, "avgpool_vec8_kernel"),
    "scalar": (F32, BF16, (2, 15, 10, 24), 2, 3, "avgpool_kernel"),
    "scalar_C12": (F16, F16, (2, 9, 8, 12), 2, 2, "avgpool_kernel"),
}


@pytest.mark.parametrize("case", list(POOL_CASES))
def test_avgpool(case, tmp_path):
    """Odd T (the last row is replicated) and F % pf != 0 (trailing columns dropped)."""
    xdt, odt, shape, pt, pf, kernel = POOL_CASES[case]
    x = (torch.randn(*shape, generator=_g(9)) * 2 + 1).to(xdt)
    xg = x.to(DEV)
    out = _one_launch(lambda: ops.avgpool(xg, pt, pf, odt), tmp_path, f"ap_{case}", kernel)
    _check(kernel, out, *ref64_mem.avgpool(x, pt, pf, odt), f"avgpool {case}")


MAXPOOL_CASES = {
    "vec8": (BF16, BF16, (2, 9, 22, 64), 4, "affine_act_maxpool_vec8_kernel"),
    "vec8_f16": (F16, F16, (2, 9, 10, 16), 2, "affine_act_maxpool_vec8_kernel"),
    "scalar": (F32, F32, (2, 9, 10, 24), 3, "affine_act_maxpool_kernel"),
    "scalar_16to32": (F16, F32, (2, 9, 10, 64), 2, "affine_act_maxpool_kernel"),
}


@pytest.mark.parametrize("case", list(MAXPOOL_CASES))
def test_affine_act_maxpool(case, tmp_path):
    """Half the channels have a negative scale (the max then comes from the smallest x); F % pf != 0."""
    xdt, odt, shape, pf, kernel = MAXPOOL_CASES[case]
    g = _g(10)
    C = shape[-1]
    x = torch.randn(*shape, generator=g).to(xdt)
    sc = torch.randn(C, generator=g).abs() + 0.1
    sc[::2] = -sc[::2]
    sh = torch.randn(C, generator=g)
    xg, scg, shg = x.to(DEV), sc.to(DEV), sh.to(DEV)
    out = _one_launch(lambda: ops.affine_act_maxpool(xg, scg, shg, 0.01, pf, odt), tmp_path, f"mp_{case}", kernel)
    _check(kernel, out, *ref64_mem.affine_act_maxpool(x, sc, sh, 0.01, pf, odt), f"maxpool {case}")


# ------------------------------------------------------------------------------------------------------------------
# direct convolution for small Cin
# ------------------------------------------------------------------------------------------------------------------
# name: (x shape [B, T, F, Cin] or [B, T, Cin], x dtype, Cout, taps, raw dtype, act dtype, outputs in odd slices,
#        bias scale, kernel)
CS_CASES = {
    "vec4_2d": ((2, 21, 20, 1), F16, 64, ops.taps_2d(3, 3, 1, 1), F32, BF16, "act", 1.0, "conv_small_vec_kernel<4>"),
    "vec4_2d_unaligned_raw": ((2, 13, 8, 3), BF16, 16, ops.taps_2d(3, 3, 1, 1), F16, F32, "raw", 1.0,
                              "conv_small_vec_kernel<4>"),
    "vec4_bias_dominated": ((2, 21, 20, 1), F32, 32, ops.taps_2d(3, 3, 1, 1), F32, F32, "", 1e3,
                            "conv_small_vec_kernel<4>"),
    "vec1_1d": ((2, 77, 16), F32, 8, ops.taps_1d(5, 2), F32, F16, "", 1.0, "conv_small_vec_kernel<1>"),
    "vec1_F5": ((2, 13, 5, 3), BF16, 16, ops.taps_2d(3, 3, 1, 1), BF16, F32, "act", 1.0, "conv_small_vec_kernel<1>"),
    "scalar_cout12": ((2, 13, 10, 3), F16, 12, ops.taps_2d(3, 3, 1, 1), F32, F16, "", 1.0, "conv_small_kernel"),
    "scalar_large_weights": ((2, 40, 16), BF16, 72, ops.taps_1d(9, 1), F32, BF16, "raw", 1.0, "conv_small_kernel"),
}


@pytest.mark.parametrize("case", list(CS_CASES))
def test_conv_small(case, tmp_path):
    """Both outputs, aligned and odd-offset ones, lens T and 9, taps past the T and F edges."""
    shape, xdt, Cout, taps, rdt, adt, odd, bscale, kernel = CS_CASES[case]
    g = _g(11 + Cout)
    Cin = shape[-1]
    x = torch.randn(*shape, generator=g)
    w = torch.randn(len(taps), Cout, Cin, generator=g) / (len(taps) * Cin) ** 0.5
    bias = torch.randn(Cout, generator=g) * bscale
    if bscale > 1:
        x = x * 1e-3
    x = x.to(xdt)
    lens = torch.tensor([shape[1], 9], dtype=torch.int32)
    sc = ops.pack_small_conv(w, bias, taps, DEV)
    xg, lg = x.to(DEV), lens.to(DEV)
    oshape = shape[:-1] + (Cout,)
    raw = _slice_out(oshape, rdt) if odd == "raw" else rdt
    act_out = _slice_out(oshape, adt) if odd == "act" else adt
    fn = lambda: ops.conv_small(xg, sc, raw=raw, act_out=act_out, act=ops.ACT_LRELU, slope=0.1, lens=lg)
    r, a = _one_launch(fn, tmp_path, f"cs_{case}", kernel)
    _check(kernel, r, *ref64_mem.conv_small(x, w, bias, taps, lens, ops.ACT_NONE, 0.0, rdt), f"conv_small {case} raw")
    _check(kernel, a, *ref64_mem.conv_small(x, w, bias, taps, lens, ops.ACT_LRELU, 0.1, adt), f"conv_small {case} act")
    _, t = ops.conv_small(xg, sc, act_out=F32, act=ops.ACT_SWISH, lens=lg)
    _check(kernel, t, *ref64_mem.conv_small(x, w, bias, taps, lens, ops.ACT_SWISH, 0.0, F32), f"conv_small {case} swish")


# ------------------------------------------------------------------------------------------------------------------
# depthwise convolution
# ------------------------------------------------------------------------------------------------------------------
# name: (x shape [B, T, (F,) Cx], x dtype, out dtype, k, stride, pad, glu, act, lens, kernel)
DW_CASES = {
    "tiled_glu_k31": ((3, 150, 128), F32, F32, (31, 1), (1, 1), (15, 0), True, ops.ACT_SWISH, True,
                      "dwconv_time_tiled_kernel"),
    "tiled_glu_k5_nolens": ((2, 70, 48), BF16, F16, (5, 1), (1, 1), (2, 0), True, ops.ACT_NONE, False,
                            "dwconv_time_tiled_kernel"),
    "tiled_k7": ((2, 100, 40), BF16, BF16, (7, 1), (1, 1), (3, 0), False, ops.ACT_LRELU, True,
                 "dwconv_time_tiled_kernel"),
    "vec8_2d_s2": ((2, 15, 20, 64), F16, F16, (3, 3), (2, 2), (1, 1), False, ops.ACT_LRELU, True,
                   "dwconv_vec8_kernel"),
    "vec8_1d_k3": ((2, 50, 32), BF16, BF16, (3, 1), (1, 1), (1, 0), False, ops.ACT_NONE, True, "dwconv_vec8_kernel"),
    "scalar_glu_k3": ((2, 50, 48), F32, F32, (3, 1), (1, 1), (1, 0), True, ops.ACT_NONE, True, "dwconv_kernel"),
    "scalar_stride2": ((2, 31, 48), F32, BF16, (3, 1), (2, 1), (1, 0), False, ops.ACT_SWISH, True, "dwconv_kernel"),
    "scalar_C12": ((2, 15, 10, 12), F16, F16, (3, 3), (1, 1), (1, 1), False, ops.ACT_LRELU, True, "dwconv_kernel"),
}


@pytest.mark.parametrize("case", list(DW_CASES))
def test_dwconv(case, tmp_path):
    """Input rows past lens_in are NaN; output rows past lens_out must be zeros (lens_out = ceil(lens_in / stride))."""
    shape, xdt, odt, k, stride, pad, glu, act, use_lens, kernel = DW_CASES[case]
    g = _g(12 + shape[-1])
    B, T = shape[0], shape[1]
    C = shape[-1] // 2 if glu else shape[-1]
    lens_in = torch.tensor([T, min(37, T // 2 + 1), 0][:B], dtype=torch.int32) if use_lens else None
    lens_out = None if lens_in is None else (lens_in + stride[0] - 1) // stride[0]
    x = torch.randn(*shape, generator=g) * 2
    if lens_in is not None:
        x = _nan_rows(x, lens_in)
    x = x.to(xdt)
    w = torch.randn(k[0] * k[1], C, generator=g) / k[0] ** 0.5
    bias = torch.randn(C, generator=g)
    xg, wg, bg = x.to(DEV), w.to(DEV), bias.to(DEV)
    lig = None if lens_in is None else lens_in.to(DEV)
    log = None if lens_out is None else lens_out.to(DEV)
    fn = lambda: ops.dwconv(xg, wg, bg, k, stride, pad, glu=glu, act=act, slope=0.2, out_dtype=odt, lens_in=lig,
                            lens_out=log)
    out = _one_launch(fn, tmp_path, f"dw_{case}", kernel)
    _check(kernel, out, *ref64_mem.dwconv(x, w, bias, k, stride, pad, glu, act, 0.2, lens_in, lens_out, odt),
           f"dwconv {case}")


# ------------------------------------------------------------------------------------------------------------------
# single-output-channel convolution (as_conv_igemm, Cout = 1)
# ------------------------------------------------------------------------------------------------------------------
def _bf(dt):
    return "true" if dt == BF16 else "false"


# name: (Cin, ntaps, dilation, T, x dtype, bias scale, path, kernel); path None: not eligible for the Cout = 1 kernels,
# the tensor-core convolution takes it
C1_CASES = {
    "mma_cin32_k7": (32, 7, 1, 1000, F16, 1.0, "mma", "conv_cout1_mma_kernel<false>"),
    "mma_cin64_k3_short": (64, 3, 1, 200, BF16, 1.0, "mma", "conv_cout1_mma_kernel<true>"),
    "mma_cin16_k8_dil9": (16, 8, 9, 777, BF16, 1.0, "mma", "conv_cout1_mma_kernel<true>"),
    "mma_bias_dominated": (32, 7, 1, 600, F16, 1e3, "mma", "conv_cout1_mma_kernel<false>"),
    "fp32_cin8": (8, 7, 1, 1500, F16, 1.0, "fp32", "conv_cout1_kernel<false>"),
    "fp32_cin24": (24, 5, 2, 1100, BF16, 1.0, "fp32", "conv_cout1_kernel<true>"),
    "fp32_cin40": (40, 3, 1, 300, F16, 1.0, "fp32", "conv_cout1_kernel<false>"),
    "fp32_cin56": (56, 7, 1, 250, BF16, 1.0, "fp32", "conv_cout1_kernel<true>"),
    "fp32_taps9": (32, 9, 1, 1030, F16, 1.0, "fp32", "conv_cout1_kernel<false>"),
    "fp32_taps16_dil4": (16, 16, 4, 2100, BF16, 1.0, "fp32", "conv_cout1_kernel<true>"),
    "fp32_bias_dominated": (24, 9, 1, 700, BF16, 1e3, "fp32", "conv_cout1_kernel<true>"),
    "igemm_cin72": (72, 7, 1, 400, F16, 1.0, None, "conv_igemm_kernel<16, 64, false>"),
    "halo_span65": (32, 6, 13, 400, BF16, 1.0, None, "conv_halo_sw_kernel<16, 32, true>"),
}


def _c1_inputs(Cin, ntaps, dil, T, xdt, bscale, seed):
    g = _g(seed)
    B = 3
    x = torch.randn(B, T, Cin, generator=g) * 0.5
    if bscale > 1:
        x = x * 1e-3
    w = (torch.randn(ntaps, 1, Cin, generator=g) / (ntaps * Cin) ** 0.5).to(xdt)
    bias = torch.randn(1, generator=g) * bscale
    lens = torch.tensor([T, 255, 0], dtype=torch.int32)
    return x.to(xdt), w, bias, ops.taps_1d(ntaps, dil), lens


def _c1_ref(x, w, bias, taps, lens, scale, act, dt, path):
    if path is None:        # tensor-core convolution: the bias is added once, in the epilogue
        return ref64.conv(x, w, taps, bias=bias, lens=lens, scale=scale, act=act, dtype=dt)
    return ref64_mem.conv_cout1(x, w, bias, taps, lens, scale, act, 0.0, dt, path)


@pytest.mark.parametrize("case", list(C1_CASES))
def test_conv_cout1(case, tmp_path):
    """lens T, 255, 0; T < 256 and T not a multiple of 256 / 1024; out_scale 0.5; raw fp32 next to a tanh output in
    fp32, fp16, bf16 and (Cout = 1 kernels only) AS_PCM16."""
    Cin, ntaps, dil, T, xdt, bscale, path, kernel = C1_CASES[case]
    x, w, bias, taps, lens = _c1_inputs(Cin, ntaps, dil, T, xdt, bscale, Cin * 100 + ntaps)
    pw = ops.pack_conv(w.float(), bias, taps, xdt, DEV)
    xg, lg = x.to(DEV), lens.to(DEV)
    act_dts = [F32, F16, BF16] + ([torch.int16] if path else [])
    for i, adt in enumerate(act_dts):
        fn = lambda: ops.conv(xg, pw, raw=F32, act_out=adt, act=ops.ACT_TANH, scale=0.5, lens=lg)
        raw, act = _one_launch(fn, tmp_path, f"c1_{case}", kernel, MEM_KERNELS + CONV_KERNELS) if i == 0 else fn()
        if i == 0:
            _check(kernel, raw, *_c1_ref(x, w, bias, taps, lens, 0.5, ops.ACT_NONE, F32, path), f"cout1 {case} raw")
        _check(kernel, act, *_c1_ref(x, w, bias, taps, lens, 0.5, ops.ACT_TANH, adt, path), f"cout1 {case} {adt}")


# ------------------------------------------------------------------------------------------------------------------
# census: the memory-bound kernels the product launches
# ------------------------------------------------------------------------------------------------------------------
CASE_TABLE = sorted({"embed_kernel", "repeat_rows_kernel", "expand_tokens_kernel", "length_regulate_kernel",
                     "transpose_cast_kernel", "global_avgpool_kernel", "log_norm_kernel"} |
                    {c[-1] for c in LN_CASES.values()} | {c[-1] for c in POOL_CASES.values()} |
                    {c[-1] for c in MAXPOOL_CASES.values()} | {c[-1] for c in CS_CASES.values()} |
                    {c[-1] for c in DW_CASES.values()} | {c[-1] for c in C1_CASES.values() if c[-2]})


def test_case_table_covers_every_dispatch_path():
    """20 kernel families: 3 LayerNorm vector widths, 2 conv_small_vec widths, 2 x 2 Cout = 1 kernels."""
    assert len(CASE_TABLE) == 25, CASE_TABLE
    assert {k.split("<")[0] for k in CASE_TABLE} == set(MEM_KERNELS)


@pytest.mark.parametrize("Tr", [240, 700])
def test_product_census(Tr, tmp_path):
    """At the benchmark's shape (16 utterances x 150 tokens) with 240- and 700-frame reference mels, every memory-bound
    or Cout = 1 kernel the product launches is in the case table."""
    import bench
    from artspeech_b200 import engine
    from tests import util
    model, gen = util.acoustic_model(0), util.generator(0)
    tok, tl, mel, ml, dur = bench.make_inputs(0, Tr=Tr)
    syn = engine.Synthesizer(model, gen, device=DEV, use_cuda_graph=False)
    _, ks = launches(lambda: syn.synthesize(tok.to(DEV), tl, mel.to(DEV), ml, dur, predict_durations=True), tmp_path,
                     f"census_{Tr}")
    census = sorted({k for k, _ in ks if k.split("<")[0] in MEM_KERNELS})
    print(f"[mem] census Tr={Tr}: {census}")
    assert census, "no memory-bound kernel in the product's trace"
    missing = sorted(set(census) - set(CASE_TABLE))
    assert not missing, f"kernels without a case: {missing}"


def test_zz_report_worst_ratios():
    """Prints the largest err / bound seen per kernel in this session (run with -s)."""
    for k in sorted(WORST):
        print(f"[mem] worst err/bound {k}: {WORST[k]:.3g}")
