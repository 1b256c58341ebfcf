"""Host-side wrappers of the C-ABI primitives (``include/artspeech_b200.h``).

Everything here is plumbing: pointer extraction from torch CUDA tensors, output allocation through
torch's caching allocator, the current stream.  The arithmetic happens in the .so.  Activations are
channels-last (``[B, T, C]`` / ``[B, T, F, C]``); a channel slice of a wider buffer is passed as a
strided torch view (``stride(-1) == 1``, row stride = the buffer's channel count), which is how
concatenations are fused away.
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass, field
from typing import Optional, Sequence

import numpy as np
import torch

from . import _lib
from ._lib import (ACT_ABS, ACT_LRELU, ACT_NONE, ACT_RELU, ACT_SWISH, ACT_TANH, AS_BF16, AS_F16,
                   AS_F32, AS_PCM16)

# torch.int16 = 16-bit PCM, accepted as the activated output of a single-output-channel convolution only
_DT = {torch.float16: AS_F16, torch.bfloat16: AS_BF16, torch.float32: AS_F32, torch.int16: AS_PCM16}

# number of kernels of ours launched since the last reset (bench.py reports it as gpu_launches)
launch_count = 0


def _count(n: int = 1) -> None:
    global launch_count
    launch_count += n


def dtype_code(dt: torch.dtype) -> int:
    try:
        return _DT[dt]
    except KeyError:
        raise _lib.AsError(f"unsupported dtype {dt}") from None


def _stream(t: torch.Tensor) -> int:
    return torch.cuda.current_stream(t.device).cuda_stream


def _require_cuda(t: torch.Tensor, name: str) -> None:
    if not t.is_cuda:
        raise _lib.AsError(f"{name}: artspeech_b200 ops need CUDA tensors (there is no CPU fallback)")


def _rows_ld(t: torch.Tensor, name: str) -> int:
    """Row stride (elements) of a channels-last tensor/view whose outer dims are dense."""
    if t.stride(-1) != 1 and t.shape[-1] != 1:
        raise _lib.AsError(f"{name}: channel stride must be 1")
    ld = t.stride(-2) if t.dim() >= 2 else t.shape[-1]
    exp = ld
    for d in range(t.dim() - 2, 0, -1):
        exp *= t.shape[d]
        if t.shape[d - 1] != 1 and t.stride(d - 1) != exp:
            raise _lib.AsError(f"{name}: outer dims must be dense (shape {tuple(t.shape)}, strides {t.stride()})")
    return ld


# --------------------------------------------------------------------------------------------
# implicit-GEMM convolution
# --------------------------------------------------------------------------------------------
@dataclass
class PackedConv:
    """Weights of one dense contraction in the kernel's layout ``[ntaps][CoutP][CinP]`` (K-major)."""
    w: torch.Tensor                 # 16-bit, device
    bias: Optional[torch.Tensor]    # fp32 [Cout], device (or None)
    ntaps: int
    Cin: int
    Cout: int
    CinP: int
    CoutP: int
    taps: Sequence[tuple]           # (dt, df) per tap
    _dt: object = field(default=None, repr=False)
    _df: object = field(default=None, repr=False)

    def __post_init__(self):
        n = len(self.taps)
        self._dt = (C.c_int32 * n)(*[int(t[0]) for t in self.taps])
        self._df = (C.c_int32 * n)(*[int(t[1]) for t in self.taps])


def conv_tile_n(cout: int) -> int:
    """Same rule as ``as_conv_tile_n`` (kept in Python so packing works without a GPU)."""
    if cout <= 16:
        return 16
    if cout <= 32:
        return 32
    if cout <= 64:
        return 64
    if cout <= 128:
        return 128
    if cout % 256 == 0:
        return 256
    if cout % 128 == 0:
        return 128
    p256 = (cout + 255) // 256 * 256
    p128 = (cout + 127) // 128 * 128
    return 128 if p128 < p256 else 256


def pack_conv(w_taps: torch.Tensor, bias: Optional[torch.Tensor], taps: Sequence[tuple],
              dtype: torch.dtype, device) -> PackedConv:
    """``w_taps`` fp32 ``[ntaps, Cout, Cin]`` -> zero-padded 16-bit ``[ntaps, CoutP, CinP]``."""
    ntaps, cout, cin = w_taps.shape
    assert ntaps == len(taps)
    bk = 64 if cin >= 64 else 32
    cinp = (cin + bk - 1) // bk * bk
    bn = conv_tile_n(cout)
    coutp = (cout + bn - 1) // bn * bn
    wp = torch.zeros(ntaps, coutp, cinp, dtype=torch.float32)
    wp[:, :cout, :cin] = w_taps.detach().float().cpu()
    wp = wp.to(dtype).to(device).contiguous()
    b = None if bias is None else bias.detach().float().to(device).contiguous()
    return PackedConv(wp, b, ntaps, cin, cout, cinp, coutp, list(taps))


def _out_arg(spec, shape, device):
    """spec: None | torch.dtype (allocate) | tensor/view (write into it)."""
    if spec is None:
        return None
    if isinstance(spec, torch.dtype):
        return torch.empty(shape, dtype=spec, device=device)
    return spec


def conv(x: torch.Tensor, pw: PackedConv, *, out_shape=None, use_bias: bool = True,
         res1: Optional[torch.Tensor] = None, res2: Optional[torch.Tensor] = None,
         scale: float = 1.0, raw=None, act_out=None, act: int = ACT_NONE, slope: float = 0.0,
         lens: Optional[torch.Tensor] = None):
    """Run ``as_conv_igemm``.

    ``x``: ``[B, T, C]`` or ``[B, T, F, C]`` 16-bit channels-last (may be a channel-slice view).
    ``out_shape``: ``(To, Fo)`` when the output grid differs from the input's ('valid' convs).
    ``raw`` / ``act_out``: ``None``, a dtype (allocate) or a tensor/view to write into.
    Returns ``(raw_tensor_or_None, act_tensor_or_None)``.
    """
    _require_cuda(x, "conv")
    lib = _lib.load()
    if x.dim() == 3:
        B, T, Cin = x.shape
        F = 1
    else:
        B, T, F, Cin = x.shape
    if Cin != pw.Cin:
        raise _lib.AsError(f"conv: input has {Cin} channels, weights expect {pw.Cin}")
    To, Fo = (T, F) if out_shape is None else out_shape
    oshape = (B, To, pw.Cout) if x.dim() == 3 else (B, To, Fo, pw.Cout)
    raw_t = _out_arg(raw, oshape, x.device)
    act_t = _out_arg(act_out, oshape, x.device)
    p = _lib.ConvParams()
    p.x = x.data_ptr(); p.x_dtype = dtype_code(x.dtype)
    p.B, p.T, p.F, p.Cin = B, T, F, Cin
    p.x_ld = _rows_ld(x, "conv.x")
    if pw.w.dtype != x.dtype:
        raise _lib.AsError(f"conv: x is {x.dtype} but weights were packed as {pw.w.dtype}")
    p.w = pw.w.data_ptr()
    p.ntaps, p.CinP, p.CoutP, p.Cout = pw.ntaps, pw.CinP, pw.CoutP, pw.Cout
    p.tap_dt = C.cast(pw._dt, _lib.c_i32_p); p.tap_df = C.cast(pw._df, _lib.c_i32_p)
    p.To, p.Fo = To, Fo
    p.bias = pw.bias.data_ptr() if (use_bias and pw.bias is not None) else None
    for name, r in (("res1", res1), ("res2", res2)):
        if r is not None:
            setattr(p, name, r.data_ptr())
            setattr(p, name + "_dtype", dtype_code(r.dtype))
            setattr(p, name + "_ld", _rows_ld(r, "conv." + name))
    p.out_scale = float(scale)
    if raw_t is not None:
        p.y_raw = raw_t.data_ptr(); p.y_raw_dtype = dtype_code(raw_t.dtype)
        p.y_raw_ld = _rows_ld(raw_t, "conv.raw")
    if act_t is not None:
        p.y_act = act_t.data_ptr(); p.y_act_dtype = dtype_code(act_t.dtype)
        p.y_act_ld = _rows_ld(act_t, "conv.act_out")
    p.act = int(act); p.slope = float(slope)
    if lens is not None:
        if lens.dtype != torch.int32:
            raise _lib.AsError("conv: lens must be int32")
        p.lens = lens.data_ptr()
    with torch.cuda.device(x.device):
        rc = lib.as_conv_igemm(C.byref(p), _stream(x))
    _lib.check(rc, "as_conv_igemm")
    _count()
    return raw_t, act_t


def resblock_pair(xa: torch.Tensor, c1: PackedConv, c2: PackedConv, k: int, dil: int, *, slope: float,
                  res2: Optional[torch.Tensor] = None, res3: Optional[torch.Tensor] = None, scale: float = 1.0,
                  out_act: int = ACT_NONE, out_slope: float = 1.0, lens: Optional[torch.Tensor] = None,
                  out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Run ``as_hifigan_resblock_pair`` on the ACTIVATED residual stream ``xa = leaky_relu(x, slope)``.

    ``xa``: ``[B, L, C]`` 16-bit channels-last, ``C`` in {32, 64, 128}; ``c1`` / ``c2``: the packed
    ``Conv1d(C, C, k, dilation=dil)`` / ``Conv1d(C, C, k)`` of one ResBlock1 iteration.  Returns
    ``out_act((conv2(lrelu(conv1(xa))) + x + res2 + res3) * scale)`` as a 16-bit ``[B, L, C]`` tensor.
    """
    _require_cuda(xa, "resblock_pair")
    lib = _lib.load()
    B, L, C_ = xa.shape
    for pw in (c1, c2):
        if (pw.Cin, pw.Cout, pw.CinP, pw.CoutP, pw.ntaps) != (C_, C_, C_, C_, k) or pw.w.dtype != xa.dtype or pw.bias is None:
            raise _lib.AsError("resblock_pair: weights must be packed [k][C][C] in the activation dtype, with bias")
    if out is None:
        out = torch.empty(B, L, C_, dtype=xa.dtype, device=xa.device)
    p = _lib.ResblockPairParams()
    p.x = xa.data_ptr(); p.x_ld = _rows_ld(xa, "resblock_pair.x"); p.dtype = dtype_code(xa.dtype)
    p.B, p.L, p.C, p.k, p.dil = B, L, C_, int(k), int(dil)
    p.w1 = c1.w.data_ptr(); p.b1 = c1.bias.data_ptr(); p.w2 = c2.w.data_ptr(); p.b2 = c2.bias.data_ptr()
    p.slope = float(slope)
    for name, r in (("res2", res2), ("res3", res3)):
        if r is not None:
            if r.dtype != xa.dtype or r.shape != xa.shape:
                raise _lib.AsError(f"resblock_pair: {name} must match x in shape and dtype")
            setattr(p, name, r.data_ptr())
            setattr(p, name + "_ld", _rows_ld(r, "resblock_pair." + name))
    p.out_scale = float(scale); p.out_act = int(out_act); p.out_slope = float(out_slope)
    p.y = out.data_ptr(); p.y_ld = _rows_ld(out, "resblock_pair.out")
    if lens is not None:
        if lens.dtype != torch.int32:
            raise _lib.AsError("resblock_pair: lens must be int32")
        p.lens = lens.data_ptr()
    with torch.cuda.device(xa.device):
        rc = lib.as_hifigan_resblock_pair(C.byref(p), _stream(xa))
    _lib.check(rc, "as_hifigan_resblock_pair")
    _count()
    return out


# tap tables -------------------------------------------------------------------------------------
def taps_1d(k: int, dilation: int = 1, padding: Optional[int] = None):
    """Conv1d taps: input index = t + j*dilation - padding ('same' padding by default)."""
    if padding is None:
        padding = (k * dilation - dilation) // 2
    return [(j * dilation - padding, 0) for j in range(k)]


def taps_2d(kt: int, kf: int, pad_t: int, pad_f: int):
    """Conv2d taps over (T, F); order matches ``w.permute`` in ``conv2d_weight_taps``."""
    return [(jt - pad_t, jf - pad_f) for jt in range(kt) for jf in range(kf)]


# --------------------------------------------------------------------------------------------
# memory-bound / small kernels
# --------------------------------------------------------------------------------------------
def _p(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _dims(x: torch.Tensor):
    """(B, T, F, C) of a channels-last 3-D or 4-D tensor."""
    if x.dim() == 3:
        return x.shape[0], x.shape[1], 1, x.shape[2]
    return tuple(x.shape)


def _i32(t: Optional[torch.Tensor], name: str):
    if t is not None and t.dtype != torch.int32:
        raise _lib.AsError(f"{name}: lens must be int32")
    return t


def _run(name: str, x: torch.Tensor, *args):
    lib = _lib.load()
    with torch.cuda.device(x.device):
        rc = getattr(lib, name)(*args, _stream(x))
    _lib.check(rc, name)
    _count()


def embed(tokens, table, scale, lens, *, out32: bool, out16=None):
    """``tokens`` int64 [B,T]; returns (fp32 [B,T,C] or None, 16-bit [B,T,C] or None)."""
    _require_cuda(tokens, "embed")
    B, T = tokens.shape
    C_ = table.shape[1]
    o32 = torch.empty(B, T, C_, dtype=torch.float32, device=tokens.device) if out32 else None
    o16 = torch.empty(B, T, C_, dtype=out16, device=tokens.device) if out16 is not None else None
    _run("as_embed", tokens, tokens.contiguous().data_ptr(), table.data_ptr(), table.shape[0], B, T, C_,
         float(scale), _p(_i32(lens, "embed")), _p(o32), _p(o16), dtype_code(out16) if out16 is not None else 0)
    return o32, o16


def layernorm(x, gamma, beta, eps, *, act=ACT_NONE, slope=0.0, lens=None, out_a=None, out_b=None):
    """Row-wise LayerNorm over channels of ``x`` [B,T,C]; ``out_a``/``out_b``: dtype or tensor."""
    _require_cuda(x, "layernorm")
    B, T, C_ = x.shape
    oa = _out_arg(out_a, (B, T, C_), x.device)
    ob = _out_arg(out_b, (B, T, C_), x.device)
    _run("as_layernorm", x, x.data_ptr(), dtype_code(x.dtype), _rows_ld(x, "layernorm.x"), B, T, C_,
         gamma.data_ptr(), beta.data_ptr(), float(eps), int(act), float(slope), _p(_i32(lens, "layernorm")),
         _p(oa), dtype_code(oa.dtype) if oa is not None else 0, _rows_ld(oa, "ln.a") if oa is not None else 0,
         _p(ob), dtype_code(ob.dtype) if ob is not None else 0, _rows_ld(ob, "ln.b") if ob is not None else 0)
    return oa, ob


def relpos_attention(qkv, emb_rel_k, emb_rel_v, window, n_heads, lens, out_dtype):
    """``qkv`` fp32 [B,T,3*H*D] -> [B,T,H*D]."""
    _require_cuda(qkv, "relpos_attention")
    B, T, C3 = qkv.shape
    HD = C3 // 3
    out = torch.empty(B, T, HD, dtype=out_dtype, device=qkv.device)
    _run("as_relpos_attention", qkv, qkv.data_ptr(), _rows_ld(qkv, "qkv"), emb_rel_k.data_ptr(),
         emb_rel_v.data_ptr(), int(window), B, T, n_heads, HD // n_heads, _p(_i32(lens, "relpos")),
         out.data_ptr(), dtype_code(out_dtype), HD)
    return out


def conformer_attention(q, k, v, pos, u_bias, v_bias, n_heads, lens, out_dtype):
    """``q,k,v`` fp32 views [B,T,H*D] with a common row stride; ``pos`` fp32 [T,H*D]."""
    _require_cuda(q, "conformer_attention")
    B, T, HD = q.shape
    ld = _rows_ld(q, "q")
    assert _rows_ld(k, "k") == ld and _rows_ld(v, "v") == ld
    out = torch.empty(B, T, HD, dtype=out_dtype, device=q.device)
    _run("as_conformer_attention", q, q.data_ptr(), k.data_ptr(), v.data_ptr(), ld, pos.data_ptr(),
         u_bias.data_ptr(), v_bias.data_ptr(), B, T, n_heads, HD // n_heads, _p(_i32(lens, "conf")),
         out.data_ptr(), dtype_code(out_dtype), HD)
    return out


def instnorm_stats(x, lens, eps=1e-5):
    """``x`` [B,T,C] -> stats fp32 [B,C,2] = (mean, rstd) over valid frames."""
    _require_cuda(x, "instnorm_stats")
    B, T, C_ = x.shape
    st = torch.empty(B, C_, 2, dtype=torch.float32, device=x.device)
    _run("as_instnorm_stats", x, x.data_ptr(), dtype_code(x.dtype), _rows_ld(x, "in.x"), B, T, C_,
         _p(_i32(lens, "instnorm")), float(eps), st.data_ptr())
    return st


def adain_apply(x, stats, gb, slope, lens, out_dtype, up_w=None, up_b=None, out=None):
    """AdaIN + LeakyReLU (+ depthwise ConvTranspose upsample).  ``gb`` fp32 view [B, 2C]."""
    _require_cuda(x, "adain_apply")
    B, T, C_ = x.shape
    To = 2 * T if up_w is not None else T
    if out is None:
        out = torch.empty(B, To, C_, dtype=out_dtype, device=x.device)
    assert gb.shape == (B, 2 * C_) and gb.stride(1) == 1
    _run("as_adain_apply", x, x.data_ptr(), dtype_code(x.dtype), _rows_ld(x, "adain.x"), B, T, C_,
         stats.data_ptr(), gb.data_ptr(), gb.stride(0), float(slope), _p(_i32(lens, "adain")), _p(up_w),
         _p(up_b), out.data_ptr(), dtype_code(out.dtype), _rows_ld(out, "adain.out"))
    return out


def adain_norm(x, gb, slope, lens, out_dtype, up_w=None, up_b=None, eps=1e-5):
    """InstanceNorm statistics + AdaIN + LeakyReLU (+ pool) in one launch (``as_adain_norm_apply``)."""
    _require_cuda(x, "adain_norm")
    B, T, C_ = x.shape
    To = 2 * T if up_w is not None else T
    out = torch.empty(B, To, C_, dtype=out_dtype, device=x.device)
    st = torch.empty(B, C_, 2, dtype=torch.float32, device=x.device)
    assert gb.shape == (B, 2 * C_) and gb.stride(1) == 1
    _run("as_adain_norm_apply", x, x.data_ptr(), dtype_code(x.dtype), _rows_ld(x, "adain.x"), B, T, C_,
         gb.data_ptr(), gb.stride(0), float(eps), float(slope), _p(_i32(lens, "adain")), _p(up_w), _p(up_b),
         out.data_ptr(), dtype_code(out.dtype), _rows_ld(out, "adain.out"), st.data_ptr())
    return out


def repeat_rows(x, rep, lens, out_dtype=None, out=None):
    _require_cuda(x, "repeat_rows")
    B, T, C_ = x.shape
    if out is None:
        out = torch.empty(B, T * rep, C_, dtype=out_dtype or x.dtype, device=x.device)
    _run("as_repeat_rows", x, x.data_ptr(), dtype_code(x.dtype), _rows_ld(x, "rep.x"), B, T, C_, int(rep),
         _p(_i32(lens, "repeat")), out.data_ptr(), dtype_code(out.dtype), _rows_ld(out, "rep.out"))
    return out


def length_regulate(x, dur, lens_t, rep, To, out=None, out_dtype=None):
    """``x`` [B,Tt,C], ``dur`` int32 [B,Tt] -> (out [B,To,C], out_lens int32 [B])."""
    _require_cuda(x, "length_regulate")
    B, Tt, C_ = x.shape
    if out is None:
        out = torch.empty(B, To, C_, dtype=out_dtype or x.dtype, device=x.device)
    olens = torch.empty(B, dtype=torch.int32, device=x.device)
    assert dur.dtype == torch.int32 and dur.is_contiguous()
    _run("as_length_regulate", x, x.data_ptr(), dtype_code(x.dtype), _rows_ld(x, "lr.x"), B, Tt, C_,
         dur.data_ptr(), _p(_i32(lens_t, "length_regulate")), int(rep), int(To), out.data_ptr(),
         dtype_code(out.dtype), _rows_ld(out, "lr.out"), olens.data_ptr())
    return out, olens


def round_durations(pred, lens_t, scale=None):
    """``pred`` fp32 [B,Tt] (the duration predictor's output) -> (dur int32 [B,Tt] = ``round(pred).clamp(min=1)``
    for ``t < lens_t[b]`` and 0 beyond, sums int32 [B]); models.py:361 on the device.  ``scale`` (prosody
    ``duration_scale``): fp32 [B,Tt'] with Tt' >= Tt, or [B] (one value per utterance); rounds ``pred * scale``."""
    _require_cuda(pred, "round_durations")
    B, Tt = pred.shape
    if pred.stride(1) != 1:
        pred = pred.contiguous()
    dur = torch.empty(B, Tt, dtype=torch.int32, device=pred.device)
    sums = torch.empty(B, dtype=torch.int32, device=pred.device)
    lens_t = _i32(lens_t, "round_durations")
    if scale is None:
        _run("as_round_durations", pred, pred.data_ptr(), pred.stride(0), B, Tt, _p(lens_t), dur.data_ptr(),
             sums.data_ptr())
        return dur, sums
    if scale.dtype != torch.float32 or scale.device != pred.device or scale.shape[0] != B or scale.dim() > 2 or \
            (scale.dim() == 2 and (scale.shape[1] < Tt or scale.stride(1) != 1)):
        raise _lib.AsError(f"round_durations: scale must be fp32 [B] or [B, >= Tt] on {pred.device}, got "
                           f"{scale.dtype} {tuple(scale.shape)} on {scale.device}")
    if scale.dim() == 1 and scale.stride(0) != 1:
        scale = scale.contiguous()
    _run("as_round_durations_scaled", pred, pred.data_ptr(), pred.stride(0), B, Tt, _p(lens_t), scale.data_ptr(),
         scale.stride(0) if scale.dim() == 2 else 0, dur.data_ptr(), sums.data_ptr())
    return dur, sums


def prosody_apply(f0, n, ema, lens, ctrl, pitch_mean: float, pitch_std: float, energy_std: float):
    """Prosody edits of the arts predictor's tracks, in place (``as_prosody_apply``; semantics in
    ``artspeech_b200.prosody``): ``f0`` / ``n`` fp32 [B,Tm,1], ``ema`` fp32 [B,Tm,10] channels-last, ``lens`` int32
    [B] valid frames, ``ctrl`` fp32 [B,24] (``prosody.pack``).  The pitch / energy statistics are host floats."""
    _require_cuda(f0, "prosody_apply")
    B, Tm, _ = f0.shape
    for t, name, ch in ((f0, "f0", 1), (n, "n", 1), (ema, "ema", 10)):
        if t.dtype != torch.float32 or t.device != f0.device or tuple(t.shape) != (B, Tm, ch):
            raise _lib.AsError(f"prosody_apply: {name} must be fp32 [{B}, {Tm}, {ch}], got {t.dtype} {tuple(t.shape)}")
    if ctrl.dtype != torch.float32 or tuple(ctrl.shape) != (B, 24) or ctrl.stride() != (24, 1) or \
            ctrl.device != f0.device:
        raise _lib.AsError(f"prosody_apply: ctrl must be a dense fp32 [{B}, 24] device tensor")
    _run("as_prosody_apply", f0, f0.data_ptr(), _rows_ld(f0, "prosody.f0"), n.data_ptr(), _rows_ld(n, "prosody.n"),
         ema.data_ptr(), _rows_ld(ema, "prosody.ema"), B, Tm, _p(_i32(lens, "prosody_apply")), ctrl.data_ptr(),
         float(pitch_mean), float(pitch_std), float(energy_std))


def resample_encode(x, lens, fmt, S_out: int, *, m0: int = 0, out=None, out_lens=None, gain=None):
    """Waveforms in an output format (``as_resample_encode``; semantics in ``artspeech_b200.audio``): ``x`` fp32
    [B, S_in] at 24 kHz (unit element stride, any row stride), ``lens`` int32 [B] device sample counts (or None: every
    row holds S_in samples), ``fmt`` an ``audio.AudioFormat``.  Returns ``[B, S_out]`` of ``fmt.dtype``: samples
    ``m0 .. m0 + S_out - 1`` at the target rate, silence beyond each utterance's ``fmt.out_samples(len)``.  ``out``:
    an optional destination; ``out_lens``: an optional int32 [B] device tensor that receives the output lengths;
    ``gain``: an optional fp32 [B] device tensor multiplied into each utterance's samples before they are encoded
    (``as_resample_encode_gain``)."""
    _require_cuda(x, "resample_encode")
    if x.dtype != torch.float32 or x.dim() != 2 or (x.stride(1) != 1 and x.shape[1] > 1):
        raise _lib.AsError(f"resample_encode: x must be fp32 [B, S] with unit sample stride, got {x.dtype} "
                           f"{tuple(x.shape)} strides {x.stride()}")
    B, S_in = x.shape
    if out is None:
        out = torch.empty(B, int(S_out), dtype=fmt.dtype, device=x.device)
    elif out.dtype != fmt.dtype or tuple(out.shape) != (B, int(S_out)) or (out.stride(1) != 1 and S_out > 1) or \
            out.device != x.device:
        raise _lib.AsError(f"resample_encode: out must be {fmt.dtype} [{B}, {S_out}] on {x.device}")
    for t, name, dt in ((lens, "lens", torch.int32), (out_lens, "out_lens", torch.int32),
                        (gain, "gain", torch.float32)):
        if t is not None and (t.dtype != dt or t.device != x.device or t.numel() != B or
                              (B > 1 and t.stride(0) != 1)):
            raise _lib.AsError(f"resample_encode: {name} must be {dt} [{B}] on {x.device}")
    table = fmt.device_table(x.device)
    one = lambda n: (int(n) + 15) // 16 * 16           # a single row's stride is free: keep rows 16-byte aligned
    args = (x.data_ptr(), x.stride(0) if B > 1 else one(S_in), B, S_in, _p(lens), table.data_ptr(), fmt.table_ld,
            fmt.up, fmt.down, fmt.K, fmt.half_len, int(m0), int(S_out), out.data_ptr(),
            out.stride(0) if B > 1 else one(S_out), fmt.code, _p(out_lens))
    if gain is None:
        _run("as_resample_encode", x, *args)
    else:
        _run("as_resample_encode_gain", x, *args, gain.data_ptr())
    return out


LOUDNESS_LAUNCHES = 3            # AS_LOUDNESS_LAUNCHES


def loudness_measure(x, lens, sample_rate: int, target: float = -23.0, ceiling: float = -1.0):
    """Integrated loudness, true peak and normalisation gain per utterance (``as_loudness_measure``; semantics in
    ``artspeech_b200.audio``): ``x`` fp32 [B, S] (unit element stride, any row stride) at ``sample_rate`` Hz, ``lens``
    int32 [B] device sample counts (or None: every row holds S samples).  Returns ``(lufs, true_peak_db, gain_db,
    gain)``: fp64 [B], fp64 [B], fp64 [B] and fp32 [B] device tensors; ``gain`` is ``10^(gain_db/20)`` rounded once,
    the factor ``resample_encode(gain=)`` takes.  Three launches, no host synchronisation."""
    from . import audio
    _require_cuda(x, "loudness_measure")
    if x.dtype != torch.float32 or x.dim() != 2 or (x.stride(1) != 1 and x.shape[1] > 1):
        raise _lib.AsError(f"loudness_measure: x must be fp32 [B, S] with unit sample stride, got {x.dtype} "
                           f"{tuple(x.shape)} strides {x.stride()}")
    B, S = x.shape
    if lens is not None and (lens.dtype != torch.int32 or lens.device != x.device or lens.numel() != B or
                             (B > 1 and lens.stride(0) != 1)):
        raise _lib.AsError(f"loudness_measure: lens must be int32 [{B}] on {x.device}")
    kw = (C.c_double * 10)(*[float(v) for v in audio.k_weighting_taps(sample_rate)])
    tp = audio.true_peak_table()
    lufs = torch.empty(B, dtype=torch.float64, device=x.device)
    tp_db, gain_db = torch.empty_like(lufs), torch.empty_like(lufs)
    gain = torch.empty(B, dtype=torch.float32, device=x.device)
    nbytes = _lib.load().as_loudness_workspace_bytes(B, S, int(sample_rate))
    ws = torch.empty(max(int(nbytes), 1), dtype=torch.uint8, device=x.device)
    _run("as_loudness_measure", x, x.data_ptr(), x.stride(0) if B > 1 else S, B, S, _p(lens), int(sample_rate), kw,
         tp.ctypes.data_as(_lib.c_f32_p), float(target), float(ceiling), ws.data_ptr(), ws.numel(), lufs.data_ptr(),
         tp_db.data_ptr(), gain_db.data_ptr(), gain.data_ptr())
    _count(LOUDNESS_LAUNCHES - 1)
    return lufs, tp_db, gain_db, gain


def _wave_rows(x, name, dtype=torch.float32):
    if x.dtype != dtype or x.dim() != 2 or (x.stride(1) != 1 and x.shape[1] > 1):
        raise _lib.AsError(f"{name}: x must be {dtype} [B, S] with unit sample stride, got {x.dtype} "
                           f"{tuple(x.shape)} strides {x.stride()}")
    return x.shape


def _lens_arg(lens, B, device, name):
    if lens is not None and (lens.dtype != torch.int32 or lens.device != device or lens.numel() != B or
                             (B > 1 and lens.stride(0) != 1)):
        raise _lib.AsError(f"{name}: lens must be int32 [{B}] on {device}")
    return _p(lens)


def watermark_embed(x, lens, wm):
    """``x`` marked with ``wm`` (an ``audio.Watermark``; ``as_watermark_embed``, semantics in
    ``artspeech_b200.audio``): ``x`` fp32 [B, S] at 24 kHz (unit element stride, any row stride), ``lens`` int32 [B]
    device sample counts (or None: every row holds S samples).  Returns a new fp32 [B, S]; zeros beyond each length."""
    _require_cuda(x, "watermark_embed")
    B, S = _wave_rows(x, "watermark_embed")
    out = torch.empty(B, S, dtype=torch.float32, device=x.device)
    pat = wm.device_pattern(x.device)
    one = lambda n: (int(n) + 3) // 4 * 4              # a single row's stride is free: keep it a multiple of 4
    _run("as_watermark_embed", x, x.data_ptr(), x.stride(0) if B > 1 else one(S), B, S,
         _lens_arg(lens, B, x.device, "watermark_embed"), pat.data_ptr(), float(wm.alpha), out.data_ptr(),
         out.stride(0) if B > 1 else one(S))
    return out


def audio_decode(x, encoding: str):
    """fp32 [B, S] samples of encoded ``x`` (``as_audio_decode``): int16 for ``"pcm16"`` (``v / 32768``), uint8
    G.711 codes for ``"mulaw"`` / ``"alaw"`` (``audioop.ulaw2lin`` / ``alaw2lin``, then ``/ 32768``)."""
    from . import audio
    _require_cuda(x, "audio_decode")
    if encoding not in ("pcm16", "mulaw", "alaw"):
        raise _lib.AsError(f"audio_decode: encoding must be pcm16, mulaw or alaw, got {encoding!r}")
    B, S = _wave_rows(x, "audio_decode", audio.DTYPES[encoding])
    out = torch.empty(B, S, dtype=torch.float32, device=x.device)
    _run("as_audio_decode", x, x.data_ptr(), x.stride(0) if B > 1 else S, B, S, audio.CODES[encoding],
         out.data_ptr(), S)
    return out


def audio_to_mono(x, lens, encoding: str):
    """Mono fp32 [B, S] of encoded samples ``x`` (``as_audio_to_mono``; semantics in ``artspeech_b200.frontend``):
    ``x`` [B, S] (one channel) or [B, S, C] (C interleaved channels, 1 <= C <= 8), float32 / int16 / uint8 for
    ``encoding`` float32 / pcm16 / mulaw, alaw; unit element stride, dense channels, any row stride.  ``lens`` int32
    [B] device samples per channel (or None: every row holds S).  Output ``(x_0 + ... + x_{C-1}) / C`` of the decoded
    samples, zeros beyond each length.  One launch, no host synchronisation."""
    from . import audio
    _require_cuda(x, "audio_to_mono")
    if encoding not in audio.ENCODINGS:
        raise _lib.AsError(f"audio_to_mono: encoding must be one of {audio.ENCODINGS}, got {encoding!r}")
    if x.dtype != audio.DTYPES[encoding] or x.dim() not in (2, 3):
        raise _lib.AsError(f"audio_to_mono: x must be {audio.DTYPES[encoding]} [B, S] or [B, S, C], got {x.dtype} "
                           f"{tuple(x.shape)}")
    B, S = x.shape[:2]
    C_ = x.shape[2] if x.dim() == 3 else 1
    if x.dim() == 3 and (x.stride(2) != 1 and C_ > 1 or x.stride(1) != C_ and S > 1):
        raise _lib.AsError(f"audio_to_mono: channels must be interleaved densely, strides {x.stride()}")
    if x.dim() == 2 and x.stride(1) != 1 and S > 1:
        raise _lib.AsError(f"audio_to_mono: x must have unit sample stride, strides {x.stride()}")
    out = torch.empty(B, S, dtype=torch.float32, device=x.device)
    _run("as_audio_to_mono", x, x.data_ptr(), x.stride(0) if B > 1 else S * C_, B, S, C_, audio.CODES[encoding],
         _lens_arg(lens, B, x.device, "audio_to_mono"), out.data_ptr(), S)
    return out


TRIM_LAUNCHES = 2                # AS_TRIM_LAUNCHES


def trim_bounds(y, lens, top_db: float):
    """Leading / trailing silence of 24 kHz fp32 ``y`` [B, S] (unit element stride, any row stride; ``as_trim_bounds``,
    semantics in ``artspeech_b200.frontend``), ``lens`` int32 [B] device sample counts (or None).  Returns int32
    [B, 2] device ``(start, end)``.  Two launches, no host synchronisation."""
    _require_cuda(y, "trim_bounds")
    B, S = _wave_rows(y, "trim_bounds")
    bounds = torch.empty(B, 2, dtype=torch.int32, device=y.device)
    nbytes = _lib.load().as_trim_workspace_bytes(B, S)
    ws = torch.empty(max(int(nbytes), 1), dtype=torch.uint8, device=y.device)
    _run("as_trim_bounds", y, y.data_ptr(), y.stride(0) if B > 1 else S, B, S, _lens_arg(lens, B, y.device,
         "trim_bounds"), float(top_db), ws.data_ptr(), ws.numel(), bounds.data_ptr())
    _count(TRIM_LAUNCHES - 1)
    return bounds


DENOISE_LAUNCHES = 3             # AS_DENOISE_LAUNCHES
DENOISE_BINS, DENOISE_N, DENOISE_HOP = 257, 512, 128
DENOISE_ALPHA, DENOISE_QUANTILE = 0.98, 0.1
_denoise_tables = {}


def _denoise_consts(device):
    """(window, twiddle, itwiddle) fp32 device tensors of ``as_denoise``, computed once per device in fp64."""
    t = _denoise_tables.get(device)
    if t is None:
        i, m = np.arange(DENOISE_N), np.arange(DENOISE_N // 2)
        ang = 2.0 * np.pi * m / DENOISE_N
        tabs = (0.5 - 0.5 * np.cos(2.0 * np.pi * i / DENOISE_N), np.stack([np.cos(ang), -np.sin(ang)], 1),
                np.stack([np.cos(ang), np.sin(ang)], 1))
        t = tuple(torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(device) for a in tabs)
        _denoise_tables[device] = t
    return t


def denoise(y, lens, reduction_db: float, *, planes: bool = False):
    """Stationary-noise suppression of 24 kHz fp32 ``y`` [B, S] (unit element stride, any row stride; ``as_denoise``,
    semantics in ``artspeech_b200.frontend`` step 2b), ``lens`` int32 [B] device sample counts (or None: every row
    holds S samples), ``reduction_db`` in [0, 60].  Returns a new fp32 [B, S], zeros beyond each length.  With
    ``planes=True`` also the workspace's ``X`` (complex64 [B, 1 + S // 128, 257]), ``lambda`` (fp64 [B, 257]) and
    ``G`` (fp32 [B, 1 + S // 128, 257]) as views; frame rows at and beyond a row's ``1 + len // 128`` are not
    written.  Three launches, no host synchronisation."""
    _require_cuda(y, "denoise")
    B, S = _wave_rows(y, "denoise")
    rdb = float(reduction_db)
    if not 0.0 <= rdb <= 60.0:
        raise _lib.AsError(f"denoise: reduction_db must be in [0, 60], got {reduction_db!r}")
    window, tw, itw = _denoise_consts(y.device)
    out = torch.empty(B, S, dtype=torch.float32, device=y.device)
    nbytes = int(_lib.load().as_denoise_workspace_bytes(B, S))
    ws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=y.device)
    alpha = DENOISE_ALPHA
    _run("as_denoise", y, y.data_ptr(), y.stride(0) if B > 1 else S, B, S, _lens_arg(lens, B, y.device, "denoise"),
         rdb, window.data_ptr(), tw.data_ptr(), itw.data_ptr(), -math.log1p(-DENOISE_QUANTILE), 10.0 ** (-rdb / 20.0),
         alpha, 1.0 - alpha, ws.data_ptr(), ws.numel(), out.data_ptr(), S)
    _count(DENOISE_LAUNCHES - 1)
    if not planes:
        return out
    F = 1 + S // DENOISE_HOP
    align = lambda v: (v + 255) // 256 * 256
    nx, ng = B * F * DENOISE_BINS * 8, B * F * DENOISE_BINS * 4
    X = ws[:nx].view(torch.complex64).view(B, F, DENOISE_BINS)
    G = ws[align(nx):align(nx) + ng].view(torch.float32).view(B, F, DENOISE_BINS)
    lo = align(nx) + align(ng)
    lam = ws[lo:lo + B * DENOISE_BINS * 8].view(torch.float64).view(B, DENOISE_BINS)
    return out, X, lam, G


WATERMARK_DETECT_LAUNCHES = 2    # AS_WM_DETECT_LAUNCHES


def watermark_detect(x, lens, key: int, threshold: float = 6.0):
    """Watermark detection (``as_watermark_detect``; semantics in ``artspeech_b200.audio``) on 8 kHz fp32 ``x``
    [B, S] (unit element stride, any row stride), ``lens`` int32 [B] device sample counts (or None).  Returns
    ``(detected bool, score fp32, lag int32, message int32)`` device tensors [B].  Two launches, no host
    synchronisation."""
    from . import audio
    _require_cuda(x, "watermark_detect")
    B, S = _wave_rows(x, "watermark_detect")
    spectra, twiddles = audio.detector_tables(key, x.device)
    score = torch.empty(B, dtype=torch.float32, device=x.device)
    lag, message = torch.empty(B, dtype=torch.int32, device=x.device), torch.empty(B, dtype=torch.int32,
                                                                                   device=x.device)
    detected = torch.empty(B, dtype=torch.bool, device=x.device)
    nbytes = _lib.load().as_watermark_workspace_bytes(B, S)
    ws = torch.empty(max(int(nbytes), 1), dtype=torch.uint8, device=x.device)
    _run("as_watermark_detect", x, x.data_ptr(), x.stride(0) if B > 1 else S, B, S,
         _lens_arg(lens, B, x.device, "watermark_detect"), spectra.data_ptr(), twiddles.data_ptr(), float(threshold),
         ws.data_ptr(), ws.numel(), score.data_ptr(), lag.data_ptr(), message.data_ptr(), detected.data_ptr())
    _count(WATERMARK_DETECT_LAUNCHES - 1)
    return detected, score, lag, message


@dataclass
class SmallConv:
    w: torch.Tensor            # fp32 [ntaps, Cout, Cin] device
    bias: Optional[torch.Tensor]
    taps: Sequence[tuple]
    _dt: object = field(default=None, repr=False)
    _df: object = field(default=None, repr=False)

    def __post_init__(self):
        n = len(self.taps)
        self._dt = (C.c_int32 * n)(*[int(t[0]) for t in self.taps])
        self._df = (C.c_int32 * n)(*[int(t[1]) for t in self.taps])


def pack_small_conv(w_taps, bias, taps, device) -> SmallConv:
    return SmallConv(w_taps.detach().float().contiguous().to(device),
                     None if bias is None else bias.detach().float().contiguous().to(device), list(taps))


def conv_small(x, sc: SmallConv, *, raw=None, act_out=None, act=ACT_NONE, slope=0.0, lens=None):
    """Direct conv for Cin <= 16.  ``x`` [B,T,Cin] or [B,T,F,Cin]."""
    _require_cuda(x, "conv_small")
    B, T, F_, Cin = _dims(x)
    ntaps, Cout, cin_w = sc.w.shape
    assert cin_w == Cin
    oshape = (B, T, Cout) if x.dim() == 3 else (B, T, F_, Cout)
    r = _out_arg(raw, oshape, x.device)
    a = _out_arg(act_out, oshape, x.device)
    _run("as_conv_small", x, x.data_ptr(), dtype_code(x.dtype), _rows_ld(x, "cs.x"), B, T, F_, Cin,
         sc.w.data_ptr(), _p(sc.bias), ntaps, C.cast(sc._dt, _lib.c_i32_p), C.cast(sc._df, _lib.c_i32_p),
         Cout, _p(_i32(lens, "conv_small")),
         _p(r), dtype_code(r.dtype) if r is not None else 0, _rows_ld(r, "cs.raw") if r is not None else 0,
         _p(a), dtype_code(a.dtype) if a is not None else 0, _rows_ld(a, "cs.act") if a is not None else 0,
         int(act), float(slope))
    return r, a


def dwconv(x, w, bias, k, stride, pad, *, glu=False, act=ACT_NONE, slope=0.0, out_dtype=None,
           lens_in=None, lens_out=None):
    """Depthwise conv.  ``x`` [B,T,(F,)C(*2 if glu)]; ``w`` fp32 [kt*kf, C]; k/stride/pad = (t, f)."""
    _require_cuda(x, "dwconv")
    B, T, F_, Cx = _dims(x)
    C_ = Cx // 2 if glu else Cx
    (kt, kf), (st, sf), (pt, pf) = k, stride, pad
    To = (T + 2 * pt - kt) // st + 1
    Fo = (F_ + 2 * pf - kf) // sf + 1
    oshape = (B, To, C_) if x.dim() == 3 else (B, To, Fo, C_)
    out = torch.empty(oshape, dtype=out_dtype or x.dtype, device=x.device)
    _run("as_dwconv", x, x.data_ptr(), dtype_code(x.dtype), _rows_ld(x, "dw.x"), B, T, F_, C_, int(glu),
         w.data_ptr(), _p(bias), kt, kf, st, sf, pt, pf, To, Fo, _p(_i32(lens_in, "dwconv")),
         _p(_i32(lens_out, "dwconv")), int(act), float(slope), out.data_ptr(), dtype_code(out.dtype),
         _rows_ld(out, "dw.out"))
    return out


def avgpool(x, pt, pf, out_dtype=None):
    _require_cuda(x, "avgpool")
    B, T, F_, C_ = _dims(x)
    To, Fo = (T + pt - 1) // pt, F_ // pf
    oshape = (B, To, C_) if x.dim() == 3 else (B, To, Fo, C_)
    out = torch.empty(oshape, dtype=out_dtype or x.dtype, device=x.device)
    _run("as_avgpool", x, x.data_ptr(), dtype_code(x.dtype), _rows_ld(x, "ap.x"), B, T, F_, C_, pt, pf,
         out.data_ptr(), dtype_code(out.dtype), _rows_ld(out, "ap.out"))
    return out


def affine_act_maxpool(x, scale, shift, slope, pf, out_dtype):
    _require_cuda(x, "affine_act_maxpool")
    B, T, F_, C_ = x.shape
    out = torch.empty(B, T, F_ // pf, C_, dtype=out_dtype, device=x.device)
    _run("as_affine_act_maxpool", x, x.data_ptr(), dtype_code(x.dtype), _rows_ld(x, "mp.x"), B, T, F_, C_,
         scale.data_ptr(), shift.data_ptr(), float(slope), int(pf), out.data_ptr(), dtype_code(out_dtype),
         _rows_ld(out, "mp.out"))
    return out


def global_avgpool(x, slope, out_dtype, t_stride=1):
    """LeakyReLU + mean over (T[::t_stride], F) -> [B, C]."""
    _require_cuda(x, "global_avgpool")
    B, T, F_, C_ = _dims(x)
    out = torch.empty(B, C_, dtype=out_dtype, device=x.device)
    _run("as_global_avgpool", x, x.data_ptr(), dtype_code(x.dtype), _rows_ld(x, "gap.x"), B, T, F_, C_,
         int(t_stride), float(slope), out.data_ptr(), dtype_code(out_dtype), C_)
    return out


def bilstm(xproj, whh_t, hidden, lens, out_dtype):
    """``xproj`` fp32 [B,T,8H]; ``whh_t`` fp32 [2,H,4H] -> [B,T,2H]."""
    _require_cuda(xproj, "bilstm")
    B, T, _ = xproj.shape
    out = torch.empty(B, T, 2 * hidden, dtype=out_dtype, device=xproj.device)
    _run("as_bilstm", xproj, xproj.data_ptr(), _rows_ld(xproj, "lstm.x"), whh_t.data_ptr(), B, T, hidden,
         _p(_i32(lens, "bilstm")), out.data_ptr(), dtype_code(out_dtype), 2 * hidden)
    return out


def lstm_onestep(xproj, hidden, out_dtype):
    _require_cuda(xproj, "lstm_onestep")
    B, T, _ = xproj.shape
    out = torch.empty(B, T, 2 * hidden, dtype=out_dtype, device=xproj.device)
    _run("as_lstm_onestep", xproj, xproj.data_ptr(), _rows_ld(xproj, "l1.x"), B * T, hidden, out.data_ptr(),
         dtype_code(out_dtype), 2 * hidden)
    return out


def log_norm(mel):
    """``mel`` fp32 [B,n_mels,T] (channels-first, contiguous) -> fp32 [B,T]."""
    _require_cuda(mel, "log_norm")
    mel = mel.contiguous()
    B, M, T = mel.shape
    out = torch.empty(B, T, dtype=torch.float32, device=mel.device)
    _run("as_log_norm", mel, mel.data_ptr(), B, M, T, out.data_ptr())
    return out


def to_channels_last(src, out_dtype, lens=None, sub=None, mul=None, out=None):
    """``src`` [B,C,T] contiguous -> [B,T,C] (``out`` may be a channel-slice view)."""
    _require_cuda(src, "to_channels_last")
    src = src.contiguous()
    B, C_, T = src.shape
    if out is None:
        out = torch.empty(B, T, C_, dtype=out_dtype, device=src.device)
    _run("as_transpose_cast", src, src.data_ptr(), dtype_code(src.dtype), out.data_ptr(), dtype_code(out.dtype),
         B, C_, T, _rows_ld(out, "tcl.out"), 1, _p(sub), _p(mul), _p(_i32(lens, "to_cl")))
    return out


def to_channels_first(src, out_dtype, lens=None, sub=None, mul=None):
    """``src`` [B,T,C] (view allowed) -> contiguous [B,C,T]."""
    _require_cuda(src, "to_channels_first")
    B, T, C_ = src.shape
    out = torch.empty(B, C_, T, dtype=out_dtype, device=src.device)
    _run("as_transpose_cast", src, src.data_ptr(), dtype_code(src.dtype), out.data_ptr(), dtype_code(out_dtype),
         B, C_, T, _rows_ld(src, "tcf.src"), 0, _p(sub), _p(mul), _p(_i32(lens, "to_cf")))
    return out


# --------------------------------------------------------------------------------------------
# stream-level concurrency for independent sub-graphs (capturable in a CUDA graph)
# --------------------------------------------------------------------------------------------
_side_streams = {}


def run_concurrently(fns, device, pool: str = "main"):
    """Run the callables ``fns`` on separate CUDA streams forked from / joined to the current one
    and return their results.  Independent branches of the model (the three encoders, the three
    predictor branches) are latency-bound chains of small kernels: overlapping them fills the SMs.
    On CPU tensors (host-logic tests) the callables simply run in order."""
    if device is None or torch.device(device).type != "cuda" or len(fns) <= 1:
        return [f() for f in fns]
    dev = torch.device(device)
    main = torch.cuda.current_stream(dev)
    # nested forks name their own pool: reusing the parent's streams would serialise the branches
    pool = _side_streams.setdefault((dev.index, pool, len(fns)), [torch.cuda.Stream(device=dev) for _ in fns])
    fork = torch.cuda.Event()
    fork.record(main)
    results, joins = [], []
    for f, st in zip(fns, pool):
        st.wait_event(fork)
        with torch.cuda.stream(st):
            r = f()
            ev = torch.cuda.Event()
            ev.record(st)
        results.append(r)
        joins.append(ev)
    for ev in joins:
        main.wait_event(ev)

    def _mark(o):
        if torch.is_tensor(o):
            if o.is_cuda:
                o.record_stream(main)
        elif isinstance(o, (tuple, list)):
            for x in o:
                _mark(x)
        elif isinstance(o, dict):
            for x in o.values():
                _mark(x)
    for r in results:
        _mark(r)
    return results
