"""ArtSpeech acoustic model on the sm_100a kernels — drop-in for the reference's ``models.py``.

Same constructors, ``state_dict`` layout and ``forward()`` signatures as ``ArtsSpeech``
(models.py:275-371), ``StyleEncoder`` (:373-472), ``Decoder`` (:474-517), ``DurationPredictor``
(:519-571) and ``ArtsPredictor`` (:573-621), plus ``build_model`` / ``load_checkpoint``
(:680-701).  Only the inference path (``step="test"``, eval, no_grad) is implemented; the training
branches stay with the reference.

Extensions (SURVEY.md §8b): ``step="test"`` accepts batches of ``B > 1`` utterances with
per-utterance lengths and reproduces *batch-1 semantics per utterance* (length-aware norms, packed
LSTMs, masked attention); ``durations=`` feeds integer durations instead of the predictor's.

Internally everything is channels-last ``[B, T, C]`` with 16-bit GEMM operands (fp16 by default —
bf16 misses the mel tolerance, SURVEY.md F7) and fp32 accumulation / statistics / recurrences.
"""
from __future__ import annotations

import math
from typing import Optional

import torch
import torch.nn as nn
from torch.nn.utils import spectral_norm, weight_norm

from . import nn_util, ops
from . import prosody as prosody_mod
from .blocks import (AdainResBlk1d, LRELU, Placeholder, ResBlk, ResBlk1d, StyleFC, run_adain_block, run_resblk1d,
                     run_resblk2d)
from .ema import EMA_Predictor
from .jdc import JDCNet
from .rel_transformer import RelTransformerEncoder


class LinearNorm(nn.Module):
    def __init__(self, in_dim, out_dim, bias=True, w_init_gain="linear"):
        super().__init__()
        self.linear_layer = nn.Linear(in_dim, out_dim, bias=bias)
        nn.init.xavier_uniform_(self.linear_layer.weight, gain=nn.init.calculate_gain(w_init_gain))


def _i32(t, device):
    return None if t is None else t.to(device=device, dtype=torch.int32)


# ============================================================================================
# Style encoder
# ============================================================================================
def _style_stack_2d(dim_in, widths, downs, last_stride):
    layers = [spectral_norm(nn.Conv2d(1, dim_in, 3, 1, 1))]
    c = dim_in
    for w, d in zip(widths, downs):
        layers.append(ResBlk(c, w, downsample=d))
        c = w
    layers += [Placeholder(), spectral_norm(nn.Conv2d(c, c, 5, last_stride, 0)), Placeholder(), Placeholder()]
    return nn.Sequential(*layers)


def _style_stack_1d(dim_in):
    layers = [spectral_norm(nn.Conv1d(1, dim_in, 3, 1, 1)), ResBlk1d(dim_in, 2 * dim_in, downsample=True, dropout_p=0.0)]
    layers += [ResBlk1d(2 * dim_in, 2 * dim_in, downsample=True, dropout_p=0.0) for _ in range(3)]
    layers += [Placeholder(), Placeholder()]
    return nn.Sequential(*layers)


def _build_stack_2d(seq, dt, device):
    blocks = [m for m in seq if isinstance(m, ResBlk)]
    last = [m for m in seq if isinstance(m, nn.Conv2d)][-1]
    return dict(first=nn_util.small_conv2d(seq[0], device, (1, 1)),
                blocks=[b.build(dt, device) for b in blocks],
                last=nn_util.pack_conv2d(last, dt, device, (0, 0)), last_stride=last.stride[0])


def _run_stack_2d(p, img, dt):
    """Mel_block / EMA_block / dur_block (models.py:385-401,530-537) on ``img`` [B,T,F,1] -> [B,C] 16-bit."""
    raw, act = ops.conv_small(img, p["first"], raw=dt, act_out=dt, act=ops.ACT_LRELU, slope=LRELU)
    for bp in p["blocks"]:
        raw, act = run_resblk2d(bp, raw, act, dt)
    B, T, F, C = act.shape
    if T < 5 or F < 5:
        raise ValueError(f"style stack: feature map {T}x{F} is smaller than the 5x5 kernel "
                         f"(the reference mel is too short)")
    y, _ = ops.conv(act, p["last"], out_shape=(T - 4, F - 4), raw=dt)
    return ops.global_avgpool(y, LRELU, dt, t_stride=p["last_stride"])


def _build_stack_1d(seq, dt, device):
    return dict(first=nn_util.small_conv1d(seq[0], device),
                blocks=[m.build(dt, device) for m in seq if isinstance(m, ResBlk1d)])


def _run_stack_1d(p, x, dt):
    """F0_block / energy_block (models.py:402-411) on ``x`` [B,T,1] -> [B,C] 16-bit."""
    raw, act = ops.conv_small(x, p["first"], raw=dt, act_out=dt, act=ops.ACT_LRELU, slope=LRELU)
    for bp in p["blocks"]:
        raw, act = run_resblk1d(bp, raw, act, dt)
    return ops.global_avgpool(raw, LRELU, dt)


class StyleEncoder(nn_util.PlanMixin, nn.Module):
    def __init__(self, dim_in=48, style_dim=48):
        super().__init__()
        # The reference loads Utils/JDC/bst.t7 and Utils/EMA/200000.pth.tar here (models.py:377-383);
        # their parameters are part of this module's state_dict, so they arrive with the checkpoint.
        self.pitch_extractor = JDCNet(num_class=1, seq_len=192)
        self.ema_extractor = EMA_Predictor()
        d = dim_in
        self.Mel_block = _style_stack_2d(d, [2 * d, 4 * d, 8 * d, 8 * d], ["half"] * 4, 1)
        self.EMA_block = _style_stack_2d(d, [2 * d, 4 * d, 4 * d], ["channelpreserve", "channelpreserve", "half"], 2)
        self.F0_block = _style_stack_1d(d)
        self.energy_block = _style_stack_1d(d)
        self.Mellinear = nn.Linear(8 * d, style_dim)
        self.EMAlinear = nn.Linear(4 * d, style_dim // 2)
        self.F0linear = nn.Linear(2 * d, style_dim // 4)
        self.Energylinear = nn.Linear(2 * d, style_dim // 4)
        self.style_dim = style_dim
        self.compute_dtype = torch.float16
        self._znorm_consts = {}
        self._init_plan()

    def _build_plan(self, device):
        dt = self.compute_dtype
        lin = lambda l: nn_util.pack_linear(l.weight, l.bias, dt, device)
        return dict(mel=_build_stack_2d(self.Mel_block, dt, device), ema=_build_stack_2d(self.EMA_block, dt, device),
                    f0=_build_stack_1d(self.F0_block, dt, device), en=_build_stack_1d(self.energy_block, dt, device),
                    heads=[lin(self.Mellinear), lin(self.EMAlinear), lin(self.F0linear), lin(self.Energylinear)])

    @torch.no_grad()
    def _forward_uniform(self, mel: torch.Tensor, distribution):
        """All utterances have the full length T.  ``mel`` fp32 [B,80,T] ->
        (f0 [B,T,1], n [B,T,1], ema [B,T,10]) fp32 channels-last z-normalised, Style [B,512] fp32."""
        dev, dt = mel.device, self.compute_dtype
        for m in (self.pitch_extractor, self.ema_extractor):
            m.compute_dtype = dt
        p = self.plan(dev)
        B, M, T = mel.shape
        n_raw = ops.log_norm(mel)                                            # [B,T]   (models.py:431)
        feat = torch.zeros(B, T, 88, dtype=dt, device=dev)                   # F0 | energy | mel (| pad)
        ops.to_channels_last(mel, dt, out=feat[..., 2:82])
        mel_cl = ops.to_channels_last(mel, dt)                               # [B,T,80]
        ops.to_channels_last(n_raw.view(B, 1, T), dt, out=feat[..., 1:2])

        # z-normalisation with the dataset statistics (:447-449)
        def znorm(x_cl, mean, std):
            C = x_cl.shape[-1]
            key = (id(mean), id(std), C, str(dev))
            cached = self._znorm_consts.get(key)
            if cached is None or cached[2] is not mean or cached[3] is not std:    # per-channel constants, built once
                sub = mean.to(dev).float().reshape(-1).expand(C).contiguous()
                mul = (1.0 / std.to(dev).float().reshape(-1)).expand(C).contiguous()
                cached = self._znorm_consts[key] = (sub, mul, mean, std)
            sub, mul = cached[0], cached[1]
            cf = ops.to_channels_first(x_cl, torch.float32, sub=sub, mul=mul)           # [B,C,T]
            return cf, ops.to_channels_last(cf, torch.float32)

        # crop to the first T-1 frames (:459-466 with equal lengths => random_start == 0)
        Tc = T - 1
        crop = lambda x_cl: x_cl[:, :Tc].contiguous()

        # Dependencies (:431-433, :447-466): the mel style stack needs only the mel, the energy stack only
        # log_norm; F0 comes from JDCNet, EMA from the conformer predictor fed with (F0, energy, mel).
        # The chain JDCNet -> EMA predictor -> EMA stack is the long one; everything else runs beside it.
        def mel_branch():
            return _run_stack_2d(p["mel"], crop(mel_cl).view(B, Tc, M, 1), dt)

        def energy_branch():
            n_cf, n_cl = znorm(n_raw.view(B, T, 1), distribution["energy_mean"], distribution["energy_std"])
            return n_cf, n_cl, _run_stack_1d(p["en"], crop(n_cl), dt)

        def pitch_chain():
            f0_raw = self.pitch_extractor.forward_cl(mel_cl.view(B, T, M, 1))    # [B,T,1] (:432)
            ops.to_channels_last(f0_raw.view(B, 1, T), dt, out=feat[..., 0:1])

            def f0_branch():
                f0_cf, f0_cl = znorm(f0_raw, distribution["pitch_mean"], distribution["pitch_std"])
                return f0_cf, f0_cl, _run_stack_1d(p["f0"], crop(f0_cl), dt)

            def ema_branch():
                ema_raw = self.ema_extractor.forward_cl(feat[..., :82])          # [B,T,10] (:433)
                ema_cf, ema_cl = znorm(ema_raw, distribution["EMA_mean"], distribution["EMA_std"])
                return ema_cf, ema_cl, _run_stack_2d(p["ema"], crop(ema_cl).view(B, Tc, 10, 1), dt)
            return ops.run_concurrently([f0_branch, ema_branch], dev, pool="style.pitch")

        pooled_mel, (n_cf, n_cl, pooled_en), ((f0_cf, f0_cl, pooled_f0), (ema_cf, ema_cl, pooled_ema)) = \
            ops.run_concurrently([mel_branch, energy_branch, pitch_chain], dev, pool="style")
        pooled = [pooled_mel, pooled_ema, pooled_f0, pooled_en]
        style = torch.empty(1, B, 2 * self.style_dim, dtype=torch.float32, device=dev)
        off = 0
        for pl, head in zip(pooled, p["heads"]):
            ops.conv(pl.view(1, B, -1), head, raw=style[..., off:off + head.Cout])
            off += head.Cout
        return (f0_cf, n_cf, ema_cf), (f0_cl, n_cl, ema_cl), style.view(B, -1)

    @torch.no_grad()
    def forward(self, mel, mel_input_length, step="second", distribution=None, epoch=20, host_lengths=None):
        """``mel`` [B,80,T], ``mel_input_length`` [B] -> (f0 [B,1,T], n [B,1,T], ema [B,10,T], Style [B,512]).

        Utterances are processed in groups of equal length so each one sees exactly what a batch-1
        call would (un-packed JDC LSTM, un-masked conformer attention, style crop ``len-1``);
        frames beyond an utterance's length come back as zeros."""
        if distribution is None:
            raise ValueError("StyleEncoder needs the normalisation statistics (Data/stats.json)")
        mel = mel.detach().float()
        B, M, T = mel.shape
        # ``host_lengths`` (python ints) avoids the device->host sync of ``.tolist()``
        lens = list(host_lengths) if host_lengths is not None else [int(v) for v in mel_input_length.tolist()]
        dev = mel.device
        if all(v == T for v in lens):
            (f0, n, ema), _, style = self._forward_uniform(mel, distribution)
            return f0, n, ema, style
        f0 = torch.zeros(B, 1, T, device=dev)
        n = torch.zeros(B, 1, T, device=dev)
        ema = torch.zeros(B, 10, T, device=dev)
        style = torch.zeros(B, 2 * self.style_dim, device=dev)
        for L in sorted(set(lens)):
            idx = [i for i, v in enumerate(lens) if v == L]
            sel = torch.tensor(idx, device=dev)
            sub = mel if (len(idx) == B and L == T) else mel.index_select(0, sel)[:, :, :L].contiguous()
            (f0_g, n_g, ema_g), _, st_g = self._forward_uniform(sub, distribution)
            if len(idx) == B and L == T:
                f0, n, ema, style = f0_g, n_g, ema_g, st_g
            else:
                f0[sel, :, :L], n[sel, :, :L], ema[sel, :, :L] = f0_g, n_g, ema_g
                style[sel] = st_g
        return f0, n, ema, style


# ============================================================================================
# Duration predictor
# ============================================================================================
class DurationPredictor(nn_util.PlanMixin, nn.Module):
    def __init__(self, style_dim, d_hid, nlayers, dropout=0.1):
        super().__init__()
        self.text_encoder = RelTransformerEncoder(n_layers=2, hidden_channels=d_hid)
        self.duration = nn.ModuleList([AdainResBlk1d(d_hid, d_hid, style_dim // 4, dropout_p=dropout) for _ in range(3)])
        self.LSTM = nn.LSTM(d_hid, d_hid // 2, 1, batch_first=True, bidirectional=True)
        self.duration_proj = LinearNorm(d_hid, 1)
        d = 64
        self.dur_block = _style_stack_2d(d, [2 * d, 2 * d, 2 * d], ["channelpreserve", "channelpreserve", "half"], 2)
        self.dur_linear = nn.Linear(2 * d, style_dim // 4)
        self.d_hid, self.style_dim = d_hid, style_dim
        self.compute_dtype = torch.float16
        self.res_dtype = torch.float32     # residual stream between AdaIN blocks
        self._init_plan()

    def _fc(self):
        fc = StyleFC(self.style_dim // 4)
        for blk in self.duration:
            fc.add(blk.norm1, 0, self.style_dim // 4)
            fc.add(blk.norm2, 0, self.style_dim // 4)
        return fc

    def _build_plan(self, device):
        dt = self.compute_dtype
        proj, whh_t = nn_util.pack_lstm(self.LSTM, dt, device)
        return dict(stack=_build_stack_2d(self.dur_block, dt, device),
                    dur_linear=nn_util.pack_linear(self.dur_linear.weight, self.dur_linear.bias, dt, device),
                    fc=self._fc().build(dt, device), blocks=[b.build(dt, device) for b in self.duration],
                    lstm_proj=proj, whh_t=whh_t,
                    out=nn_util.pack_linear(self.duration_proj.linear_layer.weight,
                                            self.duration_proj.linear_layer.bias, dt, device))

    @torch.no_grad()
    def encode_text(self, texts, text_lengths):
        """The predictor's own text encoder (models.py:546): independent of the style, so callers may run it
        beside the other encoders and hand the result to ``forward(d_text=)``."""
        self.text_encoder.compute_dtype = self.compute_dtype
        return self.text_encoder(texts, text_lengths, want_16bit=False)

    @torch.no_grad()
    def forward(self, texts, style, text_lengths, mel_input_length, host_mel_lengths=None, d_text=None):
        """``texts`` [B,Tt], ``style`` = normalised EMA [B,10,Tr] -> duration fp32 [B,Tt]
        (models.py:540-566).  Every utterance's dur_block sees its full padded EMA row, as the
        reference's per-utterance loop does (:543-545)."""
        dev, dt = texts.device, self.compute_dtype
        p = self.plan(dev)
        B, Tt = texts.shape
        lens = _i32(text_lengths, dev)
        style = style.detach().float()
        Tr = style.shape[2]
        if host_mel_lengths is not None:
            mlens = [min(int(v), Tr) for v in host_mel_lengths]
        else:
            mlens = [Tr] * B if mel_input_length is None else [min(int(v), Tr) for v in mel_input_length.tolist()]
        dstyle = torch.empty(B, self.style_dim // 4, dtype=dt, device=dev)
        for L in sorted(set(mlens)):                                          # batch-1 semantics: crop to own length
            idx = [i for i, v in enumerate(mlens) if v == L]
            whole = len(idx) == B and L == Tr
            sub = style if whole else style[idx][:, :, :L].contiguous()
            ema_cl = ops.to_channels_last(sub, dt)                            # [b,L,10]
            pooled = _run_stack_2d(p["stack"], ema_cl.view(len(idx), L, 10, 1), dt)   # [b,128]
            _, ds = ops.conv(pooled.view(1, len(idx), -1), p["dur_linear"], act_out=dt)
            if whole:
                dstyle = ds.view(B, -1)
            else:
                dstyle[idx] = ds.view(len(idx), -1)
        gbs = StyleFC.run(p["fc"], dstyle.contiguous())
        x = d_text if d_text is not None else self.encode_text(texts, text_lengths)
        rd = self.res_dtype
        for i, bp in enumerate(p["blocks"]):
            last = i == len(p["blocks"]) - 1
            x, x16, _ = run_adain_block(bp, x, gbs[2 * i], gbs[2 * i + 1], lens, dt, res_dtype=rd,
                                        out16=dt if (last and rd != dt) else None)
        if x16 is None:
            x16 = x
        xproj, _ = ops.conv(x16, p["lstm_proj"], raw=torch.float32)
        h16 = ops.bilstm(xproj, p["whh_t"], self.d_hid // 2, lens, dt)
        dur, _ = ops.conv(h16, p["out"], raw=torch.float32)                   # padded rows = bias, as in :562-565
        return dur.view(B, Tt)


# ============================================================================================
# Arts predictor (F0 / energy / EMA)
# ============================================================================================
class ArtsPredictor(nn_util.PlanMixin, nn.Module):
    def __init__(self, style_dim, d_hid, dropout=0.1):
        super().__init__()
        self.shared = AdainResBlk1d(d_hid, d_hid, style_dim * 2, dropout_p=dropout)
        h2, h4 = d_hid // 2, d_hid // 4
        branch = lambda s: nn.ModuleList([AdainResBlk1d(d_hid, d_hid, style_dim * 2, upsample=True, dropout_p=dropout),
                                          AdainResBlk1d(d_hid, h2, s, dropout_p=dropout),
                                          AdainResBlk1d(h2, h4, s, dropout_p=dropout)])
        self.F0 = branch(style_dim // 4)
        self.N = branch(style_dim // 4)
        self.EMA = branch(style_dim // 2)
        self.F0_LSTM = nn.LSTM(h4, h4, 1, batch_first=True, bidirectional=True)
        self.N_LSTM = nn.LSTM(h4, h4, 1, batch_first=True, bidirectional=True)
        self.EMA_LSTM = nn.LSTM(h4, h4, 1, batch_first=True, bidirectional=True)
        self.F0_proj = nn.Conv1d(h2, 1, 1, 1, 0)
        self.N_proj = nn.Conv1d(h2, 1, 1, 1, 0)
        self.EMA_proj = nn.Conv1d(h2, 10, 1, 1, 0)
        self.style_dim, self.d_hid = style_dim, d_hid
        self.compute_dtype = torch.float16
        self.res_dtype = torch.float32     # residual stream between AdaIN blocks
        self._init_plan()

    # style slices of the 512-d style vector (models.py:597-599)
    _SLICES = {"F0": (384, 448), "N": (448, 512), "EMA": (256, 384)}

    def _fc(self):
        S = 2 * self.style_dim
        fc = StyleFC(S)
        fc.add(self.shared.norm1, 0, S); fc.add(self.shared.norm2, 0, S)
        for name in ("F0", "N", "EMA"):
            br = getattr(self, name)
            lo, hi = self._SLICES[name]
            fc.add(br[0].norm1, 0, S); fc.add(br[0].norm2, 0, S)
            for blk in (br[1], br[2]):
                fc.add(blk.norm1, lo, hi); fc.add(blk.norm2, lo, hi)
        return fc

    def _build_plan(self, device):
        dt = self.compute_dtype
        p = dict(fc=self._fc().build(dt, device), shared=self.shared.build(dt, device), br={})
        for name in ("F0", "N", "EMA"):
            proj, whh_t = nn_util.pack_lstm(getattr(self, name + "_LSTM"), dt, device)
            p["br"][name] = dict(blocks=[b.build(dt, device) for b in getattr(self, name)], lstm_proj=proj,
                                 whh_t=whh_t, out=nn_util.pack_conv1d(getattr(self, name + "_proj"), dt, device))
        return p

    @torch.no_grad()
    def forward_cl(self, a16: torch.Tensor, style16: torch.Tensor, lens, lens_up=None):
        """``a16`` [B,L,512] (length-regulated arts-encoder output, ``res_dtype``), ``style16`` [B,512] ->
        (F0 [B,2L,1], N [B,2L,1], EMA [B,2L,10]) fp32 channels-last, lens*2 (``lens_up``: that tensor when the
        caller already has it)."""
        p = self.plan(a16.device)
        dt = self.compute_dtype
        if style16.dtype != dt:                         # only when a caller mixes compute dtypes
            style16 = style16.to(dt)
        gbs = StyleFC.run(p["fc"], style16)
        rd = self.res_dtype
        need16 = rd != dt
        xs, _, _ = run_adain_block(p["shared"], a16, gbs[0], gbs[1], lens, dt, res_dtype=rd)
        def branch(name, g):
            bp = p["br"][name]
            y, y16, l = xs, None, lens
            for j, blk in enumerate(bp["blocks"]):
                # blocks 1, 2 have a learned 1x1 shortcut (512->256->128): they need a 16-bit copy of
                # their input; the last block's 16-bit copy is the LSTM projection's operand
                y, y16, l = run_adain_block(blk, y, gbs[g + 2 * j], gbs[g + 2 * j + 1], l, dt, res_dtype=rd,
                                            x16=y16, out16=dt if need16 else None, lens_up=lens_up)
            xproj, _ = ops.conv(y16 if need16 else y, bp["lstm_proj"], raw=torch.float32)
            h16 = ops.bilstm(xproj, bp["whh_t"], self.d_hid // 4, l, dt)
            o, _ = ops.conv(h16, bp["out"], raw=torch.float32, lens=l)
            return o, l
        # the three predictor branches are independent (models.py:603-619): concurrent streams
        res = ops.run_concurrently([lambda n=n_, g=g_: branch(n, g) for n_, g_ in (("F0", 2), ("N", 8), ("EMA", 14))],
                                   a16.device)
        outs = [r[0] for r in res]
        lens2 = res[0][1]
        return outs[0], outs[1], outs[2], lens2

    @torch.no_grad()
    def forward(self, A_ens, style):
        """Reference signature (models.py:596-621): ``A_ens`` [B,512,L], ``style`` [B,512] ->
        (F0 [B,1,2L], N [B,1,2L], EMA [B,10,2L])."""
        dt = self.compute_dtype
        a_cl = ops.to_channels_last(A_ens.detach().float(), self.res_dtype)
        f0, n, ema, _ = self.forward_cl(a_cl, style.detach().to(dt).contiguous(), None)
        cf = lambda t: ops.to_channels_first(t, torch.float32)
        return cf(f0), cf(n), cf(ema)


# ============================================================================================
# Decoder
# ============================================================================================
class Decoder(nn_util.PlanMixin, nn.Module):
    def __init__(self, dec_dim=512, style_dim=64, residual_dim=64, dim_in=64, dim_out=80):
        super().__init__()
        self.dec_dim, self.style_dim, self.residual_dim, self.dim_out = dec_dim, style_dim, residual_dim, dim_out
        self.bottleneck_dim = bd = dec_dim * 2
        self.encode = AdainResBlk1d(dec_dim + 128, bd, style_dim * 2)
        self.F0_conv = weight_norm(nn.Conv1d(1, 32, kernel_size=1))
        self.N_conv = weight_norm(nn.Conv1d(1, 32, kernel_size=1))
        self.EMA_conv = weight_norm(nn.Conv1d(10, 64, kernel_size=1))
        self.asr_res = nn.Sequential(weight_norm(nn.Conv1d(dec_dim, residual_dim, kernel_size=1)))
        cat = bd + residual_dim + 128
        self.decode = nn.ModuleList([AdainResBlk1d(cat, bd, style_dim * 2), AdainResBlk1d(cat, bd, style_dim * 2),
                                     AdainResBlk1d(cat, dec_dim, style_dim * 2),
                                     AdainResBlk1d(dec_dim, dec_dim, style_dim), AdainResBlk1d(dec_dim, dec_dim, style_dim),
                                     AdainResBlk1d(dec_dim, dec_dim, style_dim)])
        self.to_out = nn.Sequential(weight_norm(nn.Conv1d(dec_dim, dim_out, 1, 1, 0)))
        self.compute_dtype = torch.float16
        self.res_dtype = torch.float32     # residual stream between AdaIN blocks (fp16 misses the mel tolerance)
        self._init_plan()

    def _fc(self):
        S = 2 * self.style_dim
        fc = StyleFC(S)
        fc.add(self.encode.norm1, 0, S); fc.add(self.encode.norm2, 0, S)
        for i, blk in enumerate(self.decode):
            hi = S if i < 3 else self.style_dim            # decode[3:] see Mel_style = Style[:, :256] (models.py:499,514)
            fc.add(blk.norm1, 0, hi); fc.add(blk.norm2, 0, hi)
        return fc

    def _build_plan(self, device):
        dt = self.compute_dtype
        return dict(fc=self._fc().build(dt, device), encode=self.encode.build(dt, device),
                    decode=[b.build(dt, device) for b in self.decode],
                    f0=nn_util.small_conv1d(self.F0_conv, device), n=nn_util.small_conv1d(self.N_conv, device),
                    ema=nn_util.small_conv1d(self.EMA_conv, device),
                    asr_res=nn_util.pack_conv1d(self.asr_res[0], dt, device),
                    to_out=nn_util.pack_conv1d(self.to_out[0], dt, device))

    def alloc_inputs(self, B, Tm, device):
        """(cat_res, cat16): the decoder's first concat buffer [B,Tm,640] in the residual-stream dtype
        and in the compute dtype (the same tensor when both dtypes agree).  The caller fills channels
        [0, 512) of both with the x2-upsampled, length-regulated text encoding."""
        W = self.dec_dim + 128
        cat16 = torch.empty(B, Tm, W, dtype=self.compute_dtype, device=device)
        if self.res_dtype == self.compute_dtype:
            return cat16, cat16
        return torch.empty(B, Tm, W, dtype=self.res_dtype, device=device), cat16

    @torch.no_grad()
    def forward_cl(self, cat_res: torch.Tensor, cat16: torch.Tensor, style16, f0_cl, n_cl, ema_cl, lens,
                   mel16_dtype=None):
        """``cat_res`` / ``cat16`` from ``alloc_inputs`` with channels [0,512) filled; F0/N/EMA fp32
        channels-last [B,Tm,{1,1,10}].  Returns mel fp32 [B,Tm,80] (zeros beyond ``lens``); with ``mel16_dtype``
        ``(mel, mel16)`` where ``mel16`` is the same tensor in that 16-bit dtype (the vocoder's operand), written
        by the same launch.

        Everything that feeds an InstanceNorm stays in ``res_dtype`` (fp32 by default): several
        concat channels (bias-dominated F0/N/EMA features) have |mean| >> std, so a 16-bit copy of
        the *pre-norm* value would lose the signal the norm then amplifies.  16-bit copies exist
        only as GEMM operands (1x1 shortcuts, asr_res)."""
        p = self.plan(cat16.device)
        dt = self.compute_dtype
        if cat16.dtype != dt or style16.dtype != dt:     # only when a caller mixes compute dtypes
            cat16, style16 = cat16.to(dt), style16.to(dt)
        B, Tm, _ = cat16.shape
        D, bd, R = self.dec_dim, self.bottleneck_dim, self.residual_dim
        rd = self.res_dtype
        need16 = cat_res.dtype != dt
        W = bd + R + 128
        big16 = torch.empty(B, Tm, W, dtype=dt, device=cat16.device)             # [x | asr_res | F0 | N | EMA]
        big = torch.empty(B, Tm, W, dtype=rd, device=cat16.device) if need16 else big16
        for (buf, buf16), base in (((cat_res, cat16), D), ((big, big16), bd + R)):   # concat fused: write slices
            for src, key, lo, hi in ((f0_cl, "f0", 0, 32), (n_cl, "n", 32, 64), (ema_cl, "ema", 64, 128)):
                ops.conv_small(src, p[key], raw=buf[..., base + lo:base + hi],
                               act_out=buf16[..., base + lo:base + hi] if need16 else None, lens=lens)
        ops.conv(cat16[..., :D], p["asr_res"], raw=big[..., bd:bd + R],
                 act_out=big16[..., bd:bd + R] if need16 else None, lens=lens)
        gbs = StyleFC.run(p["fc"], style16)
        run_adain_block(p["encode"], cat_res, gbs[0], gbs[1], lens, dt, x16=cat16, out=big[..., :bd],
                        out16=big16[..., :bd] if need16 else None)
        x = x16 = None
        for i, bp in enumerate(p["decode"]):
            g1, g2 = gbs[2 + 2 * i], gbs[3 + 2 * i]
            if i < 2:
                run_adain_block(bp, big, g1, g2, lens, dt, x16=big16, out=big[..., :bd],
                                out16=big16[..., :bd] if need16 else None)
            elif i == 2:
                x, _, _ = run_adain_block(bp, big, g1, g2, lens, dt, x16=big16, res_dtype=rd)
            else:
                last = i == len(p["decode"]) - 1
                x, x16, _ = run_adain_block(bp, x, g1, g2, lens, dt, res_dtype=rd,
                                            out16=dt if (last and need16) else None)
        if need16:
            x = x16
        mel, mel16 = ops.conv(x, p["to_out"], raw=torch.float32, act_out=mel16_dtype, lens=lens)
        return mel if mel16_dtype is None else (mel, mel16)

    @torch.no_grad()
    def forward(self, asr, Style, F0, N, EMA):
        """Reference signature (models.py:497-517): ``asr`` [B,512,L], ``Style`` [B,512],
        F0/N [B,1,2L], EMA [B,10,2L] -> mel [B,80,2L]."""
        dt = self.compute_dtype
        B, D, L = asr.shape
        cat_res, cat16 = self.alloc_inputs(B, 2 * L, asr.device)
        a_cl = ops.to_channels_last(asr.detach().float(), torch.float32)
        ops.repeat_rows(a_cl, 2, None, out=cat_res[..., :D])                   # F.interpolate(..., 2, 'nearest')
        if cat16 is not cat_res:
            ops.repeat_rows(a_cl, 2, None, out=cat16[..., :D])
        cl = lambda t: ops.to_channels_last(t.detach().float(), torch.float32)
        mel = self.forward_cl(cat_res, cat16, Style.detach().to(dt).contiguous(), cl(F0), cl(N), cl(EMA), None)
        return ops.to_channels_first(mel, torch.float32)


# ============================================================================================
# Top module
# ============================================================================================
class ArtsSpeech(nn.Module):
    def __init__(self, args, stage="first", distribution=None):
        super().__init__()
        self.stage = stage
        if stage != "first":
            self.arts_encoder = RelTransformerEncoder(n_layers=4, hidden_channels=args.hidden_dim)
            self.durationPredictor = DurationPredictor(style_dim=args.style_dim, d_hid=args.hidden_dim,
                                                       nlayers=args.n_layer, dropout=args.dropout)
            self.artsPredictor = ArtsPredictor(style_dim=args.style_dim, d_hid=args.hidden_dim, dropout=args.dropout)
        self.text_encoder = RelTransformerEncoder(n_layers=4, hidden_channels=args.hidden_dim)
        self.style_encoder = StyleEncoder(dim_in=args.dim_in, style_dim=args.style_dim)
        self.decoder = Decoder(dec_dim=args.hidden_dim, style_dim=args.style_dim, dim_out=args.n_mels)
        self.distribution = distribution if distribution is not None else {}
        self.compute_dtype = torch.float16

    def set_compute_dtype(self, dt):
        self.compute_dtype = dt
        for m in self.modules():
            if hasattr(m, "compute_dtype"):
                m.compute_dtype = dt
            if isinstance(m, nn_util.PlanMixin):
                m.invalidate_plan()

    # -- phase A: everything that does not depend on the durations -------------------------------------------
    @torch.no_grad()
    def encode(self, texts, lens_t, mels, mel_input_length, host_mel_lens=None, voice=None,
               predict_durations: bool = True, dscale: Optional[torch.Tensor] = None):
        """Text / arts / style encoders (models.py:357-359) and, when ``predict_durations``, the duration
        predictor with its device-side ``round().clamp(min=1)`` (:360-361).  ``lens_t`` int32 [B] on the device.
        ``dscale``: prosody duration scale fp32 [B,Tt] on the device, rounds ``duration * dscale`` instead.
        Returns the state ``decode`` consumes; no host synchronisation when ``host_mel_lens`` is given."""
        dev = texts.device
        dp = self.durationPredictor
        branches = [lambda: self.text_encoder(texts, lens_t),                                     # [B,Tt,512] fp32 (:357)
                    lambda: self.arts_encoder(texts, lens_t)]                                     # (:358)
        if predict_durations:
            # the predictor's own 2-layer text encoder (:546) needs only the tokens: it runs beside the others,
            # the rest of the predictor waits for the style encoder's EMA track
            branches.append(lambda: dp.encode_text(texts, lens_t))
        if voice is None:
            branches.append(lambda: self.style_encoder(mels, mel_input_length, "second", self.distribution,
                                                       host_lengths=host_mel_lens))              # (:359)
        res = ops.run_concurrently(branches, dev)
        T_en, A_en = res[0], res[1]
        # ``voice``: style-encoder outputs of the reference voice computed earlier (engine.Synthesizer.encode_voice):
        # the 30 GFLOP style encoder runs once per voice instead of once per utterance (SURVEY.md §8f)
        f0_ext, n_ext, ema_ext, style = voice if voice is not None else res[-1]
        st = dict(T_en=T_en, A_en=A_en, style=style, f0_ext=f0_ext, n_ext=n_ext, ema_ext=ema_ext, lens_t=lens_t,
                  duration=None, pred_dur=None, pred_sum=None)
        if predict_durations:
            duration = dp(texts, ema_ext, lens_t, mel_input_length, host_mel_lengths=host_mel_lens, d_text=res[2])
            st["duration"] = duration                                                             # (:360)
            if dscale is None:
                st["pred_dur"], st["pred_sum"] = ops.round_durations(duration, lens_t)            # (:361) on the device
            else:
                st["pred_dur"], st["pred_sum"] = ops.round_durations(duration, lens_t, dscale)
        return st

    # -- phase B: length regulation -> predictors -> decoder -------------------------------------------------
    @torch.no_grad()
    def decode(self, st, dur, Lmax: int, mel16_dtype=None, ctrl: Optional[torch.Tensor] = None):
        """``dur`` int32 [B,Tt] on the device (zeros or anything beyond ``lens_t``: the regulator reads
        ``dur[b, :lens_t[b]]`` only), ``Lmax`` >= max_b sum(dur[b]) (host int; a shape bucket may round it up: the
        extra rows come back as zeros).  Returns (mel_cl fp32 [B,2*Lmax,80], aux); ``mel16_dtype`` adds
        ``aux["mel16"]``, the 16-bit channels-last copy the vocoder consumes.  ``ctrl``: prosody control block fp32
        [B,24] on the device (``prosody.pack``): the F0 / energy / EMA tracks are edited before the decoder reads
        them."""
        dev, dt = dur.device, self.compute_dtype
        T_en, A_en, lens_t = st["T_en"], st["A_en"], st["lens_t"]
        B = T_en.shape[0]
        Tm = 2 * int(Lmax)
        style16 = st["style"].to(dt).contiguous()
        # length regulation as a gather (the reference multiplies by a one-hot matrix, :362-368);
        # the decoder's nearest x2 upsample (:500) is fused into the same pass.
        D = self.decoder.dec_dim
        a_reg, lens_l = ops.length_regulate(A_en, dur, lens_t, 1, int(Lmax), out_dtype=self.artsPredictor.res_dtype)
        cat_res, cat16 = self.decoder.alloc_inputs(B, Tm, dev)
        _, lens_m = ops.length_regulate(T_en, dur, lens_t, 2, Tm, out=cat_res[..., :D])
        if cat16 is not cat_res:
            ops.length_regulate(T_en, dur, lens_t, 2, Tm, out=cat16[..., :D])
        f0, n, ema, _ = self.artsPredictor.forward_cl(a_reg, style16, lens_l, lens_up=lens_m)    # (:369)
        if ctrl is not None:
            ops.prosody_apply(f0, n, ema, lens_m, ctrl, *self.prosody_constants())
        mel_cl = self.decoder.forward_cl(cat_res, cat16, style16, f0, n, ema, lens_m, mel16_dtype)   # (:370)
        mel16 = None
        if mel16_dtype is not None:
            mel_cl, mel16 = mel_cl
        return mel_cl, dict(mel_lengths=lens_m, F0=f0, N=n, EMA=ema, mel_cl=mel_cl, mel16=mel16)

    @torch.no_grad()
    def forward(self, batch, s2s_attn=None, s2s_attn_mono=None, step="test", mode="train", epoch=0,
                durations: Optional[torch.Tensor] = None, return_aux: bool = False, host_meta: Optional[dict] = None,
                voice: Optional[tuple] = None, predict_durations: Optional[bool] = None, prosody=None):
        """``step="test"`` (models.py:356-371).  ``durations`` (extension): integer durations [B,Tt] used INSTEAD of
        the predictor's (north_star: "durations are fed from the reference's integer output"); the predictor then
        runs only if ``predict_durations`` is true (its output is returned in the aux dict, the forced durations
        still drive the length regulator).
        ``host_meta`` (optional, keeps the pass free of device->host syncs so it can be captured in a CUDA graph):
        ``{"mel_lens": [int], "Lmax": int}`` = reference-mel lengths and (an upper bound of) the largest
        ``sum(durations[b, :len_b])``; ``Lmax`` requires ``durations``.
        ``voice`` (optional): ``(f0, n, ema, Style)`` as returned by the style encoder for these utterances'
        reference recordings; skips the style encoder (``mels`` is then only used for its shape).
        ``prosody`` (optional): one ``prosody.Prosody`` per utterance; with ``return_aux`` the aux dict then holds
        the edited ``F0`` / ``N`` / ``EMA`` tracks and the scaled ``pred_dur`` (``duration`` stays the predictor's
        raw output).
        Training branches (``step != "test"``) are delegated to ``self.training_delegate`` (an instance of the
        reference's own ``ArtsSpeech`` sharing this module's parameters, see ``attach_training_delegate``)."""
        if step != "test":
            if getattr(self, "training_delegate", None) is None:
                raise NotImplementedError(
                    "artspeech_b200 accelerates the synthesis path (step='test'); for the training branches "
                    "(models.py:291-354) attach the reference module with attach_training_delegate(ref_ArtsSpeech)")
            with torch.enable_grad():
                return self.training_delegate(batch, s2s_attn, s2s_attn_mono, step, mode, epoch)
        if self.stage == "first":
            raise RuntimeError("step='test' needs a second-stage model (arts_encoder / predictors)")
        texts, input_lengths, mels, mel_input_length = batch[0], batch[1], batch[2], batch[3]
        dev = texts.device
        B, Tt = texts.shape
        lens_t = _i32(input_lengths, dev)
        hm = host_meta or {}
        predict = durations is None if predict_durations is None else (bool(predict_durations) or durations is None)
        ctrl = dscale = None
        if prosody is not None:
            tl = [int(v) for v in (input_lengths.tolist() if torch.is_tensor(input_lengths) else input_lengths)]
            pros = prosody_mod.check(prosody, tl, durations is not None)
            ctrl, dscale = (t.to(dev) for t in prosody_mod.pack(pros, Tt))
        st = self.encode(texts, lens_t, mels, mel_input_length, hm.get("mel_lens"), voice, predict,
                         dscale if durations is None else None)
        if durations is None:
            dur = st["pred_dur"]
            Lmax = int(st["pred_sum"].max().item())                                       # one host sync (ref: 2*Tt+1)
            pred_dur = dur.to(torch.float32)                                              # what :361 returns
        else:
            pred_dur = durations.to(dev)
            dur = pred_dur.to(torch.int32).contiguous()
            if dur.dim() == 1:
                dur = dur.view(1, -1)
            if "Lmax" in hm:
                Lmax = int(hm["Lmax"])
            else:
                valid = torch.arange(Tt, device=dev)[None, :] < lens_t[:, None]
                Lmax = int((dur * valid).sum(dim=1).max().item())
        mel_cl, aux = self.decode(st, dur, Lmax, ctrl=ctrl)
        mel = ops.to_channels_first(mel_cl, torch.float32)                               # [B,80,Tm]
        if return_aux:
            aux.update(pred_dur=pred_dur, duration=st["duration"], predicted_dur=st["pred_dur"], style=st["style"],
                       T_en=st["T_en"], A_en=st["A_en"], f0_ext=st["f0_ext"], n_ext=st["n_ext"],
                       ema_ext=st["ema_ext"])
            return mel, aux
        return mel

    def attach_training_delegate(self, ref_module):
        """``ref_module``: an instance of the reference's ``models.ArtsSpeech`` (same args / stage).  Its parameters
        and buffers are re-pointed at this module's (same ``state_dict`` keys, SURVEY.md §8b), so optimiser steps on
        either are seen by both; ``forward(step="first"/"second")`` then runs the reference's own PyTorch training
        code (models.py:291-354) while ``step="test"`` stays on the CUDA path.  Call ``invalidate_plans()`` after
        weight updates so the folded 16-bit copies are rebuilt."""
        own_p = dict(self.named_parameters())
        own_b = dict(self.named_buffers())
        for name, mod in ref_module.named_modules():
            for k in list(mod._parameters):
                full = f"{name}.{k}" if name else k
                if mod._parameters[k] is not None and full in own_p:
                    if own_p[full].shape != mod._parameters[k].shape:
                        raise ValueError(f"training delegate: shape mismatch for {full}")
                    mod._parameters[k] = own_p[full]
            for k in list(mod._buffers):
                full = f"{name}.{k}" if name else k
                if mod._buffers[k] is not None and full in own_b:
                    mod._buffers[k] = own_b[full]
        object.__setattr__(self, "training_delegate", ref_module)     # not a sub-module: keeps state_dict unchanged
        return self

    def prosody_constants(self):
        """(pitch_mean, pitch_std, energy_std) of ``self.distribution`` as host floats, read once per distribution
        (``as_prosody_apply`` takes them by value; reading a device tensor per call would synchronise)."""
        cached = getattr(self, "_prosody_consts", None)
        if cached is None or cached[0] is not self.distribution:
            cached = (self.distribution, prosody_mod.constants(self.distribution))
            self._prosody_consts = cached
        return cached[1]

    def invalidate_plans(self):
        for m in self.modules():
            if isinstance(m, nn_util.PlanMixin):
                m.invalidate_plan()


class _Bundle(dict):
    """``Munch``-like result of build_model (attribute + item access, iterable over keys)."""
    __getattr__ = dict.__getitem__
    __setattr__ = dict.__setitem__


def build_model(args, text_aligner=None, stage="first", distribution=None):
    """models.py:680-683.  The 2-D discriminator is training-only and not built here."""
    return _Bundle(ArtsSpeech=ArtsSpeech(args, stage, distribution=distribution), text_aligner=text_aligner)


def load_checkpoint(model, optimizer, path, load_only_params=True):
    """models.py:685-701: non-strict load of ``state['net'][key]`` into ``model[key]``, eval()."""
    state = torch.load(path, map_location="cpu")
    params = state["net"]
    for key in model:
        if key in params and model[key] is not None:
            model[key].load_state_dict(params[key], False)
    for key in model:
        if model[key] is not None:
            model[key].eval()
    epoch, iters = (0, 0) if load_only_params else (state["epoch"], state["iters"])
    if not load_only_params and optimizer is not None:
        optimizer.load_state_dict(state["optimizer"])
    return model, optimizer, epoch, iters
