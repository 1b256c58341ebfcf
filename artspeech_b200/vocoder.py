"""HiFi-GAN V1 generator (24 kHz, hop 300) on the sm_100a implicit-GEMM kernels.

Drop-in for ``Vocoder/vocoder.py``: ``Generator(h)`` keeps the constructor, the ``state_dict``
layout (old-style ``weight_norm`` -> ``weight_g`` / ``weight_v``; plain ``weight`` after
``remove_weight_norm()``) and ``forward(mel[B, 80, T]) -> wav[B, 1, 300*T]`` of
``Generator`` (vocoder.py:75-125) and ``ResBlock1`` (:11-48), so ``test.py:66-73`` loads
``g_00935000`` unchanged.

How it runs (all in ``as_conv_igemm``; bf16 operands, fp32 accumulate):
  * activations are channels-last ``[B, L, C]``; every conv is one launch whose epilogue adds the
    bias and the residual(s), scales, and stores both the running residual stream and the
    LeakyReLU-ed bf16 operand of the next conv — the reference's separate leaky_relu / add /
    ``xs / 3`` passes (vocoder.py:37-41,103-111) never touch HBM on their own;
  * ``ConvTranspose1d(k=2u, stride=u)`` (:85-88) is packed as ONE 3-tap convolution with
    ``N = u*Cout`` output columns (phase-major): output row ``i`` holds the ``u`` output samples
    ``u*i .. u*i+u-1``, so the ``[B, T, u*Cout]`` result *is* the ``[B, u*T, Cout]`` tensor;
  * the three MRF branches accumulate into the stage output through the second residual input,
    the last one applying the ``1/3`` and the next stage's LeakyReLU.
Ragged batches: ``forward(mel, lengths=...)`` zeroes every activation beyond each utterance's
length (at x10/x50/x150/x300 rates), which makes the batch equal to batch-1 runs (SURVEY.md F5).
"""
from __future__ import annotations

import os
from typing import Optional

import torch
import torch.nn as nn
from torch.nn.utils import remove_weight_norm, weight_norm

from . import audio as audio_mod
from . import nn_util, ops

LRELU_SLOPE = 0.1
FUSED_PAIR_CHANNELS = (32, 64, 128)      # stages run by as_hifigan_resblock_pair (one launch per conv pair)


def get_padding(kernel_size: int, dilation: int = 1) -> int:
    return (kernel_size * dilation - dilation) // 2


def effective_weight(m: nn.Module) -> torch.Tensor:
    """fp32 weight of a (possibly old-style weight-normed) conv: ``g * v / ||v||`` over dim 0."""
    if hasattr(m, "weight_g") and hasattr(m, "weight_v"):
        v = m.weight_v.detach().float()
        g = m.weight_g.detach().float()
        norm = v.reshape(v.shape[0], -1).norm(dim=1).reshape(g.shape)
        return v * (g / norm)
    return m.weight.detach().float()


class ResBlock1(nn.Module):
    """Parameter container with the layout of vocoder.py:11-33."""

    def __init__(self, h, channels: int, kernel_size: int = 3, dilation=(1, 3, 5)):
        super().__init__()
        self.h = h
        self.kernel_size = kernel_size
        self.dilation = tuple(dilation)

        def mk(d):
            c = nn.Conv1d(channels, channels, kernel_size, 1, dilation=d,
                          padding=get_padding(kernel_size, d))
            c.weight.data.normal_(0.0, 0.01)
            return weight_norm(c)

        self.convs1 = nn.ModuleList([mk(d) for d in self.dilation])
        self.convs2 = nn.ModuleList([mk(1) for _ in self.dilation])

    def remove_weight_norm(self):
        for layer in list(self.convs1) + list(self.convs2):
            remove_weight_norm(layer)


def pack_conv_transpose(weight: torch.Tensor, bias: Optional[torch.Tensor], u: int, dtype, device):
    """Polyphase packing of ``ConvTranspose1d(k=2u, stride=u, padding=u//2+u%2)``.

    ``weight`` [Cin, Cout, k].  Output sample ``n = u*i + r`` receives ``x[i'] * W[:, :, kk]`` with
    ``kk = n - u*i' + p``; only ``i' - i in {-1, 0, +1}`` can satisfy ``0 <= kk < 2u``.
    Returns a 3-tap PackedConv with ``u*Cout`` phase-major output columns.
    """
    cin, cout, k = weight.shape
    assert k == 2 * u
    p = u // 2 + u % 2
    w = weight.detach().float().cpu()
    wt = torch.zeros(3, u * cout, cin)
    for di, d in enumerate((-1, 0, 1)):
        for r in range(u):
            kk = r + p - u * d
            if 0 <= kk < k:
                wt[di, r * cout:(r + 1) * cout, :] = w[:, :, kk].t()
    b = None if bias is None else bias.detach().float().cpu().repeat(u)
    return ops.pack_conv(wt, b, [(-1, 0), (0, 0), (1, 0)], dtype, device)


class Generator(nn.Module):
    def __init__(self, h):
        super().__init__()
        self.h = h
        self.num_kernels = len(h.resblock_kernel_sizes)
        self.num_upsamples = len(h.upsample_rates)
        if str(h.resblock) != "1":
            raise NotImplementedError("only ResBlock1 (HiFi-GAN V1, Vocoder/config.json) is implemented")
        c0 = h.upsample_initial_channel
        self.conv_pre = weight_norm(nn.Conv1d(h.num_mels, c0, 7, 1, padding=3))
        self.ups = nn.ModuleList()
        for i, (u, k) in enumerate(zip(h.upsample_rates, h.upsample_kernel_sizes)):
            ct = nn.ConvTranspose1d(c0 // (2 ** i), c0 // (2 ** (i + 1)), k, u,
                                    padding=(u // 2 + u % 2), output_padding=u % 2)
            ct.weight.data.normal_(0.0, 0.01)
            self.ups.append(weight_norm(ct))
        self.resblocks = nn.ModuleList()
        ch = c0
        for i in range(len(self.ups)):
            ch = c0 // (2 ** (i + 1))
            for k, d in zip(h.resblock_kernel_sizes, h.resblock_dilation_sizes):
                self.resblocks.append(ResBlock1(h, ch, k, d))
        post = nn.Conv1d(ch, 1, 7, 1, padding=3)
        post.weight.data.normal_(0.0, 0.01)
        self.conv_post = weight_norm(post)
        self.compute_dtype = torch.bfloat16
        self.fuse_pairs = os.environ.get("ASB_NO_FUSED_PAIRS") is None
        self._plan = None
        self.register_load_state_dict_post_hook(lambda mod, keys: mod.invalidate_plan())

    # -- reference API ------------------------------------------------------------------------
    def remove_weight_norm(self):
        for layer in self.ups:
            remove_weight_norm(layer)
        for blk in self.resblocks:
            blk.remove_weight_norm()
        remove_weight_norm(self.conv_pre)
        remove_weight_norm(self.conv_post)
        self.invalidate_plan()

    def invalidate_plan(self):
        if self._plan is not None:
            nn_util.bump_plan_epoch()
        self._plan = None

    def _apply(self, fn, *a, **kw):  # .to()/.cuda() that really move the parameters: re-pack lazily
        before = nn_util.param_signature(self)
        out = super()._apply(fn, *a, **kw)
        if nn_util.param_signature(self) != before:
            self.invalidate_plan()
        return out

    # -- weight preparation --------------------------------------------------------------------
    def _build_plan(self, device):
        dt = self.compute_dtype
        plan = {}
        w = effective_weight(self.conv_pre)                       # [512, 80, 7]
        plan["pre"] = ops.pack_conv(w.permute(2, 0, 1), self.conv_pre.bias, ops.taps_1d(7), dt, device)
        plan["ups"] = []
        for up, u in zip(self.ups, self.h.upsample_rates):
            assert up.kernel_size[0] == 2 * u, "polyphase packing assumes k = 2*stride"
            plan["ups"].append(pack_conv_transpose(effective_weight(up), up.bias, u, dt, device))
        plan["res"] = []
        for blk in self.resblocks:
            k = blk.kernel_size
            c1 = [ops.pack_conv(effective_weight(c).permute(2, 0, 1), c.bias, ops.taps_1d(k, d), dt, device)
                  for c, d in zip(blk.convs1, blk.dilation)]
            c2 = [ops.pack_conv(effective_weight(c).permute(2, 0, 1), c.bias, ops.taps_1d(k, 1), dt, device)
                  for c in blk.convs2]
            plan["res"].append((c1, c2))
        w = effective_weight(self.conv_post)                      # [1, 32, 7]
        plan["post"] = ops.pack_conv(w.permute(2, 0, 1), self.conv_post.bias, ops.taps_1d(7), dt, device)
        return plan

    # -- forward ----------------------------------------------------------------------------------
    @torch.no_grad()
    def forward(self, x: torch.Tensor, lengths: Optional[torch.Tensor] = None, pcm16: bool = False,
                audio: Optional[audio_mod.AudioFormat] = None) -> torch.Tensor:
        """``x``: mel ``[B, num_mels, T]`` -> waveform ``[B, 1, T*prod(upsample_rates)]`` (fp32).
        ``pcm16=True`` (extension): int16 samples ``rint(32767 * wav)`` straight from the conv_post kernel -- the
        samples ``soundfile.write(path, wav, 24000)`` (test.py:119) stores -- halving the device->host bytes.
        ``audio=AudioFormat(rate, encoding)`` (extension, ``artspeech_b200.audio``): the waveform resampled and
        encoded on the device, ``[B, 1, audio.out_samples(T*hop)]`` of ``audio.dtype``; with ``lengths`` each
        utterance has ``audio.out_samples(lengths[b]*hop)`` samples and silence codes beyond.  Not with ``pcm16``."""
        audio_mod.check(audio, pcm16)
        mel_cl = x.detach().transpose(1, 2).to(self.compute_dtype).contiguous()   # [B, T, 80]
        if lengths is not None:  # frames beyond an utterance's length must not leak into it
            keep = torch.arange(mel_cl.shape[1], device=mel_cl.device)[None, :] < lengths.to(mel_cl.device)[:, None]
            mel_cl = mel_cl * keep.unsqueeze(-1).to(mel_cl.dtype)
        wav = self.forward_channels_last(mel_cl, lengths, torch.int16 if pcm16 else torch.float32)
        if audio is not None:
            lens = None if lengths is None else lengths.to(device=wav.device, dtype=torch.int32) * self.hop()
            wav = ops.resample_encode(wav, lens, audio, audio.out_samples(wav.shape[1]))
        return wav.view(wav.shape[0], 1, -1)

    def hop(self) -> int:
        """24 kHz samples per mel frame (300)."""
        hop = 1
        for u in self.h.upsample_rates:
            hop *= u
        return hop

    def receptive_field_frames(self) -> int:
        """Mel frames on either side that can influence an output sample: conv_pre (k 7) + per stage the
        ConvTranspose1d reach and the widest MRF branch ``sum_d (k-1)/2 * (d + 1)`` at that stage's rate +
        conv_post (k 7), rounded up (Vocoder/vocoder.py:11-48,75-116).  14 for the V1 config."""
        import math
        rf, rate = 3.0, 1
        for i, (u, k) in enumerate(zip(self.h.upsample_rates, self.h.upsample_kernel_sizes)):
            rf += math.ceil((k - u) / 2 / u + 1) / rate       # input positions a transposed-conv output reaches
            rate *= u
            widest = max(sum((kk - 1) // 2 * (d + 1) for d in ds)
                         for kk, ds in zip(self.h.resblock_kernel_sizes, self.h.resblock_dilation_sizes))
            rf += widest / rate
        rf += 3.0 / rate
        return int(math.ceil(rf))

    @torch.no_grad()
    def stream(self, x: torch.Tensor, chunk_frames: int = 64, halo_frames: Optional[int] = None, pcm16: bool = False,
               audio: Optional[audio_mod.AudioFormat] = None):
        """Chunked vocoding for latency-bound serving (SURVEY.md §8f-3): yields ``(first_sample, wav_chunk)`` with
        ``wav_chunk`` ``[B, 1, <=chunk_frames*hop]``.  Every chunk is vocoded with ``halo_frames`` (default: the
        receptive field) of real context on both sides and only its centre is kept, so the concatenation equals
        ``forward(x)``; the first audio is available after one ``chunk_frames + halo`` pass instead of the whole
        utterance.

        ``audio=AudioFormat(...)``: chunks in that format, ``first_sample`` counted at its rate; the chunk of frames
        ``[t0, t1)`` is output samples ``[audio.out_samples(t0*hop), audio.out_samples(t1*hop))``, so the
        concatenation equals ``forward(x, audio=audio)``.  The resampling filter reaches ``ceil(half_len / up)``
        input samples (at most 30, at 8 kHz) beyond a chunk: the receptive field's ceiling (13.06 -> 14 frames for
        the V1 config) covers that.  A window starts at a multiple of ``audio.frame_align(hop)`` frames, where the
        24 kHz input and the output grid coincide."""
        audio_mod.check(audio, pcm16)
        halo = self.receptive_field_frames() if halo_frames is None else int(halo_frames)
        hop = self.hop()
        T = x.shape[2]
        align = 1 if audio is None else audio.frame_align(hop)
        for t0 in range(0, T, chunk_frames):
            t1 = min(T, t0 + chunk_frames)
            a, b = max(0, t0 - halo), min(T, t1 + halo)
            if audio is None:
                wav = self.forward(x[:, :, a:b], pcm16=pcm16)
                yield t0 * hop, wav[:, :, (t0 - a) * hop:(t1 - a) * hop]
                continue
            a -= a % align
            wav = self.forward(x[:, :, a:b])
            lo, hi = audio.out_samples(t0 * hop), audio.out_samples(t1 * hop)
            base = a * hop * audio.up // audio.down                     # output index of the window's first sample
            y = ops.resample_encode(wav.view(wav.shape[0], -1), None, audio, hi - lo, m0=lo - base)
            yield lo, y.view(y.shape[0], 1, -1)

    @torch.no_grad()
    def forward_channels_last(self, mel_cl: torch.Tensor, lengths: Optional[torch.Tensor] = None,
                              out_dtype: torch.dtype = torch.float32, return_lengths: bool = False):
        """``mel_cl``: ``[B, T, 80]`` in the compute dtype.  Returns ``[B, T*300]`` fp32 (or int16 PCM); with
        ``return_lengths`` also the utterances' sample counts, int32 [B] on the device (``lengths * 300``, computed
        with the per-stage lengths; None without ``lengths``)."""
        dev = mel_cl.device
        if self._plan is None:
            self._plan = self._build_plan(dev)
        plan = self._plan
        dt = self.compute_dtype
        B, T, _ = mel_cl.shape
        lens = None if lengths is None else lengths.to(device=dev, dtype=torch.int32)
        # per-stage lengths (frames x 10, x 50, x 150, x 300) in ONE elementwise launch instead of one per stage
        stage_lens = None
        if lens is not None:
            if plan.get("rates") is None or plan["rates"].device != dev:
                cum, r = [], 1
                for u in self.h.upsample_rates:
                    r *= u
                    cum.append(r)
                plan["rates"] = torch.tensor(cum, dtype=torch.int32, device=dev).view(-1, 1)
            stage_lens = lens.view(1, -1) * plan["rates"]

        # conv_pre, storing leaky_relu(x, 0.1): the only consumer is ups[0] (vocoder.py:101-104)
        _, a = ops.conv(mel_cl, plan["pre"], act_out=dt, act=ops.ACT_LRELU, slope=LRELU_SLOPE, lens=lens)
        L = T
        n_up = self.num_upsamples
        for i in range(n_up):
            u = self.h.upsample_rates[i]
            up = plan["ups"][i]
            cout = up.Cout // u
            last_stage = i == n_up - 1
            # the activation that follows the stage: lrelu(0.1) before ups[i+1], but the default
            # slope 0.01 before conv_post (vocoder.py:112 calls F.leaky_relu without a slope)
            next_slope = 0.01 if last_stage else LRELU_SLOPE
            if cout in FUSED_PAIR_CHANNELS and self.fuse_pairs and self.num_kernels <= 3:
                # fused path: the residual stream lives in HBM in activated form only; one launch per
                # (conv1, conv2) pair, the three MRF branches are independent until the last launch
                _, xa = ops.conv(a, up, act_out=dt, act=ops.ACT_LRELU, slope=LRELU_SLOPE, lens=lens)
                L = L * u
                xa = xa.view(B, L, cout)
                if lens is not None:
                    lens = stage_lens[i]
                done = []          # raw outputs of finished branches
                for j in range(self.num_kernels):
                    blk = self.resblocks[i * self.num_kernels + j]
                    c1s, c2s = plan["res"][i * self.num_kernels + j]
                    ra = xa
                    nconv = len(c1s)
                    for m in range(nconv):
                        kw = dict(slope=LRELU_SLOPE, lens=lens)
                        if m < nconv - 1:
                            kw.update(out_act=ops.ACT_LRELU, out_slope=LRELU_SLOPE)
                        elif j == self.num_kernels - 1:
                            kw.update(res2=done[0] if len(done) > 0 else None, res3=done[1] if len(done) > 1 else None,
                                      scale=1.0 / self.num_kernels, out_act=ops.ACT_LRELU, out_slope=next_slope)
                        ra = ops.resblock_pair(ra, c1s[m], c2s[m], blk.kernel_size, blk.dilation[m], **kw)
                    done.append(ra)
                a = done[-1]
                continue
            # ups[i]: rows of u*Cout -> viewed as [B, L*u, Cout]; keep x (residual) and lrelu(x)
            xr, xa = ops.conv(a, up, raw=dt, act_out=dt, act=ops.ACT_LRELU, slope=LRELU_SLOPE, lens=lens)
            L = L * u
            xr = xr.view(B, L, cout)
            xa = xa.view(B, L, cout)
            if lens is not None:
                lens = stage_lens[i]
            xs = None          # running sum of finished MRF branches (residual stream dtype)
            for j in range(self.num_kernels):
                c1s, c2s = plan["res"][i * self.num_kernels + j]
                r, ra = xr, xa
                nconv = len(c1s)
                for m in range(nconv):
                    _, t = ops.conv(ra, c1s[m], act_out=dt, act=ops.ACT_LRELU, slope=LRELU_SLOPE, lens=lens)
                    if m < nconv - 1:
                        r, ra = ops.conv(t, c2s[m], res1=r, raw=dt, act_out=dt, act=ops.ACT_LRELU,
                                         slope=LRELU_SLOPE, lens=lens)
                    elif j < self.num_kernels - 1:
                        # branch finished: xs += branch output (no activation needed)
                        xs, _ = ops.conv(t, c2s[m], res1=r, res2=xs, raw=torch.float32, lens=lens)
                    else:
                        # last branch: (xs + branch) / num_kernels, then the next stage's LeakyReLU
                        _, a = ops.conv(t, c2s[m], res1=r, res2=xs, scale=1.0 / self.num_kernels,
                                        act_out=dt, act=ops.ACT_LRELU, slope=next_slope, lens=lens)
        _, wav = ops.conv(a, plan["post"], act_out=out_dtype, act=ops.ACT_TANH, lens=lens)
        if return_lengths:
            return wav.view(B, L), lens
        return wav.view(B, L)
