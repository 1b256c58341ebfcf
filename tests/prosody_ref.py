"""fp64 restatement of the prosody controls (artspeech_b200/prosody.py, include/artspeech_b200.h
``as_round_durations_scaled`` / ``as_prosody_apply``), shared by the CPU and GPU prosody tests.

``install(monkeypatch)`` adds torch models of the two ops to the semantic backend of ``tests/sim_backend.py``."""
from __future__ import annotations

import math

import torch

from artspeech_b200 import ops, prosody

LN2_12 = math.log(2.0) / 12.0
LN10_10 = math.log(10.0) / 10.0


def round_scaled(pred, lens_t, scale=None):
    """-> (dur int32 [B,Tt] = round(pred * scale).clamp(min=1) for t < lens_t[b], 0 beyond; sums int32 [B]).
    ``scale`` fp32 [B, >= Tt] or [B]; the product is an fp32 multiply, as on the device."""
    B, Tt = pred.shape
    p = pred.float().cpu()
    if scale is not None:
        s = scale.float().cpu()
        p = p * (s[:, None] if s.dim() == 1 else s[:, :Tt])
    d = torch.round(p).clamp(min=1).to(torch.int32)
    if lens_t is not None:
        d = d * (torch.arange(Tt)[None, :] < lens_t.cpu()[:, None].long()).to(torch.int32)
    return d, d.sum(dim=1).to(torch.int32)


def apply_tracks(f0, n, ema, lens, ctrl, pitch_mean, pitch_std, energy_std):
    """Edited copies (fp32, CPU) of the tracks ``f0`` / ``n`` [B,Tm,1] and ``ema`` [B,Tm,10], evaluated in fp64."""
    f0, n, ema = f0.float().cpu().clone(), n.float().cpu().clone(), ema.float().cpu().clone()
    ctrl = ctrl.double().cpu()
    B, Tm, _ = f0.shape
    for b in range(B):
        L = Tm if lens is None else min(max(int(lens[b]), 0), Tm)
        c = ctrl[b]
        shift, rng, db = float(c[0]), float(c[1]), float(c[2])
        sc, off = c[4:4 + prosody.N_EMA], c[4 + prosody.N_EMA:]
        if L == 0:
            continue
        if shift != 0.0 or rng != 1.0:
            x = f0[b, :L, 0].double()
            hz = x * pitch_std + pitch_mean
            voiced = hz >= prosody.VOICING_FLOOR_HZ
            if bool(voiced.any()):
                lh = torch.log(hz.clamp_min(prosody.VOICING_FLOOR_HZ))
                mu = lh[voiced].mean()
                hz2 = torch.exp(mu + rng * (lh - mu) + shift * LN2_12)
                new = (x + (hz2 - hz) / pitch_std).float()
                f0[b, :L, 0] = torch.where(voiced, new, f0[b, :L, 0])
        if db != 0.0:
            n[b, :L, 0] = (n[b, :L, 0].double() + db * LN10_10 / energy_std).float()
        if bool((sc != 1.0).any()) or bool((off != 0.0).any()):
            e = ema[b, :L].double()
            m = e.mean(0)
            ema[b, :L] = (m + sc * (e - m) + off).float()
    return f0, n, ema


# -- semantic models of the two ops for the sim backend ------------------------------------------------------------
def sim_round_durations(pred, lens_t, scale=None):
    return round_scaled(pred, lens_t, scale)


def sim_prosody_apply(f0, n, ema, lens, ctrl, pitch_mean, pitch_std, energy_std):
    a, b, c = apply_tracks(f0, n, ema, lens, ctrl, pitch_mean, pitch_std, energy_std)
    f0.copy_(a)
    n.copy_(b)
    ema.copy_(c)


def install(monkeypatch):
    monkeypatch.setattr(ops, "round_durations", sim_round_durations)
    monkeypatch.setattr(ops, "prosody_apply", sim_prosody_apply)
