"""fp64 restatement of the loudness meter and normalisation gain (``artspeech_b200/audio.py``, ``as_loudness_measure``),
written from their definitions: K-weighting with ``scipy.signal.lfilter``, block energies and the two gates with
numpy, the true peak with ``audio_ref.resample64``; plus torch models of ``ops.loudness_measure`` and of
``ops.resample_encode(gain=)`` for host-logic tests on the CPU."""
from __future__ import annotations

import math

import numpy as np
import torch

from tests import audio_ref

# ITU-R BS.1770-4, table 1 and table 2 (48 kHz)
BS1770_SHELF = ([1.53512485958697, -2.69169618940638, 1.19839281085285], [1.0, -1.69065929318241, 0.73248077421585])
BS1770_HIGHPASS = ([1.0, -2.0, 1.0], [1.0, -1.99004745483398, 0.99007225036621])


def k_weighting(fs):
    """((b, a) shelf, (b, a) high-pass): libebur128's bilinear-transform design."""
    f0, G, Q = 1681.974450955533, 3.999843853973347, 0.7071752369554196
    K = math.tan(math.pi * f0 / fs)
    Vh = 10.0 ** (G / 20.0)
    Vb = Vh ** 0.4996667741545416
    a0 = 1.0 + K / Q + K * K
    b1 = np.array([Vh + Vb * K / Q + K * K, 2.0 * (K * K - Vh), Vh - Vb * K / Q + K * K]) / a0
    a1 = np.array([1.0, 2.0 * (K * K - 1.0) / a0, (1.0 - K / Q + K * K) / a0])
    f0, Q = 38.13547087602444, 0.5003270373238773
    K = math.tan(math.pi * f0 / fs)
    a0 = 1.0 + K / Q + K * K
    b2 = np.array([1.0, -2.0, 1.0])
    a2 = np.array([1.0, 2.0 * (K * K - 1.0) / a0, (1.0 - K / Q + K * K) / a0])
    return (b1, a1), (b2, a2)


def block_energies(x, fs):
    """The blocks' mean squares ``z`` of the K-weighted ``x`` (one block over all samples below 400 ms)."""
    from scipy.signal import lfilter
    x = np.asarray(x, dtype=np.float64)
    n = x.shape[0]
    if n == 0:
        return np.zeros(0)
    (b1, a1), (b2, a2) = k_weighting(fs)
    y = lfilter(b2, a2, lfilter(b1, a1, x))
    seg = fs // 10
    if n < 4 * seg:
        return np.array([np.mean(y * y)])
    nseg = n // seg
    E = (y[:nseg * seg] ** 2).reshape(nseg, seg).sum(1)
    return (E[:-3] + E[1:-2] + E[2:-1] + E[3:]) / (4 * seg)


def block_loudness(x, fs):
    with np.errstate(divide="ignore"):
        return -0.691 + 10.0 * np.log10(block_energies(x, fs))


def integrated(x, fs):
    z = block_energies(x, fs)
    with np.errstate(divide="ignore"):
        L = -0.691 + 10.0 * np.log10(z)
    za = z[L > -70.0]
    if za.size == 0:
        return -math.inf
    gate = -0.691 + 10.0 * math.log10(za.mean()) - 10.0
    zg = z[(L > -70.0) & (L > gate)]
    return -0.691 + 10.0 * math.log10(zg.mean())


def relative_gate(x, fs):
    """The relative gate ``G_r`` (None when no block passes the absolute gate)."""
    z = block_energies(x, fs)
    with np.errstate(divide="ignore"):
        L = -0.691 + 10.0 * np.log10(z)
    za = z[L > -70.0]
    return None if za.size == 0 else -0.691 + 10.0 * math.log10(za.mean()) - 10.0


def true_peak(x):
    """20 log10 of the largest |x| and |4x interpolation| (the resampler's filter with up 4, down 1)."""
    from artspeech_b200.audio import _design
    x = np.asarray(x, dtype=np.float64)
    if x.size == 0:
        return -math.inf
    y4, _ = audio_ref.resample64(x, _design(4, 1)[0], 4, 1, 40)
    tp = max(np.abs(x).max(), np.abs(y4).max())
    return 20.0 * math.log10(tp) if tp > 0 else -math.inf


def gain_db(L, tp, target=-23.0, ceiling=-1.0):
    return 0.0 if L == -math.inf else min(target - L, ceiling - tp)


def gain32(gdb):
    return np.float32(10.0 ** (gdb / 20.0))


# ---- torch models for host-logic tests -----------------------------------------------------------------------
def loudness_measure_model(x, lens, sample_rate, target=-23.0, ceiling=-1.0):
    B, S = x.shape
    out = torch.zeros(B, dtype=torch.float64), torch.zeros(B, dtype=torch.float64), \
        torch.zeros(B, dtype=torch.float64), torch.zeros(B, dtype=torch.float32)
    for b in range(B):
        n = S if lens is None else min(max(int(lens[b]), 0), S)
        xb = x[b, :n].double().numpy()
        L, tp = integrated(xb, sample_rate), true_peak(xb)
        g = gain_db(L, tp, target, ceiling)
        out[0][b], out[1][b], out[2][b], out[3][b] = L, tp, g, float(gain32(g))
    return out


def resample_encode_gain_model(x, lens, fmt, S_out, *, m0=0, out=None, out_lens=None, gain=None):
    """``audio_ref.resample_encode_model`` with the gain multiplied in before the encoding."""
    from artspeech_b200.audio import AudioFormat
    y = audio_ref.resample_encode_model(x, lens, AudioFormat(fmt.sample_rate), S_out, m0=m0, out_lens=out_lens)
    if gain is not None:
        y = y * gain.view(-1, 1).float()
    if fmt.encoding != "float32":
        s = torch.clamp(torch.round(y * 32767.0), -32768, 32767).to(torch.int64)
        if fmt.encoding == "pcm16":
            y = s.to(torch.int16)
        else:
            y = torch.from_numpy(audio_ref.ULAW if fmt.encoding == "mulaw" else audio_ref.ALAW)[s + 32768]
    if out is not None:
        out.copy_(y)
        return out
    return y
