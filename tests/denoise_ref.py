"""Restatement in fp64 of the enrollment noise suppressor (``artspeech_b200/frontend.py``, step 2b), written from its
definition: the centred 512-point STFT, the stationary noise profile, the decision-directed Wiener gain and the
windowed overlap-add.  Also the host model of the gain the kernel evaluates (numpy fp64, the kernel's operation order,
fed the kernel's own power), and a seeded voiced-speech generator with white, pink and mains-hum noise for the
quality tests."""
from __future__ import annotations

import math

import numpy as np
import scipy.signal as ss

N, HOP, K = 512, 128, 257
ALPHA = 0.98
Q = 0.1
C_Q = -math.log1p(-Q)                 # the 10 % quantile of an exponential with mean 1
LAMBDA_FLOOR = 1e-20


def window():
    """Periodic Hann window of N points, fp64."""
    return 0.5 - 0.5 * np.cos(2.0 * np.pi * np.arange(N) / N)


def n_frames(n):
    return 1 + n // HOP


def g_min(reduction_db):
    return 10.0 ** (-float(reduction_db) / 20.0)


def stft(y):
    """``X`` complex128 ``[F, 257]``: frame ``f`` holds ``w[i] y[128 f - 256 + i]`` (zeros outside ``[0, n)``)."""
    y = np.asarray(y, dtype=np.float64)
    n = y.size
    F = n_frames(n)
    yp = np.zeros((F - 1) * HOP + N)
    yp[N // 2:N // 2 + n] = y
    idx = np.arange(F)[:, None] * HOP + np.arange(N)[None, :]
    return np.fft.rfft(yp[idx] * window()[None, :], axis=1)


def istft(Y, n):
    """``y[t] = sum_f w[j] irfft(Y_f)[j] / sum_f w[j]^2``, ``j = t - 128 f + 256``, over the ``F`` frames of ``Y``."""
    Y = np.asarray(Y)
    F = Y.shape[0]
    w = window()
    frames = np.fft.irfft(Y, n=N, axis=1) * w[None, :]
    L = (F - 1) * HOP + N
    num, den = np.zeros(L), np.zeros(L)
    for f in range(F):
        num[f * HOP:f * HOP + N] += frames[f]
        den[f * HOP:f * HOP + N] += w * w
    return num[N // 2:N // 2 + n] / den[N // 2:N // 2 + n]


def power32(X):
    """The kernel's ``P = re^2 + im^2`` in fp32: two rounded products and one rounded add, from complex64 ``X``."""
    re = np.ascontiguousarray(X.real, dtype=np.float32)
    im = np.ascontiguousarray(X.imag, dtype=np.float32)
    return (re * re) + (im * im)


def noise_profile(P):
    """``lambda[k] = max(1e-20, P_(r)[k] / c)`` in fp64, ``P_(r)`` the ``r = F // 10``-th smallest of column k."""
    P = np.asarray(P)
    r = P.shape[0] // 10
    pr = np.partition(P, r, axis=0)[r].astype(np.float64)
    return np.maximum(LAMBDA_FLOOR, pr / C_Q)


def gains(P, lam, reduction_db):
    """fp32 ``G [F, 257]`` of the decision-directed Wiener rule, in fp64 in the kernel's order of operations."""
    P = np.asarray(P, dtype=np.float64)
    gm = g_min(reduction_db)
    one_m_alpha = 1.0 - ALPHA
    G = np.empty(P.shape, dtype=np.float32)
    A = np.zeros(P.shape[1])
    for f in range(P.shape[0]):
        gamma = P[f] / lam
        m = np.maximum(gamma - 1.0, 0.0)
        xi = m if f == 0 else ALPHA * A + one_m_alpha * m
        W = xi / (1.0 + xi)
        A = W * W * gamma
        G[f] = np.maximum(W, gm).astype(np.float32)
    return G


def denoise(y, reduction_db=18.0, planes=False):
    """The stage on one 24 kHz row, fp64 throughout (``G`` rounded to fp32 as the definition stores it)."""
    y = np.asarray(y, dtype=np.float64)
    X = stft(y)
    P = X.real ** 2 + X.imag ** 2
    lam = noise_profile(P)
    G = gains(P, lam, reduction_db)
    out = istft(G.astype(np.float64) * X, y.size)
    return (out, X, lam, G) if planes else out


# ---- voiced speech and noise ---------------------------------------------------------------------------------------
FS = 24000
EDGE_LENGTHS = (0, 1, 127, 128, 511, 512, 513)


def _resonator(fc, bw, fs=FS):
    """Two-pole resonator at ``fc`` Hz with bandwidth ``bw`` Hz, unit gain at its peak (approximately)."""
    r = math.exp(-math.pi * bw / fs)
    th = 2 * math.pi * fc / fs
    a = [1.0, -2 * r * math.cos(th), r * r]
    return [(1 - r) * math.sqrt(1 - 2 * r * math.cos(2 * th) + r * r)], a


def voiced(rng, n, fs=FS):
    """A seeded voiced-speech-like clip of ``n`` float32 samples.  Syllables of 120-350 ms separated by 60-400 ms
    pauses: a harmonic source (1/h harmonics up to 5 kHz) whose F0 glides between 85 and 260 Hz, through three formant
    resonators that move within and between syllables, with fricative bursts (high-passed noise) at some syllable
    edges.  Leading and trailing silence of 0.5-1.5 s each; peak level between -20 and -3 dBFS."""
    y = np.zeros(n)
    lead, trail = (rng.uniform(0.5, 1.5, 2) * fs).astype(int)
    t, end = int(lead), max(int(lead) + 1, n - int(trail))
    blk = fs // 100
    hp = ss.butter(4, 3000 / (fs / 2), "high")
    f0_base = rng.uniform(95, 200)
    while t < end:
        L = int(min(end - t, rng.integers(int(0.12 * fs), int(0.35 * fs))))
        k = np.arange(L)
        f0 = f0_base * np.exp(np.log(rng.uniform(0.8, 1.25)) * k / L) * (1 + 0.04 * np.sin(2 * np.pi * 5 * k / fs))
        f0 = np.clip(f0, 85, 260)
        ph = 2 * np.pi * np.cumsum(f0) / fs + rng.uniform(0, 2 * np.pi)
        src = np.zeros(L)
        for h in range(1, int(5000 / 85) + 1):
            src += np.where(h * f0 < 5000, np.sin(h * ph) / h, 0.0)
        formants = [(rng.uniform(300, 800), rng.uniform(300, 800)), (rng.uniform(900, 2200), rng.uniform(900, 2200)),
                    (rng.uniform(2300, 3300), rng.uniform(2300, 3300))]
        out = np.zeros(L)
        for (fa, fb), bw in zip(formants, (80.0, 110.0, 160.0)):
            zi = np.zeros(2)
            for s in range(0, L, blk):
                fc = fa + (fb - fa) * s / L
                b, a = _resonator(fc, bw, fs)
                seg, zi = ss.lfilter(b, a, src[s:s + blk], zi=zi)
                out[s:s + blk] += seg
        env = np.sin(np.pi * (k + 0.5) / L) ** 0.6
        syl = out * env * 10 ** (rng.uniform(-8, 0) / 20)
        if rng.random() < 0.4:                               # a fricative before or after the vowel
            fl = int(rng.integers(int(0.05 * fs), int(0.15 * fs)))
            fr = ss.lfilter(*hp, rng.standard_normal(fl)) * np.hanning(fl) * 0.3 * np.abs(syl).max()
            syl = np.concatenate([fr, syl]) if rng.random() < 0.5 else np.concatenate([syl, fr])
        m = min(syl.size, end - t)
        y[t:t + m] = syl[:m]
        t += m + int(rng.integers(int(0.06 * fs), int(0.4 * fs)))
    y *= 10 ** (rng.uniform(-20, -3) / 20) / max(1e-12, np.abs(y).max())
    return y.astype(np.float32)


def noise(rng, kind, n, fs=FS):
    """Unit-RMS stationary noise: ``white`` Gaussian, ``pink`` (1/f power from 20 Hz) or ``hum`` (50 Hz mains with
    its harmonics to 1 kHz at 1/h amplitude, random phases)."""
    if kind == "white":
        v = rng.standard_normal(n)
    elif kind == "pink":
        spec = np.fft.rfft(rng.standard_normal(n))
        f = np.fft.rfftfreq(n, 1 / fs)
        spec /= np.sqrt(np.maximum(f, 20.0))
        v = np.fft.irfft(spec, n)
    elif kind == "hum":
        t = np.arange(n) / fs
        v = sum(np.sin(2 * np.pi * 50 * h * t + rng.uniform(0, 2 * np.pi)) / h for h in range(1, 21))
    else:
        raise ValueError(kind)
    return v / max(1e-30, np.sqrt(np.mean(v ** 2)))


def mix(clean, nz, snr_db):
    """``clean + s nz`` with ``s`` such that the clip's energy over the noise's is ``snr_db``."""
    c = np.asarray(clean, np.float64)
    s = math.sqrt(np.sum(c ** 2) / np.sum(nz ** 2) / 10 ** (snr_db / 10))
    return (c + s * nz).astype(np.float32)


def snr_db(ref, y):
    ref, y = np.asarray(ref, np.float64), np.asarray(y, np.float64)
    return 10 * math.log10(np.sum(ref ** 2) / max(1e-300, np.sum((y - ref) ** 2)))


def voiced_set(seed=0, count=16):
    """``count`` seeded voiced clips of 3-12 s at 24 kHz."""
    rng = np.random.default_rng(seed)
    return [voiced(rng, int(rng.uniform(3, 12) * FS)) for _ in range(count)]
