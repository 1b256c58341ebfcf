"""fp64 restatement of the synthesis watermark (``artspeech_b200/audio.py``, ``as_watermark_embed`` /
``as_watermark_detect``), written from the definitions in ``audio.py``'s docstring: the patterns as literal cosine
sums, the envelope with ``np.interp``, the detector with numpy's FFT.  It chains with ``tests/audio_ref.py`` for the
output chain (``resample64`` and the G.711 tables) and with ``scipy.signal.resample_poly`` for the detector's
resampling; ``speech`` makes seeded speech-like test clips."""
from __future__ import annotations

import audioop
from functools import lru_cache

import numpy as np

P8, P24, NSYM = 4096, 12288, 256
BINS = np.arange(154, 1741)                   # k * 8000 / 4096 Hz inside [300, 3400]
MASK = (1 << 64) - 1


def splitmix64(x: int) -> int:
    x = (x + 0x9E3779B97F4A7C15) & MASK
    x = ((x ^ (x >> 30)) * 0xBF58476D1CE4E5B9) & MASK
    x = ((x ^ (x >> 27)) * 0x94D049BB133111EB) & MASK
    return x ^ (x >> 31)


@lru_cache(maxsize=None)
def phases(key: int, i: int) -> np.ndarray:
    hk = splitmix64(key)
    return np.array([splitmix64(hk ^ (i << 32) ^ int(k)) for k in BINS], dtype=np.float64) / 2.0 ** 64 * 2 * np.pi


@lru_cache(maxsize=None)
def pattern(key: int, i: int, n: int) -> np.ndarray:
    """``c_i^(n)[t] = sqrt(2/|K|) sum_k cos(2 pi k t / n + phi_i(k))``, summed literally."""
    t = np.arange(n, dtype=np.float64)
    c = np.zeros(n)
    ph = phases(key, i)
    for j in range(0, BINS.size, 128):
        k = BINS[j:j + 128, None].astype(np.float64)
        c += np.cos(2 * np.pi * ((k * t[None, :]) % n) / n + ph[j:j + 128, None]).sum(0)
    return c * np.sqrt(2.0 / BINS.size)


@lru_cache(maxsize=None)
def mark(key: int, message: int) -> np.ndarray:
    """The embedded 24 kHz pattern ``c`` (period 12288) of ``(key, message)``."""
    d = P24 // NSYM
    return (pattern(key, 0, P24) + np.roll(pattern(key, 1, P24), (message & 255) * d)
            + np.roll(pattern(key, 2, P24), (message >> 8) * d)) / np.sqrt(3.0)


def envelope(x, hop):
    """``e(t)`` for ``t < len(x)``: frame RMS over ``hop`` samples (zeros beyond the end), interpolated linearly between
    frame centres ``hop f + (hop - 1) / 2`` and held beyond the first and last."""
    x = np.asarray(x, dtype=np.float64)
    n = x.shape[0]
    if n == 0:
        return np.zeros(0)
    nf = -(-n // hop)
    xp = np.zeros(nf * hop)
    xp[:n] = x
    e = np.sqrt((xp.reshape(nf, hop) ** 2).sum(1) / hop)
    return np.interp(np.arange(n, dtype=np.float64), hop * np.arange(nf) + (hop - 1) / 2.0, e)


def embed(x, key, message, strength_db=-30.0, c=None):
    """The marked utterance ``y`` (fp64) of ``x`` (its ``n`` samples at 24 kHz)."""
    x = np.asarray(x, dtype=np.float64)
    c = mark(key, message) if c is None else c
    return x + 10.0 ** (strength_db / 20.0) * envelope(x, 240) * c[np.arange(x.shape[0]) % P24]


def normalise(y8):
    e = envelope(y8, 80)
    y8 = np.asarray(y8, dtype=np.float64)
    return np.where(e >= 1e-4, y8 / np.where(e >= 1e-4, e, 1.0), 0.0)


def correlations(y8, key):
    """``(r_0, r_1, r_2)``, each ``[4096]``: the whitened correlations of the 8 kHz utterance ``y8`` at every lag."""
    z = normalise(y8)
    nper = -(-z.shape[0] // P8)
    zp = np.zeros(nper * P8)
    zp[:z.shape[0]] = z
    Z = np.fft.rfft(zp.reshape(nper, P8), axis=1)[:, BINS] if nper else np.zeros((0, BINS.size), complex)
    A, S = Z.sum(0), (np.abs(Z) ** 2).sum(0)
    G = np.where(S > 0, A / np.where(S > 0, S, 1.0), 0.0)
    r = []
    for i in range(3):
        spec = np.zeros(P8, complex)
        spec[BINS] = G * np.exp(-1j * phases(key, i))
        r.append(np.real(np.fft.ifft(spec)) * P8)            # sum_k Re(G e^{-j phi} e^{j 2 pi k tau / 4096})
    return r


def detect(y8, key, threshold=6.0):
    """``(detected, score, lag, message)`` of the 8 kHz utterance ``y8``; score 0 when ``r_0`` is all zero."""
    r0, r1, r2 = correlations(y8, key)
    tau = int(np.argmax(np.abs(r0)))
    ms = np.mean(r0 ** 2)
    score = float(abs(r0[tau]) / np.sqrt(ms)) if ms > 0 else 0.0
    lags = (tau + np.arange(NSYM) * (P8 // NSYM)) % P8
    message = int(np.argmax(np.abs(r1[lags]))) | int(np.argmax(np.abs(r2[lags]))) << 8
    return score >= threshold, score, tau, message


# ---- the output chain and its inverse (what a detector receives) ----------------------------------------------
def encode(y, encoding):
    """int16 / G.711 codes of fp samples (the product's encoders), or fp32 for ``"float32"``."""
    from tests import audio_ref
    y = np.asarray(y, dtype=np.float64)
    if encoding == "float32":
        return y.astype(np.float32)
    s = np.clip(np.rint(32767.0 * y), -32768, 32767).astype(np.int64)
    if encoding == "pcm16":
        return s.astype(np.int16)
    return (audio_ref.ULAW if encoding == "mulaw" else audio_ref.ALAW)[s + 32768]


def decode(v, encoding):
    """fp64 samples of encoded ``v``: PCM16 ``v / 32768``, G.711 by ``audioop.ulaw2lin`` / ``alaw2lin`` / 32768."""
    v = np.asarray(v)
    if encoding == "float32":
        return v.astype(np.float64)
    if encoding == "pcm16":
        return v.astype(np.float64) / 32768.0
    fn = audioop.ulaw2lin if encoding == "mulaw" else audioop.alaw2lin
    return np.frombuffer(fn(v.astype(np.uint8).tobytes(), 2), "<i2").astype(np.float64) / 32768.0


def to_8k(y, rate):
    """``resample_poly(y, 8000 / g, rate / g)`` (the detector's resampling), ``y`` unchanged at 8 kHz."""
    from math import gcd
    from scipy.signal import resample_poly
    if rate == 8000:
        return np.asarray(y, dtype=np.float64)
    g = gcd(8000, rate)
    return resample_poly(np.asarray(y, dtype=np.float64), 8000 // g, rate // g)


def speech(n, rng, fs=24000):
    """A speech-like clip: pulse train (f0 90-170 Hz) through three formant resonators, syllable envelope with 20 %
    pauses, peak 0.3."""
    from scipy.signal import lfilter
    t = np.arange(n) / fs
    f0 = 120 + 30 * np.sin(2 * np.pi * 0.7 * t) + rng.uniform(-20, 20)
    y = (np.diff(np.floor(np.cumsum(f0 / fs)), prepend=0) > 0).astype(float)
    for F, bw in [(rng.uniform(400, 800), 80), (rng.uniform(1000, 2000), 120), (rng.uniform(2300, 3000), 160)]:
        r = np.exp(-np.pi * bw / fs)
        y = lfilter([1], [1, -2 * r * np.cos(2 * np.pi * F / fs), r * r], y)
    y += 0.02 * rng.standard_normal(n) * np.std(y)
    env, i = np.zeros(n), 0
    while i < n:
        m = int(fs * rng.uniform(0.1, 0.35))
        env[i:i + m] = (rng.uniform() > 0.2) * 10 ** (-rng.uniform(0, 20) / 20)
        i += m
    y *= np.convolve(env, np.ones(240) / 240, "same")
    return 0.3 * y / max(np.max(np.abs(y)), 1e-30)
