"""Restatements of voice enrollment's input stage (``artspeech_b200/frontend.py``), written from its definitions:
two independent fp64 forms of librosa 0.10's ``effects.trim`` (the librosa-shaped one pads, frames and converts to
dB as librosa does; the block-sum one is the form the kernel evaluates), a float32 numpy model of the decode and
downmix, and a seeded set of speech-like clips."""
from __future__ import annotations

import numpy as np

FRAME, HOP = 2048, 512


# ---- decode and downmix ----------------------------------------------------------------------------------------
def _ulaw2lin(u):
    u = ~int(u) & 0xFF
    t = ((u & 0xF) << 3) + 0x84
    t <<= (u & 0x70) >> 4
    return 0x84 - t if u & 0x80 else t - 0x84


def _alaw2lin(a):
    a = int(a) ^ 0x55
    t = (a & 0xF) << 4
    seg = (a & 0x70) >> 4
    if seg == 0:
        t += 8
    elif seg == 1:
        t += 0x108
    else:
        t = (t + 0x108) << (seg - 1)
    return t if a & 0x80 else -t


ULAW2LIN = np.array([_ulaw2lin(u) for u in range(256)], dtype=np.int64)     # audioop.ulaw2lin, width 2
ALAW2LIN = np.array([_alaw2lin(a) for a in range(256)], dtype=np.int64)     # audioop.alaw2lin, width 2


def decode(x, encoding):
    """float32 samples of encoded ``x`` (any shape)."""
    x = np.asarray(x)
    if encoding == "float32":
        return x.astype(np.float32)
    if encoding == "pcm16":
        v = x.astype(np.int64)
    else:
        v = (ULAW2LIN if encoding == "mulaw" else ALAW2LIN)[x.astype(np.int64)]
    return v.astype(np.float32) / np.float32(32768)


def to_mono(x, encoding):
    """numpy's float32 ``mean`` over the channels of ``x`` ``[n]`` or ``[n, C]`` after decoding: a float32 sum in
    channel order, then one float32 divide."""
    d = decode(x, encoding)
    if d.ndim == 1:
        return d
    s = d[:, 0].copy()
    for c in range(1, d.shape[1]):
        s = s + d[:, c]
    return s / np.float32(d.shape[1])


# ---- trim --------------------------------------------------------------------------------------------------------
def _bounds(nonsilent, n):
    nz = np.flatnonzero(nonsilent)
    if n == 0 or nz.size == 0:
        return 0, 0
    return int(nz[0]) * HOP, min(n, (int(nz[-1]) + 1) * HOP)


def frame_power_librosa(y):
    """fp64 mean of squares of librosa's frames: ``np.pad`` with 1024 zeros on each side, frames of 2048, hop 512."""
    y = np.asarray(y, dtype=np.float64)
    yp = np.pad(y, FRAME // 2, mode="constant")
    F = 1 + (yp.size - FRAME) // HOP
    idx = np.arange(F)[:, None] * HOP + np.arange(FRAME)[None, :]
    rms = np.sqrt(np.mean(yp[idx] ** 2, axis=1))
    return rms ** 2


def frame_power_blocks(y):
    """fp64 ``p_f = (q_{f-2} + q_{f-1} + q_f + q_{f+1}) / 2048`` from the block sums ``q_j``."""
    y = np.asarray(y, dtype=np.float64)
    n = y.size
    nblk = -(-n // HOP)
    q = np.zeros(nblk + 4)
    if n:
        yz = np.zeros(nblk * HOP)
        yz[:n] = y
        q[2:2 + nblk] = (yz.reshape(nblk, HOP) ** 2).sum(1)
    F = 1 + n // HOP
    return np.array([(q[f] + q[f + 1] + q[f + 2] + q[f + 3]) / FRAME for f in range(F)])   # q[f + 2] is q_f


def trim_librosa(y, top_db=30.0):
    """librosa.effects.trim's (start, end) in fp64: ``amplitude_to_db(rms, ref=np.max, amin=1e-5) > -top_db``."""
    n = np.asarray(y).size
    p = frame_power_librosa(y)
    db = 10.0 * np.log10(np.maximum(1e-10, p)) - 10.0 * np.log10(np.maximum(1e-10, p.max()))
    return _bounds(db > -top_db, n)


def trim_blocks(y, top_db=30.0, margin=0.0):
    """(bounds, ambiguous) from the block-sum form.  Frames whose power is within ``margin`` relative of the threshold
    ``max(1e-10, P) 10^(-top_db/10)`` may be decided either way; ``ambiguous`` is True when that changes the bounds
    (the bounds are then those with every such frame silent)."""
    n = np.asarray(y).size
    p = frame_power_blocks(y)
    pc = np.maximum(1e-10, p)
    thr = np.maximum(1e-10, p.max()) * 10.0 ** (-top_db / 10.0)
    near = np.abs(pc / thr - 1.0) <= margin
    ns = 10.0 * np.log10(pc) - 10.0 * np.log10(np.maximum(1e-10, p.max())) > -top_db
    lo, hi = _bounds(ns & ~near, n), _bounds(ns | near, n)
    return lo, lo != hi


# ---- clips -------------------------------------------------------------------------------------------------------
EDGE_LENGTHS = (0, 1, 511, 512, 513, 1025)


def speech_like(rng, n, fs=24000):
    """A seeded speech-like clip of ``n`` float32 samples: noise and tone bursts separated by pauses, with fades, an
    optional DC offset and a level between -60 and 0 dBFS; leading and trailing silence of random length, sometimes
    with a low noise floor."""
    y = np.zeros(n)
    if n == 0:
        return y.astype(np.float32)
    lead, trail = rng.integers(0, max(1, n // 4), 2)
    t = int(lead)
    end = max(t + 1, n - int(trail))
    while t < end:
        L = int(min(end - t, rng.integers(fs // 50, fs // 2)))
        k = np.arange(L)
        if rng.random() < 0.5:
            s = rng.standard_normal(L)
        else:
            s = np.sin(2 * np.pi * rng.uniform(80, 4000) / fs * k + rng.uniform(0, 2 * np.pi))
        fade = min(L // 2, int(rng.integers(1, fs // 50)))
        env = np.ones(L)
        if fade > 0:
            env[:fade] = np.linspace(0, 1, fade)
            env[L - fade:] = np.linspace(1, 0, fade)
        y[t:t + L] = s * env * 10 ** (rng.uniform(-20, 0) / 20)
        t += L + int(rng.integers(0, fs // 4))
    y *= 10 ** (rng.uniform(-60, 0) / 20) / max(1e-12, np.abs(y).max())
    if rng.random() < 0.3:
        y += rng.uniform(-0.01, 0.01)                      # DC offset over the whole recording
    if rng.random() < 0.3:
        y += rng.standard_normal(n) * 10 ** (rng.uniform(-90, -60) / 20)
    return np.clip(y, -1.0, 1.0).astype(np.float32)


def clip_set(seed=0, count=60, max_seconds=60):
    """The seeded clips: every edge length, then ``count`` clips of random length up to ``max_seconds`` at 24 kHz
    (one of exactly ``max_seconds``)."""
    rng = np.random.default_rng(seed)
    clips = [speech_like(rng, n) for n in EDGE_LENGTHS]
    lengths = [max_seconds * 24000] + [int(rng.integers(2000, 24000 * 12)) for _ in range(count - 1)]
    clips += [speech_like(rng, n) for n in lengths]
    return clips
