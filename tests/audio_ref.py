"""fp64 restatement of the output audio formats (``artspeech_b200/audio.py``, ``as_resample_encode``), written from
their definitions: the resampler from ``y[m] = sum_k h[k] * xu[m * down + half_len - k]`` and the G.711 encoders as
a literal port of CPython's audioop (``st_14linear2ulaw`` / ``st_linear2alaw``, segment search included), plus a
torch model of ``ops.resample_encode`` for host-logic tests on the CPU."""
from __future__ import annotations

import numpy as np
import torch

_SEG_UEND = (0x3F, 0x7F, 0xFF, 0x1FF, 0x3FF, 0x7FF, 0xFFF, 0x1FFF)
_SEG_AEND = (0x1F, 0x3F, 0x7F, 0xFF, 0x1FF, 0x3FF, 0x7FF, 0xFFF)


def _search(v, table):
    for i, t in enumerate(table):
        if v <= t:
            return i
    return len(table)


def _ulaw14(v):
    if v < 0:
        v, mask = -v, 0x7F
    else:
        mask = 0xFF
    v = min(v, 8159) + (0x84 >> 2)
    seg = _search(v, _SEG_UEND)
    if seg >= 8:
        return 0x7F ^ mask
    return ((seg << 4) | ((v >> (seg + 1)) & 0xF)) ^ mask


def _alaw13(v):
    if v >= 0:
        mask = 0xD5
    else:
        mask, v = 0x55, -v - 1
    seg = _search(v, _SEG_AEND)
    if seg >= 8:
        return 0x7F ^ mask
    a = seg << 4
    a |= ((v >> 1) if seg < 2 else (v >> seg)) & 0xF
    return a ^ mask


# code tables indexed by int16 + 32768 (width 2: 14-bit mu-law input s >> 2, 13-bit A-law input s >> 3)
ULAW = np.array([_ulaw14(s >> 2) for s in range(-32768, 32768)], dtype=np.uint8)
ALAW = np.array([_alaw13(s >> 3) for s in range(-32768, 32768)], dtype=np.uint8)


def resample64(x, h, up, down, half_len):
    """(y, s): the fp64 resampled signal of ``x`` (1-D) and ``s[m] = sum_j |h_j| |x_j|`` over the same terms."""
    x = np.asarray(x, dtype=np.float64)
    n_in = x.shape[0]
    n_out = -(-n_in * up // down)
    if up == 1 and down == 1:
        return x.copy(), np.abs(x)
    K = -(-len(h) // up)
    hp = np.zeros(K * up)
    hp[:len(h)] = h
    n = np.arange(n_out, dtype=np.int64) * down + half_len
    i0, p = n // up, n % up
    j = np.arange(K)
    idx = i0[:, None] - j[None, :]
    taps = hp[p[:, None] + j[None, :] * up]
    ok = (idx >= 0) & (idx < n_in)
    xv = np.where(ok, x[np.clip(idx, 0, max(n_in - 1, 0))] if n_in else 0.0, 0.0)
    return (taps * xv).sum(1), (np.abs(taps) * np.abs(xv)).sum(1)


def encode(y64, bound, encoding):
    """(want, alt): the codes of the fp64 values ``y64`` and the codes also accepted where the kernel's fp32 value
    (within ``bound`` of ``y64``) or its fp32 product with 32767 may round to the neighbouring int16."""
    if encoding == "float32":
        return y64, y64
    t = 32767.0 * y64
    s = np.clip(np.rint(t), -32768, 32767).astype(np.int64)
    near = np.abs(t - np.floor(t) - 0.5) <= 32767.0 * bound + np.abs(t) * 2.0 ** -24
    other = 2 * np.floor(t).astype(np.int64) + 1 - np.rint(t).astype(np.int64)   # the other side of the midpoint
    s2 = np.where(near, np.clip(other, -32768, 32767), s)
    if encoding == "pcm16":
        return s.astype(np.int16), s2.astype(np.int16)
    tab = ULAW if encoding == "mulaw" else ALAW
    return tab[s + 32768], tab[s2 + 32768]


# ---- torch model of ops.resample_encode (fp32, the kernel's tap order) for host-logic tests --------------------
def resample_encode_model(x, lens, fmt, S_out, *, m0=0, out=None, out_lens=None):
    B, S_in = x.shape
    table = torch.from_numpy(fmt.table().copy())
    y = torch.empty(B, int(S_out), dtype=fmt.dtype)
    m = torch.arange(int(S_out), dtype=torch.int64) + int(m0)
    for b in range(B):
        n_in = S_in if lens is None else min(max(int(lens[b]), 0), S_in)
        n_out = fmt.out_samples(n_in)
        xb = x[b, :n_in].float()
        if fmt.is_identity:
            v = torch.where(m < n_in, xb[m.clamp(0, max(n_in - 1, 0))] if n_in else torch.zeros(()),
                            torch.zeros(()))
        else:
            n = m * fmt.down + fmt.half_len
            i0, p = n // fmt.up, n % fmt.up
            v = torch.zeros(int(S_out))
            for j in range(fmt.K):
                i = i0 - j
                ok = (i >= 0) & (i < n_in)
                xv = torch.where(ok, xb[i.clamp(0, max(n_in - 1, 0))] if n_in else torch.zeros(()), torch.zeros(()))
                v = v + table[p, j] * xv
        v = torch.where(m < n_out, v, torch.zeros(()))
        if fmt.encoding == "float32":
            y[b] = v
        else:
            s = torch.clamp(torch.round(v * 32767.0), -32768, 32767).to(torch.int64)
            if fmt.encoding == "pcm16":
                y[b] = s.to(torch.int16)
            else:
                tab = torch.from_numpy(ULAW if fmt.encoding == "mulaw" else ALAW)
                y[b] = tab[s + 32768]
        if out_lens is not None:
            out_lens[b] = n_out
    if out is not None:
        out.copy_(y)
        return out
    return y
