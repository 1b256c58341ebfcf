"""Output audio formats for synthesis: any integer sample rate by polyphase resampling, and fp32 / 16-bit PCM /
ITU-T G.711 mu-law and A-law samples, computed on the GPU after the vocoder (``as_resample_encode``).

``AudioFormat(sample_rate, encoding)`` names a format; the vocoder's own is ``AudioFormat(24000, "float32")``.

Semantics (per utterance of ``n_in`` samples at 24 kHz):

- **Rate.**  ``up / down = sample_rate / 24000`` reduced by their gcd; ``n_out = ceil(n_in * up / down)``.  The
  filter is ``scipy.signal.resample_poly``'s default design: ``half_len = 10 * max(up, down)``,
  ``h = firwin(2 * half_len + 1, 1 / max(up, down), window=("kaiser", 5.0)) * up`` (designed here in fp64 with numpy:
  windowed sinc, unit DC gain, times ``up``), and ``y[m] = sum_k h[k] * xu[m * down + half_len - k]`` with ``xu`` the
  input zero-stuffed by ``up`` and zero outside ``[0, n_in)``.  The kernel evaluates it from the fp32 polyphase table
  ``table[p][j] = h[p + j * up]`` (``K = ceil(len(h) / up)`` taps per output) as one fp32 fma chain over
  ``j = 0 .. K-1``.  24 kHz is the identity.
- **Encoding.**  ``"float32"``: ``y``.  ``"pcm16"``: ``clamp(rint(32767 * y), -32768, 32767)``, the expression of the
  vocoder's ``pcm16=True`` output.  ``"mulaw"`` / ``"alaw"``: the uint8 G.711 code of that int16 value (the codes of
  ``audioop.lin2ulaw`` / ``lin2alaw`` with width 2).  Samples beyond an utterance's ``n_out`` hold the encoding's code
  for 0 (``silence``): 0, 0, 0xFF, 0xD5.

A rate whose filter does not fit the kernel's shared-memory budget (``smem_bytes`` above ``SMEM_MAX``: very low rates
and rates with a large ``up``, e.g. 44101 Hz) is refused on construction.
"""
from __future__ import annotations

import math
import operator
from dataclasses import dataclass
from functools import lru_cache
from typing import Dict, Tuple

import numpy as np
import torch

NATIVE_RATE = 24000
ENCODINGS = ("float32", "pcm16", "mulaw", "alaw")
CODES = {"float32": 0, "pcm16": 1, "mulaw": 2, "alaw": 3}            # AS_AUDIO_F32 .. AS_AUDIO_ALAW
DTYPES = {"float32": torch.float32, "pcm16": torch.int16, "mulaw": torch.uint8, "alaw": torch.uint8}
SILENCE = {"float32": 0, "pcm16": 0, "mulaw": 0xFF, "alaw": 0xD5}
TILE = 1024                      # AS_AUDIO_TILE: output samples per CTA work item
SMEM_MAX = 96 * 1024             # AS_AUDIO_SMEM_MAX
KAISER_BETA = 5.0


@lru_cache(maxsize=None)
def _design(up: int, down: int) -> Tuple[np.ndarray, np.ndarray]:
    """(h fp64 [2 * half_len + 1], polyphase table fp32 [up, table_ld]) of the ratio ``up / down``."""
    mx = max(up, down)
    half_len = 10 * mx
    n = 2 * half_len + 1
    cutoff = 1.0 / mx
    m = np.arange(n, dtype=np.float64) - half_len
    h = cutoff * np.sinc(cutoff * m) * np.kaiser(n, KAISER_BETA)
    h = h / h.sum() * up
    K = -(-n // up)
    table = np.zeros((up, (K + 3) // 4 * 4), dtype=np.float32)
    hp = np.zeros(up * K)
    hp[:n] = h
    table[:, :K] = hp.reshape(K, up).T
    return h, table


def smem_bytes(up: int, down: int, K: int, table_ld: int) -> int:
    """Shared memory of one ``as_resample_encode`` CTA (``as_resample_smem_bytes``): table, input window of a tile,
    encoded tile."""
    ident = up == 1 and down == 1
    if ident:
        K, table_ld = 1, 4
    win = ((TILE - 1) * down + up - 1) // up + K + 8
    win = (win + 3) // 4 * 4
    return 4 * ((0 if ident else up * table_ld) + win) + 4 * TILE


_TABLES: Dict[tuple, torch.Tensor] = {}


@dataclass(frozen=True)
class AudioFormat:
    """An output format: integer ``sample_rate`` (Hz) and ``encoding`` in ``ENCODINGS``; validated on
    construction (``ValueError``)."""
    sample_rate: int = NATIVE_RATE
    encoding: str = "float32"

    def __post_init__(self):
        rate = self.sample_rate
        if isinstance(rate, bool):
            raise ValueError(f"AudioFormat.sample_rate: expected an integer, got {rate!r}")
        try:
            rate = operator.index(rate)
        except TypeError:
            raise ValueError(f"AudioFormat.sample_rate: expected an integer, got {rate!r}") from None
        if rate <= 0:
            raise ValueError(f"AudioFormat.sample_rate: must be positive, got {rate}")
        if self.encoding not in ENCODINGS:
            raise ValueError(f"AudioFormat.encoding: expected one of {ENCODINGS}, got {self.encoding!r}")
        object.__setattr__(self, "sample_rate", rate)
        if smem_bytes(self.up, self.down, self.K, self.table_ld) > SMEM_MAX:
            raise ValueError(f"AudioFormat.sample_rate: {rate} Hz (up {self.up}, down {self.down}) needs "
                             f"{smem_bytes(self.up, self.down, self.K, self.table_ld)} bytes of shared memory for its "
                             f"polyphase filter, more than the kernel's {SMEM_MAX}")

    # -- the ratio and the filter --------------------------------------------------------------------------------
    @property
    def up(self) -> int:
        return self.sample_rate // math.gcd(self.sample_rate, NATIVE_RATE)

    @property
    def down(self) -> int:
        return NATIVE_RATE // math.gcd(self.sample_rate, NATIVE_RATE)

    @property
    def is_identity(self) -> bool:
        """24 kHz: the kernel only encodes."""
        return self.up == 1 and self.down == 1

    @property
    def half_len(self) -> int:
        return 0 if self.is_identity else 10 * max(self.up, self.down)

    @property
    def K(self) -> int:
        """Taps per output sample."""
        return 1 if self.is_identity else -(-(2 * self.half_len + 1) // self.up)

    @property
    def table_ld(self) -> int:
        return (self.K + 3) // 4 * 4

    def filter64(self) -> np.ndarray:
        """The fp64 prototype filter ``h`` (``2 * half_len + 1`` taps, DC gain ``up``)."""
        if self.is_identity:
            return np.ones(1)
        return _design(self.up, self.down)[0]

    def table(self) -> np.ndarray:
        """The fp32 polyphase table ``[up, table_ld]``: ``table[p][j] = h[p + j * up]``, zero beyond."""
        if self.is_identity:
            return np.array([[1.0, 0.0, 0.0, 0.0]], dtype=np.float32)
        return _design(self.up, self.down)[1]

    def device_table(self, device) -> torch.Tensor:
        """The table on ``device`` (cached per ratio and device)."""
        device = torch.device(device)
        key = (self.up, self.down, device)
        t = _TABLES.get(key)
        if t is None:
            t = torch.from_numpy(self.table().copy()).to(device)
            _TABLES[key] = t
        return t

    # -- sizes and types -----------------------------------------------------------------------------------------
    def out_samples(self, n_in: int) -> int:
        """Output samples of an utterance of ``n_in`` samples at 24 kHz: ``ceil(n_in * up / down)``."""
        return -(-int(n_in) * self.up // self.down)

    @property
    def dtype(self) -> torch.dtype:
        return DTYPES[self.encoding]

    @property
    def code(self) -> int:
        return CODES[self.encoding]

    @property
    def silence(self) -> int:
        return SILENCE[self.encoding]

    def frame_align(self, hop: int) -> int:
        """Frames (of ``hop`` samples at 24 kHz) between input positions whose output offset is an integer: a window
        of the input starting at a multiple of this many frames is resampled on the same output grid."""
        return self.down // math.gcd(self.down, hop)


NATIVE = AudioFormat()


def check(audio, pcm16: bool):
    """Validate an ``audio=`` argument: None or an ``AudioFormat``; ``pcm16=True`` together with a format is a
    ``ValueError`` (the format names the encoding)."""
    if audio is None:
        return None
    if not isinstance(audio, AudioFormat):
        raise ValueError(f"audio: expected an AudioFormat, got {type(audio).__name__}")
    if pcm16:
        raise ValueError("audio= and pcm16=True: choose the encoding with AudioFormat(..., encoding='pcm16')")
    return audio
