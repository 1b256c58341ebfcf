"""Output audio formats for synthesis: any integer sample rate by polyphase resampling, and fp32 / 16-bit PCM /
ITU-T G.711 mu-law and A-law samples, computed on the GPU after the vocoder (``as_resample_encode``); loudness
normalisation; and the synthesis watermark.

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

**Loudness normalisation** (``Loudness(target_lufs, max_true_peak_db)``, ``as_loudness_measure``).  The meter, for
one utterance of ``n`` fp32 samples at ``fs`` Hz (the engine meters at 24 kHz; ``measure_loudness`` takes any multiple
of 10 Hz from 8000 to 192000):

1. **K-weighting** (ITU-R BS.1770): two cascaded biquads with zero initial state, designed by the bilinear transform
   as libebur128 does and evaluated in fp64 on the host (``k_weighting``).  Shelf: ``f0 = 1681.974450955533``,
   ``G = 3.999843853973347``, ``Q = 0.7071752369554196``, ``K = tan(pi f0 / fs)``, ``Vh = 10^(G/20)``,
   ``Vb = Vh^0.4996667741545416``, ``a0 = 1 + K/Q + K^2``, ``b = [Vh + Vb K/Q + K^2, 2 (K^2 - Vh),
   Vh - Vb K/Q + K^2] / a0``, ``a = [1, 2 (K^2 - 1) / a0, (1 - K/Q + K^2) / a0]``.  High-pass:
   ``f0 = 38.13547087602444``, ``Q = 0.5003270373238773``, ``b = [1, -2, 1]``, ``a`` as above.  At 48 kHz these are
   BS.1770-4's table.
2. **Blocks.**  Segments of ``fs/10`` samples (100 ms); block ``j`` covers segments ``j .. j+3`` (400 ms, 75 %
   overlap) for ``j = 0 .. nseg - 4``, ``nseg = n // (fs/10)``; samples after the last complete segment feed no
   block.  ``z_j`` is the mean of the squared K-weighted output over the block, ``L_j = -0.691 + 10 log10 z_j``.
   An utterance shorter than one block (``n < 4 fs/10``, e.g. a single word) is one block over all ``n`` samples;
   BS.1770 defines no value for such signals.
3. **Gating.**  ``J_a = {j : L_j > -70}``, ``G_r = -0.691 + 10 log10(mean_{J_a} z) - 10``,
   ``J_g = {j in J_a : L_j > G_r}``, integrated loudness ``L = -0.691 + 10 log10(mean_{J_g} z)`` (LUFS); ``-inf``
   when ``J_a`` is empty or ``n = 0``.
4. **True peak.**  ``TP = max(max_i |x_i|, max_m |y4_m|)`` with ``y4`` the 4x interpolation by this module's
   resampler math (``_design(4, 1)``: 81 taps, ``half_len`` 40, fp32 polyphase table ``true_peak_table()``), ``x``
   zero outside ``[0, n)``, ``m < 4 n``; ``true_peak_db = 20 log10 TP`` (``-inf`` for 0).  At 24 kHz this is a 96 kHz
   peak: BS.1770 asks 4x for 48 kHz input, so an inter-sample peak close to Nyquist can read low.
5. **Gain.**  ``gain_db = 0`` if ``L = -inf``, else ``min(target_lufs - L, max_true_peak_db - true_peak_db)``;
   ``g = fp32(10^(gain_db/20))`` (computed in fp64, rounded once).  The format stage outputs ``encode(g * y)``: one
   fp32 multiply after the resampler's value ``y`` (after ``x`` at 24 kHz), before the encoding; silence codes are
   unchanged.  A single gain, like ffmpeg ``loudnorm`` in linear mode: no limiter or dynamic range control.
6. **Measurement point.**  The engine meters the vocoder's 24 kHz fp32 waveform once per utterance, whatever the
   output format, so one utterance requested in two formats gets the same gain and no extra pass at the target rate
   is needed.  A meter run at a lower delivery rate (8 kHz) reads somewhat lower, because the band above that rate's
   Nyquist frequency is removed.  Normalisation sets the overall level, so it overrides the overall-level effect of
   ``Prosody.energy_db`` (the energy contour's shape stays).

**Watermark** (``Watermark(key, message, strength_db)``, ``as_watermark_embed`` / ``as_watermark_detect``).  A mark in
the samples that says "synthetic" and carries a 16-bit ``message``, keyed by a 64-bit secret ``key``.  Detectors
deployed later depend on this exact format:

1. **Pattern.**  ``K`` = DFT bins ``k = 154 .. 1740`` of a 4096-point period at 8 kHz (``k 8000 / 4096`` Hz inside
   [300, 3400] Hz, the telephone band; 1587 bins).  Pattern ``i`` in {0, 1, 2} (sync, data 1, data 2) has the phases
   ``phi_i(k) = 2 pi h(h(key) ^ (i << 32) ^ k) / 2^64`` with ``h`` splitmix64 (add ``0x9E3779B97F4A7C15``, then
   ``x ^= x >> 30; x *= 0xBF58476D1CE4E5B9; x ^= x >> 27; x *= 0x94D049BB133111EB; x ^= x >> 31``, mod 2^64).  With
   ``n`` samples per 0.512 s period, ``c_i^(n)[t] = sqrt(2/|K|) sum_{k in K} cos(2 pi k t / n + phi_i(k))``: unit
   RMS, band-limited, periodic; ``c^(12288)[3t] = c^(4096)[t]``.
2. **Embedding** (24 kHz, utterance of ``n`` samples).  ``s1 = message & 255``, ``s2 = message >> 8``;
   ``c[t] = (c_0[t] + c_1[(t - 48 s1) mod 12288] + c_2[(t - 48 s2) mod 12288]) / sqrt(3)``, computed in fp64 and
   rounded once to fp32 (``watermark_mark``, cached per key, message and device).  ``e_f`` is the RMS of the
   240-sample frame ``f`` (10 ms; zeros at and beyond ``n``), ``e(t)`` interpolates linearly between the frame centres
   ``240 f + 119.5`` and is held beyond the first and last.  ``y[t] = x[t] + (alpha e(t)) c[t mod 12288]`` (one fp32
   fma) for ``t < n``, ``alpha = 10^(strength_db/20)``, and 0 beyond ``n``.  The mark follows the speech envelope: it
   vanishes in digital silence and its power relative to the signal is ``strength_db`` (default -30 dB).  It depends
   only on the utterance's own samples and ``t``.
3. **Detection** (8 kHz fp32, utterance of ``n`` samples).  (a) ``z[t] = y[t] / e(t)`` where ``e(t) >= 1e-4``, else
   0, with the envelope of 80-sample frames.  (b) Period ``p`` is ``z[4096 p .. 4096 p + 4095]`` (zeros beyond ``n``),
   ``Z_p(k)`` its DFT at ``k in K``.  (c) Whitening: ``A(k) = sum_p Z_p(k)``, ``S(k) = sum_p |Z_p(k)|^2``,
   ``G = A / S`` (0 where ``S = 0``).  (d) ``r_i[tau] = sum_k Re(G(k) e^{-j phi_i(k)} e^{j 2 pi k tau / 4096})`` for
   every ``tau < 4096``: a crop is a circular lag, found without a search.  (e) ``tau* = argmax |r_0|`` (lowest on
   ties), ``score = |r_0[tau*]| / sqrt(mean r_0^2)`` (0 when ``r_0`` is 0), ``detected = score >= threshold``
   (default 6: about 2 4096 Q(6) = 8e-6 false positives per clip under a Gaussian null); polarity and gain do not
   matter.  (f) ``s_i = argmax_{s < 256} |r_i[(tau* + 16 s) mod 4096]|``, ``message = s1 | s2 << 8``.
4. **Input formats.**  ``detect_watermark`` decodes PCM16 as ``v / 32768`` and G.711 as ``audioop.ulaw2lin`` /
   ``alaw2lin`` then ``/ 32768``, and resamples to 8 kHz with this module's resampler (``ToDetectionRate``:
   ``resample_poly``'s filter for ``8000 / rate``; a ratio whose filter does not fit the kernel is refused).
5. **Measured robustness** (fp64 reference, tests/test_watermark_cpu.py): seeded speech-like clips of 2-12 s through
   every ``AudioFormat`` rate and encoding, cropped, polarity-flipped and loudness-normalised, are all detected with
   their message; unmarked, wrong-key, white-noise and silent clips score at most about 5.  Not covered: lossy codecs
   (MP3, Opus, AAC), time-stretch, pitch-shift, deliberate removal or forgery (the periodic pattern can be estimated
   by averaging many marked clips: this is a compliance label, not a security mechanism), listening tests, and
   ``Generator.stream`` / ``pcm16=True`` engines, which are not marked.
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


# ---- loudness --------------------------------------------------------------------------------------------------
_SHELF = (1681.974450955533, 3.999843853973347, 0.7071752369554196)
_HIGHPASS = (38.13547087602444, 0.5003270373238773)
TRUE_PEAK_UP = 4


def _rate_ok(fs) -> bool:
    return not isinstance(fs, bool) and isinstance(fs, (int, np.integer)) and 8000 <= fs <= 192000 and fs % 10 == 0


@lru_cache(maxsize=None)
def k_weighting(fs: int) -> Tuple[Tuple[np.ndarray, np.ndarray], Tuple[np.ndarray, np.ndarray]]:
    """((b, a) of the shelf, (b, a) of the high-pass) of BS.1770's K-weighting at ``fs`` Hz, fp64."""
    f0, G, Q = _SHELF
    K = math.tan(math.pi * f0 / fs)
    Vh = 10.0 ** (G / 20.0)
    Vb = Vh ** 0.4996667741545416
    a0 = 1.0 + K / Q + K * K
    shelf = (np.array([(Vh + Vb * K / Q + K * K) / a0, 2.0 * (K * K - Vh) / a0, (Vh - Vb * K / Q + K * K) / a0]),
             np.array([1.0, 2.0 * (K * K - 1.0) / a0, (1.0 - K / Q + K * K) / a0]))
    f0, Q = _HIGHPASS
    K = math.tan(math.pi * f0 / fs)
    a0 = 1.0 + K / Q + K * K
    hp = (np.array([1.0, -2.0, 1.0]), np.array([1.0, 2.0 * (K * K - 1.0) / a0, (1.0 - K / Q + K * K) / a0]))
    return shelf, hp


def k_weighting_taps(fs: int) -> np.ndarray:
    """The 10 doubles ``as_loudness_measure`` takes: b0 b1 b2 a1 a2 of the shelf, then of the high-pass."""
    (bs, as_), (bh, ah) = k_weighting(int(fs))
    return np.concatenate([bs, as_[1:], bh, ah[1:]])


def true_peak_table() -> np.ndarray:
    """The fp32 polyphase table ``[4, 24]`` of the 4x true-peak interpolator (``_design(4, 1)``: 21 taps a phase)."""
    return _design(TRUE_PEAK_UP, 1)[1]


@dataclass(frozen=True)
class Loudness:
    """Loudness normalisation of each utterance to ``target_lufs`` (integrated loudness, ITU-R BS.1770) with its true
    peak at most ``max_true_peak_db`` dBTP: one gain per utterance, applied before the output encoding.  The default is
    EBU R128 (-23 LUFS, -1 dBTP); ATSC A/85 is -24, streaming platforms use -14 to -16."""
    target_lufs: float = -23.0
    max_true_peak_db: float = -1.0

    def __post_init__(self):
        for name in ("target_lufs", "max_true_peak_db"):
            v = getattr(self, name)
            if isinstance(v, bool) or not isinstance(v, (int, float, np.integer, np.floating)) or \
                    not math.isfinite(float(v)):
                raise ValueError(f"Loudness.{name}: expected a finite number, got {v!r}")
            object.__setattr__(self, name, float(v))
        if self.target_lufs >= 0.0:
            raise ValueError(f"Loudness.target_lufs: must be negative, got {self.target_lufs}")
        if self.max_true_peak_db > 0.0:
            raise ValueError(f"Loudness.max_true_peak_db: must be at most 0 dBTP, got {self.max_true_peak_db}")


def check_loudness(loudness, pcm16: bool):
    """Validate a ``loudness=`` argument: None or a ``Loudness``; with ``pcm16=True`` a ``ValueError`` (the meter and
    the gain read the fp32 waveform)."""
    if loudness is None:
        return None
    if not isinstance(loudness, Loudness):
        raise ValueError(f"loudness: expected a Loudness, got {type(loudness).__name__}")
    if pcm16:
        raise ValueError("loudness= and pcm16=True: the meter reads the fp32 waveform; use Synthesizer(pcm16=False) "
                         "with audio=AudioFormat(24000, 'pcm16')")
    return loudness


def measure_loudness(wav: torch.Tensor, lengths=None, sample_rate: int = NATIVE_RATE):
    """``(lufs, true_peak_db)`` of each row of ``wav`` (fp32 [B, S] or [S], CUDA) as fp64 [B] device tensors, measured
    on the GPU as stated in this module's docstring.  ``lengths``: per-row sample counts (int tensor or sequence;
    None: every row holds S samples); ``sample_rate``: a multiple of 10 Hz from 8000 to 192000."""
    from . import ops
    if not _rate_ok(sample_rate):
        raise ValueError(f"measure_loudness: sample_rate must be a multiple of 10 Hz in [8000, 192000], "
                         f"got {sample_rate!r}")
    x = wav.view(1, -1) if wav.dim() == 1 else wav
    if lengths is not None:
        lengths = torch.as_tensor(lengths).to(device=x.device, dtype=torch.int32).contiguous()
    lufs, tp, _, _ = ops.loudness_measure(x, lengths, int(sample_rate))
    return lufs, tp


# ---- watermark -------------------------------------------------------------------------------------------------
WM_PERIOD = 4096                 # AS_WM_PERIOD: samples per pattern period at 8 kHz (0.512 s)
WM_PERIOD_24K = 12288            # AS_WM_PERIOD_24K
WM_RATE = 8000                   # the detector's rate
WM_BINS = np.arange(154, 1741)   # AS_WM_K_LO ..: bins k * 8000 / 4096 Hz inside [300, 3400]
WM_BINS_LD = 1588                # AS_WM_BINS_LD
WM_SYMBOLS = 256                 # AS_WM_SYMBOLS
WM_THRESHOLD = 6.0
_MASK64 = (1 << 64) - 1


def splitmix64(x: int) -> int:
    """One splitmix64 output of the 64-bit state ``x``."""
    x = (x + 0x9E3779B97F4A7C15) & _MASK64
    x = ((x ^ (x >> 30)) * 0xBF58476D1CE4E5B9) & _MASK64
    x = ((x ^ (x >> 27)) * 0x94D049BB133111EB) & _MASK64
    return x ^ (x >> 31)


@lru_cache(maxsize=64)
def watermark_phases(key: int) -> np.ndarray:
    """fp64 ``[3, 1587]``: ``phi_i(k) = 2 pi h(h(key) ^ (i << 32) ^ k) / 2^64`` of the sync and the two data
    patterns."""
    hk = splitmix64(int(key))
    return np.array([[splitmix64(hk ^ (i << 32) ^ int(k)) for k in WM_BINS] for i in range(3)],
                    dtype=np.float64) / 2.0 ** 64 * (2.0 * math.pi)


def watermark_pattern(key: int, i: int, n: int) -> np.ndarray:
    """fp64 ``c_i^(n)``: ``sqrt(2/|K|) sum_k cos(2 pi k t / n + phi_i(k))``, ``t < n`` (one period, unit RMS)."""
    spec = np.zeros(n // 2 + 1, dtype=np.complex128)
    spec[WM_BINS] = np.exp(1j * watermark_phases(key)[i])
    return np.fft.irfft(spec, n) * (n / 2.0) * math.sqrt(2.0 / WM_BINS.size)


@lru_cache(maxsize=64)
def watermark_mark(key: int, message: int) -> np.ndarray:
    """The fp32 24 kHz pattern ``[12288]`` of ``(key, message)``: ``(c_0[t] + c_1[(t - 48 s1) mod 12288] +
    c_2[(t - 48 s2) mod 12288]) / sqrt(3)`` in fp64, rounded once."""
    d = WM_PERIOD_24K // WM_SYMBOLS
    c = (watermark_pattern(key, 0, WM_PERIOD_24K) + np.roll(watermark_pattern(key, 1, WM_PERIOD_24K), (message & 255) * d)
         + np.roll(watermark_pattern(key, 2, WM_PERIOD_24K), (message >> 8) * d)) / math.sqrt(3.0)
    return c.astype(np.float32)


def watermark_spectra(key: int) -> np.ndarray:
    """fp32 ``[3, 1588, 2]``: ``e^{-j phi_i(k)}`` of the three patterns (the detector's table; the last row is 0)."""
    out = np.zeros((3, WM_BINS_LD, 2), dtype=np.float32)
    ph = watermark_phases(key)
    out[:, :WM_BINS.size, 0] = np.cos(ph)
    out[:, :WM_BINS.size, 1] = -np.sin(ph)
    return out


def watermark_twiddles() -> np.ndarray:
    """fp32 ``[2048, 2]``: ``(cos, -sin)(2 pi m / 4096)`` of the detector's FFT."""
    a = 2.0 * math.pi * np.arange(WM_PERIOD // 2, dtype=np.float64) / WM_PERIOD
    return np.stack([np.cos(a), -np.sin(a)], 1).astype(np.float32)


_WM_TABLES: Dict[tuple, torch.Tensor] = {}


def _wm_table(name, args, device, make):
    device = torch.device(device)
    k = (name, args, device)
    t = _WM_TABLES.get(k)
    if t is None:
        if len(_WM_TABLES) >= 256:
            _WM_TABLES.clear()
        t = torch.from_numpy(np.ascontiguousarray(make())).to(device)
        _WM_TABLES[k] = t
    return t


def _int_in(v, lo, hi, what):
    if isinstance(v, bool) or not isinstance(v, (int, np.integer)) or not lo <= int(v) < hi:
        raise ValueError(f"{what}: expected an integer in [{lo}, {hi}), got {v!r}")
    return int(v)


@dataclass(frozen=True)
class Watermark:
    """A keyed watermark for synthesis: 64-bit secret ``key``, 16-bit ``message`` (e.g. a deployment or model-version
    id) and ``strength_db``, the mark's power relative to the speech (-40 to -15 dB, default -30).  Validated on
    construction (``ValueError``)."""
    key: int
    message: int = 0
    strength_db: float = -30.0

    def __post_init__(self):
        object.__setattr__(self, "key", _int_in(self.key, 0, 1 << 64, "Watermark.key"))
        object.__setattr__(self, "message", _int_in(self.message, 0, 1 << 16, "Watermark.message"))
        v = self.strength_db
        if isinstance(v, bool) or not isinstance(v, (int, float, np.integer, np.floating)) or \
                not math.isfinite(float(v)) or not -40.0 <= float(v) <= -15.0:
            raise ValueError(f"Watermark.strength_db: expected a number in [-40, -15], got {v!r}")
        object.__setattr__(self, "strength_db", float(v))

    @property
    def alpha(self) -> float:
        return 10.0 ** (self.strength_db / 20.0)

    def device_pattern(self, device) -> torch.Tensor:
        """``watermark_mark(key, message)`` on ``device`` (cached per key, message and device)."""
        return _wm_table("mark", (self.key, self.message), device, lambda: watermark_mark(self.key, self.message))


def detector_tables(key: int, device) -> Tuple[torch.Tensor, torch.Tensor]:
    """(pattern spectra, twiddles) of ``key`` on ``device`` (cached)."""
    key = _int_in(key, 0, 1 << 64, "key")
    return (_wm_table("spectra", key, device, lambda: watermark_spectra(key)),
            _wm_table("twiddles", None, device, watermark_twiddles))


def check_watermark(watermark, pcm16: bool):
    """Validate a ``watermark=`` argument: None or a ``Watermark``; with ``pcm16=True`` a ``ValueError`` (the mark is
    added to the fp32 waveform)."""
    if watermark is None:
        return None
    if not isinstance(watermark, Watermark):
        raise ValueError(f"watermark: expected a Watermark, got {type(watermark).__name__}")
    if pcm16:
        raise ValueError("watermark= and pcm16=True: the mark is added to the fp32 waveform; use "
                         "Synthesizer(pcm16=False) with audio=AudioFormat(24000, 'pcm16')")
    return watermark


class ToDetectionRate(AudioFormat):
    """The detector's resampler: ``sample_rate`` Hz to 8 kHz fp32 with ``resample_poly``'s filter for ``8000 / rate``
    (``_design``), run by ``as_resample_encode``.  A rate whose filter does not fit the kernel is a ``ValueError``."""

    @property
    def up(self) -> int:
        return WM_RATE // math.gcd(self.sample_rate, WM_RATE)

    @property
    def down(self) -> int:
        return self.sample_rate // math.gcd(self.sample_rate, WM_RATE)


class ToNativeRate(AudioFormat):
    """The enrollment resampler: ``sample_rate`` Hz to the model's 24 kHz fp32 with ``resample_poly``'s filter for
    ``24000 / rate`` (``_design``), run by ``as_resample_encode``.  A rate whose filter does not fit the kernel is a
    ``ValueError``.  This is not librosa's default resampler (``soxr_hq``): the two differ in the transition band near
    12 kHz, which the top mel filters see."""

    @property
    def up(self) -> int:
        return NATIVE_RATE // math.gcd(self.sample_rate, NATIVE_RATE)

    @property
    def down(self) -> int:
        return self.sample_rate // math.gcd(self.sample_rate, NATIVE_RATE)


def to_native_rate(sample_rate) -> ToNativeRate:
    if not _rate_ok_any(sample_rate):
        raise ValueError(f"sample_rate must be a positive integer, got {sample_rate!r}")
    try:
        return ToNativeRate(int(sample_rate), "float32")
    except ValueError as e:
        raise ValueError(f"cannot resample {sample_rate!r} Hz to 24 kHz: {e}") from None


def to_detection_rate(sample_rate: int) -> ToDetectionRate:
    try:
        return ToDetectionRate(sample_rate, "float32")
    except ValueError as e:
        raise ValueError(f"detect_watermark: cannot resample {sample_rate!r} Hz to 8 kHz: {e}") from None


def embed_watermark(wav: torch.Tensor, lengths, wm: Watermark) -> torch.Tensor:
    """Marked copy of 24 kHz fp32 waveforms ``wav`` ([B, S] or [S], CUDA), as stated in this module's docstring;
    ``lengths``: per-row sample counts (int tensor or sequence; None: every row holds S samples).  Samples beyond a
    row's length are 0."""
    from . import ops
    if not isinstance(wm, Watermark):
        raise ValueError(f"embed_watermark: expected a Watermark, got {type(wm).__name__}")
    x = wav.view(1, -1) if wav.dim() == 1 else wav
    if lengths is not None:
        lengths = torch.as_tensor(lengths).to(device=x.device, dtype=torch.int32).contiguous()
    y = ops.watermark_embed(x, lengths, wm)
    return y.view(-1) if wav.dim() == 1 else y


def detect_watermark(x: torch.Tensor, lengths, sample_rate: int, key: int, encoding: str = "float32",
                     threshold: float = WM_THRESHOLD):
    """``(detected bool, score fp32, message int32)`` device tensors ``[B]`` of the audio ``x`` ([B, S] or [S], CUDA;
    fp32, int16 or uint8 for ``encoding`` float32, pcm16, mulaw / alaw) at ``sample_rate`` Hz, for ``key``.  The
    samples are decoded to fp32 (``ops.audio_decode``), resampled to 8 kHz (``ToDetectionRate``) and detected
    (``ops.watermark_detect``), as stated in this module's docstring; no host synchronisation."""
    from . import ops
    if encoding not in ENCODINGS:
        raise ValueError(f"detect_watermark: encoding must be one of {ENCODINGS}, got {encoding!r}")
    if not _rate_ok_any(sample_rate):
        raise ValueError(f"detect_watermark: sample_rate must be a positive integer, got {sample_rate!r}")
    key = _int_in(key, 0, 1 << 64, "detect_watermark: key")
    if isinstance(threshold, bool) or not isinstance(threshold, (int, float)) or not math.isfinite(threshold):
        raise ValueError(f"detect_watermark: threshold must be a finite number, got {threshold!r}")
    rs = to_detection_rate(int(sample_rate))
    x = x.view(1, -1) if x.dim() == 1 else x
    if x.dtype != DTYPES[encoding]:
        raise ValueError(f"detect_watermark: {encoding} samples must be {DTYPES[encoding]}, got {x.dtype}")
    if lengths is not None:
        lengths = torch.as_tensor(lengths).to(device=x.device, dtype=torch.int32).contiguous()
    if encoding != "float32":
        x = ops.audio_decode(x, encoding)
    if not rs.is_identity:
        n8 = torch.empty(x.shape[0], dtype=torch.int32, device=x.device)
        x = ops.resample_encode(x, lengths, rs, rs.out_samples(x.shape[1]), out_lens=n8)
        lengths = n8
    detected, score, _, message = ops.watermark_detect(x, lengths, key, float(threshold))
    return detected, score, message


def _rate_ok_any(fs) -> bool:
    return not isinstance(fs, bool) and isinstance(fs, (int, np.integer)) and fs > 0
