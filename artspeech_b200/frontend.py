"""Log-mel front-end on the GPU — drop-in for the reference's ``to_mel`` / ``preprocess``
(``test.py:40-47``, ``meldataset.py:42-49``): ``torchaudio.transforms.MelSpectrogram(n_mels=80,
n_fft=2048, win_length=1200, hop_length=300)`` followed by ``(log(1e-5 + mel) + 4) / 4``.

The transform's constants (periodic Hann window zero-padded to ``n_fft``, HTK triangular filterbank with
torchaudio's default ``sample_rate=16000`` — the reference never passes its 24 kHz rate, which is kept for
checkpoint compatibility — and the FFT twiddles) are computed once on the host; the arithmetic is one
launch of ``as_log_mel`` (``csrc/frontend.cu``) for a whole batch of recordings.

**Voice enrollment from recordings** (``reference_mels``, ``Synthesizer.enroll``): what the reference does to a
reference recording before that log-mel (``test.py:100-108``: ``librosa.load(path, sr=24000)``,
``librosa.effects.trim(wave, top_db=30)``, ``preprocess``), on the GPU.  Input: a batch of B recordings, ``x`` ``[B, S]``
(mono) or ``[B, S, C]`` (C interleaved channels, 1 <= C <= 8); ``lengths[b] <= S`` samples per channel at
``sample_rate`` Hz; ``encoding`` ``float32``, ``pcm16``, ``mulaw`` or ``alaw`` (the dtypes of ``audio.DTYPES``).

1. **Decode and downmix** (``as_audio_to_mono``).  Each sample is decoded as ``audio.detect_watermark`` decodes
   (``v / 32768``, or ``audioop.ulaw2lin`` / ``alaw2lin`` then ``/ 32768``), then ``m[t] = (x_0[t] + ... +
   x_{C-1}[t]) / C``: an fp32 sum in channel order and one fp32 divide, numpy's float32 ``mean(axis=0)`` that
   librosa's ``to_mono`` uses.  fp32 mono input takes no launch.
2. **Resample to 24 kHz** (``audio.ToNativeRate``, ``as_resample_encode``).  ``resample_poly``'s filter for
   ``24000 / rate``; ``n24 = ceil(n up / down)`` samples.  24 kHz takes no launch; a rate whose filter does not fit
   the kernel is a ``ValueError`` (8, 11.025, 12, 16, 22.05, 32, 44.1, 48, 88.2, 96 and 192 kHz fit).  This is not
   librosa's resampler (``soxr_hq``): the two differ in the transition band near 12 kHz, which the top mel filters see.

2b. **Noise reduction** (``as_denoise``; ``noise_reduction_db``, default ``None``: no stage, exactly the launches and
   bits of the chain without it; the standalone stage is ``denoise``).  A stationary-noise spectral suppressor on each
   whole 24 kHz row ``y[0 .. n)``, before the trim, so that the leading and trailing noise informs the noise estimate;
   the trim and the log-mel then read the denoised row.  With ``reduction_db`` in [0, 60]:

   1. STFT: N = 512, hop 128, periodic Hann window ``w``; frame ``f < F = 1 + n // 128`` holds ``w[i] y[128 f - 256 +
      i]`` with zeros outside ``[0, n)``, and ``X[f, k]`` is its 257-bin real FFT (``torch.stft(center=True,
      pad_mode="constant", onesided=True)``).
   2. Power ``P = re^2 + im^2`` in fp32, two rounded products and one rounded add.
   3. Noise profile (stationary, from the whole recording): ``lambda[k] = max(1e-20, P_(r)[k] / c)`` in fp64, where
      ``P_(r)[k]`` is the ``r``-th smallest (0-based) of ``P[0 .. F), k]``, ``r = F // 10``, and ``c = -log1p(-0.1)``
      is the 10 % quantile of an exponential with mean 1: for Gaussian noise, ``lambda`` estimates the noise PSD
      without bias.
   4. Decision-directed Wiener gain (Ephraim-Malah), fp64, ``alpha = 0.98``: ``gamma = P / lambda``, ``xi_0 =
      max(gamma_0 - 1, 0)``, ``xi_f = alpha A_{f-1} + (1 - alpha) max(gamma_f - 1, 0)``, ``W_f = xi_f / (1 + xi_f)``,
      ``A_f = W_f W_f gamma_f``, ``G_f = max(W_f, g_min)`` stored as fp32, ``g_min = 10^(-reduction_db / 20)``.  The
      host computes ``c``, ``g_min``, ``alpha`` and ``1 - alpha`` in fp64; the kernel evaluates each operation rounded
      once in this order, so ``G`` is bit-equal to a numpy float64 model fed the kernel's ``P``.
   5. Synthesis: ``y'[t] = sum_f w[j] irfft(G_f X_f)[j] / sum_f w[j]^2``, ``j = t - 128 f + 256``, over the frames
      covering ``t`` in ascending ``f`` (``torch.istft(length=n)``); zeros beyond ``n``.  At ``reduction_db = 0``,
      ``g_min = 1`` and this is the STFT round trip.

   A row's output depends only on its own samples, bit for bit.  Digital silence stays silence.  A recording whose
   quietest tenth of frames is digital silence is left almost unchanged (``lambda`` is at its floor).  Non-stationary
   noise (babble, music) is not tracked.  Three launches, no read-back.
3. **Trim** (``as_trim_bounds``; ``top_db``, default 30, ``None`` for no trim).  librosa 0.10's ``effects.trim``
   with its defaults (frame 2048, hop 512), evaluated at 24 kHz in fp64: ``q_j`` is the sum of ``y^2`` over block
   ``[512 j, 512 j + 512)`` (zeros at and beyond ``n``); frame ``f < F = 1 + n // 512`` has the power
   ``p_f = (q_{f-2} + q_{f-1} + q_f + q_{f+1}) / 2048`` (blocks out of range count 0: ``feature.rms(center=True,
   pad_mode="constant")`` squared); ``P = max_f p_f``; frame ``f`` is non-silent iff ``10 log10(max(1e-10, p_f)) -
   10 log10(max(1e-10, P)) > -top_db`` (``amplitude_to_db(ref=np.max, amin=1e-5)``); ``start = 512 first``,
   ``end = min(n, 512 (last + 1))``, and ``(0, 0)`` for ``n = 0``.  As in librosa, digital silence is entirely
   non-silent and keeps ``(0, n)``.  The one known difference: librosa sums in fp32, so a frame within about 1e-6 dB
   of the threshold can be decided differently.
4. **Log-mel of the span** (``as_log_mel_span``).  Exactly ``LogMel`` of ``y[start:end]``, reflect-padded at the
   span's own ends: ``1 + L // 300`` frames for ``L = end - start``.  A row with ``L <= 1024`` is a ``ValueError``
   naming the row (``torch.stft``'s reflect padding, and so the reference, cannot take it).

Outputs: ``mels`` fp32 ``[B, 80, T_max]`` with zeros beyond each row's frames, ``mel_lens`` int64 ``[B]`` on the host
(what ``synthesize`` / ``encode_voice`` take), ``bounds`` int32 ``[B, 2]`` on the device, ``(start, end)`` in 24 kHz
samples.  A row's outputs depend only on its own samples, bit for bit: not on the batch, the padding or the row
stride.  The call makes at most five launches, eight with noise reduction, and one device-to-host read-back (the B
bounds, into pinned memory, between the trim and the log-mel: it sizes ``T_max`` and finds short rows).  Container
formats (WAV, FLAC, MP3 headers) are the caller's: it hands over sample arrays.
"""
from __future__ import annotations

import math
import numbers
from typing import Optional, Sequence, Union

import numpy as np
import torch
import torch.nn as nn

from . import _lib, audio, ops

N_FFT, WIN_LENGTH, HOP_LENGTH, N_MELS = 2048, 1200, 300, 80
LOG_EPS, MEAN, STD = 1e-5, -4.0, 4.0


def hann_window_padded(n_fft: int = N_FFT, win_length: int = WIN_LENGTH) -> torch.Tensor:
    w = torch.hann_window(win_length, periodic=True, dtype=torch.float64)
    out = torch.zeros(n_fft, dtype=torch.float64)
    left = (n_fft - win_length) // 2
    out[left:left + win_length] = w
    return out.float()


def htk_filterbank(n_freqs: int, n_mels: int, sample_rate: int = 16000) -> torch.Tensor:
    """Triangular HTK mel filters without normalisation, ``[n_freqs, n_mels]`` (f_min 0, f_max sample_rate/2)."""
    freqs = torch.linspace(0, sample_rate // 2, n_freqs)
    to_mel = lambda f: 2595.0 * math.log10(1.0 + f / 700.0)
    m_pts = torch.linspace(to_mel(0.0), to_mel(sample_rate / 2.0), n_mels + 2)
    f_pts = 700.0 * (10.0 ** (m_pts / 2595.0) - 1.0)
    f_diff = f_pts[1:] - f_pts[:-1]
    slopes = f_pts.unsqueeze(0) - freqs.unsqueeze(1)
    down = (-1.0 * slopes[:, :-2]) / f_diff[:-1]
    up = slopes[:, 2:] / f_diff[1:]
    return torch.clamp(torch.min(down, up), min=0.0)


def filter_ranges(fb: torch.Tensor) -> torch.Tensor:
    """int32 ``[n_mels, 2]``: first bin and number of bins with a non-zero weight per filter."""
    out = torch.zeros(fb.shape[1], 2, dtype=torch.int32)
    for m in range(fb.shape[1]):
        nz = torch.nonzero(fb[:, m] > 0).flatten()
        if nz.numel():
            out[m, 0] = int(nz[0])
            out[m, 1] = int(nz[-1]) - int(nz[0]) + 1
    return out


class LogMel(nn.Module):
    """``forward(wave [B, N] fp32 CUDA, lengths=None) -> [B, 80, 1 + N // 300]`` normalised log-mel.

    ``starts=`` (int32 [B] device, with ``lengths``) takes recording ``b`` as the ``lengths[b]`` samples from
    ``wave[b, starts[b]]`` (``as_log_mel_span``), with the bits ``LogMel`` gives for those samples copied to the start
    of a row; ``n_frames`` then sets the output's frame count (default ``1 + N // 300``)."""

    def __init__(self, n_mels: int = N_MELS, n_fft: int = N_FFT, win_length: int = WIN_LENGTH,
                 hop_length: int = HOP_LENGTH, mean: float = MEAN, std: float = STD):
        super().__init__()
        if n_fft != 2048:
            raise NotImplementedError("as_log_mel implements the reference's n_fft = 2048")
        self.n_mels, self.n_fft, self.hop_length, self.mean, self.std = n_mels, n_fft, hop_length, mean, std
        fb = htk_filterbank(n_fft // 2 + 1, n_mels)
        k = np.arange(n_fft // 2, dtype=np.float64)
        tw = np.stack([np.cos(2 * np.pi * k / n_fft), -np.sin(2 * np.pi * k / n_fft)], axis=1)
        self.register_buffer("window", hann_window_padded(n_fft, win_length), persistent=False)
        self.register_buffer("fb", fb.contiguous(), persistent=False)
        self.register_buffer("fb_range", filter_ranges(fb), persistent=False)
        self.register_buffer("twiddle", torch.from_numpy(tw.astype(np.float32)).contiguous(), persistent=False)

    @torch.no_grad()
    def forward(self, wave: torch.Tensor, lengths: Optional[torch.Tensor] = None,
                starts: Optional[torch.Tensor] = None, n_frames: Optional[int] = None) -> torch.Tensor:
        ops._require_cuda(wave, "log_mel")
        if wave.dim() == 1:
            wave = wave.unsqueeze(0)
        wave = wave.float()
        if wave.stride(-1) != 1:
            wave = wave.contiguous()
        B, N = wave.shape
        if n_frames is None:
            n_frames = 1 + N // self.hop_length
        out = torch.empty(B, self.n_mels, n_frames, dtype=torch.float32, device=wave.device)
        lens = None if lengths is None else lengths.to(device=wave.device, dtype=torch.int32).contiguous()
        consts = (self.window.data_ptr(), self.twiddle.data_ptr(), self.fb.data_ptr(), self.fb_range.data_ptr(),
                  self.n_fft, self.hop_length, self.n_mels, float(LOG_EPS), float(self.mean), float(self.std),
                  out.data_ptr(), n_frames)
        if starts is None:
            ops._run("as_log_mel", wave, wave.data_ptr(), wave.stride(0), ops._p(lens), B, N, *consts)
        else:
            if lens is None:
                raise ValueError("LogMel: starts= needs lengths")
            st = starts.to(device=wave.device, dtype=torch.int32).contiguous()
            ops._run("as_log_mel_span", wave, wave.data_ptr(), wave.stride(0), st.data_ptr(), lens.data_ptr(), B, N,
                     *consts)
        return out


_default = {}


def preprocess(wave, device="cuda") -> torch.Tensor:
    """The reference's ``preprocess(wave)`` (test.py:43-47): numpy / tensor ``[N]`` -> ``[1, 80, T]`` on ``device``."""
    dev = torch.device(device)
    if dev not in _default:
        _default[dev] = LogMel().to(dev)
    w = torch.from_numpy(wave) if isinstance(wave, np.ndarray) else wave
    return _default[dev](w.to(dev))


# ---- voice enrollment from recordings -----------------------------------------------------------------------------
MIN_SPAN = N_FFT // 2            # a trimmed span must be longer than this (reflect padding of the first frame)


def _check_top_db(top_db):
    if top_db is None:
        return None
    if isinstance(top_db, bool) or not isinstance(top_db, numbers.Real) or not math.isfinite(float(top_db)) or \
            float(top_db) <= 0.0:
        raise ValueError(f"top_db must be a finite positive number or None, got {top_db!r}")
    return float(top_db)


def trim_bounds(wave: torch.Tensor, lengths=None, top_db: float = 30.0) -> torch.Tensor:
    """``(start, end)`` int32 ``[B, 2]`` device tensor of the non-silent span of each row of 24 kHz fp32 ``wave``
    (``[B, S]`` or ``[S]``, CUDA) as step 3 of this module's docstring states; ``lengths``: per-row sample counts (int
    tensor or sequence; None: every row holds S samples).  Two launches, no host synchronisation."""
    top_db = _check_top_db(top_db)
    if top_db is None:
        raise ValueError("trim_bounds: top_db must be a finite positive number")
    x = wave.view(1, -1) if wave.dim() == 1 else wave
    if lengths is not None:
        lengths = torch.as_tensor(lengths).to(device=x.device, dtype=torch.int32).contiguous()
    return ops.trim_bounds(x, lengths, top_db)


def _check_reduction_db(v, name="reduction_db"):
    if v is None:
        return None
    if isinstance(v, bool) or not isinstance(v, numbers.Real) or not math.isfinite(float(v)) or \
            not 0.0 <= float(v) <= 60.0:
        raise ValueError(f"{name} must be a finite number in [0, 60], got {v!r}")
    return float(v)


def denoise(wave: torch.Tensor, lengths=None, reduction_db: float = 18.0) -> torch.Tensor:
    """Stationary-noise suppression of 24 kHz fp32 ``wave`` (``[B, S]`` or ``[S]``, CUDA) as step 2b of this module's
    docstring states; ``lengths``: per-row sample counts (int tensor or sequence; None: every row holds S samples).
    Returns the denoised rows in ``wave``'s shape, zeros beyond each length: listen to them, or feed them to
    ``LogMel``.  Three launches, no host synchronisation."""
    reduction_db = _check_reduction_db(reduction_db)
    if reduction_db is None:
        raise ValueError("denoise: reduction_db must be a finite number in [0, 60]")
    ops._require_cuda(wave, "denoise")
    x = wave.unsqueeze(0) if wave.dim() == 1 else wave
    x = x.float()
    if x.stride(-1) != 1 and x.shape[-1] > 1:
        x = x.contiguous()
    if lengths is not None:
        lengths = torch.as_tensor(lengths).to(device=x.device, dtype=torch.int32).contiguous()
    out = ops.denoise(x, lengths, reduction_db)
    return out[0] if wave.dim() == 1 else out


def _read_back(t: torch.Tensor) -> torch.Tensor:
    """Host copy of a small device tensor through pinned memory: the one synchronisation of ``reference_mels``."""
    if not t.is_cuda:
        return t.clone()
    h = torch.empty(t.shape, dtype=t.dtype).pin_memory()
    h.copy_(t, non_blocking=True)
    torch.cuda.current_stream(t.device).synchronize()
    return h


def _host_lengths(lengths, B: int, S: int) -> torch.Tensor:
    if lengths is None:
        return torch.full((B,), S, dtype=torch.int64)
    if isinstance(lengths, torch.Tensor):
        if lengths.is_cuda:
            raise ValueError("lengths: expected a host tensor or sequence (reading a device tensor would synchronise)")
        if lengths.is_floating_point() or lengths.dtype == torch.bool:
            raise ValueError(f"lengths: expected integers, got {lengths.dtype}")
        L = lengths.to(torch.int64).flatten()
    else:
        vals = list(lengths)
        if any(isinstance(v, bool) or not isinstance(v, (numbers.Integral, np.integer)) for v in vals):
            raise ValueError(f"lengths: expected integers, got {vals!r}")
        L = torch.tensor([int(v) for v in vals], dtype=torch.int64)
    if L.numel() != B:
        raise ValueError(f"lengths: expected {B} values, got {L.numel()}")
    if B and (int(L.min()) < 0 or int(L.max()) > S):
        raise ValueError(f"lengths: every length must be in [0, {S}], got {L.tolist()}")
    return L


_enroll_logmel = {}


def reference_mels(x: torch.Tensor, lengths: Union[Sequence[int], torch.Tensor, None], sample_rate: int,
                   encoding: str = "float32", top_db: Optional[float] = 30.0, device=None,
                   noise_reduction_db: Optional[float] = None):
    """Reference mels of recordings, as this module's docstring states: ``x`` ``[B, S]`` or ``[B, S, C]`` (host or
    CUDA) of ``audio.DTYPES[encoding]`` at ``sample_rate`` Hz, ``lengths`` host samples per channel (None: S).
    Returns ``(mels fp32 [B, 80, T_max] device, mel_lens int64 [B] host, bounds int32 [B, 2] device)``.  ``device``:
    where to run when ``x`` is on the host (default ``cuda``).  ``noise_reduction_db``: None (no noise reduction) or
    the ``reduction_db`` of step 2b, in [0, 60].  At most five launches (eight with noise reduction), one read-back."""
    if encoding not in audio.ENCODINGS:
        raise ValueError(f"encoding must be one of {audio.ENCODINGS}, got {encoding!r}")
    rs = audio.to_native_rate(sample_rate)
    top_db = _check_top_db(top_db)
    noise_reduction_db = _check_reduction_db(noise_reduction_db, "noise_reduction_db")
    if not isinstance(x, torch.Tensor) or x.dim() not in (2, 3):
        raise ValueError(f"x: expected a [B, S] or [B, S, C] tensor, got {getattr(x, 'shape', type(x))}")
    if x.dtype != audio.DTYPES[encoding]:
        raise ValueError(f"x: {encoding} samples must be {audio.DTYPES[encoding]}, got {x.dtype}")
    B, S = x.shape[:2]
    C = x.shape[2] if x.dim() == 3 else 1
    if not 1 <= C <= 8:
        raise ValueError(f"x: 1 to 8 interleaved channels, got {C}")
    n = _host_lengths(lengths, B, S)
    dev = x.device if x.is_cuda else torch.device(device if device is not None else "cuda")
    if B == 0:
        return (torch.zeros(0, N_MELS, 0, device=dev), torch.zeros(0, dtype=torch.int64),
                torch.zeros(0, 2, dtype=torch.int32, device=dev))
    if not x.is_cuda:
        x = x.contiguous().to(dev, non_blocking=False)
    lens = n.to(torch.int32).to(dev)
    m = x if x.dim() == 2 else x[..., 0]
    if encoding != "float32" or C > 1:
        m = ops.audio_to_mono(x, lens, encoding)
    if rs.is_identity:
        y, n24, n24_host = m, lens, n
    else:
        n24 = torch.empty(B, dtype=torch.int32, device=dev)
        y = ops.resample_encode(m, lens, rs, rs.out_samples(S), out_lens=n24)
        n24_host = torch.tensor([rs.out_samples(int(v)) for v in n], dtype=torch.int64)
    if noise_reduction_db is not None:
        y = ops.denoise(y, n24, noise_reduction_db)
    if top_db is None:
        host = torch.stack([torch.zeros_like(n24_host), n24_host], 1).to(torch.int32)
        bounds = host.to(dev)
    else:
        bounds = ops.trim_bounds(y, n24, top_db)
        host = _read_back(bounds)
    span = (host[:, 1] - host[:, 0]).to(torch.int64)
    short = [b for b in range(B) if int(span[b]) <= MIN_SPAN]
    if short:
        raise ValueError(f"reference_mels: rows {short} keep {[int(span[b]) for b in short]} samples at 24 kHz after "
                         f"the trim; a log-mel needs more than {MIN_SPAN}")
    mel_lens = 1 + span // HOP_LENGTH
    starts_lens = torch.stack([host[:, 0], span.to(torch.int32)]).to(dev)
    if dev not in _enroll_logmel:
        _enroll_logmel[dev] = LogMel().to(dev)
    mels = _enroll_logmel[dev](y, starts_lens[1], starts=starts_lens[0], n_frames=int(mel_lens.max()))
    return mels, mel_lens, bounds
