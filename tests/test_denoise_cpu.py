"""Noise reduction for voice enrollment without a GPU: the fp64 restatement against ``torch.stft`` / ``torch.istft``,
the noise profile of white noise, hand cases of the gain, the quality of the stage on voiced speech in white, pink and
mains-hum noise, input validation, and the host logic of ``reference_mels`` / ``enroll`` with semantic models."""
import math
import types

import numpy as np
import pytest
import torch

from artspeech_b200 import audio, engine, frontend, ops
from oracle import frontend_oracle as fo
from tests import audio_ref
from tests import denoise_ref as D
from tests import enroll_ref as R
from tests.test_enroll_cpu import _clip, _Models


def _torch_stft(y):
    w = torch.hann_window(D.N, periodic=True, dtype=torch.float64)
    return torch.stft(torch.from_numpy(np.asarray(y, np.float64)), D.N, D.HOP, window=w, center=True,
                      pad_mode="constant", onesided=True, return_complex=True).T.numpy()


def _torch_istft(Y, n):
    w = torch.hann_window(D.N, periodic=True, dtype=torch.float64)
    return torch.istft(torch.from_numpy(Y.T.copy()), D.N, D.HOP, window=w, center=True, length=n).numpy()


@pytest.mark.parametrize("n", list(D.EDGE_LENGTHS) + [1000, 24000 + 77])
def test_framing_and_synthesis_are_torchs(n):
    rng = np.random.default_rng(n)
    y = rng.standard_normal(n)
    X = D.stft(y)
    assert X.shape == (D.n_frames(n), D.K)
    if n:
        Xt = _torch_stft(y)
        assert np.abs(X - Xt).max() <= 1e-12 * max(1.0, np.abs(Xt).max())
        Y = X * rng.uniform(0.0, 1.0, X.shape)                 # any gain: the synthesis is torch.istft
        assert np.abs(D.istft(Y, n) - _torch_istft(Y, n)).max() <= 1e-12
    out = D.denoise(y, 0.0)                                   # g_min = 1: the STFT round trip
    assert out.shape == (n,) and (n == 0 or np.abs(out - y).max() <= 1e-12)
    assert not D.denoise(np.zeros(n), 18.0).any()             # digital silence stays silence


def test_noise_profile_of_white_noise_is_its_psd():
    rng = np.random.default_rng(7)
    sigma = 0.01
    X = D.stft(rng.standard_normal(60 * D.FS) * sigma)
    lam = D.noise_profile(X.real ** 2 + X.imag ** 2)
    psd = sigma ** 2 * np.sum(D.window() ** 2)                # E|X[k]|^2 for 0 < k < 256
    err_db = 10 * math.log10(np.mean(lam[1:256]) / psd)
    assert abs(err_db) <= 0.5, err_db
    assert np.abs(10 * np.log10(lam[1:256] / psd)).max() <= 1.5   # and no bin is far off


def test_gain_hand_cases():
    P = np.array([[4.0, 0.0, 1.0], [4.0, 0.0, 1.0]])
    lam = np.array([1.0, 1e-20, 1.0])
    G = D.gains(P, lam, 20.0)
    assert G.dtype == np.float32 and G.shape == (2, 3)
    assert G[0, 0] == np.float32(0.75)                        # xi_0 = gamma - 1 = 3, W = 3 / 4
    A = 0.75 * 0.75 * 4.0
    xi = D.ALPHA * A + (1 - D.ALPHA) * 3.0
    assert G[1, 0] == np.float32(xi / (1 + xi))
    assert G[0, 1] == G[1, 1] == np.float32(0.1)              # no energy: g_min
    assert G[0, 2] == np.float32(0.1)                         # gamma = 1: xi = 0, W = 0
    assert np.array_equal(D.noise_profile(np.arange(25.0)[:, None]), [2.0 / D.C_Q])   # r = 25 // 10
    X = np.array([[3 + 4j, 1e-3 + 1e10j]], np.complex64)
    im2 = np.float32(1e10) * np.float32(1e10)
    assert D.power32(X).tolist() == [[25.0, float(np.float32(1e-3) * np.float32(1e-3) + im2)]]


# Measured with this module's generators, 16 voiced clips of 3-12 s at 18 dB reduction, fp64 reference (mean over
# clips; min SNR gain / max log-mel L1 ratio over clips in brackets):
#   noise  SNR in | SNR gain             | log-mel L1 noisy -> denoised     | trim error, mean
#   white   0 dB  | +10.3 (+9.27)        | 2.078 -> 1.399 (ratio <= 0.714)  | 1.95 -> 1.93 s
#   white  10 dB  |  +7.8 (+6.41)        | 1.614 -> 1.028 (<= 0.696)        | 1.95 -> 0.01 s
#   white  20 dB  |  +6.6 (+5.02)        | 1.204 -> 0.672 (<= 0.640)        | 1.36 -> 0.00 s
#   pink    0 dB  |  +7.0 (+4.65)        | 2.002 -> 1.333 (<= 0.706)        | 1.95 -> 1.94 s
#   pink   10 dB  |  +6.0 (+3.68)        | 1.537 -> 0.968 (<= 0.695)        | 1.95 -> 1.19 s
#   pink   20 dB  |  +5.1 (+2.82)        | 1.128 -> 0.604 (<= 0.626)        | 1.71 -> 0.00 s
#   hum     0 dB  |  +8.6 (+4.19)        | 0.484 -> 0.339 (<= 0.794)        | 1.95 -> 1.94 s
#   hum    10 dB  |  +7.9 (+3.21)        | 0.372 -> 0.239 (<= 0.726)        | 1.95 -> 0.00 s
#   hum    20 dB  |  +7.1 (+2.29)        | 0.277 -> 0.148 (<= 0.622)        | 1.33 -> 0.00 s
# The margins below are those numbers, rounded towards failure by a small step.
MARGINS = {  # (kind, snr): (min SNR gain dB, max log-mel L1 ratio)
    ("white", 0): (9.0, 0.74), ("white", 10): (6.0, 0.72), ("white", 20): (4.7, 0.67),
    ("pink", 0): (4.3, 0.73), ("pink", 10): (3.4, 0.72), ("pink", 20): (2.5, 0.65),
    ("hum", 0): (3.9, 0.82), ("hum", 10): (2.9, 0.75), ("hum", 20): (2.0, 0.65),
}


@pytest.fixture(scope="module")
def voiced_clips():
    return D.voiced_set(0, 16)


def _log_mel(y):
    return fo.log_mel(torch.from_numpy(np.ascontiguousarray(y, np.float32)))[0].double().numpy()


def _trim_error(bounds, clean_bounds):
    return (abs(bounds[0] - clean_bounds[0]) + abs(bounds[1] - clean_bounds[1])) / D.FS


@pytest.mark.parametrize("kind", ["white", "pink", "hum"])
def test_quality_on_voiced_speech(voiced_clips, kind):
    for snr in (0, 10, 20):
        min_gain, max_ratio = MARGINS[(kind, snr)]
        err_noisy, err_clean = [], []
        for i, c in enumerate(voiced_clips):
            x = D.mix(c, D.noise(np.random.default_rng(1000 + i), kind, c.size), snr)
            y = D.denoise(x, 18.0).astype(np.float32)
            gain = D.snr_db(c, y) - D.snr_db(c, x)
            assert gain >= min_gain, (kind, snr, i, gain)
            st, en = R.trim_blocks(c, 30.0)[0]
            ref = _log_mel(c[st:en])
            l1_noisy = np.mean(np.abs(_log_mel(x[st:en]) - ref))
            l1_denoised = np.mean(np.abs(_log_mel(y[st:en]) - ref))
            assert l1_denoised <= max_ratio * l1_noisy, (kind, snr, i, l1_noisy, l1_denoised)
            err_noisy.append(_trim_error(R.trim_blocks(x, 30.0)[0], (st, en)))
            err_clean.append(_trim_error(R.trim_blocks(y, 30.0)[0], (st, en)))
        if kind != "pink" and snr >= 10:                      # the trim bounds move to the clean clip's
            assert np.mean(err_noisy) >= 1.0 and np.mean(err_clean) <= 0.05, (kind, snr, err_noisy, err_clean)
            assert all(d <= e for d, e in zip(err_clean, err_noisy))


def test_validation():
    x = torch.zeros(2, 3000)
    for v in (math.nan, math.inf, -math.inf, -1.0, 60.5, True, False, "18", 1j):
        with pytest.raises(ValueError):
            frontend.reference_mels(x, [3000, 2000], 16000, device="cpu", noise_reduction_db=v)
        with pytest.raises(ValueError):
            frontend.denoise(x, None, v)
    with pytest.raises(ValueError):
        frontend.denoise(x, None, None)
    for v in (0, 0.0, 18, np.float64(60.0)):
        assert frontend._check_reduction_db(v) == float(v)


# ---- host logic with semantic models --------------------------------------------------------------------------
def _models(monkeypatch):
    m = _Models(monkeypatch)

    def denoise(y, lens, reduction_db, planes=False):
        m.calls.append("denoise")
        out = torch.zeros(y.shape)
        for b in range(y.shape[0]):
            n = int(lens[b]) if lens is not None else y.shape[1]
            out[b, :n] = torch.from_numpy(D.denoise(y[b, :n].numpy(), reduction_db).astype(np.float32))
        return out
    monkeypatch.setattr(ops, "denoise", denoise)
    return m


def _noisy(rng, n, lead, trail, C=1):
    y = _clip(rng, n, lead, trail, C)
    return (y + 0.01 * rng.standard_normal(y.shape)).astype(np.float32)


@pytest.mark.parametrize("rate,encoding,C", [(8000, "mulaw", 1), (16000, "pcm16", 1), (44100, "pcm16", 2),
                                             (24000, "float32", 1)])
def test_reference_mels_host_logic(monkeypatch, rate, encoding, C):
    m = _models(monkeypatch)
    rng = np.random.default_rng(rate)
    lens = [rate // 2, rate // 3]
    S = max(lens) + 37
    x = np.zeros((2, S, C), np.float32)
    for b, n in enumerate(lens):
        x[b, :n] = _noisy(rng, n, n // 4, n // 3, C)
    if encoding == "float32":
        xt = torch.from_numpy(x)
    else:
        s = np.clip(np.rint(32767 * x), -32768, 32767).astype(np.int64)
        xt = torch.from_numpy(s.astype(np.int16)) if encoding == "pcm16" else \
            torch.from_numpy(audio_ref.ULAW[s + 32768])
    if C == 1:
        xt = xt[..., 0].contiguous()
    base = (["audio_to_mono"] if encoding != "float32" or C > 1 else []) + \
        (["resample_encode"] if rate != 24000 else [])
    mels0, ml0, b0 = frontend.reference_mels(xt, lens, rate, encoding, device="cpu")
    assert m.calls == base + ["trim_bounds", "read_back", "log_mel_span"]
    m.calls.clear()
    mels, mel_lens, bounds = frontend.reference_mels(xt, lens, rate, encoding, device="cpu", noise_reduction_db=18)
    assert m.calls == base + ["denoise", "trim_bounds", "read_back", "log_mel_span"]
    assert m.calls.count("read_back") == 1
    fmt = audio.to_native_rate(rate)
    for b, n in enumerate(lens):
        y = R.to_mono(xt[b, :n].numpy(), encoding)
        y24 = audio_ref.resample64(y, fmt.filter64(), fmt.up, fmt.down, fmt.half_len)[0] if rate != 24000 else y
        y24 = D.denoise(np.asarray(y24, np.float32), 18.0).astype(np.float32)
        st, en = R.trim_blocks(y24, 30.0)[0]
        assert (int(bounds[b, 0]), int(bounds[b, 1])) == (st, en)
        assert int(mel_lens[b]) == 1 + (en - st) // 300
        ref = fo.log_mel(torch.from_numpy(y24[st:en].copy()))[0]
        assert (mels[b, :, :ref.shape[1]] - ref).abs().max().item() <= 1e-4
    assert mels.shape == (2, 80, int(mel_lens.max()))
    assert not torch.equal(mels0[:, :, :mels.shape[2]], mels[:, :, :mels0.shape[2]])


def test_enroll_passes_noise_reduction(monkeypatch):
    m = _models(monkeypatch)
    seen = []
    syn = types.SimpleNamespace(device=torch.device("cpu"),
                                encode_voice=lambda mels, ml: seen.append((mels, ml)) or "voice")
    x = torch.from_numpy(_noisy(np.random.default_rng(2), 16000, 3000, 3000)[:, 0]).view(1, -1)
    mels, mel_lens, voice = engine.Synthesizer.enroll(syn, x, [16000], 16000, noise_reduction_db=12.0)
    assert voice == "voice" and seen[0][0] is mels and seen[0][1] is mel_lens
    assert m.calls == ["resample_encode", "denoise", "trim_bounds", "read_back", "log_mel_span"]
    m.calls.clear()
    engine.Synthesizer.enroll(syn, x, [16000], 16000)
    assert m.calls == ["resample_encode", "trim_bounds", "read_back", "log_mel_span"]
