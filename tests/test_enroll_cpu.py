"""Voice enrollment without a GPU: the two fp64 trim restatements against each other and on hand-derivable cases,
the ``ToNativeRate`` filter against scipy, input validation, and the host logic of ``reference_mels`` / ``enroll``
with semantic models of the new ops."""
import math
import types

import numpy as np
import pytest
import scipy.signal as ss
import torch

from artspeech_b200 import audio, engine, frontend, ops
from oracle import frontend_oracle as fo
from tests import audio_ref
from tests import enroll_ref as R

MARGIN = 1e-9
RATES = (8000, 11025, 12000, 16000, 22050, 32000, 44100, 48000, 88200, 96000, 192000)


def test_trim_restatements_agree_on_the_clip_set():
    clips = R.clip_set()
    excluded, trimmed = 0, 0
    for i, y in enumerate(clips):
        b, ambiguous = R.trim_blocks(y, 30.0, MARGIN)
        if ambiguous:
            excluded += 1
            continue
        assert R.trim_librosa(y, 30.0) == b, (i, y.size)
        trimmed += b != (0, y.size)
    assert excluded <= 1, excluded
    assert trimmed >= len(clips) // 2, trimmed                # the set exercises the trim, not just (0, n)
    assert [y.size for y in clips[:len(R.EDGE_LENGTHS)]] == list(R.EDGE_LENGTHS)


@pytest.mark.parametrize("trim", [R.trim_librosa, lambda y, t: R.trim_blocks(y, t)[0]])
def test_trim_hand_cases(trim):
    n = 512 * 50
    y = np.zeros(n, np.float32)
    y[512 * 10:512 * 30] = 0.5                                 # a burst over blocks 10 .. 29
    # frames 9 .. 31 overlap the burst (frame f covers blocks f-2 .. f+1); frame 9 holds one block of four, -6 dB
    assert trim(y, 30.0) == (512 * 9, 512 * 32)
    assert trim(np.zeros(n, np.float32), 30.0) == (0, n)      # digital silence is kept whole, as librosa does
    tone = (0.3 * np.sin(0.05 * np.arange(n))).astype(np.float32)
    assert trim(tone, 30.0) == (0, n)
    assert trim(tone[:700], 30.0) == (0, 700)                 # one frame
    assert trim(tone[:1], 30.0) == (0, 1)
    assert trim(np.zeros(0, np.float32), 30.0) == (0, 0)
    quiet = y * np.float32(10 ** (-70 / 20))
    quiet[512 * 40] = 0.5                                     # one click in block 40, 37 dB above the burst's frames
    assert trim(quiet, 30.0) == (512 * 39, 512 * 43)


def test_native_rate_filter_is_resample_polys():
    rng = np.random.default_rng(1)
    x = rng.standard_normal(4000)
    for fs in RATES + (24000,):
        r = audio.to_native_rate(fs)
        assert r.out_samples(fs) == 24000
        if r.is_identity:
            continue
        mx = max(r.up, r.down)
        h = ss.firwin(2 * 10 * mx + 1, 1.0 / mx, window=("kaiser", 5.0)) * r.up
        assert np.abs(r.filter64() - h).max() <= 1e-15 * r.up, fs
        y = audio_ref.resample64(x, r.filter64(), r.up, r.down, r.half_len)[0]
        assert np.abs(y - ss.resample_poly(x, r.up, r.down)).max() <= 1e-12, fs
        assert audio.smem_bytes(r.up, r.down, r.K, r.table_ld) <= audio.SMEM_MAX
    assert max(audio.smem_bytes(r.up, r.down, r.K, r.table_ld) for r in map(audio.to_native_rate, RATES)) == 38176
    for fs in (7999, 44101, 0, -8000, 8000.0, True, "8000"):
        with pytest.raises(ValueError):
            audio.to_native_rate(fs)


def test_validation():
    x = torch.zeros(2, 3000)
    bad = [dict(encoding="mp3"), dict(encoding="pcm16"), dict(x=torch.zeros(2, 3000, 9)),
           dict(x=torch.zeros(2, 3000, 0)), dict(lengths=[-1, 5]), dict(lengths=[3001, 5]), dict(lengths=[5]),
           dict(lengths=[1.5, 2]), dict(top_db=0.0), dict(top_db=-3.0), dict(top_db=math.inf), dict(top_db=math.nan),
           dict(top_db=True), dict(top_db="30"), dict(sample_rate=True), dict(sample_rate=0), dict(sample_rate=16000.0),
           dict(sample_rate=44101), dict(x=torch.zeros(3000)), dict(x=torch.zeros(2, 3000, dtype=torch.int16))]
    for kw in bad:
        args = dict(x=x, lengths=[3000, 2000], sample_rate=16000, encoding="float32", top_db=30.0, device="cpu")
        args.update(kw)
        with pytest.raises(ValueError):
            frontend.reference_mels(**args)
    with pytest.raises(ValueError):
        frontend.trim_bounds(torch.zeros(2, 100), None, None)


# ---- host logic with semantic models --------------------------------------------------------------------------
class _Models:
    """Torch / numpy models of the new ops on the CPU, recording the launch sequence and the read-backs."""

    def __init__(self, monkeypatch):
        self.calls = []
        me = self

        def to_mono(x, lens, encoding):
            me.calls.append("audio_to_mono")
            B, S = x.shape[:2]
            out = torch.zeros(B, S)
            for b in range(B):
                n = int(lens[b])
                xb = x[b, :n].numpy()
                out[b, :n] = torch.from_numpy(R.to_mono(xb, encoding))
            return out

        def resample(x, lens, fmt, S_out, **kw):
            me.calls.append("resample_encode")
            return audio_ref.resample_encode_model(x, lens, fmt, S_out, **kw)

        def trim(y, lens, top_db):
            me.calls.append("trim_bounds")
            return torch.tensor([R.trim_blocks(y[b, :int(lens[b])].numpy(), top_db)[0] for b in range(y.shape[0])],
                                dtype=torch.int32).view(-1, 2)

        def log_mel(mod, wave, lengths=None, starts=None, n_frames=None):
            me.calls.append("log_mel_span")
            out = torch.zeros(wave.shape[0], 80, n_frames)
            for b in range(wave.shape[0]):
                s, n = int(starts[b]), int(lengths[b])
                m = fo.log_mel(wave[b, s:s + n].clone())[0]
                out[b, :, :m.shape[1]] = m
            return out

        real_read_back = frontend._read_back

        def read_back(t):
            me.calls.append("read_back")
            return real_read_back(t)
        monkeypatch.setattr(ops, "audio_to_mono", to_mono)
        monkeypatch.setattr(ops, "resample_encode", resample)
        monkeypatch.setattr(ops, "trim_bounds", trim)
        monkeypatch.setattr(frontend.LogMel, "forward", log_mel)
        monkeypatch.setattr(frontend, "_read_back", read_back)


def _clip(rng, n, lead, trail, C=1):
    y = np.zeros((n, C), np.float32)
    k = np.arange(n - lead - trail)
    for c in range(C):
        y[lead:n - trail, c] = 0.3 * np.sin(0.07 * (c + 1) * k)
    return y


@pytest.mark.parametrize("rate,encoding,C", [(8000, "mulaw", 1), (16000, "pcm16", 1), (44100, "pcm16", 2),
                                             (24000, "float32", 1), (48000, "float32", 2), (24000, "alaw", 1)])
def test_reference_mels_host_logic(monkeypatch, rate, encoding, C):
    m = _Models(monkeypatch)
    rng = np.random.default_rng(rate)
    lens = [rate // 2, rate // 3]
    S = max(lens) + 37
    x = np.zeros((2, S, C), np.float32)
    for b, n in enumerate(lens):
        x[b, :n] = _clip(rng, n, n // 4, n // 3, C)
    if encoding == "float32":
        xt = torch.from_numpy(x)
    else:
        s = np.clip(np.rint(32767 * x), -32768, 32767).astype(np.int64)
        if encoding == "pcm16":
            xt = torch.from_numpy(s.astype(np.int16))
        else:
            xt = torch.from_numpy((audio_ref.ULAW if encoding == "mulaw" else audio_ref.ALAW)[s + 32768])
    if C == 1:
        xt = xt[..., 0].contiguous()
    mels, mel_lens, bounds = frontend.reference_mels(xt, lens, rate, encoding, device="cpu")
    want = (["audio_to_mono"] if encoding != "float32" or C > 1 else []) + \
        (["resample_encode"] if rate != 24000 else []) + ["trim_bounds", "read_back", "log_mel_span"]
    assert m.calls == want
    assert len(want) - 1 <= 5
    assert mel_lens.dtype == torch.int64 and not mel_lens.is_cuda
    fmt = audio.to_native_rate(rate)
    for b, n in enumerate(lens):
        y = R.to_mono(xt[b, :n].numpy(), encoding)
        y24 = audio_ref.resample64(y, fmt.filter64(), fmt.up, fmt.down, fmt.half_len)[0] if rate != 24000 else y
        st, en = R.trim_blocks(y24, 30.0)[0]
        assert (int(bounds[b, 0]), int(bounds[b, 1])) == (st, en)
        assert 0 < st and en < fmt.out_samples(n)              # the silence was cut at both ends
        assert int(mel_lens[b]) == 1 + (en - st) // 300
    assert mels.shape == (2, 80, int(mel_lens.max()))
    b = int(mel_lens.argmin())
    assert float(mels[b, :, int(mel_lens[b]):].abs().max()) == 0.0


def test_reference_mels_without_trim_and_short_rows(monkeypatch):
    m = _Models(monkeypatch)
    x = torch.from_numpy(_clip(None, 6000, 2000, 2000)[:, 0]).view(1, -1)
    mels, mel_lens, bounds = frontend.reference_mels(x, None, 24000, top_db=None, device="cpu")
    assert m.calls == ["log_mel_span"] and bounds.tolist() == [[0, 6000]] and mel_lens.tolist() == [21]
    m.calls.clear()
    x = torch.zeros(3, 4000)
    x[0, :4000] = 0.1
    x[1, 1000:1900] = 0.5                                     # trimmed to 2048 samples: fine
    x[2, 3950:] = 0.5                                         # frames 6 and 7: (3072, 4000), too short
    with pytest.raises(ValueError, match=r"rows \[2\]"):
        frontend.reference_mels(x, [4000, 4000, 4000], 24000, device="cpu")
    assert m.calls == ["trim_bounds", "read_back"]
    with pytest.raises(ValueError, match=r"rows \[0\]"):
        frontend.reference_mels(x, [1000, 4000, 4000], 24000, top_db=None, device="cpu")


def test_enroll_is_reference_mels_then_encode_voice(monkeypatch):
    m = _Models(monkeypatch)
    seen = []
    syn = types.SimpleNamespace(device=torch.device("cpu"),
                                encode_voice=lambda mels, ml: seen.append((mels, ml)) or "voice")
    x = torch.from_numpy(_clip(None, 16000, 3000, 3000)[:, 0]).view(1, -1)
    mels, mel_lens, voice = engine.Synthesizer.enroll(syn, x, [16000], 16000)
    assert voice == "voice" and seen[0][0] is mels and seen[0][1] is mel_lens
    assert m.calls == ["resample_encode", "trim_bounds", "read_back", "log_mel_span"]
