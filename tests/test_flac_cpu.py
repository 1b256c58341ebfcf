"""FLAC output without a GPU: the restatement (tests/flac_ref.py) against catalogue CRC values and a hand-derived file,
round trips through the separately written reader over edge lengths, full-scale signals and speech-like clips at every
delivery rate, the choice of every subframe kind, the size bound, the compression ratio, validation, and the engine's
host logic with a torch model of ``ops.flac_encode``."""
import types

import numpy as np
import pytest
import torch

from artspeech_b200 import audio, engine, ops
from artspeech_b200.audio import AudioFormat, Loudness, Watermark
from tests import audio_ref, denoise_ref, enroll_ref, loudness_ref
from tests import flac_ref as F

RATES = (8000, 12000, 16000, 22050, 24000, 44100, 48000)
LENGTHS = (0, 1, 15, 16, 17, 4095, 4096, 4097, 12293)


def test_crc_catalogue_values():
    assert F.crc8(b"123456789") == 0xF4                 # CRC-8/SMBUS
    assert F.crc16(b"123456789") == 0xFEE8              # CRC-16/UMTS


def test_sixteen_zero_samples_by_hand():
    """RFC 9639 field by field: the header, STREAMINFO and one 13-byte CONSTANT frame."""
    streaminfo = bytes([0x10, 0x00, 0x10, 0x00,          # min / max block size 4096
                        0x00, 0x00, 0x0D, 0x00, 0x00, 0x0D,   # min / max frame size 13
                        # 20-bit rate 24000 = 0x05DC0, 3-bit channels-1 = 0, 5-bit bps-1 = 15, 36-bit total 16
                        0x05, 0xDC, 0x00, 0xF0, 0x00, 0x00, 0x00, 0x10]) + bytes(16)   # MD5 not computed
    head = b"fLaC" + bytes([0x80, 0x00, 0x00, 0x22]) + streaminfo  # last block, type 0, length 34
    fh = bytes([0xFF, 0xF8,                              # sync, reserved 0, fixed block size
                0x77,                                    # block size 0b0111 (16-bit bs-1 follows), rate 0b0111 24 kHz
                0x08,                                    # channels 0b0000, 16 bits 0b100, reserved 0
                0x00,                                    # frame number 0
                0x00, 0x0F])                             # bs - 1 = 15
    crc8 = 0
    for b in fh:                                          # CRC-8, poly 0x07, bit by bit
        crc8 ^= b
        for _ in range(8):
            crc8 = ((crc8 << 1) ^ 0x07) & 0xFF if crc8 & 0x80 else (crc8 << 1) & 0xFF
    frame = fh + bytes([crc8, 0x00, 0x00, 0x00])          # subframe: pad 0, CONSTANT 000000, no wasted bits, value 0
    crc16 = 0
    for b in frame:
        crc16 ^= b << 8
        for _ in range(8):
            crc16 = ((crc16 << 1) ^ 0x8005) & 0xFFFF if crc16 & 0x8000 else (crc16 << 1) & 0xFFFF
    want = head + frame + crc16.to_bytes(2, "big")
    assert len(head) == 42 and len(frame) + 2 == 13
    got = F.encode(np.zeros(16, np.int16), 24000)
    assert got == want, (got.hex(), want.hex())
    assert np.array_equal(F.decode(got)[0], np.zeros(16, np.int16))


def _signals(n, rng):
    t = np.arange(n)
    sine = np.clip(np.rint(40000.0 * np.sin(2 * np.pi * 440.0 * t / 24000)), -32768, 32767)
    return {"silence": np.zeros(n), "constant": np.full(n, -1234), "square": np.where((t // 37) % 2, 32767, -32768),
            "sine": sine, "noise": rng.integers(-32768, 32768, n)}


def _pcm16(y):
    return np.clip(np.rint(32767.0 * np.asarray(y, np.float64)), -32768, 32767).astype(np.int16)


def _check(x, rate, stats=None, kinds=None):
    f = F.encode(x, rate, stats)
    assert len(f) <= F.bound(x.size) == audio.flac_max_bytes(x.size)
    info = {}
    y, r = F.decode(f, info)
    assert r == rate and np.array_equal(y, x)
    assert info["total"] == x.size and info["md5"] == 0 and info["min_block"] == info["max_block"] == 4096
    if kinds is not None:
        kinds.extend(info["kinds"])
    return f, info


@pytest.mark.parametrize("n", LENGTHS)
def test_round_trip_full_scale(n):
    rng = np.random.default_rng(n)
    for name, v in _signals(n, rng).items():
        x = np.asarray(v, dtype=np.int64).astype(np.int16)
        if name in ("square", "sine") and n >= 4096:
            assert x.min() == -32768 and x.max() == 32767
        f, info = _check(x, 24000)
        # the first block (blocks below 16 samples can be smaller as FIXED 0)
        if n >= 16 and name in ("silence", "constant"):
            assert info["kinds"][0] == ("constant", 0), name
        if name == "noise" and n >= 16:
            assert info["kinds"][0] == ("verbatim", 0), info["kinds"]
        if n == 0:
            assert len(f) == 42 and info["min_frame"] == info["max_frame"] == 0


def _speech_clips():
    rng = np.random.default_rng(9)
    clips = [c[:3 * 24000] for c in denoise_ref.voiced_set(seed=3, count=2)]
    clips += [enroll_ref.speech_like(rng, int(2.5 * 24000)) for _ in range(2)]
    return clips


@pytest.fixture(scope="module")
def speech_corpus():
    """(rate, int16 clip) pairs: the seeded clips taken from 24 kHz to every rate by the resampler's fp64 model and
    quantised as pcm16."""
    out = []
    for rate in RATES:
        fmt = AudioFormat(rate, "pcm16")
        for c in _speech_clips():
            y, _ = audio_ref.resample64(c, fmt.filter64(), fmt.up, fmt.down, fmt.half_len)
            out.append((rate, _pcm16(y)))
    return out


def test_speech_round_trip_and_every_subframe_kind(speech_corpus):
    stats, kinds = {}, []
    raw = packed = 0
    for rate, x in speech_corpus:
        f, _ = _check(x, rate, stats, kinds)
        raw += 2 * x.size
        packed += len(f)
    rng = np.random.default_rng(5)
    for n in (4096, 4097, 12293):                        # full-scale signals add CONSTANT and VERBATIM
        for v in _signals(n, rng).values():
            _check(np.asarray(v, np.int64).astype(np.int16), 16000, stats, kinds)
    chosen = set(stats)
    assert {("constant", 0), ("verbatim", 0)} <= chosen
    assert {("fixed", o) for o in range(5)} & chosen
    assert {("lpc", p) for p in range(1, 9)} <= chosen, sorted(chosen)
    assert set(kinds) == chosen
    ratio = packed / raw
    print(f"speech-like corpus: {packed} bytes of FLAC for {raw} bytes of PCM16 (ratio {ratio:.3f}); {sorted(stats)}")
    # measured 0.232 on this seeded corpus (synthetic clips: real speech compresses less)
    assert ratio < 0.25


def test_reader_rejects_corruption():
    x = _pcm16(denoise_ref.voiced(np.random.default_rng(2), 9000))
    f = bytearray(F.encode(x, 16000))
    for pos in (43, 47, 60, len(f) - 1):
        g = bytearray(f)
        g[pos] ^= 0x10
        with pytest.raises(F.DecodeError):
            F.decode(bytes(g))
    with pytest.raises(F.DecodeError):
        F.decode(bytes(f[:-3]))


def test_validation():
    f = AudioFormat(16000, "pcm16", container="flac")
    assert f.dtype == torch.uint8 and f.raw == AudioFormat(16000, "pcm16") and f.raw.container == "raw"
    assert f.out_bytes(24000) == F.bound(16000)
    assert AudioFormat(12000, "pcm16", "flac").out_bytes(0) == 42
    assert audio.ENCODINGS == ("float32", "pcm16", "mulaw", "alaw")
    for enc in ("float32", "mulaw", "alaw"):
        with pytest.raises(ValueError):
            AudioFormat(8000, enc, container="flac")
    for bad in ("ogg", "FLAC", None, 1):
        with pytest.raises(ValueError):
            AudioFormat(8000, "pcm16", container=bad)
    with pytest.raises(ValueError):
        AudioFormat(96000, "pcm16", container="flac")
    AudioFormat(96000, "pcm16")                          # the raw format keeps its range
    x = torch.zeros(2, 100, dtype=torch.int16)
    for bad in (0, 65536, 8000.0, True, "8000"):
        with pytest.raises(ValueError):
            audio.encode_flac(x, None, bad)
    for bad in (torch.zeros(2, 100), torch.zeros(2, 3, 4, dtype=torch.int16), np.zeros(4, np.int16)):
        with pytest.raises(ValueError):
            audio.encode_flac(bad, None, 8000)
    with pytest.raises(Exception):                       # ops.resample_encode writes samples, never a container
        ops.resample_encode(torch.zeros(1, 10), None, f, 7)


# ---- engine host logic -------------------------------------------------------------------------------------------
class _Recorder:
    def __init__(self, monkeypatch):
        self.calls = []
        rec = self

        def wrap(name, fn):
            def g(*a, **k):
                rec.calls.append((name, a, dict(k)))
                return fn(*a, **k)
            monkeypatch.setattr(ops, name, g)
        wrap("resample_encode", loudness_ref.resample_encode_gain_model)
        wrap("loudness_measure", loudness_ref.loudness_measure_model)
        wrap("flac_encode", F.encode_model)
        wrap("watermark_embed", lambda x, lens, wm: x.clone())


def _fake_syn(wav_lengths):
    syn = types.SimpleNamespace(last=dict(wav_lengths=wav_lengths, graph=True), last_stream=None, launches_per_call=10,
                                _slot_done={})
    syn._format_stage = types.MethodType(engine.Synthesizer._format_stage, syn)
    return syn


@pytest.mark.parametrize("rate,loud,wm", [(8000, None, None), (24000, Loudness(), None),
                                          (12000, Loudness(-16.0), Watermark(7, 3))])
def test_format_stage_encodes_the_pcm16_samples(sim, monkeypatch, rate, loud, wm):
    rec = _Recorder(monkeypatch)
    t = torch.arange(30000, dtype=torch.float64)
    wav = torch.stack([0.3 * torch.sin(0.05 * t), 0.05 * torch.sin(0.11 * t)]).float()
    lens = torch.tensor([30000, 21000], dtype=torch.int32)
    fmt = AudioFormat(rate, "pcm16", container="flac")
    syn = _fake_syn(lens)
    y, _, _ = syn._format_stage((wav, None, None), fmt, None, loud, **({"wm": wm} if wm else {}))
    names = [c[0] for c in rec.calls]
    assert names == (["watermark_embed"] if wm else []) + (["loudness_measure"] if loud else []) + \
        ["resample_encode", "flac_encode"]
    rs = [c for c in rec.calls if c[0] == "resample_encode"][0]
    assert rs[1][2] == AudioFormat(rate, "pcm16") and rs[1][3] == fmt.out_samples(30000)
    assert syn.launches_per_call == 10 + 1 + ops.FLAC_LAUNCHES + (ops.LOUDNESS_LAUNCHES if loud else 0) + \
        (1 if wm else 0)
    assert y.dtype == torch.uint8 and tuple(y.shape) == (2, fmt.out_bytes(30000))
    nb = syn.last["byte_lengths"]
    n = syn.last["sample_lengths"]
    pcm = loudness_ref.resample_encode_gain_model(wav, lens, AudioFormat(rate, "pcm16"), fmt.out_samples(30000),
                                                  gain=rs[2].get("gain"))
    for b in range(2):
        x, r = F.decode(bytes(y[b, :int(nb[b])].numpy()))
        assert r == rate and np.array_equal(x, pcm[b, :int(n[b])].numpy())
        assert not y[b, int(nb[b]):].any()


class _FakeEngine:
    """``synthesize_many``'s view of ``Synthesizer`` on the CPU."""
    pcm16 = False
    pipeline_depth = 1
    frame_quantum = 40
    device = torch.device("cpu")
    last_stream = None
    _out_format = engine.Synthesizer._out_format

    def __init__(self):
        self.calls = []

    def synthesize(self, tok, tl, mel, ml, dur, defer=False, prosody=None, audio=None):
        frames = [2 * int(dur[b, :tl[b]].sum()) for b in range(len(tl))]
        S = 300 * max(frames)
        wav = torch.zeros(len(tl), S)
        for b, fr in enumerate(frames):
            wav[b, :300 * fr] = (0.1 + 0.1 * int(tok[b, 0])) * torch.sin(torch.arange(300 * fr) * 0.05)
        lens = torch.tensor(frames, dtype=torch.int32) * 300
        self.calls.append(audio)
        self.last = dict(frames=frames, wav_lengths=lens, graph=False)
        self._format_stage = types.MethodType(engine.Synthesizer._format_stage, self)
        y, _, _ = self._format_stage((wav, None, None), audio)
        return y, torch.tensor(frames, dtype=torch.int32), None

    def finish(self, t):
        return t

    def join(self):
        pass


def test_synthesize_many_returns_whole_files(sim, monkeypatch):
    _Recorder(monkeypatch)
    monkeypatch.setattr(torch.Tensor, "pin_memory", lambda self, *a, **k: self)
    monkeypatch.setattr(torch.cuda, "current_stream", lambda *a: types.SimpleNamespace(synchronize=lambda: None))
    durs = [torch.tensor([3, 1, 4]), torch.tensor([2] * 7), torch.tensor([5]), torch.tensor([1, 1])]
    toks = [torch.full((d.shape[0],), i + 1, dtype=torch.long) for i, d in enumerate(durs)]
    mels = [torch.zeros(80, 10) for _ in durs]
    fmt = AudioFormat(16000, "pcm16", container="flac")
    for to_host in (False, True):
        syn = _FakeEngine()
        files, frames = engine.synthesize_many(syn, toks, mels, durations=durs, max_batch=2, audio=fmt,
                                               to_host=to_host)
        raw, _ = engine.synthesize_many(_FakeEngine(), toks, mels, durations=durs, max_batch=2,
                                        audio=AudioFormat(16000, "pcm16"))
        assert all(c == fmt for c in syn.calls)
        for i in range(len(durs)):
            one, _ = engine.synthesize_many(_FakeEngine(), [toks[i]], [mels[i]], durations=[durs[i]], audio=fmt)
            assert files[i].dtype == torch.uint8 and torch.equal(files[i], one[0])
            x, r = F.decode(bytes(files[i].numpy()))
            assert r == 16000 and np.array_equal(x, raw[i].numpy())
    pcm = _FakeEngine()
    pcm.pcm16 = True
    with pytest.raises(ValueError):
        engine.synthesize_many(pcm, toks, mels, durations=durs, audio=fmt)
