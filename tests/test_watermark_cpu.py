"""The synthesis watermark without a GPU: the patterns' properties, the product's host tables against the fp64
restatement (tests/watermark_ref.py), ``Watermark`` validation, a robustness matrix of the design through every output
format, the null distribution, and the engine's host logic with torch models of the new ops."""
import math
import types

import numpy as np
import pytest
import torch

from artspeech_b200 import audio, engine, ops
from artspeech_b200.audio import AudioFormat, Loudness, Watermark
from tests import audio_ref, loudness_ref
from tests import watermark_ref as W

KEY, MSG = 0x0123456789ABCDEF, 0xBEEF


@pytest.mark.parametrize("i", [0, 1, 2])
def test_pattern_properties(i):
    for n in (W.P8, W.P24):
        c = W.pattern(KEY, i, n)
        assert abs(np.sqrt(np.mean(c ** 2)) - 1.0) <= 1e-12
        spec = np.abs(np.fft.rfft(c)) ** 2
        out = np.ones(spec.size, bool)
        out[W.BINS] = False
        assert spec[out].sum() <= 1e-20 * spec.sum()
        assert np.abs(audio.watermark_pattern(KEY, i, n) - c).max() <= 1e-12       # irfft == the literal sum
    assert np.abs(W.pattern(KEY, i, W.P24)[::3] - W.pattern(KEY, i, W.P8)).max() <= 1e-12


def test_patterns_are_nearly_orthogonal_at_every_lag():
    cs = [np.fft.rfft(W.pattern(KEY, i, W.P8)) for i in range(3)]
    worst = 0.0
    for a in range(3):
        for b in range(3):
            if a != b:
                x = np.fft.irfft(cs[a] * np.conj(cs[b]), W.P8) / W.P8          # normalised circular cross-correlation
                worst = max(worst, np.abs(x).max())
    other = np.fft.rfft(W.pattern(KEY + 1, 0, W.P8))
    worst = max(worst, np.abs(np.fft.irfft(cs[0] * np.conj(other), W.P8) / W.P8).max())
    print(f"largest cross-correlation between patterns: {worst:.4f}")
    assert worst <= 0.12


def test_product_tables_match_the_reference():
    assert audio.splitmix64(0) == W.splitmix64(0) == 0xE220A8397B1DCDAF        # splitmix64's first output from 0
    assert np.array_equal(audio.watermark_phases(KEY)[1], W.phases(KEY, 1))
    m = audio.watermark_mark(KEY, MSG)
    assert m.dtype == np.float32 and m.shape == (W.P24,)
    assert np.abs(m.astype(np.float64) - W.mark(KEY, MSG)).max() <= 2.0 ** -24 * np.abs(W.mark(KEY, MSG)).max() * 2
    sp = audio.watermark_spectra(KEY)
    assert sp.shape == (3, 1588, 2) and not sp[:, 1587].any()
    ph = W.phases(KEY, 2)
    assert np.abs(sp[2, :1587, 0] - np.cos(ph)).max() <= 1e-7 and np.abs(sp[2, :1587, 1] + np.sin(ph)).max() <= 1e-7
    tw = audio.watermark_twiddles()
    assert tw.shape == (2048, 2) and tw[512, 0] == np.float32(np.cos(np.pi / 4))


def test_watermark_validation():
    for kw in (dict(key=-1), dict(key=1 << 64), dict(key=1.0), dict(key=True), dict(key="1"),
               dict(key=1, message=-1), dict(key=1, message=1 << 16), dict(key=1, message=2.0),
               dict(key=1, strength_db=-14.9), dict(key=1, strength_db=-40.1), dict(key=1, strength_db=math.nan),
               dict(key=1, strength_db=False), dict(key=1, strength_db="-30")):
        with pytest.raises(ValueError):
            Watermark(**kw)
    w = Watermark(np.uint64((1 << 64) - 1), np.int32(65535), -15)
    assert w.key == (1 << 64) - 1 and w.message == 65535 and w.strength_db == -15.0
    assert Watermark(5) == Watermark(5, 0, -30.0) and abs(Watermark(5).alpha - 10 ** -1.5) < 1e-15
    with pytest.raises(ValueError):
        audio.check_watermark(Watermark(1), pcm16=True)
    with pytest.raises(ValueError):
        audio.check_watermark(1, pcm16=False)
    assert audio.check_watermark(None, pcm16=True) is None


def test_detection_resampler_ratios():
    """Every named output rate fits the kernel at its ratio to 8 kHz; 44.1 kHz is the largest, at 62976 bytes."""
    sizes = {}
    for fs in (8000, 11025, 16000, 22050, 24000, 32000, 44100, 48000):
        r = audio.to_detection_rate(fs)
        assert r.out_samples(fs) == 8000 and np.array_equal(r.filter64(), audio._design(r.up, r.down)[0]) or fs == 8000
        sizes[fs] = audio.smem_bytes(r.up, r.down, r.K, r.table_ld)
    assert max(sizes, key=sizes.get) == 44100 and sizes[44100] == 62976
    for fs in (44101, 0, -8000, 8000.0, True):
        with pytest.raises(ValueError):
            audio.detect_watermark(torch.zeros(8), None, fs, KEY)


# ---- the design through the output chain ---------------------------------------------------------------------
RATES = (8000, 11025, 16000, 22050, 24000, 32000, 44100, 48000)
ENCODINGS = ("float32", "pcm16", "mulaw", "alaw")


def _deliver(y24, fmt, target):
    """What a detector receives: ``y24`` normalised to ``target`` LUFS (-1 dBTP) at 24 kHz, resampled to the
    format's rate (fp64), encoded, decoded and resampled to 8 kHz."""
    L, tp = loudness_ref.integrated(y24, 24000), loudness_ref.true_peak(y24.astype(np.float32))
    g = 10 ** (loudness_ref.gain_db(L, tp, target, -1.0) / 20)
    f = AudioFormat(fmt[0], "float32")
    y = audio_ref.resample64(g * y24, f.filter64(), f.up, f.down, f.half_len)[0]
    return W.to_8k(W.decode(W.encode(y, fmt[1]), fmt[1]), fmt[0])


@pytest.mark.parametrize("rate", RATES)
def test_robustness_matrix(rate):
    """Seeded speech-like clips of 2-12 s at -30 dB, cropped at a random offset, polarity-flipped or not, normalised to
    -23 or -14 LUFS and delivered in each encoding: every clip is detected with its exact message."""
    rng = np.random.default_rng(rate)
    scores = []
    for j, enc in enumerate(ENCODINGS):
        dur = [2.0, 3.5, 7.0, 12.0][(j + RATES.index(rate)) % 4]
        msg = int(rng.integers(0, 1 << 16))
        x = W.speech(int(dur * 24000) + 12000, rng)
        y = W.embed(x, KEY, msg)[int(rng.integers(0, 12000)):]
        y = y[:int(dur * 24000)] * (-1.0 if j % 2 else 1.0)
        d, s, _, m = W.detect(_deliver(y, (rate, enc), (-23.0, -14.0)[j % 2]), KEY)
        scores.append(s)
        assert d and m == msg, (rate, enc, dur, s, hex(m), hex(msg))
    print(f"{rate} Hz: scores {np.round(scores, 2).tolist()}")


def test_null_scores_stay_below_the_threshold():
    """Unmarked speech, the wrong key, white noise and silence: 240 clips, all below 6."""
    rng = np.random.default_rng(11)
    worst = {}
    for j in range(60):
        dur = 2.0 + 10.0 * rng.uniform()
        n = int(dur * 24000)
        x = W.speech(n, rng)
        fmt = (RATES[j % len(RATES)], ENCODINGS[j % 4])
        cases = {"unmarked": (_deliver(x, fmt, -23.0), KEY),
                 "wrong key": (_deliver(W.embed(x, KEY, j), fmt, -23.0), KEY ^ (1 << (j % 64))),
                 "white noise": (0.1 * rng.standard_normal(int(dur * 8000)), KEY),
                 "silence": (np.zeros(int(dur * 8000)), KEY)}
        for name, (y8, key) in cases.items():
            d, s, _, _ = W.detect(y8, key)
            worst[name] = max(worst.get(name, 0.0), s)
            assert not d, (name, j, s)
    print("largest null scores:", {k: round(v, 2) for k, v in worst.items()})
    assert worst["silence"] == 0.0


def test_strength_is_the_watermark_to_signal_ratio():
    rng = np.random.default_rng(3)
    x = W.speech(24000 * 5, rng)
    for db in (-30.0, -20.0):
        y = W.embed(x, KEY, MSG, db)
        assert abs(10 * np.log10(np.sum((y - x) ** 2) / np.sum(x ** 2)) - db) <= 0.5
    z = np.zeros(24000)
    z[9000:15000] = x[9000:15000]
    y = W.embed(z, KEY, MSG)
    assert not y[:8000].any() and not y[16000:].any()                        # silence stays digital silence


# ---- engine host logic -------------------------------------------------------------------------------------------
def _embed_model(x, lens, wm):
    y = torch.zeros_like(x)
    for b in range(x.shape[0]):
        n = x.shape[1] if lens is None else min(int(lens[b]), x.shape[1])
        y[b, :n] = torch.from_numpy(W.embed(x[b, :n].double().numpy(), wm.key, wm.message, wm.strength_db)).float()
    return y


class _Recorder:
    def __init__(self, monkeypatch):
        self.calls = []
        rec = self

        def wrap(name, fn):
            def f(*a, **k):
                rec.calls.append((name, a, dict(k)))
                return fn(*a, **k)
            monkeypatch.setattr(ops, name, f)
        wrap("watermark_embed", _embed_model)
        wrap("resample_encode", loudness_ref.resample_encode_gain_model)
        wrap("loudness_measure", loudness_ref.loudness_measure_model)


def _fake_syn(wav_lengths):
    syn = types.SimpleNamespace(last=dict(wav_lengths=wav_lengths, graph=True), last_stream=None, launches_per_call=10,
                                _slot_done={})
    syn._format_stage = types.MethodType(engine.Synthesizer._format_stage, syn)
    return syn


def _waves():
    t = torch.arange(30000, dtype=torch.float64)
    wav = torch.stack([0.3 * torch.sin(0.05 * t), 0.05 * torch.sin(0.11 * t) + 0.02 * torch.sin(0.013 * t)]).float()
    return wav, torch.tensor([30000, 21000], dtype=torch.int32)


@pytest.mark.parametrize("fmt,loud", [(None, None), (AudioFormat(8000, "mulaw"), None), (AudioFormat(), Loudness()),
                                      (AudioFormat(16000, "pcm16"), Loudness(-14.0))])
def test_output_stage_marks_first(sim, monkeypatch, fmt, loud):
    rec = _Recorder(monkeypatch)
    wav, lens = _waves()
    syn = _fake_syn(lens)
    wm = Watermark(KEY, MSG)
    y, _, _ = syn._format_stage((wav, None, None), fmt, None, loud, wm=wm)
    names = [c[0] for c in rec.calls]
    want = ["watermark_embed"] + (["loudness_measure"] if loud else []) + (["resample_encode"] if fmt else [])
    assert names == want
    _, a, _ = rec.calls[0]
    assert a[0] is wav and a[1] is lens and a[2] is wm
    marked = _embed_model(wav, lens, wm)
    assert syn.launches_per_call == 10 + 1 + (ops.LOUDNESS_LAUNCHES if loud else 0) + (1 if fmt else 0)
    if fmt is None:
        assert torch.equal(y, marked) and "sample_lengths" not in syn.last
    else:
        for c in rec.calls[1:]:
            assert torch.equal(c[1][0], marked)                  # the meter and the format read the marked samples
        assert "sample_lengths" in syn.last


def test_deferred_ticket_carries_the_watermark(sim, monkeypatch):
    seen = []
    syn = _fake_syn(None)
    syn._format_stage = lambda res, fmt, side, loud, wm=None: seen.append((fmt, side, loud, wm)) or res
    out = dict(wav=torch.zeros(2, 300 * 40), mel_lengths=torch.tensor([40, 30]), mel=torch.zeros(2, 80, 40))
    eb = types.SimpleNamespace(graph=types.SimpleNamespace(replay=lambda: None), out=out, launches=5)
    syn._lookup = lambda slot, key: eb
    syn.stats = dict(replays=0)
    syn.frame_quantum = 40
    monkeypatch.setattr(ops, "_count", lambda n=1: None)
    for fmt in (None, AudioFormat(8000, "alaw")):
        t = engine._Ticket()
        t.ent = types.SimpleNamespace(pin_meta=torch.tensor([20, 15], dtype=torch.int32), uid=1,
                                      state=dict(duration=None, pred_dur=None))
        t.got = types.SimpleNamespace(synchronize=lambda: None)
        t.B, t.slot, t.launches, t.is_side, t.run_stream = 2, 0, 7, False, None
        t.fmt, t.wm = fmt, Watermark(7, 3)
        engine.Synthesizer.finish(syn, t)
    assert seen == [(None, None, None, Watermark(7, 3)), (AudioFormat(8000, "alaw"), None, None, Watermark(7, 3))]
    # an unmarked, unformatted ticket has no output stage at all
    seen.clear()
    t = engine._Ticket()
    t.ent = types.SimpleNamespace(pin_meta=torch.tensor([20, 15], dtype=torch.int32), uid=1,
                                  state=dict(duration=None, pred_dur=None))
    t.got = types.SimpleNamespace(synchronize=lambda: None)
    t.B, t.slot, t.launches, t.is_side, t.run_stream = 2, 0, 7, False, None
    engine.Synthesizer.finish(syn, t)
    assert seen == []


class _FakeEngine:
    """``synthesize_many``'s view of ``Synthesizer`` on the CPU, with ``watermark``."""
    pcm16 = False
    pipeline_depth = 1
    frame_quantum = 40
    device = torch.device("cpu")
    last_stream = None
    _out_format = engine.Synthesizer._out_format

    def __init__(self):
        self.calls = []

    def synthesize(self, tok, tl, mel, ml, dur, defer=False, prosody=None, audio=None, watermark=None):
        frames = [2 * int(dur[b, :tl[b]].sum()) for b in range(len(tl))]
        S = 300 * max(frames)
        wav = torch.zeros(len(tl), S)
        for b, fr in enumerate(frames):
            wav[b, :300 * fr] = (0.1 + 0.1 * int(tok[b, 0])) * torch.sin(torch.arange(300 * fr) * 0.05)
        lens = torch.tensor(frames, dtype=torch.int32) * 300
        self.calls.append((audio, watermark))
        wav = _embed_model(wav, lens, watermark)
        if audio is not None:
            wav = ops.resample_encode(wav, lens, audio, audio.out_samples(S))
        self.last = dict(frames=frames)
        return wav, torch.tensor(frames, dtype=torch.int32), None

    def finish(self, t):
        return t

    def join(self):
        pass


def test_synthesize_many_with_watermark(sim, monkeypatch):
    _Recorder(monkeypatch)
    monkeypatch.setattr(torch.Tensor, "pin_memory", lambda self, *a, **k: self)
    durs = [torch.tensor([3, 1, 4]), torch.tensor([2] * 7), torch.tensor([5]), torch.tensor([1, 1])]
    toks = [torch.full((d.shape[0],), i + 1, dtype=torch.long) for i, d in enumerate(durs)]
    mels = [torch.zeros(80, 10) for _ in durs]
    wm = Watermark(KEY, 77)
    for f in (AudioFormat(8000, "mulaw"), None):
        syn = _FakeEngine()
        wavs, frames = engine.synthesize_many(syn, toks, mels, durations=durs, max_batch=2, audio=f, watermark=wm)
        assert all(c == (f, wm) for c in syn.calls)
        for i in range(len(durs)):
            one, _ = engine.synthesize_many(_FakeEngine(), [toks[i]], [mels[i]], durations=[durs[i]], audio=f,
                                            watermark=wm)
            assert torch.equal(wavs[i], one[0])
    pcm = _FakeEngine()
    pcm.pcm16 = True
    with pytest.raises(ValueError):
        engine.synthesize_many(pcm, toks, mels, durations=durs, watermark=wm)
