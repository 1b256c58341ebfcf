"""Loudness normalisation without a GPU: the K-weighting design against BS.1770's table, the fp64 meter
(tests/loudness_ref.py) against known readings (full-scale sine, EBU Tech 3341, a true-peak reference point),
``Loudness`` validation, and the engine's host logic (format stage, deferred tickets, ``synthesize_many``) with torch
models of the new ops."""
import math
import types

import numpy as np
import pytest
import torch

from artspeech_b200 import _lib, audio, engine, ops
from artspeech_b200.audio import AudioFormat, Loudness
from tests import loudness_ref


def _tone(dbfs, seconds, fs, freq=1000.0):
    """A mono sine at ``dbfs`` + 3.01 dB: EBU Tech 3341 states its levels for two channels."""
    t = np.arange(int(round(seconds * fs))) / fs
    return 10.0 ** ((dbfs + 10 * math.log10(2)) / 20.0) * np.sin(2 * np.pi * freq * t)


@pytest.mark.parametrize("design", ["product", "reference"])
def test_coefficients_match_bs1770_at_48k(design):
    (bs, as_), (bh, ah) = audio.k_weighting(48000) if design == "product" else loudness_ref.k_weighting(48000)
    assert np.abs(bs - loudness_ref.BS1770_SHELF[0]).max() <= 1e-12
    assert np.abs(as_ - loudness_ref.BS1770_SHELF[1]).max() <= 1e-12
    assert np.abs(bh - loudness_ref.BS1770_HIGHPASS[0]).max() <= 1e-12
    assert np.abs(ah - loudness_ref.BS1770_HIGHPASS[1]).max() <= 1e-12


@pytest.mark.parametrize("fs", [8000, 16000, 24000, 44100, 48000, 192000])
def test_product_design_equals_the_reference(fs):
    (p1, p2), (r1, r2) = audio.k_weighting(fs), loudness_ref.k_weighting(fs)
    for a, b in zip(p1 + p2, r1 + r2):
        assert np.abs(a - b).max() <= 1e-15
    taps = audio.k_weighting_taps(fs)
    assert taps.tolist() == [*p1[0], *p1[1][1:], *p2[0], *p2[1][1:]]


def test_full_scale_997hz_sine_reads_minus_3_01():
    fs = 48000
    x = np.sin(2 * np.pi * 997 * np.arange(10 * fs) / fs)
    assert abs(loudness_ref.integrated(x, fs) - (-3.01)) <= 0.01


EBU_3341 = {
    1: [(-23, 20)],
    3: [(-36, 10), (-23, 60), (-36, 10)],
    4: [(-72, 10), (-36, 10), (-23, 60), (-36, 10), (-72, 10)],
    5: [(-26, 20), (-20, 20.1), (-26, 20)],
}


@pytest.mark.parametrize("fs", [48000, 24000])
@pytest.mark.parametrize("case", sorted(EBU_3341))
def test_ebu_tech_3341(case, fs):
    x = np.concatenate([_tone(db, s, fs) for db, s in EBU_3341[case]])
    assert abs(loudness_ref.integrated(x, fs) - (-23.0)) <= 0.1


def test_true_peak_reference_point():
    """A 6 kHz sine at 24 kHz, amplitude 0.5, 45 degree phase: samples at -9.03 dB, true peak -6.006 dBTP.  The ends
    are faded over 10 ms: an abrupt start rings in the interpolator (-5.9 dBTP)."""
    n = np.arange(24000)
    fade = np.ones(n.size)
    ramp = 0.5 - 0.5 * np.cos(np.pi * np.arange(240) / 240)
    fade[:240], fade[-240:] = ramp, ramp[::-1]
    x = 0.5 * np.sin(np.pi / 2 * n + np.pi / 4) * fade
    assert abs(20 * math.log10(np.abs(x).max()) - (-9.03)) <= 0.005
    assert abs(loudness_ref.true_peak(x) - (-6.006)) <= 0.001


def test_silence_and_empty_read_minus_inf():
    assert loudness_ref.integrated(np.zeros(48000), 24000) == -math.inf
    assert loudness_ref.integrated(np.zeros(0), 24000) == -math.inf
    assert loudness_ref.integrated(_tone(-80, 2, 24000), 24000) == -math.inf
    assert loudness_ref.gain_db(-math.inf, -math.inf) == 0.0


def test_loudness_validation():
    for kw in (dict(target_lufs=0.0), dict(target_lufs=3.0), dict(max_true_peak_db=0.5), dict(target_lufs=math.nan),
               dict(target_lufs=-math.inf), dict(max_true_peak_db=math.inf), dict(target_lufs=True),
               dict(max_true_peak_db=False), dict(target_lufs="-23"), dict(target_lufs=None)):
        with pytest.raises(ValueError):
            Loudness(**kw)
    assert Loudness() == Loudness(-23.0, -1.0)
    assert Loudness(np.int64(-24), 0).target_lufs == -24.0 and Loudness(-16, 0).max_true_peak_db == 0.0
    with pytest.raises(ValueError):
        audio.check_loudness(Loudness(), pcm16=True)
    with pytest.raises(ValueError):
        audio.check_loudness(-23.0, pcm16=False)
    assert audio.check_loudness(None, pcm16=True) is None


def test_measure_loudness_rejects_rates():
    for fs in (7990, 8005, 192010, 44100.0, True):
        with pytest.raises(ValueError):
            audio.measure_loudness(torch.zeros(8), sample_rate=fs)


def test_workspace_bytes():
    lib = _lib.load()
    assert lib.as_loudness_workspace_bytes(0, 1000, 24000) == 0
    assert lib.as_loudness_workspace_bytes(1, 1000, 7000) == 0
    a = lib.as_loudness_workspace_bytes(16, 240000, 24000)
    assert a > 0 and a % 256 == 0
    assert lib.as_loudness_workspace_bytes(16, 1440000, 24000) > a
    assert audio.true_peak_table().shape == (4, 24) and audio.true_peak_table().dtype == np.float32


# ---- engine host logic --------------------------------------------------------------------------------------------
class _Recorder:
    """Records the calls of the two ops, answering with their torch models."""

    def __init__(self, monkeypatch):
        self.calls = []
        rec = self

        def resample_encode(*a, **k):
            rec.calls.append(("resample_encode", a, dict(k)))
            return loudness_ref.resample_encode_gain_model(*a, **k)

        def loudness_measure(*a, **k):
            rec.calls.append(("loudness_measure", a, dict(k)))
            return loudness_ref.loudness_measure_model(*a, **k)
        monkeypatch.setattr(ops, "resample_encode", resample_encode)
        monkeypatch.setattr(ops, "loudness_measure", loudness_measure)


def _fake_syn(wav_lengths):
    syn = types.SimpleNamespace(last=dict(wav_lengths=wav_lengths, graph=True), last_stream=None, launches_per_call=10,
                                _slot_done={})
    syn._format_stage = types.MethodType(engine.Synthesizer._format_stage, syn)
    return syn


def _waves():
    t = torch.arange(30000, dtype=torch.float64)
    wav = torch.stack([0.3 * torch.sin(0.05 * t), 0.05 * torch.sin(0.11 * t) + 0.02 * torch.sin(0.013 * t)]).float()
    return wav, torch.tensor([30000, 21000], dtype=torch.int32)


def test_format_stage_without_loudness_calls_what_it_called_before(sim, monkeypatch):
    rec = _Recorder(monkeypatch)
    wav, lens = _waves()
    syn = _fake_syn(lens)
    f = AudioFormat(8000, "mulaw")
    y, _, _ = syn._format_stage((wav, None, None), f)
    assert [c[0] for c in rec.calls] == ["resample_encode"]
    _, a, k = rec.calls[0]
    assert a[0] is wav and a[1] is lens and a[2] == f and a[3] == f.out_samples(30000)
    assert sorted(k) == ["out_lens"]                        # no gain= keyword
    assert syn.launches_per_call == 11 and "loudness" not in syn.last


@pytest.mark.parametrize("fmt", [AudioFormat(), AudioFormat(16000, "pcm16")])
def test_format_stage_with_loudness(sim, monkeypatch, fmt):
    rec = _Recorder(monkeypatch)
    wav, lens = _waves()
    syn = _fake_syn(lens)
    loud = Loudness(-20.0, -2.0)
    y, _, _ = syn._format_stage((wav, None, None), fmt, None, loud)
    assert [c[0] for c in rec.calls] == ["loudness_measure", "resample_encode"]
    _, a, k = rec.calls[0]
    assert a[0] is wav and a[1] is lens and a[2:] == (24000, -20.0, -2.0)
    gain = rec.calls[1][2]["gain"]
    assert syn.launches_per_call == 10 + ops.LOUDNESS_LAUNCHES + 1
    for b in range(2):
        n = int(lens[b])
        L, tp = loudness_ref.integrated(wav[b, :n].double().numpy(), 24000), loudness_ref.true_peak(wav[b, :n].numpy())
        assert float(syn.last["loudness"][b]) == L and float(syn.last["true_peak"][b]) == tp
        gdb = loudness_ref.gain_db(L, tp, -20.0, -2.0)
        assert float(syn.last["gain_db"][b]) == gdb and float(gain[b]) == float(loudness_ref.gain32(gdb))
    assert torch.equal(y, loudness_ref.resample_encode_gain_model(wav, lens, fmt, fmt.out_samples(30000), gain=gain))


def test_deferred_ticket_carries_the_loudness(sim, monkeypatch):
    rec = _Recorder(monkeypatch)
    wav, lens = _waves()
    seen = []
    syn = _fake_syn(lens)
    syn._format_stage = lambda res, fmt, side, loud: seen.append((fmt, side, loud)) or res
    out = dict(wav=torch.zeros(2, 300 * 40), mel_lengths=torch.tensor([40, 30]), mel=torch.zeros(2, 80, 40))
    eb = types.SimpleNamespace(graph=types.SimpleNamespace(replay=lambda: None), out=out, launches=5)
    syn._lookup = lambda slot, key: eb
    syn.stats = dict(replays=0)
    syn.frame_quantum = 40
    t = engine._Ticket()
    t.ent = types.SimpleNamespace(pin_meta=torch.tensor([20, 15], dtype=torch.int32), uid=1,
                                  state=dict(duration=None, pred_dur=None))
    t.got = types.SimpleNamespace(synchronize=lambda: None)
    t.B, t.slot, t.launches, t.is_side, t.run_stream = 2, 0, 7, False, None
    t.fmt, t.loud = AudioFormat(), Loudness()
    monkeypatch.setattr(ops, "_count", lambda n=1: None)
    engine.Synthesizer.finish(syn, t)
    assert seen == [(AudioFormat(), None, Loudness())]


class _FakeEngine:
    """``synthesize_many``'s view of ``Synthesizer`` on the CPU (as in test_audio_format_cpu.py), with ``loudness``."""
    pcm16 = False
    pipeline_depth = 1
    frame_quantum = 40
    device = torch.device("cpu")
    last_stream = None
    _out_format = engine.Synthesizer._out_format

    def __init__(self):
        self.calls = []

    def synthesize(self, tok, tl, mel, ml, dur, defer=False, prosody=None, audio=None, loudness=None):
        frames = [2 * int(dur[b, :tl[b]].sum()) for b in range(len(tl))]
        S = 300 * max(frames)
        wav = torch.zeros(len(tl), S)
        for b, fr in enumerate(frames):
            wav[b, :300 * fr] = (0.1 + 0.1 * int(tok[b, 0])) * torch.sin(torch.arange(300 * fr) * 0.05)
        lens = torch.tensor(frames, dtype=torch.int32) * 300
        self.calls.append((audio, loudness))
        fmt = audio
        if loudness is not None:
            fmt = fmt or AudioFormat()
            gain = ops.loudness_measure(wav, lens, 24000, loudness.target_lufs, loudness.max_true_peak_db)[3]
            wav = ops.resample_encode(wav, lens, fmt, fmt.out_samples(S), gain=gain)
        elif fmt is not None:
            wav = ops.resample_encode(wav, lens, fmt, fmt.out_samples(S))
        self.last = dict(frames=frames)
        return wav, torch.tensor(frames, dtype=torch.int32), None

    def finish(self, t):
        return t

    def join(self):
        pass


def test_synthesize_many_with_loudness(sim, monkeypatch):
    _Recorder(monkeypatch)
    monkeypatch.setattr(torch.Tensor, "pin_memory", lambda self, *a, **k: self)
    durs = [torch.tensor([3, 1, 4]), torch.tensor([2] * 7), torch.tensor([5]), torch.tensor([1, 1])]
    toks = [torch.full((d.shape[0],), i + 1, dtype=torch.long) for i, d in enumerate(durs)]
    mels = [torch.zeros(80, 10) for _ in durs]
    loud = Loudness(-18.0)
    for f in (AudioFormat(8000, "mulaw"), None):
        syn = _FakeEngine()
        wavs, frames = engine.synthesize_many(syn, toks, mels, durations=durs, max_batch=2, audio=f, loudness=loud)
        want_fmt = f or AudioFormat()
        assert all(c == (want_fmt, loud) for c in syn.calls)
        for i in range(len(durs)):
            assert wavs[i].dtype == want_fmt.dtype and wavs[i].shape[0] == want_fmt.out_samples(300 * frames[i])
            one, _ = engine.synthesize_many(_FakeEngine(), [toks[i]], [mels[i]], durations=[durs[i]], audio=f,
                                            loudness=loud)
            assert torch.equal(wavs[i], one[0])
    # without loudness the engine is called as before: no loudness keyword at all
    syn = _FakeEngine()
    syn.synthesize = lambda tok, tl, mel, ml, dur, defer=False, prosody=None, audio=None: \
        _FakeEngine.synthesize(syn, tok, tl, mel, ml, dur, defer, prosody, audio)
    engine.synthesize_many(syn, toks, mels, durations=durs, max_batch=2)
    assert all(c == (None, None) for c in syn.calls)
    pcm = _FakeEngine()
    pcm.pcm16 = True
    with pytest.raises(ValueError):
        engine.synthesize_many(pcm, toks, mels, durations=durs, loudness=loud)
