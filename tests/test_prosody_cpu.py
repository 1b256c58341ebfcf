"""Prosody controls without a GPU: validation and packing of ``Prosody``, the fp64 restatement's arithmetic, and the
model's wiring of the two ops on the semantic backend (``sim`` plus the models of tests/prosody_ref.py)."""
import math

import pytest
import torch

from artspeech_b200 import prosody
from artspeech_b200.prosody import Prosody
from tests import prosody_ref, util

PM, PS, ES = 137.0945846179066, 78.25457848323684, 3.110472802617481


@pytest.mark.parametrize("kw", [
    dict(duration_scale=0.0), dict(duration_scale=-1.0), dict(duration_scale=float("nan")),
    dict(duration_scale=[1.0, 0.0, 1.0]), dict(duration_scale=[1.0, float("inf")]), dict(duration_scale=[]),
    dict(duration_scale="fast"), dict(pitch_shift=float("inf")), dict(pitch_shift=None),
    dict(pitch_range=-0.1), dict(pitch_range=float("nan")), dict(energy_db=float("-inf")),
    dict(articulation_scale=[1.0] * 9), dict(articulation_scale=[1.0] * 11),
    dict(articulation_offset=[0.0] * 9 + [float("nan")]), dict(articulation_offset=3.0),
])
def test_prosody_rejects_bad_values(kw):
    with pytest.raises(ValueError):
        Prosody(**kw)


def test_prosody_normalises_and_defaults_to_identity():
    p = Prosody()
    assert not p.scales_durations and p.ctrl_row() == [0.0, 1.0, 0.0, 0.0] + [1.0] * 10 + [0.0] * 10
    q = Prosody(duration_scale=torch.tensor([1.0, 2.0, 3.0]), pitch_shift=2, articulation_scale=torch.full((10,), 1.5))
    assert q.duration_scale == (1.0, 2.0, 3.0) and q.scales_durations and q.mean_duration_scale(2) == 1.5
    assert Prosody(duration_scale=[1.0, 1.0]).scales_durations is False
    assert Prosody(pitch_range=0.0).pitch_range == 0.0           # monotone voice is allowed


def test_check_batch_rules():
    assert prosody.check(None, [3, 4], False) is None
    with pytest.raises(ValueError):
        prosody.check([Prosody()], [3, 4], False)                  # one per utterance
    with pytest.raises(ValueError):
        prosody.check([Prosody(), "slow"], [3, 4], False)
    with pytest.raises(ValueError):
        prosody.check([Prosody(), Prosody(duration_scale=[1.0] * 3)], [3, 4], False)   # shorter than the utterance
    with pytest.raises(ValueError):
        prosody.check([Prosody(duration_scale=1.2), Prosody()], [3, 4], True)          # caller owns the durations
    ok = prosody.check([Prosody(duration_scale=[1.0] * 5), Prosody(pitch_shift=3)], [3, 4], True)
    assert len(ok) == 2 and prosody.check(Prosody(), [7], False) == [Prosody()]


def test_pack_layout():
    ps = [Prosody(duration_scale=1.5, pitch_shift=-2, pitch_range=0.5, energy_db=3,
                  articulation_scale=[float(i) for i in range(10)], articulation_offset=[0.1 * i for i in range(10)]),
          Prosody(duration_scale=[0.5, 2.0, 3.0])]
    ctrl, ds = prosody.pack(ps, 5)
    assert ctrl.dtype == torch.float32 and ctrl.shape == (2, prosody.CTRL_WIDTH) and ds.shape == (2, 5)
    assert ctrl[0, :4].tolist() == [-2.0, 0.5, 3.0, 0.0]
    assert ctrl[0, 4:14].tolist() == [float(i) for i in range(10)]
    assert torch.allclose(ctrl[0, 14:], torch.tensor([0.1 * i for i in range(10)]))
    assert ctrl[1].tolist() == Prosody().ctrl_row()
    assert ds[0].tolist() == [1.5] * 5 and ds[1].tolist() == [0.5, 2.0, 3.0, 1.0, 1.0]
    _, ds2 = prosody.pack(ps, 2)
    assert ds2[1].tolist() == [0.5, 2.0]


def _tracks(B, Tm, seed):
    g = torch.Generator().manual_seed(seed)
    f0 = torch.randn(B, Tm, 1, generator=g) * 0.8
    f0[:, ::3] = -1.5                                              # hz = 137 - 117 = 20 Hz: unvoiced
    return f0, torch.randn(B, Tm, 1, generator=g), torch.randn(B, Tm, 10, generator=g)


def test_restatement_arithmetic():
    """The restatement against the formulas, evaluated independently on single frames."""
    B, Tm = 3, 40
    f0, n, ema = _tracks(B, Tm, 0)
    f0[2] = -1.5                                                   # no voiced frame at all
    lens = torch.tensor([40, 17, 30])
    ctrl, _ = prosody.pack([Prosody(pitch_shift=12.0, energy_db=10.0, articulation_scale=[0.0] * 10),
                            Prosody(pitch_range=0.0, articulation_offset=[1.0] * 10),
                            Prosody(pitch_shift=5.0)], 1)
    f1, n1, e1 = prosody_ref.apply_tracks(f0, n, ema, lens, ctrl, PM, PS, ES)
    hz = lambda x: x.double() * PS + PM
    v0 = hz(f0[0, :, 0]) >= 50
    # +12 semitones with range 1: every voiced frame an octave higher, unvoiced frames untouched
    assert torch.allclose(hz(f1[0, v0, 0]), 2 * hz(f0[0, v0, 0]), rtol=1e-6)
    assert torch.equal(f1[0, ~v0], f0[0, ~v0])
    # +10 dB: n + ln(10) / energy_std
    assert torch.allclose(n1[0], n[0] + math.log(10) / ES, atol=1e-6)
    # articulation scale 0: every channel flat at its mean
    assert torch.allclose(e1[0], ema[0].mean(0, keepdim=True).expand(Tm, 10), atol=1e-6)
    # range 0: voiced frames collapse to exp(mean ln hz); frames beyond the length untouched; offset in std units
    v1 = hz(f0[1, :17, 0]) >= 50
    want = torch.exp(torch.log(hz(f0[1, :17, 0])[v1]).mean())
    assert torch.allclose(hz(f1[1, :17, 0])[v1], want.expand(int(v1.sum())), rtol=1e-6)
    assert torch.equal(f1[1, 17:], f0[1, 17:]) and torch.equal(e1[1, 17:], ema[1, 17:])
    assert torch.allclose(e1[1, :17], ema[1, :17] + 1.0, atol=1e-6)
    # no voiced frame: F0 unchanged; identity energy / EMA not written
    assert torch.equal(f1[2], f0[2]) and torch.equal(n1[1:], n[1:]) and torch.equal(e1[2], ema[2])


def _model(sim, monkeypatch):
    prosody_ref.install(monkeypatch)
    monkeypatch.setattr(sim, "EMULATE_FP16_RECURRENCE", False)
    g = util.load_golden("acoustic_small.pt")
    model = util.acoustic_model(g["checkpoint_seed"])
    model.set_compute_dtype(torch.float32)
    return model, g


def _ragged(g):
    cs = [g["cases"][k] for k in ("b_forced_dur", "c_short")]
    Tt = max(c["tokens"].shape[1] for c in cs)
    Tr = max(c["ref_mel"].shape[2] for c in cs)
    tok = torch.zeros(2, Tt, dtype=torch.long)
    mel = torch.zeros(2, 80, Tr)
    dur = torch.ones(2, Tt, dtype=torch.long)
    for i, c in enumerate(cs):
        tok[i, :c["tokens"].shape[1]] = c["tokens"][0]
        mel[i, :, :c["ref_mel"].shape[2]] = c["ref_mel"][0]
        dur[i, :c["tokens"].shape[1]] = c["out"]["pred_dur"].view(-1)
    tl = torch.tensor([c["tokens"].shape[1] for c in cs])
    ml = torch.tensor([c["ref_mel"].shape[2] for c in cs])
    return [tok, tl, mel, ml], dur


def test_forward_prosody_equals_decoder_on_edited_tracks(sim, monkeypatch):
    """ArtsSpeech.forward(prosody=...) == the decoder run on the restatement-edited predictor tracks."""
    from artspeech_b200 import ops
    model, g = _model(sim, monkeypatch)
    batch, dur = _ragged(g)
    pros = [Prosody(pitch_shift=3.0, pitch_range=1.2, energy_db=2.0, articulation_scale=[1.1] * 10),
            Prosody(pitch_range=0.0, articulation_offset=[0.05 * i for i in range(10)])]
    _, aux0 = model(batch, step="test", durations=dur, return_aux=True)
    mel, aux = model(batch, step="test", durations=dur, return_aux=True, prosody=pros)
    ctrl, _ = prosody.pack(pros, 1)
    want = prosody_ref.apply_tracks(aux0["F0"], aux0["N"], aux0["EMA"], aux0["mel_lengths"], ctrl,
                                    *model.prosody_constants())
    for k, w in zip(("F0", "N", "EMA"), want):
        assert torch.equal(aux[k], w), k
        assert not torch.equal(aux[k], aux0[k]), k
    assert model.prosody_constants() == (float(model.distribution["pitch_mean"]),
                                         float(model.distribution["pitch_std"]),
                                         float(model.distribution["energy_std"]))
    # the decoder (reference signature) on the edited tracks
    L = int(aux["mel_lengths"].max()) // 2
    a_cl, _ = ops.length_regulate(aux["T_en"], dur.to(torch.int32), batch[1].to(torch.int32), 1, L)
    cf = lambda t: t.transpose(1, 2)
    for b in range(2):                                             # batch-1 decoder runs at each utterance's length
        Tm = int(aux["mel_lengths"][b])
        ref = model.decoder(cf(a_cl[b:b + 1, :Tm // 2]), aux["style"][b:b + 1],
                            *(cf(w[b:b + 1, :Tm]) for w in want))
        assert (mel[b, :, :Tm] - ref[0]).abs().max().item() < 1e-4, b
    with pytest.raises(ValueError):
        model(batch, step="test", durations=dur, prosody=[Prosody(duration_scale=2.0), Prosody()])


def test_identity_prosody_equals_no_prosody(sim, monkeypatch):
    model, g = _model(sim, monkeypatch)
    c = g["cases"]["a_pred_dur"]
    batch = [c["tokens"], torch.tensor([c["tokens"].shape[1]]), c["ref_mel"], torch.tensor([c["ref_mel"].shape[2]])]
    mel0, aux0 = model(batch, step="test", return_aux=True)
    mel1, aux1 = model(batch, step="test", return_aux=True, prosody=[Prosody()])
    assert torch.equal(mel0, mel1)
    for k in ("F0", "N", "EMA", "pred_dur", "duration", "mel_lengths"):
        assert torch.equal(aux0[k], aux1[k]), k


def test_duration_scale_on_predicted_durations(sim, monkeypatch):
    """pred_dur = round(duration * scale).clamp(min=1); ``duration`` stays the predictor's raw output."""
    model, g = _model(sim, monkeypatch)
    c = g["cases"]["a_pred_dur"]
    Tt = c["tokens"].shape[1]
    batch = [c["tokens"], torch.tensor([Tt]), c["ref_mel"], torch.tensor([c["ref_mel"].shape[2]])]
    _, aux0 = model(batch, step="test", return_aux=True)
    per_token = [4.0 + 0.5 * (i % 12) for i in range(Tt + 3)]     # the random-init predictor gives ~0.1-0.3
    for p in (Prosody(duration_scale=9.0), Prosody(duration_scale=per_token)):
        mel, aux = model(batch, step="test", return_aux=True, prosody=[p])
        _, ds = prosody.pack([p], Tt)
        want, sums = prosody_ref.round_scaled(aux0["duration"], torch.tensor([Tt]), ds)
        assert torch.equal(aux["duration"], aux0["duration"])
        assert torch.equal(aux["pred_dur"], want.float())
        assert int(aux["mel_lengths"][0]) == 2 * int(sums[0]) == mel.shape[2]
        assert int(sums[0]) != int(aux0["pred_dur"].sum())
