"""Prosody controls on the GPU: ``as_prosody_apply`` and ``as_round_durations_scaled`` against the fp64 restatement
(tests/prosody_ref.py), per-utterance batch invariance of the edits, and the controls as graph inputs of the serving
engine."""
import pytest
import torch

from artspeech_b200 import checkpoint, ops, prosody
from artspeech_b200.prosody import Prosody
from tests import prosody_ref, util

pytestmark = pytest.mark.gpu
DEV = "cuda"
CONSTS = prosody.constants(checkpoint.default_distribution())


def _tracks(B, Tm, seed):
    g = torch.Generator().manual_seed(seed)
    f0 = torch.randn(B, Tm, 1, generator=g) * 0.8
    f0[torch.rand(B, Tm, 1, generator=g) < 0.3] = -1.5             # 20 Hz: unvoiced
    n = torch.randn(B, Tm, 1, generator=g) * 2
    ema = torch.randn(B, Tm, 10, generator=g) + torch.linspace(-0.5, 0.5, 10)
    return f0, n, ema


def _apply(f0, n, ema, lens, ctrl):
    out = [t.to(DEV).contiguous() for t in (f0, n, ema)]
    ops.prosody_apply(*out, lens.to(DEV, torch.int32), ctrl.to(DEV), *CONSTS)
    torch.cuda.synchronize()
    return [t.cpu() for t in out]


def test_prosody_apply_matches_restatement_and_is_batch_invariant():
    B, Tm = 7, 300
    f0, n, ema = _tracks(B, Tm, 0)
    f0[3] = -1.5                                                   # no voiced frame
    lens = torch.tensor([300, 1, 157, 240, 299, 64, 300])
    pros = [Prosody(pitch_shift=3.0, pitch_range=1.2, energy_db=2.0, articulation_scale=[1.1] * 10),
            Prosody(pitch_shift=-5.0, energy_db=-6.0, articulation_offset=[0.3] * 10),
            Prosody(pitch_range=0.0),                                              # monotone, other tracks identity
            Prosody(pitch_shift=7.0, articulation_scale=[0.5 + 0.1 * i for i in range(10)]),
            Prosody(energy_db=1.5),                                                # energy only
            Prosody(),                                                             # identity: nothing written
            Prosody(pitch_shift=12.0, pitch_range=0.3, energy_db=-3.0,
                    articulation_scale=[0.0] * 10, articulation_offset=[-0.2 * i for i in range(10)])]
    ctrl, _ = prosody.pack(pros, 1)
    got = _apply(f0, n, ema, lens, ctrl)
    want = prosody_ref.apply_tracks(f0, n, ema, lens, ctrl, *CONSTS)
    for name, g_, w, x in zip(("F0", "N", "EMA"), got, want, (f0, n, ema)):
        for b in range(B):
            L = int(lens[b])
            torch.testing.assert_close(g_[b, :L], w[b, :L], rtol=1e-5, atol=1e-12, msg=f"{name} utterance {b}")
            assert torch.equal(g_[b, L:], x[b, L:]), (name, b)                     # beyond the length: untouched
    assert torch.equal(got[0][3], f0[3])                                           # no voiced frame
    assert torch.equal(got[1][2], n[2]) and torch.equal(got[2][2], ema[2]) and torch.equal(got[2][4], ema[4])
    assert torch.equal(got[0][4], f0[4]) and all(torch.equal(g_[5], x[5]) for g_, x in zip(got, (f0, n, ema)))
    assert not torch.equal(got[0][0], f0[0]) and not torch.equal(got[2][6], ema[6])
    # the same utterance alone, and inside a larger frame bucket with other batch-mates: the same bits
    for b in (0, 2, 6):
        L = int(lens[b])
        alone = _apply(f0[b:b + 1, :L], n[b:b + 1, :L], ema[b:b + 1, :L], lens[b:b + 1], ctrl[b:b + 1])
        big = [torch.cat([torch.randn(2, 480, t.shape[2]), torch.zeros(1, 480, t.shape[2])]) for t in (f0, n, ema)]
        for t, x in zip(big, (f0, n, ema)):
            t[2, :Tm] = x[b]
        inb = _apply(*big, torch.tensor([480, 333, L]), torch.cat([ctrl[[6, 1]], ctrl[b:b + 1]]))
        for a, c, g_ in zip(alone, inb, got):
            assert torch.equal(a[0], g_[b, :L]) and torch.equal(c[2, :L], g_[b, :L]), b


def test_round_durations_scaled():
    g = torch.Generator().manual_seed(0)
    B, Tt = 7, 93
    pred = torch.randn(B, Tt, generator=g) * 3 + 2
    pred[0, :6] = torch.tensor([0.25, 0.75, 1.25, -0.5, 0.1, 3.0])
    lens = torch.tensor([93, 1, 50, 92, 33, 64, 2], dtype=torch.int32)
    per_token = torch.rand(B, Tt + 4, generator=g) * 3 + 0.2
    per_token[0, :6] = torch.tensor([2.0, 2.0, 2.0, 1.0, 4.0, 0.5])   # ties: 0.5, 1.5, 2.5
    per_utt = torch.rand(B, generator=g) * 2 + 0.5
    for scale in (per_token, per_utt):
        dur, sums = ops.round_durations(pred.to(DEV), lens.to(DEV), scale.to(DEV))
        want, wsum = prosody_ref.round_scaled(pred, lens, scale)
        assert torch.equal(dur.cpu(), want) and torch.equal(sums.cpu(), wsum)
    d0, s0 = ops.round_durations(pred.to(DEV), lens.to(DEV))
    d1, s1 = ops.round_durations(pred.to(DEV), lens.to(DEV), torch.ones(B, Tt, device=DEV))
    assert torch.equal(d0, d1) and torch.equal(s0, s1)


@pytest.fixture(scope="module")
def model_gpu():
    g = util.load_golden("acoustic_small.pt")
    m = util.acoustic_model(g["checkpoint_seed"])
    m.set_compute_dtype(torch.float16)
    m = m.to(DEV)
    m.distribution = {k: v.to(DEV) for k, v in m.distribution.items()}
    yield m, util.generator(0).to(DEV)
    util._MODELS.clear()


def _inputs(seed, tl, Tr=110):
    gsrc = torch.Generator().manual_seed(seed)
    B, Tt = len(tl), max(tl)
    tok = torch.randint(1, 178, (B, Tt), generator=gsrc)
    for b in range(B):
        tok[b, tl[b]:] = 0
    mel = (torch.randn(B, 80, Tr, generator=gsrc) * 0.5).clamp(-2, 2)
    dur = torch.randint(1, 4, (B, Tt), generator=gsrc)
    return tok, mel, dur


def _random_prosody(gsrc, n_tokens, scale_durations=False):
    r = lambda lo, hi: float(lo + (hi - lo) * torch.rand((), generator=gsrc))
    return Prosody(duration_scale=[r(4.0, 8.0) for _ in range(n_tokens)] if scale_durations else 1.0,
                   pitch_shift=r(-6, 6), pitch_range=r(0, 1.5), energy_db=r(-4, 4),
                   articulation_scale=[r(0.7, 1.3) for _ in range(10)],
                   articulation_offset=[r(-0.2, 0.2) for _ in range(10)])


def test_one_graph_serves_changing_prosody(model_gpu):
    """Forced durations: ONE captured graph serves calls whose controls change every call, each equal to the eager
    pass; a controlled graph has one launch more than the uncontrolled one, which keeps its own launch count."""
    from artspeech_b200 import engine
    model, gen = model_gpu
    tl = [40, 33, 12]
    plain = engine.Synthesizer(model, gen, device=DEV, use_cuda_graph=True)
    tok, mel, dur = _inputs(3, tl)
    dur[0] = 3
    plain.synthesize(tok.to(DEV), tl, mel.to(DEV), [110] * 3, dur)
    base_launches = plain.launches_per_call
    graph = engine.Synthesizer(model, gen, device=DEV, use_cuda_graph=True)
    eager = engine.Synthesizer(model, gen, device=DEV, use_cuda_graph=False)
    gsrc = torch.Generator().manual_seed(5)
    for step in range(4):
        pros = [_random_prosody(gsrc, t) for t in tl]
        if step == 2:
            pros[1] = Prosody()                                            # identity beside edited utterances
        wg, lg, mg = graph.synthesize(tok.to(DEV), tl, mel.to(DEV), [110] * 3, dur, prosody=pros)
        wg, mg = wg.clone(), mg.clone()
        assert graph.launches_per_call == base_launches + 1
        we, le, me = eager.synthesize(tok.to(DEV), tl, mel.to(DEV), [110] * 3, dur, prosody=pros)
        assert lg.tolist() == le.tolist()
        for b in range(3):
            n = int(lg[b])
            assert (mg[b, :, :n] - me[b, :, :n]).abs().max().item() <= 2e-3, (step, b)
            assert util.snr_db(wg[b, :300 * n].cpu(), we[b, :300 * n].cpu()) >= 50.0, (step, b)
        graph.synthesize(tok.to(DEV), tl, mel.to(DEV), [110] * 3, dur)      # uncontrolled calls in between
        assert graph.launches_per_call == base_launches
    assert graph.stats["captures"] == 2 and graph.stats["eager"] == 0        # one controlled + one plain graph
    with pytest.raises(ValueError):
        graph.synthesize(tok.to(DEV), tl, mel.to(DEV), [110] * 3, dur, prosody=[Prosody(duration_scale=2.0)] * 3)


def test_identity_prosody_is_bit_identical(model_gpu):
    from artspeech_b200 import engine
    model, gen = model_gpu
    tl = [40, 25]
    tok, mel, _ = _inputs(7, tl)
    syn = engine.Synthesizer(model, gen, device=DEV, use_cuda_graph=True)
    for _ in range(2):
        w0, l0, m0 = syn.synthesize(tok.to(DEV), tl, mel.to(DEV), [110] * 2, None)
        w0, l0, m0, d0 = w0.clone(), l0.clone(), m0.clone(), syn.last["pred_dur"].clone()
        w1, l1, m1 = syn.synthesize(tok.to(DEV), tl, mel.to(DEV), [110] * 2, None, prosody=[Prosody()] * 2)
        assert torch.equal(w0, w1) and torch.equal(m0, m1) and torch.equal(l0, l1)
        assert torch.equal(d0, syn.last["pred_dur"])


def test_duration_scale_sets_frame_counts(model_gpu):
    """Predicted durations with duration_scale: 2 * sum(round(pred * scale)) frames on the two-graph path and on the
    bounded single-graph path."""
    from artspeech_b200 import engine
    model, gen = model_gpu
    tl = [40, 25, 33]
    tok, mel, _ = _inputs(11, tl)
    gsrc = torch.Generator().manual_seed(2)
    pros = [Prosody(duration_scale=6.0), _random_prosody(gsrc, 25, True), Prosody(duration_scale=4.5, pitch_shift=2)]
    two = engine.Synthesizer(model, gen, device=DEV, use_cuda_graph=True)
    bounded = engine.Synthesizer(model, gen, device=DEV, use_cuda_graph=True, duration_bound=4.0)
    _, ds = prosody.pack(pros, 40)
    for _ in range(2):
        w, lens, _ = two.synthesize(tok.to(DEV), tl, mel.to(DEV), [110] * 3, None, prosody=pros)
        want, sums = prosody_ref.round_scaled(two.last["duration"][:, :40].cpu(), torch.tensor(tl), ds)
        assert two.last["frames"] == [2 * int(s) for s in sums] and lens.tolist() == two.last["frames"]
        assert torch.equal(two.last["pred_dur"][:, :40].cpu(), want)
        wb, lb, _ = bounded.synthesize(tok.to(DEV), tl, mel.to(DEV), [110] * 3, None, prosody=pros)
        torch.cuda.synchronize()
        assert lb.tolist() == two.last["frames"] and int(bounded.last["pred_sum"].max()) * 2 <= bounded.last["frame_bound"]
        for b in range(3):
            n = two.last["frames"][b]
            assert util.snr_db(wb[b, :300 * n].cpu(), w[b, :300 * n].cpu()) >= 50.0, b
    assert two.stats["eager"] == 0 and bounded.stats["eager"] == 0


def test_synthesize_many_gives_each_utterance_its_own_prosody(model_gpu):
    """pipeline_depth=2 with a different Prosody per utterance: every utterance equals its own batch-1 call."""
    from artspeech_b200 import engine
    model, gen = model_gpu
    syn = engine.Synthesizer(model, gen, device=DEV, use_cuda_graph=True, pipeline_depth=2)
    one = engine.Synthesizer(model, gen, device=DEV, use_cuda_graph=False)
    gsrc = torch.Generator().manual_seed(21)
    tl = [15, 90, 33, 61, 47, 120, 18]
    toks = [torch.randint(1, 178, (t,), generator=gsrc) for t in tl]
    mels = [(torch.randn(80, 120, generator=gsrc) * 0.5).clamp(-2, 2) for _ in tl]
    pros = [_random_prosody(gsrc, t, scale_durations=i % 2 == 0) for i, t in enumerate(tl)]
    for _ in range(2):
        wavs, frames = engine.synthesize_many(syn, toks, mels, None, max_batch=3, to_host=True, prosody=pros)
    for i in range(len(tl)):
        w1, _, _ = one.synthesize(toks[i].view(1, -1).to(DEV), [tl[i]], mels[i].unsqueeze(0).to(DEV), [120], None,
                                  prosody=[pros[i]])
        assert frames[i] == one.last["frames"][0] and wavs[i].numel() == 300 * frames[i], i
        assert util.snr_db(wavs[i], w1[0, :300 * frames[i]].cpu()) >= 50.0, i
