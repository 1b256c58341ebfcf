"""The synthesis watermark on the GPU: ``as_watermark_embed`` against the fp64 restatement (tests/watermark_ref.py)
with NaN guards, ``as_audio_decode`` against audioop, ``as_watermark_detect`` against the restatement, the bitwise
batch invariance of both, and the engine's watermark stage end to end (every output format detected on the GPU)."""
import audioop

import numpy as np
import pytest
import torch

from artspeech_b200 import engine, ops
from artspeech_b200.audio import AudioFormat, Loudness, Watermark, detect_watermark, embed_watermark
from tests import util
from tests import watermark_ref as W

pytestmark = pytest.mark.gpu
DEV = "cuda"
KEY, MSG = 0x0123456789ABCDEF, 0xBEEF
GUARD = 16


def _rows(sigs, S, guard=GUARD):
    """[B, guard + S + guard] fp32 with NaN everywhere but each row's signal; returns (buffer, the [B, S] view)."""
    buf = torch.full((len(sigs), guard + S + guard), float("nan"))
    for b, v in enumerate(sigs):
        buf[b, guard:guard + len(v)] = torch.from_numpy(np.asarray(v, dtype=np.float32))
    return buf.to(DEV), buf.to(DEV)[:, guard:guard + S]


LENS = (0, 1, 119, 239, 240, 241, 7679, 7680, 7681, 12289, 72017, 1440000)


def test_embed_against_the_reference():
    rng = np.random.default_rng(0)
    wm = Watermark(KEY, MSG, -30.0)
    S = max(LENS) + 37
    sigs = [W.speech(n, rng) if n > 480 else 0.2 * rng.standard_normal(n) for n in LENS]
    _, x = _rows(sigs, S)
    lens = torch.tensor(LENS, dtype=torch.int32, device=DEV)
    y = ops.watermark_embed(x, lens, wm).cpu().numpy()
    c = W.mark(KEY, MSG)
    worst = 0.0
    for b, n in enumerate(LENS):
        assert not y[b, n:].any(), b                                       # zeros beyond n, NaN guards never read
        if n == 0:
            continue
        xs = np.asarray(sigs[b], dtype=np.float32).astype(np.float64)
        ref = W.embed(xs, KEY, MSG, -30.0)
        mark = wm.alpha * W.envelope(xs, 240) * np.abs(c[np.arange(n) % W.P24])
        bound = 2.0 ** -23 * np.abs(xs) + 1e-4 * mark + 1e-30
        err = np.abs(y[b, :n] - ref) / bound
        worst = max(worst, err.max())
        assert err.max() <= 1.0, (n, err.max())
    print(f"embed: largest err / bound {worst:.3f}")


def test_embed_is_batch_invariant():
    rng = np.random.default_rng(1)
    lens = [50000, 12345, 0, 99999]
    sigs = [W.speech(n, rng) if n else np.zeros(0) for n in lens]
    wm = Watermark(KEY, 0x1234, -20.0)
    _, x = _rows(sigs, 100003)
    y = ops.watermark_embed(x, torch.tensor(lens, dtype=torch.int32, device=DEV), wm)
    for b, n in enumerate(lens):
        for S, g in ((n, 0), (n + 5, 3)):
            _, xb = _rows([sigs[b]], S, guard=g + 4 if g else 4)
            yb = ops.watermark_embed(xb, torch.tensor([n], dtype=torch.int32, device=DEV), wm)
            assert torch.equal(yb[0, :n], y[b, :n]), (b, S)
    assert not y[2].any()


def test_decode_against_audioop():
    codes = torch.arange(256, dtype=torch.uint8).view(1, -1).repeat(3, 1)
    for enc, fn in (("mulaw", audioop.ulaw2lin), ("alaw", audioop.alaw2lin)):
        got = ops.audio_decode(codes.to(DEV), enc).cpu().numpy()
        want = np.frombuffer(fn(bytes(range(256)), 2), "<i2") / 32768.0
        assert np.array_equal(got[1], want), enc
    v = torch.tensor([[-32768, -1, 0, 1, 32767, 1234, -4321]], dtype=torch.int16)
    assert torch.equal(ops.audio_decode(v.to(DEV), "pcm16").cpu(), v.float() / 32768.0)


def _clips(seed, specs):
    """8 kHz fp32 clips (fp64 reference chain through 24 kHz -> 8 kHz) of ``specs`` = [(seconds, marked, msg)]."""
    rng = np.random.default_rng(seed)
    out = []
    for dur, marked, msg in specs:
        x = W.speech(int(dur * 24000) + 6000, rng)
        y = W.embed(x, KEY, msg) if marked else x
        y = -0.5 * y[int(rng.integers(0, 6000)):][:int(dur * 24000)]
        out.append(W.to_8k(y, 24000).astype(np.float32))
    return out


def test_detect_against_the_reference():
    specs = [(2.0, True, 1), (3.0, True, 0xBEEF), (10.0, True, 0xFFFF), (5.5, True, 0x0100), (4.0, False, 0),
             (9.0, False, 0), (0.0, False, 0), (0.3, True, 7)]
    clips = _clips(2, specs)
    S = max(len(c) for c in clips) + 100
    _, x = _rows(clips, S)
    lens = torch.tensor([len(c) for c in clips], dtype=torch.int32, device=DEV)
    det, score, lag, msg = [t.cpu() for t in ops.watermark_detect(x, lens, KEY)]
    worst = 0.0
    for b, c in enumerate(clips):
        d, s, tau, m = W.detect(c.astype(np.float64), KEY)
        if s == 0.0:
            assert float(score[b]) == 0.0 and not bool(det[b])
            continue
        rel = abs(float(score[b]) - s) / s
        worst = max(worst, rel)
        assert rel <= 1e-3, (b, float(score[b]), s)
        if abs(s - 6.0) > 0.1:
            assert bool(det[b]) == d, b
        if specs[b][1] and s >= 7.0:
            assert int(lag[b]) == tau and int(msg[b]) == m == specs[b][2], (b, int(lag[b]), tau, int(msg[b]), m)
    print(f"detect: largest relative score error {worst:.2e}; scores {score.tolist()}")
    # batch invariance: each row alone, another S and row stride, gives the same bits
    for b, c in enumerate(clips):
        _, xb = _rows([c], len(c) + 4096 * (b % 3), guard=4)
        r = ops.watermark_detect(xb, torch.tensor([len(c)], dtype=torch.int32, device=DEV), KEY)
        assert float(r[1][0]) == float(score[b]) and int(r[2][0]) == int(lag[b]) and int(r[3][0]) == int(msg[b]), b


@pytest.mark.parametrize("rate,enc", [(8000, "mulaw"), (8000, "alaw"), (16000, "pcm16"), (48000, "float32"),
                                      (44100, "mulaw"), (22050, "pcm16")])
def test_detect_watermark_through_the_product_chain(rate, enc):
    """GPU embed -> GPU format (resample + encode) -> GPU detect_watermark: the key and message come back, unmarked
    audio stays below the threshold."""
    rng = np.random.default_rng(rate)
    sigs = [W.speech(n, rng) for n in (24000 * 3, 24000 * 7 + 11, 24000 * 12)]
    _, x = _rows(sigs, max(len(s) for s in sigs))
    lens = torch.tensor([len(s) for s in sigs], dtype=torch.int32, device=DEV)
    f = AudioFormat(rate, enc)
    wm = Watermark(KEY, 0x5A17)
    for marked in (True, False):
        y = embed_watermark(x, lens, wm) if marked else torch.nan_to_num(x, nan=0.0)
        n = torch.empty(3, dtype=torch.int32, device=DEV)
        out = ops.resample_encode(y, lens, f, f.out_samples(x.shape[1]), out_lens=n)
        det, score, msg = detect_watermark(out, n, rate, KEY, encoding=enc)
        assert det.tolist() == [marked] * 3, (marked, score.tolist())
        if marked:
            assert msg.tolist() == [0x5A17] * 3
        else:
            assert score.max().item() < 6.0


# ---- engine -------------------------------------------------------------------------------------------------------
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
    dur = torch.randint(2, 6, (B, Tt), generator=gsrc)
    return tok, mel, dur


@pytest.mark.parametrize("depth", [1, 2])
@pytest.mark.parametrize("mode", ["forced", "predicted", "bounded"])
def test_engine_watermark_stage(model_gpu, mode, depth):
    """A marked call is its unmarked pass plus one embed launch: bit-identical to ``embed_watermark`` of that pass's
    waveform; every format's bytes give the key and message back on the GPU; unmarked calls are not detected."""
    model, gen = model_gpu
    tl = [100, 80, 60]
    tok, mel, dur = _inputs(5 + depth, tl)
    dur = dur if mode == "forced" else None
    kw = dict(duration_bound=6.0) if mode == "bounded" else {}
    syn = engine.Synthesizer(model, gen, device=DEV, use_cuda_graph=True, pipeline_depth=depth, **kw)
    args = (tok.to(DEV), tl, mel.to(DEV), [110] * 3, dur)
    for _ in range(depth):
        syn.synthesize(*args)
    base, caps = syn.launches_per_call, syn.stats["captures"]
    wm = Watermark(KEY, 0x0B0E)
    w0, l0, _ = syn.synthesize(*args)
    syn.join()
    w0 = w0.clone()
    n24 = [300 * int(v) for v in l0.cpu()]
    y, l1, _ = syn.synthesize(*args, watermark=wm)
    assert syn.launches_per_call == base + 1 and "sample_lengths" not in syn.last
    syn.join()
    y = y.clone()
    torch.cuda.synchronize()
    assert torch.equal(l0, l1)
    assert torch.equal(y, embed_watermark(w0, torch.tensor(n24, dtype=torch.int32), wm))
    long_enough = [n >= 2 * 24000 for n in n24]
    det, _, msg = detect_watermark(y, torch.tensor(n24, dtype=torch.int32), 24000, KEY)
    for b in range(3):
        if long_enough[b]:
            assert bool(det[b]) and int(msg[b]) == 0x0B0E, (mode, b)
    det0, s0, _ = detect_watermark(torch.nan_to_num(w0), torch.tensor(n24, dtype=torch.int32), 24000, KEY)
    assert not det0.any(), s0.tolist()
    for f, loud in ((AudioFormat(8000, "mulaw"), None), (AudioFormat(16000, "pcm16"), Loudness(-16.0)),
                    (AudioFormat(48000, "float32"), None), (AudioFormat(8000, "alaw"), Loudness())):
        y, _, _ = syn.synthesize(*args, audio=f, watermark=wm, **({"loudness": loud} if loud else {}))
        assert syn.launches_per_call == base + 2 + (ops.LOUDNESS_LAUNCHES if loud else 0)
        syn.join()
        y = y.clone()
        n = syn.last["sample_lengths"].clone()
        torch.cuda.synchronize()
        det, score, msg = detect_watermark(y, n, f.sample_rate, KEY, encoding=f.encoding)
        for b in range(3):
            if long_enough[b]:
                assert bool(det[b]) and int(msg[b]) == 0x0B0E, (mode, f, b, score.tolist())
        y0, _, _ = syn.synthesize(*args, audio=f)
        syn.join()
        y0 = y0.clone()
        torch.cuda.synchronize()
        det0, s0, _ = detect_watermark(y0, n, f.sample_rate, KEY, encoding=f.encoding)
        assert not det0.any(), (mode, f, s0.tolist())
    assert syn.stats["captures"] == caps


def test_synthesize_many_mulaw_watermark(model_gpu):
    model, gen = model_gpu
    f = AudioFormat(8000, "mulaw")
    syn = engine.Synthesizer(model, gen, device=DEV, use_cuda_graph=True, pipeline_depth=2)
    gsrc = torch.Generator().manual_seed(41)
    tl = [60, 150, 90, 120, 75]
    toks = [torch.randint(1, 178, (t,), generator=gsrc) for t in tl]
    mels = [(torch.randn(80, 120, generator=gsrc) * 0.5).clamp(-2, 2) for _ in tl]
    durs = [torch.randint(2, 6, (t,), generator=gsrc) for t in tl]
    wm = Watermark(KEY, 4242)
    wavs, frames = engine.synthesize_many(syn, toks, mels, durs, max_batch=2, to_host=True, audio=f, watermark=wm)
    torch.cuda.synchronize()
    for i in range(len(tl)):
        assert wavs[i].dtype == torch.uint8 and wavs[i].numel() == f.out_samples(300 * frames[i]), i
        det, score, msg = detect_watermark(wavs[i].to(DEV), None, 8000, KEY, encoding="mulaw")
        assert bool(det[0]) and int(msg[0]) == 4242, (i, float(score[0]))
