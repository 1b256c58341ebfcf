"""Voice enrollment on the GPU: ``as_audio_to_mono`` against the float32 numpy model bit for bit, ``as_trim_bounds``
against the fp64 reference exactly, ``LogMel(starts=)`` against the compacted span bit for bit, batch invariance,
the whole chain stage by stage, and the engine's ``enroll`` against ``encode_voice`` and ``synthesize``."""
import numpy as np
import pytest
import torch

from artspeech_b200 import audio, engine, frontend, ops
from oracle import frontend_oracle as fo
from tests import audio_ref, util
from tests import enroll_ref as R

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 2e-3                   # test_frontend's bound on the normalised log-mel
MARGIN = 1e-9


def _encode(y, encoding):
    """Encoded samples of float32 ``y`` (any shape) as a torch tensor of ``audio.DTYPES[encoding]``."""
    if encoding == "float32":
        return torch.from_numpy(np.ascontiguousarray(y, dtype=np.float32))
    s = np.clip(np.rint(32767 * np.asarray(y, np.float64)), -32768, 32767).astype(np.int64)
    if encoding == "pcm16":
        return torch.from_numpy(s.astype(np.int16))
    return torch.from_numpy((audio_ref.ULAW if encoding == "mulaw" else audio_ref.ALAW)[s + 32768])


def _guarded(rows, S, C, dtype, offset=0):
    """[B, S(, C)] device tensor holding ``rows`` (each [n] or [n, C]) after ``offset`` padding elements, NaN (or the
    largest code) everywhere else: beyond each length, in the row padding and before the first row."""
    fill = float("nan") if dtype == torch.float32 else (127 if dtype == torch.uint8 else 32767)
    B = len(rows)
    ld = S * C + 3                                           # a row stride that is not a multiple of 4
    buf = torch.full((offset + B * ld,), fill, dtype=dtype)
    for b, r in enumerate(rows):
        r = r.reshape(-1)
        buf[offset + b * ld:offset + b * ld + r.numel()] = r
    t = buf.to(DEV)[offset:].as_strided((B, S, C), (ld, C, 1))
    return t[..., 0] if C == 1 else t


@pytest.mark.parametrize("encoding", audio.ENCODINGS)
@pytest.mark.parametrize("C", [1, 2, 3, 6])
def test_audio_to_mono_is_numpys_float32_mean(encoding, C):
    rng = np.random.default_rng(C)
    lens = [0, 1, 1023, 1024, 1025, 4099, 20000]
    S = max(lens) + 5
    rows = [_encode(np.clip(rng.standard_normal((n, C)) * 0.3, -1, 1), encoding) for n in lens]
    for offset in (0, 1):
        x = _guarded(rows, S, C, audio.DTYPES[encoding], offset)
        lt = torch.tensor(lens, dtype=torch.int32, device=DEV)
        out = ops.audio_to_mono(x, lt, encoding).cpu().numpy()
        for b, n in enumerate(lens):
            want = R.to_mono(rows[b].numpy(), encoding)
            assert np.array_equal(out[b, :n].view(np.int32), want.view(np.int32)), (b, n, offset)
            assert not out[b, n:].any()
    if C == 1 and encoding != "float32":                     # as_audio_decode is the C = 1 case, unchanged results
        d = ops.audio_decode(x, encoding).cpu().numpy()
        for b, n in enumerate(lens):
            assert np.array_equal(d[b, :n], R.decode(rows[b].numpy().reshape(-1), encoding))


def _trim_rows(ys, pad=0, stride_extra=0):
    S = max(y.size for y in ys) + pad
    ld = S + stride_extra
    buf = torch.full((len(ys), ld), float("nan"))
    for b, y in enumerate(ys):
        buf[b, :y.size] = torch.from_numpy(y)
    x = buf.to(DEV)[:, :S]
    lens = torch.tensor([y.size for y in ys], dtype=torch.int32, device=DEV)
    return x, lens


def test_trim_bounds_equals_the_fp64_reference():
    clips = R.clip_set()
    excluded = 0
    for start in range(0, len(clips), 16):
        batch = clips[start:start + 16]
        x, lens = _trim_rows(batch, pad=1000, stride_extra=1)
        got = frontend.trim_bounds(x, lens, 30.0).cpu().tolist()
        for y, g in zip(batch, got):
            want, ambiguous = R.trim_blocks(y, 30.0, MARGIN)
            if ambiguous:
                excluded += 1
                continue
            assert tuple(g) == want, (y.size, g, want)
            assert R.trim_librosa(y, 30.0) == want
    assert excluded <= 1
    for top_db in (10.0, 60.0):
        got = frontend.trim_bounds(*_trim_rows(clips[6:14]), top_db=top_db).cpu().tolist()
        for y, g in zip(clips[6:14], got):
            want, ambiguous = R.trim_blocks(y, top_db, MARGIN)
            assert ambiguous or tuple(g) == want


def test_log_mel_span_is_log_mel_of_the_compacted_span():
    rng = np.random.default_rng(3)
    fe = frontend.LogMel().to(DEV)
    spans = [(0, 24000), (517, 9000), (12345, 1025), (3, 30001)]
    S = max(s + n for s, n in spans) + 77
    rows = torch.full((len(spans), S + 5), float("nan"))
    compact = []
    for b, (s, n) in enumerate(spans):
        y = torch.from_numpy((rng.standard_normal(n) * 0.2).astype(np.float32))
        rows[b, s:s + n] = y
        compact.append(y)
    x = rows.to(DEV)[:, :S]
    starts = torch.tensor([s for s, _ in spans], dtype=torch.int32, device=DEV)
    lens = torch.tensor([n for _, n in spans], dtype=torch.int32, device=DEV)
    T = 1 + max(n for _, n in spans) // 300
    out = fe(x, lens, starts=starts, n_frames=T).cpu()
    for b, (s, n) in enumerate(spans):
        alone = fe(compact[b].to(DEV)).cpu()[0]
        nf = 1 + n // 300
        assert torch.equal(out[b, :, :nf], alone), b
        assert float(out[b, :, nf:].abs().max() if nf < T else 0.0) == 0.0
        assert (alone - fo.log_mel(compact[b])[0]).abs().max().item() <= TOL


def _ragged(recs, C, encoding, pad, stride_extra):
    """Host [B, S(, C)] of ``recs`` padded to their longest plus ``pad`` and viewed with a wider row stride."""
    S = max(r.shape[0] for r in recs) + pad
    buf = torch.zeros((len(recs), S + stride_extra) + ((C,) if C > 1 else ()), dtype=audio.DTYPES[encoding])
    for b, r in enumerate(recs):
        buf[b, :r.shape[0]] = r
    return buf[:, :S], [r.shape[0] for r in recs]


def _recording(rng, seconds, rate, C, encoding):
    n = int(seconds * rate)
    y = np.zeros((n, C))
    lead, trail = int(rng.uniform(0.2, 0.6) * rate), int(rng.uniform(0.2, 0.6) * rate)
    k = np.arange(n - lead - trail)
    for c in range(C):
        y[lead:n - trail, c] = 0.3 * np.sin(2 * np.pi * (150 + 40 * c) / rate * k) * \
            (1 + 0.5 * np.sin(2 * np.pi * 3 / rate * k))
    y += rng.standard_normal((n, C)) * 1e-4
    return _encode(np.clip(y if C > 1 else y[:, 0], -1, 1), encoding)


def test_batch_invariance():
    rng = np.random.default_rng(5)
    recs = [_recording(rng, s, 44100, 2, "pcm16") for s in (1.3, 2.7, 0.9)]
    x, lens = _ragged(recs, 2, "pcm16", 0, 0)
    mels, ml, bounds = frontend.reference_mels(x, lens, 44100, "pcm16")
    x2, lens2 = _ragged(recs[::-1] + recs[:1], 2, "pcm16", 4321, 7)
    mels2, ml2, bounds2 = frontend.reference_mels(x2.to(DEV), lens2, 44100, "pcm16")
    for b in range(3):
        alone, ml1, b1 = frontend.reference_mels(recs[b][None].to(DEV), None, 44100, "pcm16")
        j = 2 - b
        assert torch.equal(bounds[b].cpu(), b1[0].cpu()) and torch.equal(bounds2[j].cpu(), b1[0].cpu())
        n = int(ml1[0])
        assert int(ml[b]) == int(ml2[j]) == n
        assert torch.equal(mels[b, :, :n], alone[0]) and torch.equal(mels2[j, :, :n], alone[0])
        assert float(mels[b, :, n:].abs().max() if n < mels.shape[2] else 0) == 0.0
    tb = frontend.trim_bounds(torch.zeros(1, 1, device=DEV), None)       # a lone row of one sample
    assert tb.cpu().tolist() == [[0, 1]]


CASES = [(8000, "mulaw", 1), (8000, "alaw", 1), (16000, "pcm16", 1), (22050, "float32", 1), (44100, "pcm16", 2),
         (48000, "float32", 2), (24000, "float32", 1)]


@pytest.mark.parametrize("rate,encoding,C", CASES)
def test_chain_stage_by_stage(rate, encoding, C):
    rng = np.random.default_rng(rate + C)
    recs = [_recording(rng, s, rate, C, encoding) for s in (2.2, 1.1, 3.4)]
    x, lens = _ragged(recs, C, encoding, 100, 3)
    dev_x = x.to(DEV)
    mels, mel_lens, bounds = frontend.reference_mels(dev_x, lens, rate, encoding)
    fmt = audio.to_native_rate(rate)
    lt = torch.tensor(lens, dtype=torch.int32, device=DEV)
    mono = ops.audio_to_mono(dev_x, lt, encoding) if encoding != "float32" or C > 1 else dev_x
    if fmt.is_identity:
        y24, n24 = mono, lt
    else:
        n24 = torch.empty(3, dtype=torch.int32, device=DEV)
        y24 = ops.resample_encode(mono, lt, fmt, fmt.out_samples(x.shape[1]), out_lens=n24)
    mono_h, y24_h, n24_h, b_h = mono.cpu().numpy(), y24.cpu().numpy(), n24.cpu().tolist(), bounds.cpu().tolist()
    for b, n in enumerate(lens):
        m_ref = R.to_mono(recs[b].numpy(), encoding)
        assert np.array_equal(mono_h[b, :n], m_ref)                          # stage 1: bit for bit
        y64, bound = audio_ref.resample64(mono_h[b, :n], fmt.filter64(), fmt.up, fmt.down, fmt.half_len)
        assert n24_h[b] == fmt.out_samples(n) == y64.size
        assert np.all(np.abs(y24_h[b, :y64.size] - y64) <= (fmt.K + 2) * 2.0 ** -24 * bound)   # stage 2
        want, ambiguous = R.trim_blocks(y24_h[b, :y64.size], 30.0, MARGIN)   # stage 3 on the kernel's 24 kHz
        assert ambiguous or tuple(b_h[b]) == want
        assert 0 < want[0] and want[1] < y64.size                            # both silences were cut
        L = want[1] - want[0]
        assert int(mel_lens[b]) == 1 + L // 300
        ref = fo.log_mel(torch.from_numpy(y24_h[b, want[0]:want[1]].copy()))[0]   # stage 4
        assert ref.shape[1] == int(mel_lens[b])
        assert (mels[b, :, :ref.shape[1]].cpu() - ref).abs().max().item() <= TOL
    assert mels.shape == (3, 80, int(mel_lens.max()))


def test_native_rate_without_silence_equals_preprocess():
    rng = np.random.default_rng(11)
    n = 24000 * 2 + 123
    y = (0.3 * np.sin(2 * np.pi * 220 / 24000 * np.arange(n)) + rng.standard_normal(n) * 0.01).astype(np.float32)
    mels, mel_lens, bounds = frontend.reference_mels(torch.from_numpy(y)[None], None, 24000)
    assert bounds.cpu().tolist() == [[0, n]] and mel_lens.tolist() == [1 + n // 300]
    assert torch.equal(mels, frontend.preprocess(y))


@pytest.fixture(scope="module")
def model_gpu():
    g = util.load_golden("acoustic_small.pt")
    m = util.acoustic_model(g["checkpoint_seed"])
    m.set_compute_dtype(torch.float16)
    m = m.to(DEV)
    m.distribution = {k: v.to(DEV) for k, v in m.distribution.items()}
    yield m
    util._MODELS.clear()


def test_enroll_feeds_synthesize(model_gpu):
    gen = util.generator(0).to(DEV)
    rng = np.random.default_rng(13)
    recs = [_recording(rng, s, 16000, 1, "pcm16") for s in (4.0, 3.1)]     # ~3 s spans, as the benchmark's voices
    x, lens = _ragged(recs, 1, "pcm16", 0, 0)
    B, Tt = 2, 24
    gsrc = torch.Generator().manual_seed(9)
    tok = torch.randint(1, 178, (B, Tt), generator=gsrc).to(DEV)
    tl = torch.full((B,), Tt)
    dur = torch.randint(1, 4, (B, Tt), generator=gsrc)
    for use_graph in (False, True):
        syn = engine.Synthesizer(model_gpu, gen, device=DEV, use_cuda_graph=use_graph)
        mels, mel_lens, voice = syn.enroll(x, lens, 16000, "pcm16")
        assert mel_lens[0] != mel_lens[1]                                    # a ragged batch of voices
        again = syn.encode_voice(mels, mel_lens)
        assert len(voice) == len(again) == 4 and all(torch.equal(a, b) for a, b in zip(voice, again))
        full, _, mel_full = syn.synthesize(tok, tl, mels, mel_lens, dur)
        full, mel_full = full.clone(), mel_full.clone()
        for _ in range(2):
            cached, _, mel_cached = syn.synthesize(tok, tl, mels, mel_lens, dur, voice=voice)
        assert torch.equal(mel_cached, mel_full) and torch.equal(cached, full), f"graph={use_graph}"
