"""FLAC output on the GPU: ``ops.flac_encode`` byte for byte against the restatement (tests/flac_ref.py), its
invariance to batch composition, padding and row stride, and the engine's FLAC format end to end (decoded files equal
the raw PCM16 of the same call, with loudness and the watermark, on the eager, graph and pipelined paths)."""
import numpy as np
import pytest
import torch

from artspeech_b200 import engine, ops
from artspeech_b200.audio import AudioFormat, Loudness, Watermark, detect_watermark, encode_flac
from tests import audio_ref, denoise_ref, enroll_ref, util
from tests import flac_ref as F

pytestmark = pytest.mark.gpu
DEV = "cuda"
GUARD = 8
KEY = 0x0123456789ABCDEF


def _pcm16(y):
    return np.clip(np.rint(32767.0 * np.asarray(y, np.float64)), -32768, 32767).astype(np.int16)


def _rows(sigs, S, guard=GUARD, seed=0):
    """[B, guard + S + guard] int16 with random values everywhere but each row's signal; returns the [B, S] view."""
    rng = np.random.default_rng(seed)
    buf = torch.from_numpy(rng.integers(-32768, 32768, (len(sigs), guard + S + guard)).astype(np.int16))
    for b, v in enumerate(sigs):
        buf[b, guard:guard + len(v)] = torch.from_numpy(np.asarray(v, dtype=np.int16))
    return buf.to(DEV)[:, guard:guard + S]


def _check_against_reference(sigs, rate, S=None):
    S = max(len(s) for s in sigs) + 5 if S is None else S
    x = _rows(sigs, S)
    lens = torch.tensor([len(s) for s in sigs], dtype=torch.int32, device=DEV)
    out, nb = ops.flac_encode(x, lens, rate)
    out, nb = out.cpu(), nb.cpu()
    assert out.shape == (len(sigs), F.bound(S))
    for b, s in enumerate(sigs):
        want = F.encode(np.asarray(s, np.int16), rate)
        got = bytes(out[b, :int(nb[b])].numpy())
        assert int(nb[b]) == len(want) and got == want, (rate, b, len(s), int(nb[b]), len(want))
        assert not out[b, int(nb[b]):].any()
    return out, nb


def test_corpus_matches_the_reference():
    rng = np.random.default_rng(1)
    t = np.arange(12293)
    edge = [rng.integers(-32768, 32768, n) for n in (0, 1, 15, 16, 17, 4095, 4096, 4097, 12293)]
    edge += [np.zeros(5000), np.full(4200, -1234), np.where((t // 37) % 2, 32767, -32768),
             np.clip(np.rint(40000.0 * np.sin(2 * np.pi * 440.0 * t / 24000)), -32768, 32767)]
    _check_against_reference(edge, 24000)
    clips = [c[:3 * 24000] for c in denoise_ref.voiced_set(seed=3, count=2)]
    clips += [enroll_ref.speech_like(rng, int(2.5 * 24000)) for _ in range(2)]
    for rate in (8000, 12000, 16000, 22050, 24000, 44100, 48000):
        fmt = AudioFormat(rate, "pcm16")
        sigs = [_pcm16(audio_ref.resample64(c, fmt.filter64(), fmt.up, fmt.down, fmt.half_len)[0]) for c in clips]
        _check_against_reference(sigs, rate)


@pytest.mark.parametrize("B,seconds", [(16, 10), (8, 60)])
def test_long_batches_match_the_reference(B, seconds):
    rng = np.random.default_rng(B)
    n = 24000 * seconds
    sigs = [_pcm16(enroll_ref.speech_like(rng, n - int(rng.integers(0, 24000)))) for _ in range(B)]
    _check_against_reference(sigs, 24000, S=n)


def test_rows_do_not_depend_on_their_batch():
    rng = np.random.default_rng(7)
    sigs = [_pcm16(denoise_ref.voiced(rng, n) if n else np.zeros(0)) for n in (50000, 12345, 0, 99999, 4096)]
    x = _rows(sigs, 100003)
    lens = torch.tensor([len(s) for s in sigs], dtype=torch.int32, device=DEV)
    out, nb = ops.flac_encode(x, lens, 16000)
    for b, s in enumerate(sigs):
        n = len(s)
        for S, g in ((n, 0), (n + 5, 3), (n + 4097, 1)):
            xb = _rows([s], S, guard=g + 4, seed=b + S)
            o1, n1 = ops.flac_encode(xb, torch.tensor([n], dtype=torch.int32, device=DEV), 16000)
            assert int(n1[0]) == int(nb[b]) and torch.equal(o1[0, :int(nb[b])], out[b, :int(nb[b])]), (b, S)
            assert not o1[0, int(n1[0]):].any()
    # no lengths: every row holds S samples; a [S] tensor is one row
    full = torch.from_numpy(sigs[4]).to(DEV)
    o2, n2 = encode_flac(full, None, 16000)
    assert bytes(o2[0, :int(n2[0])].cpu().numpy()) == F.encode(sigs[4], 16000)
    assert int(nb[2]) == 42


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


def _decode_rows(y, nb):
    y, nb = y.cpu(), nb.cpu()
    return [F.decode(bytes(y[b, :int(nb[b])].numpy())) for b in range(y.shape[0])]


@pytest.mark.parametrize("graph,depth", [(False, 1), (True, 1), (True, 2)])
def test_engine_flac_decodes_to_the_raw_samples(model_gpu, graph, depth):
    model, gen = model_gpu
    tl = [90, 70, 50]
    tok, mel, dur = _inputs(11 + depth, tl)
    syn = engine.Synthesizer(model, gen, device=DEV, use_cuda_graph=graph, pipeline_depth=depth)
    args = (tok.to(DEV), tl, mel.to(DEV), [110] * 3, dur)
    for _ in range(depth + 1):
        syn.synthesize(*args)
    syn.join()
    caps = syn.stats["captures"]
    wm = Watermark(KEY, 0x0F1A)
    for rate, kw in ((16000, {}), (12000, {}), (24000, {"loudness": Loudness(-16.0)}),
                     (8000, {"loudness": Loudness(), "watermark": wm})):
        raw_fmt = AudioFormat(rate, "pcm16")
        fmt = AudioFormat(rate, "pcm16", container="flac")
        raw, _, _ = syn.synthesize(*args, audio=raw_fmt, **kw)
        base = syn.launches_per_call
        syn.join()
        raw = raw.clone()
        n = syn.last["sample_lengths"].clone()
        y, _, _ = syn.synthesize(*args, audio=fmt, **kw)
        syn.join()
        if graph:
            assert syn.launches_per_call == base + ops.FLAC_LAUNCHES
        y, nb = y.clone(), syn.last["byte_lengths"].clone()
        torch.cuda.synchronize()
        assert y.dtype == torch.uint8 and y.shape[1] == F.bound(raw.shape[1])
        assert torch.equal(syn.last["sample_lengths"].cpu(), n.cpu())
        for b, (x, r) in enumerate(_decode_rows(y, nb)):
            assert r == rate and np.array_equal(x, raw[b, :int(n[b])].cpu().numpy()), (rate, b)
            assert not y[b, int(nb[b]):].any()
        if "watermark" in kw:
            for b, (x, _) in enumerate(_decode_rows(y, nb)):
                if x.size >= 2 * rate:
                    det, score, msg = detect_watermark(torch.from_numpy(x).to(DEV), None, rate, KEY,
                                                       encoding="pcm16")
                    assert bool(det[0]) and int(msg[0]) == 0x0F1A, (b, float(score[0]))
    assert syn.stats["captures"] == caps


def test_synthesize_many_files_equal_single_calls(model_gpu):
    model, gen = model_gpu
    fmt = AudioFormat(16000, "pcm16", container="flac")
    syn = engine.Synthesizer(model, gen, device=DEV, use_cuda_graph=True, pipeline_depth=2)
    gsrc = torch.Generator().manual_seed(43)
    tl = [60, 150, 90, 120, 75]
    toks = [torch.randint(1, 178, (t,), generator=gsrc) for t in tl]
    mels = [(torch.randn(80, 120, generator=gsrc) * 0.5).clamp(-2, 2) for _ in tl]
    durs = [torch.randint(2, 6, (t,), generator=gsrc) for t in tl]
    for to_host in (True, False):
        files, frames = engine.synthesize_many(syn, toks, mels, durs, max_batch=2, to_host=to_host, audio=fmt)
        torch.cuda.synchronize()
        for i in range(len(tl)):
            one, _ = engine.synthesize_many(syn, [toks[i]], [mels[i]], [durs[i]], to_host=True, audio=fmt)
            assert files[i].dtype == torch.uint8 and torch.equal(files[i].cpu(), one[0].cpu()), i
            x, r = F.decode(bytes(files[i].cpu().numpy()))
            assert r == 16000 and x.size == fmt.out_samples(300 * frames[i])
