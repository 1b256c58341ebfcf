"""Output audio formats on the GPU: ``as_resample_encode`` against the fp64 restatement (tests/audio_ref.py) for every
listed rate and encoding with out-of-range guards, its bit-for-bit invariants (batch position, bucket size, output
window, 24 kHz PCM equal to the vocoder's own), and the format stage of the serving engine."""
import numpy as np
import pytest
import torch

from artspeech_b200 import engine, ops
from artspeech_b200.audio import ENCODINGS, AudioFormat
from tests import audio_ref, util

pytestmark = pytest.mark.gpu
DEV = "cuda"
RATES = (8000, 11025, 16000, 22050, 24000, 32000, 44100, 48000)
LENS = (0, 1, 299, 300, 24007, 240000)
GUARD = 16                                    # NaN floats before each input row (keeps rows 16-byte aligned)
SENTINEL = {"float32": 1234.5, "pcm16": 0x5A5A, "mulaw": 0xA5, "alaw": 0xA5}


def _signal(lens, S_in, seed, guard=GUARD):
    """[B, guard + S_in + guard] fp32 with NaN everywhere but each row's first ``lens[b]`` samples (a band-limited
    mix with peaks beyond full scale, to exercise saturation); returns (buffer, the [B, S_in] view)."""
    g = torch.Generator().manual_seed(seed)
    B = len(lens)
    buf = torch.full((B, guard + S_in + guard), float("nan"))
    for b, n in enumerate(lens):
        t = torch.arange(n, dtype=torch.float64)
        f = 0.002 + 0.3 * torch.rand((), generator=g, dtype=torch.float64)
        v = 0.6 * torch.sin(f * t) + 0.3 * torch.randn(n, generator=g, dtype=torch.float64)
        v[n // 3:n // 3 + 50] *= 4.0
        buf[b, guard:guard + n] = v.float()
    return buf, buf[:, guard:guard + S_in]


def _run(x, lens, fmt, S_out, m0=0, pad=16):
    """The kernel into a sentinel-padded output; returns (out [B, S_out] on the CPU, out_lens, tail sentinel ok)."""
    B = x.shape[0]
    buf = torch.full((B, S_out + pad), SENTINEL[fmt.encoding], dtype=fmt.dtype, device=DEV)
    n = torch.full((B,), -7, dtype=torch.int32, device=DEV)
    lt = None if lens is None else torch.tensor(lens, dtype=torch.int32, device=DEV)
    ops.resample_encode(x, lt, fmt, S_out, m0=m0, out=buf[:, :S_out], out_lens=n)
    torch.cuda.synchronize()
    buf = buf.cpu()
    return buf[:, :S_out], n.cpu(), bool((buf[:, S_out:] == SENTINEL[fmt.encoding]).all())


@pytest.mark.parametrize("rate", RATES)
def test_kernel_matches_fp64_restatement(rate):
    S_in = max(LENS) + 5
    xbuf, x = _signal(LENS, S_in, rate)
    xd = xbuf.to(DEV)[:, GUARD:GUARD + S_in]
    f0 = AudioFormat(rate)
    refs = [audio_ref.resample64(x[b, :L].double().numpy(), f0.filter64(), f0.up, f0.down, f0.half_len)
            for b, L in enumerate(LENS)]
    for enc in ENCODINGS:
        f = AudioFormat(rate, enc)
        S_out = f.out_samples(S_in)
        got, n, tail_ok = _run(xd, list(LENS), f, S_out)
        assert tail_ok, "write beyond S_out"
        assert n.tolist() == [f.out_samples(v) for v in LENS]
        worst = (0.0, None)
        for b, L in enumerate(LENS):
            y64, s = refs[b]
            bound = (f.K + 2) * 2.0 ** -24 * s
            nb = y64.shape[0]
            g = got[b, :nb].numpy()
            if enc == "float32":
                err = np.abs(g.astype(np.float64) - y64)
                ratio = err / np.maximum(bound, 1e-300)
                if nb and ratio.max() > worst[0]:
                    worst = (float(ratio.max()), (b, int(ratio.argmax()), float(err.max())))
                assert (err <= bound).all(), (enc, b, worst)
            else:
                want, alt = audio_ref.encode(y64, bound, enc)
                ok = (g == want) | (g == alt)
                assert ok.all(), (enc, b, int((~ok).sum()), np.nonzero(~ok)[0][:5])
            assert (got[b, nb:] == f.silence).all(), (enc, b)
        if enc == "float32":
            print(f"{rate} Hz fp32: worst err/bound {worst[0]:.3g} at (utterance, sample, |err|) {worst[1]}")


def test_unaligned_rows_and_row_strides():
    """Input and output rows that are not 16-byte aligned take the element-wise paths: same bits."""
    lens = [24007, 3001, 0]
    xbuf, _ = _signal(lens, 24011, 3, guard=3)
    xa = _signal(lens, 24011, 3)[0].to(DEV)[:, GUARD:GUARD + 24011]
    xu = xbuf.to(DEV)[:, 3:3 + 24011]
    for f in (AudioFormat(16000, "mulaw"), AudioFormat(44100, "float32"), AudioFormat(24000, "pcm16")):
        S_out = f.out_samples(24011)
        a, _, ok_a = _run(xa, lens, f, S_out)
        u, _, ok_u = _run(xu, lens, f, S_out, pad=3)
        assert ok_a and ok_u and torch.equal(a, u), f


@pytest.mark.parametrize("rate,enc", [(8000, "mulaw"), (11025, "alaw"), (22050, "float32"), (48000, "pcm16")])
def test_bitwise_invariants(rate, enc):
    f = AudioFormat(rate, enc)
    lens = [48000, 7, 30011, 47999]
    xbuf, _ = _signal(lens, 48000, 11)
    xd = xbuf.to(DEV)[:, GUARD:GUARD + 48000]
    full, n, _ = _run(xd, lens, f, f.out_samples(48000))
    for b in (0, 2, 3):
        L = lens[b]
        alone, _, _ = _run(xd[b:b + 1, :L].contiguous(), None, f, f.out_samples(L))
        assert torch.equal(alone[0], full[b, :f.out_samples(L)]), ("alone", b)
        # inside a larger bucket, at another batch position, beside other utterances
        big = torch.full((3, 90000), float("nan"), device=DEV)
        big[2, :L] = xd[b, :L]
        big[0, :9000] = 0.25
        inb, _, _ = _run(big, [9000, 0, L], f, f.out_samples(90000))
        assert torch.equal(inb[2, :f.out_samples(L)], full[b, :f.out_samples(L)]), ("bucket", b)
        assert (inb[2, f.out_samples(L):] == f.silence).all()
    # an output window (m0, S_out) is the same slice of the one-shot output
    for m0, S in ((0, 1000), (1, 1), (777, 4096), (f.out_samples(30011) - 5, 40)):
        win, _, ok = _run(xd, lens, f, S, m0=m0)
        assert ok and torch.equal(win, full[:, m0:m0 + S]), (m0, S)


@pytest.fixture(scope="module")
def model_gpu():
    g = util.load_golden("acoustic_small.pt")
    m = util.acoustic_model(g["checkpoint_seed"])
    m.set_compute_dtype(torch.float16)
    m = m.to(DEV)
    m.distribution = {k: v.to(DEV) for k, v in m.distribution.items()}
    yield m, util.generator(0).to(DEV)
    util._MODELS.clear()


def test_generator_formats(model_gpu):
    """24 kHz pcm16 through the format kernel == the vocoder's own AS_PCM16 output; forward(lengths) cuts each
    utterance; stream(audio=) concatenates to forward(audio=)."""
    _, gen = model_gpu
    mel = (torch.randn(2, 80, 50, generator=torch.Generator().manual_seed(4)) * 0.7).to(DEV)
    assert torch.equal(gen(mel, audio=AudioFormat(24000, "pcm16")), gen(mel, pcm16=True))
    assert torch.equal(gen(mel, audio=AudioFormat()), gen(mel))
    lengths = torch.tensor([50, 21], device=DEV)
    for f in (AudioFormat(8000, "mulaw"), AudioFormat(44100, "float32")):
        y = gen(mel, lengths=lengths, audio=f)
        w = gen(mel, lengths=lengths)
        want, _, _ = _run(w.view(2, -1), [15000, 6300], f, f.out_samples(15000))
        assert torch.equal(y.view(2, -1).cpu(), want)
        assert (y[1, 0, f.out_samples(6300):] == f.silence).all()
        full = gen(mel, audio=f)
        parts = list(gen.stream(mel, chunk_frames=8, audio=f))
        assert [p[0] for p in parts] == [f.out_samples(300 * t) for t in range(0, 50, 8)]
        cat = torch.cat([p[1] for p in parts], dim=2)
        assert cat.shape == full.shape
        if f.encoding == "float32":
            assert util.snr_db(cat.cpu(), full.cpu()) >= 60.0
        else:
            assert (cat != full).float().mean().item() < 0.05


def _inputs(seed, tl, Tr=110):
    gsrc = torch.Generator().manual_seed(seed)
    B, Tt = len(tl), max(tl)
    tok = torch.randint(1, 178, (B, Tt), generator=gsrc)
    for b in range(B):
        tok[b, tl[b]:] = 0
    mel = (torch.randn(B, 80, Tr, generator=gsrc) * 0.5).clamp(-2, 2)
    dur = torch.randint(1, 4, (B, Tt), generator=gsrc)
    return tok, mel, dur


@pytest.mark.parametrize("depth", [1, 2])
@pytest.mark.parametrize("mode", ["forced", "predicted", "bounded"])
def test_engine_format_stage(model_gpu, mode, depth):
    """A formatted call is its unformatted pass plus one format launch: equal to the kernel on that pass's output, on
    the graph and the eager path; graphs are shared with unformatted calls (no new captures)."""
    model, gen = model_gpu
    tl = [40, 17, 33]
    tok, mel, dur = _inputs(3 + depth, tl)
    dur = dur if mode == "forced" else None
    kw = dict(duration_bound=6.0) if mode == "bounded" else {}
    graph = engine.Synthesizer(model, gen, device=DEV, use_cuda_graph=True, pipeline_depth=depth, **kw)
    eager = engine.Synthesizer(model, gen, device=DEV, use_cuda_graph=False, **kw)
    args = (tok.to(DEV), tl, mel.to(DEV), [110] * 3, dur)
    for _ in range(depth):                                      # every pipeline slot has its graphs
        graph.synthesize(*args)
    base, caps = graph.launches_per_call, graph.stats["captures"]
    for f in (AudioFormat(8000, "mulaw"), AudioFormat(16000, "pcm16"), AudioFormat(48000, "float32"),
              AudioFormat(24000, "pcm16")):
        outs = []
        for syn in (graph, eager):
            w0, l0, _ = syn.synthesize(*args)
            with torch.cuda.stream(syn.last_stream):
                w0 = w0.clone()
            if syn is graph:
                assert syn.launches_per_call == base
            y, l1, _ = syn.synthesize(*args, audio=f)
            if syn is graph:
                assert syn.launches_per_call == base + 1
            syn.join()
            y = y.clone()                                       # consumed on the current stream after join()
            torch.cuda.synchronize()
            assert torch.equal(l0, l1) and y.dtype == f.dtype
            sl = syn.last["sample_lengths"].cpu()
            assert sl.tolist() == [f.out_samples(300 * int(v)) for v in l1.cpu()]
            assert y.shape == (3, f.out_samples(w0.shape[1]))
            want, _, _ = _run(w0, [300 * int(v) for v in l0.cpu()], f, y.shape[1])
            assert torch.equal(y.cpu(), want), (mode, f, syn is graph)
            outs.append((y.cpu(), sl))
        (yg, sg), (ye, se) = outs
        assert torch.equal(sg, se)
        if f.encoding in ("float32", "pcm16"):
            for b in range(3):
                n = int(sg[b])
                assert util.snr_db(yg[b, :n].double(), ye[b, :n].double()) >= 45.0, (mode, f, b)
    assert graph.stats["captures"] == caps and graph.stats["eager"] == 0
    assert graph.launches_per_call == base + 1


def test_pcm16_engine_equals_the_pcm16_format(model_gpu):
    model, gen = model_gpu
    tl = [40, 25]
    tok, mel, dur = _inputs(9, tl)
    fp = engine.Synthesizer(model, gen, device=DEV, use_cuda_graph=True)
    pcm = engine.Synthesizer(model, gen, device=DEV, use_cuda_graph=True, pcm16=True)
    for _ in range(2):
        a, _, _ = fp.synthesize(tok.to(DEV), tl, mel.to(DEV), [110] * 2, dur, audio=AudioFormat(24000, "pcm16"))
        a = a.clone()
        b, _, _ = pcm.synthesize(tok.to(DEV), tl, mel.to(DEV), [110] * 2, dur)
        assert pcm.launches_per_call == fp.launches_per_call - 1
        assert torch.equal(a, b)
        # the pcm16 engine's native format takes the unformatted path; other formats are refused
        c, _, _ = pcm.synthesize(tok.to(DEV), tl, mel.to(DEV), [110] * 2, dur, audio=AudioFormat(24000, "pcm16"))
        assert torch.equal(c, b) and "sample_lengths" not in pcm.last
    with pytest.raises(ValueError):
        pcm.synthesize(tok.to(DEV), tl, mel.to(DEV), [110] * 2, dur, audio=AudioFormat(8000, "mulaw"))


@pytest.mark.parametrize("bound", [None, 4.0])
def test_synthesize_many_mulaw(model_gpu, bound):
    """Each utterance has exactly out_samples(300 * frames) codes and equals its batch-1 run bit for bit."""
    model, gen = model_gpu
    f = AudioFormat(8000, "mulaw")
    syn = engine.Synthesizer(model, gen, device=DEV, use_cuda_graph=True, pipeline_depth=2, duration_bound=bound)
    one = engine.Synthesizer(model, gen, device=DEV, use_cuda_graph=True)
    gsrc = torch.Generator().manual_seed(31)
    tl = [15, 90, 33, 61, 47, 120, 18]
    toks = [torch.randint(1, 178, (t,), generator=gsrc) for t in tl]
    mels = [(torch.randn(80, 120, generator=gsrc) * 0.5).clamp(-2, 2) for _ in tl]
    durs = [torch.randint(1, 5, (t,), generator=gsrc) for t in tl]
    for to_host in (True, False):
        wavs, frames = engine.synthesize_many(syn, toks, mels, durs, max_batch=3, to_host=to_host, audio=f)
        torch.cuda.synchronize()
        for i in range(len(tl)):
            assert frames[i] == 2 * int(durs[i].sum())
            assert wavs[i].dtype == torch.uint8 and wavs[i].numel() == f.out_samples(300 * frames[i]), i
            w1, _, _ = one.synthesize(toks[i].view(1, -1).to(DEV), [tl[i]], mels[i].unsqueeze(0).to(DEV), [120],
                                      durs[i].view(1, -1), audio=f)
            w1 = w1[0, :f.out_samples(300 * frames[i])].cpu()
            # the acoustic model's batch-1 semantics are within noise of the batch (tests/test_serving_gpu.py):
            # the codes of the same 24 kHz samples are the same, so compare through the 24 kHz pass
            assert (wavs[i].cpu() == w1).float().mean().item() >= 0.95, i
    # predicted durations through the bounded single-graph path (and its exact re-run) also cut at out_samples
    wavs, frames = engine.synthesize_many(syn, toks, mels, None, max_batch=3, to_host=True, audio=f)
    assert all(wavs[i].numel() == f.out_samples(300 * frames[i]) for i in range(len(tl)))
