"""Loudness normalisation on the GPU: ``as_loudness_measure`` against the fp64 meter (tests/loudness_ref.py) with NaN
guards around every row, its bitwise batch invariance, the gain in ``as_resample_encode_gain`` (bit-identical at 1,
against the fp64 encode otherwise), and the engine's loudness stage."""
import math

import numpy as np
import pytest
import torch

from artspeech_b200 import audio, engine, ops
from artspeech_b200.audio import ENCODINGS, AudioFormat, Loudness
from tests import audio_ref, loudness_ref, util

pytestmark = pytest.mark.gpu
DEV = "cuda"
LENS = (0, 1, 599, 9599, 9600, 9601, 24007, 240000, 1440000)
GUARD = 16
MARGIN = 0.05                                  # LU between every block and either gate


def _true_peak64(x, chunk=100000):
    """``loudness_ref.true_peak`` in chunks of ``audio_ref.resample64`` (each with the filter's 10-sample context)."""
    x = np.asarray(x, dtype=np.float64)
    if x.size == 0:
        return -math.inf
    h = audio._design(4, 1)[0]
    tp = np.abs(x).max()
    for a in range(0, x.size, chunk):
        lo, hi = max(0, a - 10), min(x.size, a + chunk + 10)
        y4, _ = audio_ref.resample64(x[lo:hi], h, 4, 1, 40)
        y4 = y4[4 * (a - lo):4 * (min(x.size, a + chunk) - lo)]
        tp = max(tp, np.abs(y4).max())
    return 20.0 * math.log10(tp) if tp > 0 else -math.inf


def _gates_clear(v, fs):
    L = loudness_ref.block_loudness(v, fs)
    g = loudness_ref.relative_gate(v, fs)
    return not (np.abs(L + 70.0) < MARGIN).any() and (g is None or not (np.abs(L - g) < MARGIN).any())


def _speechlike(n, fs, g):
    """Tones and noise under a 50-400 ms step envelope spanning ~45 dB (some blocks fall to the relative gate)."""
    t = torch.arange(n, dtype=torch.float64) / fs
    f = 100.0 + 3000.0 * torch.rand(3, generator=g, dtype=torch.float64)
    v = sum(torch.sin(2 * math.pi * fk * t + k) for k, fk in enumerate(f)) / 3 + \
        0.2 * torch.randn(n, generator=g, dtype=torch.float64)
    env = torch.empty(n, dtype=torch.float64)
    i = 0
    while i < n:
        m = int(fs * (0.05 + 0.35 * float(torch.rand((), generator=g))))
        env[i:i + m] = 10.0 ** (-45.0 * float(torch.rand((), generator=g)) / 20.0)
        i += m
    return 0.6 * v * env


def _signal(lens, S, seed, fs, guard=GUARD):
    """[B, guard + S + guard] fp32, NaN everywhere but each row's first ``lens[b]`` samples; a row whose blocks come
    within MARGIN of a gate is drawn again (a rescale would move the relative gate with the blocks)."""
    g = torch.Generator().manual_seed(seed)
    buf = torch.full((len(lens), guard + S + guard), float("nan"))
    for b, n in enumerate(lens):
        for _ in range(50):
            v = _speechlike(n, fs, g)
            if n == 0 or _gates_clear(v.float().double().numpy(), fs):
                break
        else:
            raise AssertionError("no signal clear of the gates")
        buf[b, guard:guard + n] = v.float()
    return buf, buf[:, guard:guard + S]


def _meter(x, lens, fs, target=-23.0, ceiling=-1.0):
    lt = None if lens is None else torch.tensor(lens, dtype=torch.int32, device=DEV)
    out = ops.loudness_measure(x, lt, fs, target, ceiling)
    torch.cuda.synchronize()
    return [t.cpu() for t in out]


@pytest.mark.parametrize("fs", [24000, 16000, 48000])
def test_meter_matches_fp64_reference(fs):
    S = max(LENS) + 3
    xbuf, x = _signal(LENS, S, fs, fs)
    xd = xbuf.to(DEV)[:, GUARD:GUARD + S]
    L, tp, gdb, gain = _meter(xd, list(LENS), fs)
    worst_l = worst_tp = 0.0
    for b, n in enumerate(LENS):
        xb = x[b, :n].double().numpy()
        Lr, tpr = loudness_ref.integrated(xb, fs), _true_peak64(xb)
        if n == 0:
            assert L[b] == -math.inf and tp[b] == -math.inf and gdb[b] == 0.0 and gain[b] == 1.0
            continue
        assert (float(L[b]) == -math.inf) == (Lr == -math.inf), (n, float(L[b]), Lr)
        assert abs(float(tp[b]) - tpr) <= 0.01, (n, float(tp[b]), tpr)
        if Lr == -math.inf:
            continue
        worst_l, worst_tp = max(worst_l, abs(float(L[b]) - Lr)), max(worst_tp, abs(float(tp[b]) - tpr))
        assert abs(float(L[b]) - Lr) <= 0.01, (n, float(L[b]), Lr)
        want = loudness_ref.gain_db(float(L[b]), float(tp[b]))
        assert float(gdb[b]) == pytest.approx(want, abs=1e-12)
        assert float(gain[b]) == float(loudness_ref.gain32(float(gdb[b])))
    print(f"{fs} Hz: largest |dL| {worst_l:.2e} LU, |dTP| {worst_tp:.2e} dB")


def test_silence_and_quiet_read_minus_inf():
    n = 48000
    x = torch.zeros(3, n, device=DEV)
    x[1] = 1e-5 * torch.sin(torch.arange(n, device=DEV) * 0.1)            # about -100 LUFS
    x[2, :5] = 1e-6
    L, tp, gdb, gain = _meter(x, None, 24000)
    assert (L == -math.inf).all() and (gdb == 0.0).all() and (gain == 1.0).all()
    assert tp[0] == -math.inf and math.isfinite(tp[1]) and math.isfinite(tp[2])


def test_batch_invariance():
    fs = 24000
    lens = [240000, 7, 30011, 9600, 0]
    xbuf, _ = _signal(lens, 240000, 5, fs)
    xd = xbuf.to(DEV)[:, GUARD:GUARD + 240000]
    full = _meter(xd, lens, fs)
    fmt = AudioFormat(8000, "mulaw")

    def encode(x, ln, gain):
        lt = None if ln is None else torch.tensor(ln, dtype=torch.int32, device=DEV)
        return ops.resample_encode(x, lt, fmt, fmt.out_samples(x.shape[1]), gain=gain.to(DEV)).cpu()
    full_y = encode(xd, lens, full[3])
    for b in (0, 1, 2, 3):
        L = lens[b]
        alone = _meter(xd[b:b + 1, :L].contiguous(), None, fs)
        big = torch.full((4, 300007), float("nan"), device=DEV)
        big[3, :L] = xd[b, :L]
        big[0, :9000] = 0.25
        big[1, :200000] = torch.randn(200000, device=DEV) * 0.1
        inb = _meter(big, [9000, 200000, 0, L], fs)
        for k in range(4):
            assert torch.equal(alone[k][0], full[k][b]) and torch.equal(inb[k][3], full[k][b]), (b, k)
        n_out = fmt.out_samples(L)
        y_alone = encode(xd[b:b + 1, :L].contiguous(), None, alone[3])
        y_big = encode(big, [9000, 200000, 0, L], inb[3])
        assert torch.equal(y_alone[0, :n_out], full_y[b, :n_out]) and torch.equal(y_big[3, :n_out], full_y[b, :n_out])


@pytest.mark.parametrize("rate", [8000, 11025, 16000, 22050, 24000, 44100, 48000])
def test_unit_gain_is_bit_identical(rate):
    lens = [24007, 1, 0, 9600]
    xbuf, _ = _signal(lens, 24011, rate, 24000)
    xd = xbuf.to(DEV)[:, GUARD:GUARD + 24011]
    lt = torch.tensor(lens, dtype=torch.int32, device=DEV)
    one = torch.ones(4, device=DEV)
    for enc in ENCODINGS:
        f = AudioFormat(rate, enc)
        S = f.out_samples(24011)
        a = ops.resample_encode(xd, lt, f, S)
        b = ops.resample_encode(xd, lt, f, S, gain=one)
        assert torch.equal(a, b), f


@pytest.mark.parametrize("rate,enc", [(8000, "mulaw"), (16000, "pcm16"), (24000, "float32"), (44100, "float32"),
                                      (48000, "alaw"), (24000, "pcm16")])
def test_gain_matches_fp64_encode(rate, enc):
    f = AudioFormat(rate, enc)
    lens = [24007, 3001, 0]
    xbuf, x = _signal(lens, 24011, 7, 24000)
    xd = xbuf.to(DEV)[:, GUARD:GUARD + 24011]
    gains = torch.tensor([0.37, 2.9, 1.5])
    S = f.out_samples(24011)
    got = ops.resample_encode(xd, torch.tensor(lens, dtype=torch.int32, device=DEV), f, S,
                              gain=gains.to(DEV)).cpu()
    for b, n in enumerate(lens):
        y64, s = audio_ref.resample64(x[b, :n].double().numpy(), f.filter64(), f.up, f.down, f.half_len)
        g = float(gains[b])
        y64 = g * y64
        bound = g * (f.K + 2) * 2.0 ** -24 * s + np.abs(y64) * 2.0 ** -24
        nb = y64.shape[0]
        if enc == "float32":
            assert (np.abs(got[b, :nb].numpy().astype(np.float64) - y64) <= bound).all(), b
        else:
            want, alt = audio_ref.encode(y64, bound, enc)
            ok = (got[b, :nb].numpy() == want) | (got[b, :nb].numpy() == alt)
            assert ok.all(), (b, int((~ok).sum()))
        assert (got[b, nb:] == f.silence).all()


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
    dur = torch.randint(1, 4, (B, Tt), generator=gsrc)
    return tok, mel, dur


@pytest.mark.parametrize("depth", [1, 2])
@pytest.mark.parametrize("mode", ["forced", "predicted", "bounded"])
def test_engine_loudness_stage(model_gpu, mode, depth):
    """A normalised call is its unformatted pass plus the meter and one format launch: equal to
    ``resample_encode(gain=)`` on that pass's 24 kHz output with the call's own gain; no new captures."""
    model, gen = model_gpu
    tl = [40, 17, 33]
    tok, mel, dur = _inputs(3 + depth, tl)
    dur = dur if mode == "forced" else None
    kw = dict(duration_bound=6.0) if mode == "bounded" else {}
    graph = engine.Synthesizer(model, gen, device=DEV, use_cuda_graph=True, pipeline_depth=depth, **kw)
    eager = engine.Synthesizer(model, gen, device=DEV, use_cuda_graph=False, **kw)
    args = (tok.to(DEV), tl, mel.to(DEV), [110] * 3, dur)
    for _ in range(depth):
        graph.synthesize(*args)
    base, caps = graph.launches_per_call, graph.stats["captures"]
    cases = ((None, Loudness(-30.0, -1.0)), (AudioFormat(8000, "mulaw"), Loudness()),
             (AudioFormat(48000, "float32"), Loudness(-5.0, -1.0)), (AudioFormat(24000, "pcm16"), Loudness(-16.0)))
    for f, loud in cases:
        fo = f or audio.NATIVE
        for syn in (graph, eager):
            w0, l0, _ = syn.synthesize(*args)
            with torch.cuda.stream(syn.last_stream):
                w0 = w0.clone()
            y, l1, _ = syn.synthesize(*args, audio=f, loudness=loud)
            if syn is graph:
                assert syn.launches_per_call == base + ops.LOUDNESS_LAUNCHES + 1
            syn.join()
            y = y.clone()
            torch.cuda.synchronize()
            assert torch.equal(l0, l1) and y.dtype == fo.dtype and y.shape == (3, fo.out_samples(w0.shape[1]))
            n24 = [300 * int(v) for v in l0.cpu()]
            lt = torch.tensor(n24, dtype=torch.int32, device=DEV)
            Lm, tpm, gdbm, gm = ops.loudness_measure(w0, lt, 24000, loud.target_lufs, loud.max_true_peak_db)
            gdb = syn.last["gain_db"].cpu()
            assert torch.equal(gdb, gdbm.cpu()) and torch.equal(syn.last["loudness"].cpu(), Lm.cpu())
            assert torch.equal(syn.last["true_peak"].cpu(), tpm.cpu())
            g = torch.tensor([float(loudness_ref.gain32(float(v))) for v in gdb], device=DEV)
            assert torch.equal(g, gm)
            want = ops.resample_encode(w0, lt, fo, y.shape[1], gain=g)
            assert torch.equal(y, want), (mode, f, syn is graph)
            if f is None:                                    # the normalised 24 kHz output, read by the fp64 meter
                for b in range(3):
                    yb = y[b, :n24[b]].double().cpu().numpy()
                    L, tp = float(syn.last["loudness"][b]), float(syn.last["true_peak"][b])
                    if float(gdb[b]) == loud.target_lufs - L:
                        assert abs(loudness_ref.integrated(yb, 24000) - loud.target_lufs) <= 0.05
                    else:
                        assert float(gdb[b]) == loud.max_true_peak_db - tp
                        assert abs(_true_peak64(yb) - loud.max_true_peak_db) <= 0.01
            if f == AudioFormat(48000, "float32"):          # a high target: the ceiling binds
                for b in range(3):
                    assert float(gdb[b]) == loud.max_true_peak_db - float(syn.last["true_peak"][b])
                    yb = ops.resample_encode(w0[b:b + 1, :n24[b]].contiguous(), None, audio.NATIVE, n24[b],
                                             gain=g[b:b + 1]).double().cpu().numpy()[0]
                    assert abs(_true_peak64(yb) - loud.max_true_peak_db) <= 0.01
    assert graph.stats["captures"] == caps and graph.stats["eager"] == 0
    assert graph.launches_per_call == base + ops.LOUDNESS_LAUNCHES + 1


def test_loudness_with_pcm16_engine_is_refused(model_gpu):
    model, gen = model_gpu
    tok, mel, dur = _inputs(9, [20])
    pcm = engine.Synthesizer(model, gen, device=DEV, use_cuda_graph=True, pcm16=True)
    with pytest.raises(ValueError):
        pcm.synthesize(tok.to(DEV), [20], mel.to(DEV), [110], dur, loudness=Loudness())


def test_synthesize_many_mulaw_loudness(model_gpu):
    """Each utterance has out_samples(300 * frames) codes, normalised by the meter's gain on its own waveform."""
    model, gen = model_gpu
    f = AudioFormat(8000, "mulaw")
    syn = engine.Synthesizer(model, gen, device=DEV, use_cuda_graph=True, pipeline_depth=2)
    gsrc = torch.Generator().manual_seed(31)
    tl = [15, 90, 33, 61, 47, 120, 18]
    toks = [torch.randint(1, 178, (t,), generator=gsrc) for t in tl]
    mels = [(torch.randn(80, 120, generator=gsrc) * 0.5).clamp(-2, 2) for _ in tl]
    durs = [torch.randint(1, 5, (t,), generator=gsrc) for t in tl]
    raw, frames0 = engine.synthesize_many(syn, toks, mels, durs, max_batch=3)
    syn.join()
    torch.cuda.synchronize()
    raw = [w.clone() for w in raw]
    wavs, frames = engine.synthesize_many(syn, toks, mels, durs, max_batch=3, to_host=True, audio=f,
                                          loudness=Loudness(-20.0))
    torch.cuda.synchronize()
    assert frames == frames0
    for i in range(len(tl)):
        assert wavs[i].dtype == torch.uint8 and wavs[i].numel() == f.out_samples(300 * frames[i]), i
        w = raw[i].view(1, -1).contiguous()
        _, _, _, g = ops.loudness_measure(w, None, 24000, -20.0, -1.0)
        want = ops.resample_encode(w, None, f, f.out_samples(w.shape[1]), gain=g).cpu()[0]
        assert torch.equal(wavs[i], want), i
