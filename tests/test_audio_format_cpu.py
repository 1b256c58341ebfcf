"""Output audio formats without a GPU: validation of ``AudioFormat``, the fp64 filter against scipy's design, the
fp64 restatement against ``scipy.signal.resample_poly`` and ``audioop``, the chunk grid of the streaming path, and
the host logic of ``Generator.forward / stream(audio=)`` and ``synthesize_many(audio=)`` on the semantic backend
(``sim`` plus the torch model of ``ops.resample_encode`` in tests/audio_ref.py)."""
import multiprocessing as mp
import os
import socket
import types
import warnings

import numpy as np
import pytest
import torch

from artspeech_b200 import audio, engine, ops
from artspeech_b200.audio import AudioFormat
from tests import audio_ref, util

RATES = (8000, 11025, 16000, 22050, 24000, 32000, 44100, 48000)
K_WANT = {8000: 61, 11025: 44, 16000: 31, 22050: 22, 32000: 21, 44100: 21, 48000: 21}


def test_validation():
    for kw in (dict(encoding="opus"), dict(encoding="PCM16"), dict(sample_rate=16000.0), dict(sample_rate=8000.5),
               dict(sample_rate="8000"), dict(sample_rate=True), dict(sample_rate=0), dict(sample_rate=-8000),
               dict(sample_rate=44101), dict(sample_rate=1000)):
        with pytest.raises(ValueError):
            AudioFormat(**kw)
    assert AudioFormat(np.int64(16000)).sample_rate == 16000
    assert AudioFormat() == AudioFormat(24000, "float32") and AudioFormat().is_identity
    f = AudioFormat(11025, "alaw")
    assert (f.up, f.down, f.K, f.table_ld, f.dtype, f.silence) == (147, 320, 44, 44, torch.uint8, 0xD5)
    assert f.table().nbytes == 147 * 44 * 4                       # the largest table of the listed rates
    assert audio.smem_bytes(1, 24, 481, 484) > audio.SMEM_MAX     # 1 kHz: the input window does not fit


def test_audio_with_pcm16_is_refused():
    gen = util.generator()
    with pytest.raises(ValueError):
        gen(torch.zeros(1, 80, 4), pcm16=True, audio=AudioFormat(16000))
    with pytest.raises(ValueError):
        next(gen.stream(torch.zeros(1, 80, 4), pcm16=True, audio=AudioFormat(16000)))
    with pytest.raises(ValueError):
        gen(torch.zeros(1, 80, 4), audio="mulaw")
    pcm_engine = types.SimpleNamespace(pcm16=True)
    with pytest.raises(ValueError):
        engine.Synthesizer._out_format(pcm_engine, AudioFormat(8000, "mulaw"))
    # the native formats take the unformatted path
    assert engine.Synthesizer._out_format(pcm_engine, AudioFormat(24000, "pcm16")) is None
    fp_engine = types.SimpleNamespace(pcm16=False)
    assert engine.Synthesizer._out_format(fp_engine, AudioFormat()) is None
    assert engine.Synthesizer._out_format(fp_engine, AudioFormat(24000, "pcm16")) == AudioFormat(24000, "pcm16")


@pytest.mark.parametrize("rate", [r for r in RATES if r != 24000])
def test_filter_matches_scipy_firwin(rate):
    from scipy.signal import firwin
    f = AudioFormat(rate)
    mx = max(f.up, f.down)
    assert f.half_len == 10 * mx and f.K == K_WANT[rate]
    want = firwin(2 * f.half_len + 1, 1.0 / mx, window=("kaiser", 5.0)) * f.up
    assert np.abs(f.filter64() - want).max() <= 1e-12
    # the fp32 polyphase table: table[p][j] = h[p + j * up], zero beyond the filter
    t, h = f.table(), f.filter64()
    for p in (0, f.up // 2, f.up - 1):
        for j in range(f.table_ld):
            k = p + j * f.up
            assert t[p, j] == (np.float32(h[k]) if j < f.K and k < len(h) else 0.0)


@pytest.mark.parametrize("rate", RATES)
def test_restatement_matches_resample_poly(rate):
    from scipy.signal import resample_poly
    f = AudioFormat(rate)
    rng = np.random.default_rng(rate)
    for n in (0, 1, 2, f.K - 1, f.K, 1000, 240007):
        if n < 0:
            continue
        x = rng.standard_normal(n)
        y, _ = audio_ref.resample64(x, f.filter64(), f.up, f.down, f.half_len)
        want = resample_poly(x, f.up, f.down)
        assert y.shape == want.shape and f.out_samples(n) == want.shape[0], (n, y.shape, want.shape)
        if n:
            assert np.abs(y - want).max() <= 1e-12, n


def test_g711_tables_match_audioop():
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", DeprecationWarning)
        audioop = pytest.importorskip("audioop")
    pcm = np.arange(-32768, 32768, dtype=np.int16).tobytes()
    assert np.array_equal(audio_ref.ULAW, np.frombuffer(audioop.lin2ulaw(pcm, 2), dtype=np.uint8))
    assert np.array_equal(audio_ref.ALAW, np.frombuffer(audioop.lin2alaw(pcm, 2), dtype=np.uint8))
    assert audio_ref.ULAW[32768] == audio.SILENCE["mulaw"] and audio_ref.ALAW[32768] == audio.SILENCE["alaw"]


def test_encode_accepts_the_neighbour_only_at_midpoints():
    y = np.array([0.5 / 32767, 0.25 / 32767, 1.0, -2.0, 100.5 / 32767])
    want, alt = audio_ref.encode(y, np.full(5, 1e-9), "pcm16")
    assert want.tolist() == [0, 0, 32767, -32768, 100]
    assert alt.tolist() == [1, 0, 32767, -32768, 101]


@pytest.mark.parametrize("rate", RATES)
def test_chunk_ranges_partition_the_output(rate):
    f = AudioFormat(rate)
    for T in (1, 57, 203):
        for chunk in (1, 7, 64):
            edges = [f.out_samples(300 * t0) for t0 in range(0, T, chunk)] + [f.out_samples(300 * T)]
            assert edges[0] == 0 and all(a <= b for a, b in zip(edges, edges[1:]))
            assert edges[-1] == f.out_samples(300 * T)
            # the window start of each chunk is on the output grid
            a = 300 * (max(0, 37 - 14) // f.frame_align(300) * f.frame_align(300))
            assert a * f.up % f.down == 0


# ---- host logic on the semantic backend ---------------------------------------------------------------------------
@pytest.fixture
def fmt_model(sim, monkeypatch):
    monkeypatch.setattr(ops, "resample_encode", audio_ref.resample_encode_model)
    return sim


def _framewise_generator(monkeypatch):
    """The vocoder with its network replaced by a frame-local map (sample ``300 t + k`` depends on mel frame ``t``
    only): every window then gives the same samples, so the chunked and one-shot outputs must agree bit for bit
    and only the host logic (chunk grid, window alignment, ``m0``) is under test."""
    gen = util.generator()
    ramp = torch.linspace(-1.0, 1.0, 300)

    def fcl(mel_cl, lengths=None, out_dtype=torch.float32, return_lengths=False):
        B, T, _ = mel_cl.shape
        wav = torch.tanh(mel_cl.float().mean(2, keepdim=True) * 3.0 + ramp).reshape(B, T * 300)
        if lengths is not None:
            wav = wav * (torch.arange(T * 300)[None, :] < 300 * lengths.view(-1, 1))
        return wav
    monkeypatch.setattr(gen, "forward_channels_last", fcl)
    return gen


@pytest.mark.parametrize("rate,encoding", [(8000, "mulaw"), (11025, "float32"), (22050, "pcm16"), (48000, "alaw"),
                                           (44100, "mulaw"), (24000, "float32")])
def test_stream_concatenates_to_forward(fmt_model, monkeypatch, rate, encoding):
    gen = _framewise_generator(monkeypatch)
    f = AudioFormat(rate, encoding)
    g = torch.Generator().manual_seed(rate)
    mel = torch.randn(2, 80, 45, generator=g)
    full = gen(mel, audio=f)
    assert full.dtype == f.dtype and full.shape == (2, 1, f.out_samples(300 * 45))
    for chunk in (1, 7, 64):
        parts = list(gen.stream(mel, chunk_frames=chunk, audio=f))
        assert [p[0] for p in parts] == [f.out_samples(300 * t0) for t0 in range(0, 45, chunk)]
        assert torch.equal(torch.cat([p[1] for p in parts], dim=2), full), chunk


def test_forward_with_lengths_cuts_each_utterance(fmt_model, monkeypatch):
    gen = _framewise_generator(monkeypatch)
    f = AudioFormat(16000, "mulaw")
    mel = torch.randn(2, 80, 12, generator=torch.Generator().manual_seed(1))
    y = gen(mel, lengths=torch.tensor([12, 5]), audio=f)
    one = gen(mel[1:, :, :5], audio=f)
    n = f.out_samples(300 * 5)
    assert y.shape == (2, 1, f.out_samples(3600)) and one.shape == (1, 1, n)
    assert bool((y[1, 0, n:] == 0xFF).all()) and torch.equal(y[1, 0, :n], one[0, 0])


class _FakeEngine:
    """The surface of ``Synthesizer`` that ``synthesize_many`` uses, on the CPU: utterance ``i`` of a batch gets
    ``frames = 2 * sum(durations)`` mel frames and a 24 kHz waveform of ``300 * frames`` samples, formatted by the
    model of ``ops.resample_encode``."""
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
            wav[b, :300 * fr] = torch.sin(torch.arange(300 * fr) * (0.01 + 0.003 * int(tok[b, 0])))
        res = (wav, torch.tensor(frames, dtype=torch.int32), None)
        self.calls.append(audio)
        if audio is not None:
            n = torch.empty(len(tl), dtype=torch.int32)
            res = (ops.resample_encode(wav, torch.tensor(frames, dtype=torch.int32) * 300, audio,
                                       audio.out_samples(S), out_lens=n), res[1], None)
        self.last = dict(frames=frames)
        return res

    def finish(self, t):
        return t

    def join(self):
        pass


def test_synthesize_many_cuts_each_utterance(fmt_model, monkeypatch):
    monkeypatch.setattr(torch.Tensor, "pin_memory", lambda self, *a, **k: self)     # no CUDA host allocator here
    f = AudioFormat(8000, "mulaw")
    durs = [torch.tensor([3, 1, 4]), torch.tensor([2] * 7), torch.tensor([5]), torch.tensor([1, 1])]
    toks = [torch.full((d.shape[0],), i + 1, dtype=torch.long) for i, d in enumerate(durs)]
    mels = [torch.zeros(80, 10) for _ in durs]
    syn = _FakeEngine()
    wavs, frames = engine.synthesize_many(syn, toks, mels, durations=durs, max_batch=2, audio=f)
    assert frames == [2 * int(d.sum()) for d in durs]
    assert all(a == f for a in syn.calls)
    for i, d in enumerate(durs):
        assert wavs[i].dtype == torch.uint8 and wavs[i].shape[0] == f.out_samples(300 * frames[i])
        # batch-1 run of the same utterance
        one, _ = engine.synthesize_many(_FakeEngine(), [toks[i]], [mels[i]], durations=[d], audio=f)
        assert torch.equal(wavs[i], one[0])
    native, _ = engine.synthesize_many(syn, toks, mels, durations=durs, max_batch=2, audio=AudioFormat())
    assert syn.calls[-1] is None and native[0].dtype == torch.float32 and native[0].shape[0] == 300 * frames[0]


# ---- gather of uint8 payloads -------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _gather_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        B, S = (3, 101) if rank == 0 else (2, 64)
        g = torch.Generator().manual_seed(rank)
        wav = torch.randint(0, 256, (B, S), generator=g, dtype=torch.int64).to(torch.uint8)
        lens = torch.tensor([S - 3 * b for b in range(B)], dtype=torch.int64)
        wavs, lns = engine.gather_waveforms(wav, lens, dst=0)
        gat = engine.WaveformGatherer("cpu", [(3, 101), (2, 64)], torch.uint8, dst=0)
        gat.submit(wav, lens)
        wavs2, lns2 = gat.results()
        if rank == 0:
            ok = True
            for r in range(world):
                gr = torch.Generator().manual_seed(r)
                Br, Sr = (3, 101) if r == 0 else (2, 64)
                want = torch.randint(0, 256, (Br, Sr), generator=gr, dtype=torch.int64).to(torch.uint8)
                ok &= wavs[r].dtype == torch.uint8 and torch.equal(wavs[r], want) and torch.equal(wavs2[r], want)
                ok &= lns[r].tolist() == [Sr - 3 * b for b in range(Br)] and torch.equal(lns[r], lns2[r])
            q.put(bool(ok))
    finally:
        dist.destroy_process_group()


def test_gather_uint8_payload_gloo_world2():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_gather_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    assert q.get(timeout=5) is True


def test_shared_memory_budget_matches_the_library():
    """``AudioFormat`` refuses exactly the filters the kernel's launch would refuse (the library loads without a
    GPU)."""
    from artspeech_b200 import _lib
    lib = _lib.load()
    for rate in RATES + (4000, 6000, 12000, 96000, 192000, 44101, 2000):
        up, down = rate // np.gcd(rate, 24000), 24000 // np.gcd(rate, 24000)
        K = 1 if up == down == 1 else -(-(20 * max(up, down) + 1) // up)
        ld = (K + 3) // 4 * 4
        assert lib.as_resample_smem_bytes(up, down, K, ld) == audio.smem_bytes(up, down, K, ld), rate
        fits = audio.smem_bytes(up, down, K, ld) <= audio.SMEM_MAX
        if fits:
            assert AudioFormat(rate).K == K
        else:
            with pytest.raises(ValueError):
                AudioFormat(rate)
