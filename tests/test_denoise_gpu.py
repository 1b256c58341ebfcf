"""Noise reduction for voice enrollment on the GPU: ``as_denoise``'s planes against the fp64 restatement (``X`` within a
bound of the fp64 STFT, ``lambda`` and ``G`` bit for bit from the kernel's own power), the output against the fp64
overlap-add of the kernel's ``G X``, the round trip at 0 dB, invariance and edge cases, ``reference_mels`` with
noise reduction stage by stage, and ``enroll`` feeding ``synthesize``."""
import numpy as np
import pytest
import torch

from artspeech_b200 import audio, engine, frontend, ops
from oracle import frontend_oracle as fo
from tests import denoise_ref as D
from tests import enroll_ref as R
from tests import util
from tests.test_enroll_gpu import CASES, _encode, _ragged, _recording

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 2e-3                   # test_frontend's bound on the normalised log-mel
MARGIN = 1e-9
X_TOL = 1e-5                 # |X - X64| <= X_TOL * sqrt(sum_i (w_i y_i)^2), the frame's energy
OUT_TOL = 2e-5               # |out - overlap-add64(G X)| <= OUT_TOL * the row's peak
ID_TOL = 1e-5                # |out - y| <= ID_TOL * the row's peak at reduction_db = 0


def _rows(ys, pad=0, stride_extra=0, offset=0):
    """[B, S] device view of ``ys`` with NaN beyond each length, in the padding and before the first row."""
    S = max([y.size for y in ys] + [1]) + pad
    ld = S + stride_extra
    buf = torch.full((offset + len(ys) * ld,), float("nan"))
    for b, y in enumerate(ys):
        buf[offset + b * ld:offset + b * ld + y.size] = torch.from_numpy(np.asarray(y, np.float32))
    x = buf.to(DEV)[offset:].as_strided((len(ys), S), (ld, 1))
    lens = torch.tensor([y.size for y in ys], dtype=torch.int32, device=DEV)
    return x, lens


def _noisy_voiced(seed, seconds, kind="white", snr=10.0):
    rng = np.random.default_rng(seed)
    c = D.voiced(rng, int(seconds * D.FS))
    return D.mix(c, D.noise(rng, kind, c.size), snr)


def _clips():
    rng = np.random.default_rng(4)
    edge = [(rng.standard_normal(n) * 0.1).astype(np.float32) for n in D.EDGE_LENGTHS]
    return edge + [np.zeros(3000, np.float32), _noisy_voiced(1, 2.3), _noisy_voiced(2, 4.1, "pink", 0.0),
                   _noisy_voiced(3, 3.2, "hum", 20.0), _noisy_voiced(5, 61.0)]


def _check_row(y, n, out, X, lam, G, reduction_db):
    F = D.n_frames(n)
    y = np.asarray(y, np.float32)
    Xk = X[:F].astype(np.complex64)
    # X: within X_TOL of the fp64 STFT of the same fp32 samples, relative to each frame's energy
    ref = D.stft(y.astype(np.float64))
    yp = np.zeros((F - 1) * D.HOP + D.N)
    yp[D.N // 2:D.N // 2 + n] = y
    frames = yp[np.arange(F)[:, None] * D.HOP + np.arange(D.N)[None, :]] * D.window()[None, :]
    energy = np.sqrt(np.sum(frames ** 2, axis=1))
    err = np.abs(Xk.astype(np.complex128) - ref).max(axis=1)
    assert np.all(err <= X_TOL * energy), (n, float(np.max(err / np.maximum(energy, 1e-300))))
    # lambda and G: bit for bit from the kernel's own power
    P = D.power32(Xk)
    assert np.array_equal(lam.view(np.int64), D.noise_profile(P).view(np.int64)), n
    assert np.array_equal(G[:F].view(np.int32), D.gains(P, lam, reduction_db).view(np.int32)), n
    # the output: the fp64 overlap-add of the kernel's G X
    want = D.istft(G[:F].astype(np.float64) * Xk.astype(np.complex128), n)
    peak = np.abs(want).max() if n else 0.0
    assert np.all(np.abs(out[:n] - want) <= OUT_TOL * peak), (n, float(np.abs(out[:n] - want).max()), peak)
    return want


@pytest.mark.parametrize("reduction_db", [18.0, 6.0, 60.0])
def test_planes_and_output_against_the_fp64_reference(reduction_db):
    ys = _clips()
    x, lens = _rows(ys, pad=1000, stride_extra=3, offset=1)
    out, X, lam, G = ops.denoise(x, lens, reduction_db, planes=True)
    out, X, lam, G = out.cpu().numpy(), X.cpu().numpy(), lam.cpu().numpy(), G.cpu().numpy()
    assert not np.isnan(out).any()
    for b, y in enumerate(ys):
        _check_row(y, y.size, out[b], X[b], lam[b], G[b], reduction_db)
        assert not out[b, y.size:].any()
    silent = len(D.EDGE_LENGTHS)                               # the all-zero row: floor, g_min, silence
    assert np.all(lam[silent] == 1e-20) and np.all(G[silent, :D.n_frames(3000)] == np.float32(D.g_min(reduction_db)))
    assert not out[silent].any() and not out[0].any()           # and the zero-length row


def test_zero_reduction_is_the_round_trip():
    ys = _clips()
    x, lens = _rows(ys, stride_extra=1)
    out = ops.denoise(x, lens, 0.0).cpu().numpy()
    for b, y in enumerate(ys):
        peak = np.abs(y).max() if y.size else 0.0
        assert np.all(np.abs(out[b, :y.size] - y) <= ID_TOL * peak), (b, float(np.abs(out[b, :y.size] - y).max()))


def test_bitwise_invariance_and_determinism():
    ys = _clips()
    x, lens = _rows(ys)
    first = ops.denoise(x, lens, 18.0)
    assert torch.equal(first, ops.denoise(x, lens, 18.0))      # two calls
    perm = [9, 3, 11, 0, 8, 10, 7]
    x2, lens2 = _rows([ys[i] for i in perm], pad=5000, stride_extra=13, offset=2)
    second = ops.denoise(x2, lens2, 18.0)
    for j, i in enumerate(perm):
        n = ys[i].size
        assert torch.equal(second[j, :n], first[i, :n]), i
        alone = frontend.denoise(torch.from_numpy(ys[i]).to(DEV), reduction_db=18.0)
        assert alone.shape == (n,) and torch.equal(alone, first[i, :n]), i
    assert ops.denoise(torch.zeros(0, 100, device=DEV), None, 18.0).shape == (0, 100)
    assert ops.denoise(torch.zeros(2, 0, device=DEV), None, 18.0).shape == (2, 0)


def _noisy_recording(rng, seconds, rate, C, encoding):
    """``_recording``'s tone bursts with white noise 20 dB below them, encoded."""
    clean = _recording(rng, seconds, rate, C, "float32").numpy().astype(np.float64)
    y = clean + rng.standard_normal(clean.shape) * 0.3 / np.sqrt(2) * 10 ** (-20 / 20)
    return _encode(np.clip(y, -1, 1).astype(np.float32), encoding)


@pytest.mark.parametrize("rate,encoding,C", CASES)
def test_chain_with_noise_reduction_stage_by_stage(rate, encoding, C):
    rng = np.random.default_rng(rate + C + 1)
    recs = [_noisy_recording(rng, s, rate, C, encoding) for s in (2.2, 1.1, 3.4)]
    x, lens = _ragged(recs, C, encoding, 100, 3)
    dev_x = x.to(DEV)
    before = ops.launch_count
    mels, mel_lens, bounds = frontend.reference_mels(dev_x, lens, rate, encoding, noise_reduction_db=18)
    with_nr = ops.launch_count - before
    before = ops.launch_count
    plain = frontend.reference_mels(dev_x, lens, rate, encoding)
    assert with_nr == ops.launch_count - before + ops.DENOISE_LAUNCHES
    none = frontend.reference_mels(dev_x, lens, rate, encoding, noise_reduction_db=None)
    assert all(torch.equal(a.cpu(), b.cpu()) for a, b in zip(plain, none))     # None: today's call, bit for bit
    fmt = audio.to_native_rate(rate)
    lt = torch.tensor(lens, dtype=torch.int32, device=DEV)
    mono = ops.audio_to_mono(dev_x, lt, encoding) if encoding != "float32" or C > 1 else dev_x
    if fmt.is_identity:
        y24, n24 = mono, lt
    else:
        n24 = torch.empty(3, dtype=torch.int32, device=DEV)
        y24 = ops.resample_encode(mono, lt, fmt, fmt.out_samples(x.shape[1]), out_lens=n24)
    den = ops.denoise(y24, n24, 18.0)
    assert torch.equal(frontend.trim_bounds(den, n24), bounds)
    y24_h, den_h, n24_h, b_h = y24.cpu().numpy(), den.cpu().numpy(), n24.cpu().tolist(), bounds.cpu().tolist()
    for b in range(3):
        n = n24_h[b]
        want = D.denoise(y24_h[b, :n], 18.0)                    # stage 2b in fp64 on the kernel's 24 kHz samples
        assert np.abs(den_h[b, :n] - want).max() <= OUT_TOL * np.abs(want).max()
        tb, ambiguous = R.trim_blocks(den_h[b, :n], 30.0, MARGIN)
        assert ambiguous or tuple(b_h[b]) == tb
        assert 0 < tb[0] and tb[1] < n                           # the noise did not stop the trim
        ref = fo.log_mel(torch.from_numpy(den_h[b, b_h[b][0]:b_h[b][1]].copy()))[0]
        assert int(mel_lens[b]) == ref.shape[1]
        assert (mels[b, :, :ref.shape[1]].cpu() - ref).abs().max().item() <= TOL


@pytest.fixture(scope="module")
def model_gpu():
    g = util.load_golden("acoustic_small.pt")
    m = util.acoustic_model(g["checkpoint_seed"])
    m.set_compute_dtype(torch.float16)
    m = m.to(DEV)
    m.distribution = {k: v.to(DEV) for k, v in m.distribution.items()}
    yield m
    util._MODELS.clear()


def test_enroll_with_noise_reduction_feeds_synthesize(model_gpu):
    gen = util.generator(0).to(DEV)
    rng = np.random.default_rng(17)
    recs = [_noisy_recording(rng, s, 16000, 1, "pcm16") for s in (4.0, 3.1)]
    x, lens = _ragged(recs, 1, "pcm16", 0, 0)
    B, Tt = 2, 24
    gsrc = torch.Generator().manual_seed(9)
    tok = torch.randint(1, 178, (B, Tt), generator=gsrc).to(DEV)
    tl = torch.full((B,), Tt)
    dur = torch.randint(1, 4, (B, Tt), generator=gsrc)
    for use_graph in (False, True):
        syn = engine.Synthesizer(model_gpu, gen, device=DEV, use_cuda_graph=use_graph)
        mels, mel_lens, voice = syn.enroll(x, lens, 16000, "pcm16", noise_reduction_db=12.0)
        want = frontend.reference_mels(x, lens, 16000, "pcm16", noise_reduction_db=12.0)
        assert torch.equal(mels, want[0]) and torch.equal(mel_lens, want[1])
        again = syn.encode_voice(mels, mel_lens)
        assert len(voice) == len(again) == 4 and all(torch.equal(a, b) for a, b in zip(voice, again))
        full, _, mel_full = syn.synthesize(tok, tl, mels, mel_lens, dur)
        full, mel_full = full.clone(), mel_full.clone()
        for _ in range(2):
            cached, _, mel_cached = syn.synthesize(tok, tl, mels, mel_lens, dur, voice=voice)
        assert torch.equal(mel_cached, mel_full) and torch.equal(cached, full), f"graph={use_graph}"
        assert torch.isfinite(full).all()
