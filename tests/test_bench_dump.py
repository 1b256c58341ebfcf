"""bench.py --dump-outputs: the arrays a caller of the timed path receives, as float32 / float64 .npy files, capped
in size by a seeded sample of utterances; --steps sets the timed steps and must be positive."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench

BENCH = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bench.py")


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}


def test_dump_outputs_dtypes_and_sampling(tmp_path, monkeypatch):
    g = torch.Generator().manual_seed(0)
    wav = torch.randn(6, 3000, generator=g)
    mel = torch.randn(6, 80, 10, generator=g).half()
    lens = torch.tensor([10, 9, 8, 7, 6, 5], dtype=torch.int32)
    bench.dump_outputs(str(tmp_path / "all"), wav, lens, mel)
    a = _load(tmp_path / "all")
    assert sorted(a) == ["mel", "mel_lengths", "wav"]
    assert a["wav"].dtype == np.float32 and np.array_equal(a["wav"], wav.numpy())
    assert a["mel"].dtype == np.float32 and np.array_equal(a["mel"], mel.float().numpy())
    assert a["mel_lengths"].dtype == np.float64 and a["mel_lengths"].tolist() == lens.tolist()

    row = (3000 + 80 * 10) * 4 + 8
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 4 * row)
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), wav, lens, mel)
    s1, s2 = _load(tmp_path / "s1"), _load(tmp_path / "s2")
    assert sum(os.path.getsize(tmp_path / "s1" / f) for f in os.listdir(tmp_path / "s1")) < 4 * row + 4 * 128
    idx = s1["utterance_index"].astype(np.int64)
    assert len(idx) == 3 and all(np.array_equal(s1[k], s2[k]) for k in s1)          # the same sample every run
    assert np.array_equal(s1["wav"], wav.numpy()[idx]) and s1["mel_lengths"].tolist() == lens[idx].tolist()


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]])
def test_bad_arguments_are_rejected(argv, tmp_path):
    r = subprocess.run([sys.executable, BENCH, *argv], capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode == 2 and argv[-2] in r.stderr and not os.listdir(tmp_path)


@pytest.mark.gpu
def test_cuda_arm_dumps_its_last_timed_step(tmp_path):
    """Two timed steps on different input sets: the dump equals a fresh engine's output on the last one's inputs."""
    from artspeech_b200 import checkpoint, engine
    steps, warmup, depth = 2, 3, 2
    r = subprocess.run([sys.executable, BENCH, "--steps", str(steps), "--warmup", str(warmup), "--pipeline", str(depth),
                        "--skip-configs", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    a = _load(tmp_path)
    assert sorted(a) == ["mel", "mel_lengths", "wav"]

    dev = torch.device("cuda:0")
    syn = engine.Synthesizer(checkpoint.build_random_artsspeech(0), checkpoint.build_random_generator(0), device=dev,
                             pipeline_depth=depth)
    last = (bench.warmup_calls(warmup, depth) + steps - 1) % bench.N_INPUT_SETS
    tok, tl, mel, ml, dur = bench.make_inputs(0, bench.B_PER_GPU, last)
    wav, lens, mel_out = syn.synthesize(tok.to(dev), tl, mel.to(dev), ml, dur, predict_durations=True)
    syn.join()
    torch.cuda.synchronize()
    assert a["mel_lengths"].tolist() == lens.cpu().tolist()
    for name, want in (("wav", wav), ("mel", mel_out)):
        want = want.float().cpu().numpy()
        assert a[name].shape == want.shape, name
        assert np.array_equal(a[name], want), (name, float(np.abs(a[name] - want).max()))
