"""Cost and yield of FLAC output for synthesis (``as_flac_encode``, format in artspeech_b200/audio.py) on the GPU.

    python tools/prof_flac.py [--out FILE] [--launches N] [--calls K] [--bench-steps S] [--no-bench]

1. The stage alone (``ops.flac_encode``, three launches) at 16 x 10 s and 8 x 60 s of seeded speech-like PCM16 at 8,
   16, 24 and 48 kHz: one CUDA graph of back-to-back calls replayed to >= ``--launches`` calls between two CUDA
   events; consecutive calls read different input sets (together more than twice the 126 MB L2).
2. Each kernel's mean device time under ``torch.profiler`` (a run of its own), against its byte floor at 7.7 TB/s:
   analysis and emit read 2 B per sample, emit and layout write the output row (the bound, zeros included).
3. Compression ratio and device->host bytes per audio-second against PCM16, on the seeded speech-like clips and on the
   random-weight model's 24 kHz output (not representative of trained speech).
4. The benchmark step (``bench.py --gpus 1``) in a subprocess of the same run: the benchmark does not call this code.

Writes one JSON object (with the GPU's name and power limit, read in the same run) to ``--out`` or stdout."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

from artspeech_b200 import audio, checkpoint, engine, ops
from tests import enroll_ref
from tools.prof_denoise import bench_step
from tools.prof_enroll import graph_time
from tools.prof_prosody import gpu_info

HBM_TBS = 7.7
L2_BYTES = 126 << 20


def clips(B, seconds, rate, seed):
    """[B, S] int16 host rows of seeded speech-like audio generated at ``rate``."""
    rng = np.random.default_rng(seed)
    S = rate * seconds
    y = np.stack([enroll_ref.speech_like(rng, S, fs=rate) for _ in range(B)]).astype(np.float64)
    return torch.from_numpy(np.clip(np.rint(32767 * y), -32768, 32767).astype(np.int16))


def kernel_times(x, lens, rate, calls):
    ops.flac_encode(x, lens, rate)
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            ops.flac_encode(x, lens, rate)
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        if "flac_" in ev.key:
            out[ev.key.split("(")[0].split("::")[-1]] = round(ev.device_time_total / max(1, ev.count), 2)
    return out


def case(dev, B, seconds, rate, launches, calls):
    x0 = clips(B, seconds, rate, B * 1000 + rate)
    S = x0.shape[1]
    row = audio.flac_max_bytes(S)
    set_bytes = B * S * 2 + B * row
    nsets = max(2, -(-2 * L2_BYTES // set_bytes) + 1)
    xs = [x0.to(dev)] + [torch.roll(x0, 4099 * i, 1).to(dev) for i in range(1, nsets)]
    lens = torch.full((B,), S, dtype=torch.int32, device=dev)
    us = graph_time(dev, [lambda x=x: ops.flac_encode(x, lens, rate) for x in xs], launches, per_graph=8)
    out, nb = ops.flac_encode(xs[0], lens, rate)
    nbytes = int(nb.sum())
    kt = kernel_times(xs[0], lens, rate, calls)
    floors = {"flac_analysis_kernel": B * S * 2, "flac_layout_kernel": B * row - nbytes,
              "flac_emit_kernel": B * S * 2 + nbytes}
    kernels = {k: {"us": v, "byte_floor_us": round(floors.get(k, 0) / (HBM_TBS * 1e6), 2),
                   "share_of_byte_floor": round(floors.get(k, 0) / (HBM_TBS * 1e6) / v, 3) if v else None}
               for k, v in kt.items()}
    return {"B": B, "seconds": seconds, "rate": rate, "input_sets": nsets, "us_per_call": round(us, 2),
            "audio_s_per_s": round(B * seconds / (us * 1e-6), 1), "kernels": kernels,
            "compression_ratio": round(nbytes / (2 * B * S), 4),
            "flac_bytes_per_audio_s": round(nbytes / (B * seconds), 1), "pcm16_bytes_per_audio_s": 2 * rate}


def model_output(dev):
    """Compression of the random-weight model's output at 24 kHz (16 utterances, forced durations)."""
    model = checkpoint.build_random_artsspeech(0)
    gen = checkpoint.build_random_generator(0)
    syn = engine.Synthesizer(model, gen, device=dev, use_cuda_graph=False)
    g = torch.Generator().manual_seed(5)
    tl = [120] * 16
    tok = torch.randint(1, 178, (16, 120), generator=g)
    mel = (torch.randn(16, 80, 110, generator=g) * 0.5).clamp(-2, 2)
    dur = torch.randint(2, 6, (16, 120), generator=g)
    fmt = audio.AudioFormat(24000, "pcm16", container="flac")
    syn.synthesize(tok.to(dev), tl, mel.to(dev), [110] * 16, dur, audio=fmt)
    nb = syn.last["byte_lengths"].cpu()
    n = syn.last["sample_lengths"].cpu()
    sec = float(n.sum()) / 24000
    return {"utterances": 16, "audio_s": round(sec, 2), "compression_ratio": round(float(nb.sum()) / (2 * float(n.sum())), 4),
            "flac_bytes_per_audio_s": round(float(nb.sum()) / sec, 1), "pcm16_bytes_per_audio_s": 48000,
            "note": "random weights: not representative of trained speech"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--bench-steps", type=int, default=10)
    ap.add_argument("--no-bench", action="store_true")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    res = {"gpu": gpu_info(dev), "cases": []}
    for B, sec in ((16, 10), (8, 60)):
        for rate in (8000, 16000, 24000, 48000):
            res["cases"].append(case(dev, B, sec, rate, args.launches, args.calls))
            print(json.dumps(res["cases"][-1]), file=sys.stderr)
    res["model_output"] = model_output(dev)
    if not args.no_bench:
        res["bench"] = bench_step(args.bench_steps, 3)
    text = json.dumps(res, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
