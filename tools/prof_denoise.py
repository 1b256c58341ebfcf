"""Cost of enrollment noise reduction (artspeech_b200/frontend.py step 2b, ``as_denoise``) on the GPU.

    python tools/prof_denoise.py [--out FILE] [--launches N] [--calls K] [--bench-steps S] [--no-bench]

For 16 recordings of 10 s and of 60 s (seeded tone bursts over white noise, 16 kHz PCM16 mono):

1. The stage alone (``ops.denoise`` on the 24 kHz rows, three launches): one CUDA graph of back-to-back calls, replayed
   to >= ``--launches`` calls between two CUDA events.  Consecutive calls read different 24 kHz input sets (together
   more than twice the 126 MB L2); the X and G planes the stage writes and reads back are its own working set.
2. Each kernel: its mean device time under ``torch.profiler`` (CUDA activities, a run of its own over ``--calls``
   eager calls), and its share of its byte floor at 7.7 TB/s.  Floors: the STFT reads 4 B per sample and writes X
   (8 B per bin and frame); the profile and gain kernel reads X and writes G (4 B per bin and frame), but it is a
   latency-bound chain (one fp64 divide per frame and bin in sequence), so its time per frame is reported too; the
   synthesis reads X and G and writes 4 B per sample.
3. The whole ``frontend.reference_mels`` call with and without ``noise_reduction_db=18`` (host clock over whole
   calls, each ending in its read-back; the timed loop ends in a device synchronise), with the input on the device.
4. The benchmark step (``bench.py --gpus 1``) in a subprocess of the same run: the benchmark does not call this code.

Writes one JSON object (with the GPU's name and power limit, read in the same run) to ``--out`` or stdout."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

from artspeech_b200 import audio, frontend, ops
from tools.prof_enroll import graph_time
from tools.prof_prosody import gpu_info

HBM_TBS = 7.7
L2_BYTES = 126 << 20
B, RATE = 16, 16000
BINS, HOP = ops.DENOISE_BINS, ops.DENOISE_HOP


def recordings(seconds, seed):
    """[B, S] int16 host samples: tone bursts between 0.5-1.5 s of leading and trailing white noise, 20 dB below."""
    rng = np.random.default_rng(seed)
    S = RATE * seconds
    y = rng.standard_normal((B, S)) * 0.02
    for b in range(B):
        lead, trail = (rng.uniform(0.5, 1.5, 2) * RATE).astype(int)
        k = np.arange(S - lead - trail)
        y[b, lead:S - trail] += 0.3 * np.sin(2 * np.pi * rng.uniform(100, 300) / RATE * k) * \
            (0.6 + 0.4 * np.sin(2 * np.pi * 4 / RATE * k))
    return torch.from_numpy(np.clip(np.rint(32767 * np.clip(y, -1, 1)), -32768, 32767).astype(np.int16))


def kernel_times(dev, y, n24, calls):
    """Mean device microseconds per launch of each denoise kernel under torch.profiler."""
    ops.denoise(y, n24, 18.0)
    torch.cuda.synchronize(dev)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            ops.denoise(y, n24, 18.0)
        torch.cuda.synchronize(dev)
    out = {}
    for ev in prof.key_averages():
        if "denoise_" in ev.key:
            total = getattr(ev, "device_time_total", None)
            if total is None:
                total = ev.cuda_time_total
            name = ev.key.split("(")[0].split("::")[-1].split("<")[0]
            out[name] = {"launches": ev.count, "us_per_launch": round(total / ev.count, 2)}
    return out


def floor(name, us, floor_bytes, extra=None):
    fl = floor_bytes / (HBM_TBS * 1e6)
    d = {"us_per_launch": us, "byte_floor": int(floor_bytes), "byte_floor_us": round(fl, 2),
         "share_of_byte_floor": round(fl / us, 3) if us else None}
    d.update(extra or {})
    return d


def profile_case(dev, seconds, args):
    x0 = recordings(seconds, seconds)
    S = x0.shape[1]
    fmt = audio.to_native_rate(RATE)
    S24 = fmt.out_samples(S)
    lens = torch.full((B,), S, dtype=torch.int32, device=dev)
    n24 = torch.empty(B, dtype=torch.int32, device=dev)
    nsets = max(2, -(-2 * L2_BYTES // (B * S24 * 4)) + 1)
    xs = [x0.to(dev)] + [torch.roll(x0, 97 * i, 1).to(dev) for i in range(1, nsets)]
    y24s = [ops.resample_encode(ops.audio_to_mono(x, lens, "pcm16"), lens, fmt, S24, out_lens=n24) for x in xs]
    F = 1 + S24 // HOP
    res = {"input": f"{B} x {seconds} s, {RATE} Hz pcm16 mono, noise 20 dB below the bursts",
           "samples_24k_per_row": S24, "frames_per_row": F, "buffer_sets_rotated": nsets,
           "workspace_bytes": int(ops._lib.load().as_denoise_workspace_bytes(B, S24))}
    us = graph_time(dev, [lambda y=y: ops.denoise(y, n24, 18.0) for y in y24s], args.launches)
    res["stage_us_per_call"] = round(us, 2)
    kt = kernel_times(dev, y24s[0], n24, args.calls)
    plane = B * F * BINS
    kernels = {}
    for name, v in kt.items():
        if "stft" in name:
            kernels[name] = floor(name, v["us_per_launch"], B * S24 * 4 + plane * 8)
        elif "gain" in name:
            kernels[name] = floor(name, v["us_per_launch"], plane * 12, {
                "bound": "latency: a sequential fp64 scan over the frames per (row, bin), one divide on the chain",
                "ns_per_frame_of_the_chain": round(v["us_per_launch"] * 1e3 / F, 1)})
        else:
            kernels[name] = floor(name, v["us_per_launch"], plane * 12 + B * S24 * 4)
    res["kernels_profiler"] = kernels
    res["reference_mels_ms"] = {}
    for label, nr in (("without noise reduction", None), ("noise_reduction_db=18", 18.0)):
        frontend.reference_mels(xs[0], None, RATE, "pcm16", noise_reduction_db=nr)
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for _ in range(args.calls):
            frontend.reference_mels(xs[0], None, RATE, "pcm16", noise_reduction_db=nr)
        torch.cuda.synchronize(dev)
        res["reference_mels_ms"][label] = round((time.perf_counter() - t0) * 1e3 / args.calls, 3)
    return res


def bench_step(steps, warmup):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup",
           str(warmup)]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True)
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    if r.returncode != 0 or not lines:
        return {"command": " ".join(cmd[1:]), "error": f"exit {r.returncode}", "stderr_tail": r.stderr[-2000:]}
    out = json.loads(lines[-1])
    return {"command": " ".join(["bench.py"] + cmd[2:]), "ms_per_step": out.get("ms_per_step"),
            "value": out.get("value"), "unit": out.get("unit")}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--bench-steps", type=int, default=10)
    ap.add_argument("--no-bench", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("prof_denoise.py: needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res = {"gpu": gpu_info(dev),
           "timing": "stage: CUDA events around graph replays of back-to-back calls with rotated input sets (launch "
                     "gaps included); kernels: torch.profiler device time, eager calls; reference_mels: host clock "
                     "over whole calls, each ending in its read-back",
           "cases": [profile_case(dev, s, args) for s in (10, 60)]}
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
