"""Cost of the output audio formats (artspeech_b200/audio.py, ``as_resample_encode``) on the GPU.

    python tools/prof_audio_format.py [--out FILE] [--rounds R] [--steps K] [--launches N]

1. ``as_resample_encode`` alone for every listed rate x encoding at 16 x 10 s and 8 x 60 s of 24 kHz input: one CUDA
   graph of back-to-back launches, replayed to >= ``--launches`` launches between two CUDA events.  Consecutive
   launches read and write different buffers: the input/output sets together exceed twice the 126 MB L2, so every
   launch streams from HBM.  Achieved bandwidth = (4 * sum n_in + elem * sum n_out) / time, against 7.7 TB/s.
2. The benchmark's step (BASELINE configs[1], two calls in flight, as bench.py) in alternating arms: without the
   format stage (24 kHz fp32) and with it, for 8 kHz mu-law and 16 kHz PCM.  Per round every arm times K steps with
   CUDA events (the order rotates between rounds).  In the same rounds each arm also times the device->host copy of
   one step's waveforms into pinned memory.

Writes one JSON object (with the GPU's name and power limit, read in the same run) to ``--out`` or stdout."""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import bench
from artspeech_b200 import checkpoint, engine, ops
from artspeech_b200.audio import ENCODINGS, AudioFormat
from tools.prof_prosody import gpu_info

RATES = (8000, 11025, 16000, 22050, 24000, 32000, 44100, 48000)
HBM_TBS = 7.7
L2_BYTES = 126 << 20


def kernel_time(dev, fmt, B, seconds, launches, per_graph=50):
    S_in = 24000 * seconds
    S_out = fmt.out_samples(S_in)
    es = torch.empty((), dtype=fmt.dtype).element_size()
    set_bytes = B * (S_in * 4 + S_out * es)
    nsets = max(2, -(-2 * L2_BYTES // set_bytes) + 1)
    g = torch.Generator(device=dev).manual_seed(0)
    xs = [torch.rand(B, S_in, device=dev, generator=g) * 1.6 - 0.8 for _ in range(nsets)]
    ys = [torch.empty(B, S_out, dtype=fmt.dtype, device=dev) for _ in range(nsets)]
    lens = torch.full((B,), S_in, dtype=torch.int32, device=dev)
    s = torch.cuda.Stream(device=dev)
    s.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(s):
        for x, y in zip(xs, ys):
            ops.resample_encode(x, lens, fmt, S_out, out=y)
    torch.cuda.current_stream(dev).wait_stream(s)
    torch.cuda.synchronize(dev)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for i in range(per_graph):
            ops.resample_encode(xs[i % nsets], lens, fmt, S_out, out=ys[i % nsets])
    graph.replay()
    torch.cuda.synchronize(dev)
    reps = -(-launches // per_graph)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        graph.replay()
    e1.record()
    torch.cuda.synchronize(dev)
    total = reps * per_graph
    us = e0.elapsed_time(e1) * 1e3 / total
    nbytes = B * (S_in * 4 + S_out * es)
    return {"rate": fmt.sample_rate, "encoding": fmt.encoding, "B": B, "seconds": seconds, "K": fmt.K,
            "launches": total, "us_per_launch": round(us, 3), "bytes": nbytes,
            "GB_per_s": round(nbytes / us / 1e3, 1), "share_of_7p7_TBs": round(nbytes / us / 1e6 / HBM_TBS, 3),
            "hbm_floor_us": round(nbytes / (HBM_TBS * 1e6), 2), "buffer_sets_rotated": nsets}


def step_arms(dev, rounds, steps):
    model = checkpoint.build_random_artsspeech(0)
    gen = checkpoint.build_random_generator(0)
    syn = engine.Synthesizer(model, gen, device=dev, pipeline_depth=2)
    B = bench.B_PER_GPU
    sets = [bench.make_inputs(0, B, i) for i in range(bench.N_INPUT_SETS)]
    tl, ml = sets[0][1], sets[0][3]
    dev_sets = [(t.to(dev), m.to(dev), d) for t, _, m, _, d in sets]
    arms = {"native_24k_f32": None, "8k_mulaw": AudioFormat(8000, "mulaw"), "16k_pcm16": AudioFormat(16000, "pcm16")}
    calls = [0]

    def step(fmt):
        t, m, d = dev_sets[calls[0] % len(dev_sets)]
        calls[0] += 1
        return syn.synthesize(t, tl, m, ml, d, predict_durations=True, audio=fmt)

    info = {}
    for name, fmt in arms.items():                      # warm-up: every arm's graphs and kernels
        for _ in range(4):
            step(fmt)
        syn.join()
        w, _, _ = step(fmt)
        syn.join()
        info[name] = {"launches_per_call": syn.launches_per_call, "bytes_per_step": w.numel() * w.element_size(),
                      "shape": list(w.shape), "dtype": str(w.dtype)}
    torch.cuda.synchronize(dev)
    captures = syn.stats["captures"]
    pinned = {k: torch.empty(v["bytes_per_step"], dtype=torch.uint8).pin_memory() for k, v in info.items()}
    times = {k: [] for k in arms}
    copies = {k: [] for k in arms}
    names = list(arms)
    for r in range(rounds):
        order = names[r % len(names):] + names[:r % len(names)]
        for name in order:
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                w, _, _ = step(arms[name])
            syn.join()
            e1.record()
            torch.cuda.synchronize(dev)
            times[name].append(e0.elapsed_time(e1) / steps)
            # the device->host copy of the last step's waveforms (pinned destination), timed alone
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            src = w.contiguous().view(-1).view(torch.uint8)
            torch.cuda.synchronize(dev)
            c0.record()
            pinned[name].copy_(src, non_blocking=True)
            c1.record()
            torch.cuda.synchronize(dev)
            copies[name].append(c0.elapsed_time(c1))
    assert syn.stats["captures"] == captures, "the timed steps must replay graphs"
    res = {"workload": f"bench.py step: {B} x {bench.TT} tokens, Tr = {bench.TR}, sum(dur) = {bench.SUM_DUR}, "
                       "predict_durations=True, pipeline_depth=2, 8 seeded input sets cycled",
           "rounds": rounds, "steps_per_round": steps, "arms": {}}
    for name in names:
        ts, cs = times[name], copies[name]
        res["arms"][name] = dict(info[name], mean_step_ms=sum(ts) / len(ts), min_round_ms=min(ts),
                                 max_round_ms=max(ts), round_ms=ts, mean_d2h_copy_ms=sum(cs) / len(cs),
                                 d2h_copy_ms=cs)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--launches", type=int, default=1000)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("prof_audio_format.py: needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res = {"gpu": gpu_info(dev)}
    res["as_resample_encode"] = {
        "timing": "CUDA events around graph replays of back-to-back launches (launch gaps included); input and "
                  "output buffer sets rotated so that each launch's set was evicted from L2 by the others",
        "runs": [kernel_time(dev, AudioFormat(r, e), B, s, args.launches)
                 for B, s in ((16, 10), (8, 60)) for r in RATES for e in ENCODINGS]}
    res["step"] = step_arms(dev, args.rounds, args.steps)
    text = json.dumps(res, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
