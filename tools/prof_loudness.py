"""Cost of loudness normalisation (artspeech_b200/audio.py, ``as_loudness_measure``) on the GPU.

    python tools/prof_loudness.py [--out FILE] [--rounds R] [--steps K] [--launches N]

1. The meter alone (its three launches) at 16 x 10 s and 8 x 60 s of 24 kHz input: one CUDA graph of back-to-back
   meter calls, replayed to >= ``--launches`` calls between two CUDA events.  Consecutive calls read different input
   buffers: the sets together exceed twice the 126 MB L2, so every call streams from HBM.  The byte floor is two
   reads of 4 bytes per sample (the two filter passes) at 7.7 TB/s.
2. The benchmark's step (BASELINE configs[1], two calls in flight, as bench.py) in alternating arms: unformatted;
   loudness-normalised 24 kHz fp32; loudness-normalised 8 kHz mu-law.  Per round every arm times K steps with CUDA
   events (the order rotates between rounds).

Writes one JSON object (with the GPU's name and power limit, read in the same run) to ``--out`` or stdout."""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import bench
from artspeech_b200 import checkpoint, engine, ops
from artspeech_b200.audio import AudioFormat, Loudness
from tools.prof_prosody import gpu_info

HBM_TBS = 7.7
L2_BYTES = 126 << 20


def meter_time(dev, B, seconds, launches, per_graph=50):
    S = 24000 * seconds
    set_bytes = B * S * 4
    nsets = max(2, -(-2 * L2_BYTES // set_bytes) + 1)
    g = torch.Generator(device=dev).manual_seed(0)
    xs = [(torch.rand(B, S, device=dev, generator=g) * 1.6 - 0.8) for _ in range(nsets)]
    lens = torch.full((B,), S, dtype=torch.int32, device=dev)
    s = torch.cuda.Stream(device=dev)
    s.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(s):
        for x in xs:
            ops.loudness_measure(x, lens, 24000)
    torch.cuda.current_stream(dev).wait_stream(s)
    torch.cuda.synchronize(dev)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for i in range(per_graph):
            ops.loudness_measure(xs[i % nsets], lens, 24000)
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
    floor_bytes = 2 * 4 * B * S
    return {"B": B, "seconds": seconds, "samples": B * S, "calls": total, "launches_per_call": ops.LOUDNESS_LAUNCHES,
            "us_per_call": round(us, 3), "byte_floor": floor_bytes,
            "byte_floor_us": round(floor_bytes / (HBM_TBS * 1e6), 2),
            "share_of_byte_floor": round(floor_bytes / (HBM_TBS * 1e6) / us, 3), "buffer_sets_rotated": nsets}


def step_arms(dev, rounds, steps):
    model = checkpoint.build_random_artsspeech(0)
    gen = checkpoint.build_random_generator(0)
    syn = engine.Synthesizer(model, gen, device=dev, pipeline_depth=2)
    B = bench.B_PER_GPU
    sets = [bench.make_inputs(0, B, i) for i in range(bench.N_INPUT_SETS)]
    tl, ml = sets[0][1], sets[0][3]
    dev_sets = [(t.to(dev), m.to(dev), d) for t, _, m, _, d in sets]
    arms = {"unformatted": (None, None), "loudness_24k_f32": (None, Loudness()),
            "loudness_8k_mulaw": (AudioFormat(8000, "mulaw"), Loudness())}
    calls = [0]

    def step(arm):
        fmt, loud = arms[arm]
        t, m, d = dev_sets[calls[0] % len(dev_sets)]
        calls[0] += 1
        kw = {} if loud is None else dict(loudness=loud)
        return syn.synthesize(t, tl, m, ml, d, predict_durations=True, audio=fmt, **kw)

    info = {}
    for name in arms:
        for _ in range(4):
            step(name)
        syn.join()
        w, _, _ = step(name)
        syn.join()
        info[name] = {"launches_per_call": syn.launches_per_call, "shape": list(w.shape), "dtype": str(w.dtype)}
    torch.cuda.synchronize(dev)
    captures = syn.stats["captures"]
    times = {k: [] for k in arms}
    names = list(arms)
    for r in range(rounds):
        order = names[r % len(names):] + names[:r % len(names)]
        for name in order:
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                step(name)
            syn.join()
            e1.record()
            torch.cuda.synchronize(dev)
            times[name].append(e0.elapsed_time(e1) / steps)
    assert syn.stats["captures"] == captures, "the timed steps must replay graphs"
    res = {"workload": f"bench.py step: {B} x {bench.TT} tokens, Tr = {bench.TR}, sum(dur) = {bench.SUM_DUR}, "
                       "predict_durations=True, pipeline_depth=2, 8 seeded input sets cycled",
           "rounds": rounds, "steps_per_round": steps, "arms": {}}
    for name in names:
        ts = times[name]
        res["arms"][name] = dict(info[name], mean_step_ms=sum(ts) / len(ts), min_round_ms=min(ts),
                                 max_round_ms=max(ts), round_ms=ts)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--launches", type=int, default=500)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("prof_loudness.py: needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res = {"gpu": gpu_info(dev)}
    res["as_loudness_measure"] = {
        "timing": "CUDA events around graph replays of back-to-back meter calls (launch gaps included); input buffer "
                  "sets rotated so that each call's input was evicted from L2 by the others",
        "runs": [meter_time(dev, B, s, args.launches) for B, s in ((16, 10), (8, 60))]}
    res["step"] = step_arms(dev, args.rounds, args.steps)
    text = json.dumps(res, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
