"""Cost of the prosody controls (artspeech_b200/prosody.py) on the GPU.

    python tools/prof_prosody.py [--out FILE] [--rounds R] [--steps K]

1. The benchmark's step (BASELINE configs[1]: 16 utterances x 150 tokens, 240-frame reference mels, seeded durations
   summing to 400, the duration predictor inside the graph, two calls in flight) in three arms that alternate within
   one process: no prosody, identity prosody, and edited prosody (pitch +3 semitones, range 1.2, +2 dB, articulation
   scale 1.1, duration_scale 1 so the frame counts match).  Each round times K steps of every arm with CUDA events
   (the arm order rotates between rounds); the mean step time per arm is over all rounds.
2. ``as_prosody_apply`` alone at 16 x 800 and 8 x 4800 frames: one CUDA graph of back-to-back launches, replayed to
   >= 1000 launches between two CUDA events.  The controls alternate with their inverse, so the tracks stay bounded.

Writes one JSON object (with the GPU's name and power limit, read in the same run) to ``--out`` or stdout."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import bench
from artspeech_b200 import checkpoint, engine, ops, prosody
from artspeech_b200.prosody import Prosody

EDIT = dict(pitch_shift=3.0, pitch_range=1.2, energy_db=2.0, articulation_scale=[1.1] * 10)
INVERSE = dict(pitch_shift=-3.0, pitch_range=1 / 1.2, energy_db=-2.0, articulation_scale=[1 / 1.1] * 10)


def gpu_info(dev):
    info = {"name": torch.cuda.get_device_name(dev)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                            "-i", str(dev.index or 0)], capture_output=True, text=True, timeout=30).stdout.strip()
        pl, mx = [v.strip() for v in q.split(",")]
        info.update(power_limit_w=float(pl), sm_max_mhz=int(float(mx)))
    except Exception as e:                              # reported, not guessed
        info.update(power_limit_w="not measured", sm_max_mhz="not measured", query_error=repr(e))
    return info


def step_arms(dev, rounds, steps):
    model = checkpoint.build_random_artsspeech(0)
    gen = checkpoint.build_random_generator(0)
    syn = engine.Synthesizer(model, gen, device=dev, pipeline_depth=2)
    B = bench.B_PER_GPU
    sets = [bench.make_inputs(0, B, i) for i in range(bench.N_INPUT_SETS)]
    tl, ml = sets[0][1], sets[0][3]
    dev_sets = [(t.to(dev), m.to(dev), d) for t, _, m, _, d in sets]
    arms = {"none": None, "identity": [Prosody()] * B, "edited": [Prosody(**EDIT)] * B}
    calls = [0]

    def step(pros):
        t, m, d = dev_sets[calls[0] % len(dev_sets)]
        calls[0] += 1
        return syn.synthesize(t, tl, m, ml, d, predict_durations=True, prosody=pros)

    outs = {}
    for name, pros in arms.items():                     # warm-up: capture every arm's graphs, keep one result each
        calls[0] = 0
        for _ in range(4):
            step(pros)
        syn.join()
        calls[0] = 0
        w, lens, _ = step(pros)
        syn.join()
        outs[name] = (w.clone(), lens.clone(), syn.launches_per_call)
    torch.cuda.synchronize(dev)
    captures = syn.stats["captures"]
    times = {k: [] for k in arms}
    names = list(arms)
    for r in range(rounds):
        order = names[r % 3:] + names[:r % 3]
        for name in order:
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                step(arms[name])
            syn.join()
            e1.record()
            torch.cuda.synchronize(dev)
            times[name].append(e0.elapsed_time(e1) / steps)
    assert syn.stats["captures"] == captures, "the timed steps must replay graphs"
    w0, l0, _ = outs["none"]
    res = {"workload": f"bench.py step: {B} x {bench.TT} tokens, Tr = {bench.TR}, sum(dur) = {bench.SUM_DUR}, "
                       "predict_durations=True, pipeline_depth=2, 8 seeded input sets cycled",
           "rounds": rounds, "steps_per_round": steps, "arms": {}}
    for name in names:
        w, l, launches = outs[name]
        ts = times[name]
        res["arms"][name] = {"mean_step_ms": sum(ts) / len(ts), "min_round_ms": min(ts), "max_round_ms": max(ts),
                             "round_ms": ts, "launches_per_call": launches,
                             "frames_equal_to_none": bool(torch.equal(l, l0)),
                             "wav_bit_identical_to_none": bool(torch.equal(w, w0))}
    res["edited_prosody"] = EDIT
    return res


def kernel_time(dev, B, Tm, launches=1000, per_graph=100):
    g = torch.Generator().manual_seed(0)
    f0 = (torch.randn(B, Tm, 1, generator=g) * 0.8).to(dev)
    n = torch.randn(B, Tm, 1, generator=g).to(dev)
    ema = torch.randn(B, Tm, 10, generator=g).to(dev)
    lens = torch.full((B,), Tm, dtype=torch.int32, device=dev)
    ctrls = [prosody.pack([Prosody(**kw)] * B, 1)[0].to(dev) for kw in (EDIT, INVERSE)]
    consts = prosody.constants(checkpoint.default_distribution())
    s = torch.cuda.Stream(device=dev)
    s.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(s):
        for c in ctrls:
            ops.prosody_apply(f0, n, ema, lens, c, *consts)
    torch.cuda.current_stream(dev).wait_stream(s)
    torch.cuda.synchronize(dev)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for i in range(per_graph):
            ops.prosody_apply(f0, n, ema, lens, ctrls[i % 2], *consts)
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
    assert bool(torch.isfinite(f0).all()) and bool(torch.isfinite(ema).all())
    return {"B": B, "frames_per_utterance": Tm, "launches": total, "us_per_launch": us,
            "bytes_per_launch": B * Tm * 12 * 4 * 2,
            "timing": "CUDA events around graph replays of back-to-back launches (launch gaps included)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--steps", type=int, default=30)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("prof_prosody.py: needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res = {"gpu": gpu_info(dev)}
    res["step"] = step_arms(dev, args.rounds, args.steps)
    res["as_prosody_apply"] = [kernel_time(dev, 16, 800), kernel_time(dev, 8, 4800)]
    text = json.dumps(res, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
