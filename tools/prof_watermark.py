"""Cost of the synthesis watermark (artspeech_b200/audio.py, ``as_watermark_embed`` / ``as_watermark_detect``) on the
GPU.

    python tools/prof_watermark.py [--out FILE] [--rounds R] [--steps K] [--launches N] [--clips C]

1. The embedder alone at 16 x 10 s and 8 x 60 s of 24 kHz input: one CUDA graph of back-to-back embed calls, replayed
   to >= ``--launches`` calls between two CUDA events.  Consecutive calls read different input buffers (the sets
   together exceed twice the 126 MB L2).  The byte floor is 8 bytes per sample (read x, write y) at 7.7 TB/s.
2. The detector on a scan-sized batch (``--clips`` clips of 10 s) delivered as 8 kHz mu-law and as 48 kHz fp32:
   clips per second of the whole ``detect_watermark`` call (CUDA events), and the time of each launch (decode,
   resample, the two detector launches) from a separate ``torch.profiler`` run.
3. The benchmark's step (BASELINE configs[1], two calls in flight, as bench.py) in alternating arms: no watermark;
   watermark; watermark + loudness + 8 kHz mu-law.  Per round every arm times K steps with CUDA events (the order
   rotates between rounds).

Writes one JSON object (with the GPU's name and power limit, read in the same run) to ``--out`` or stdout."""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import bench
from artspeech_b200 import checkpoint, engine, ops
from artspeech_b200.audio import AudioFormat, Loudness, Watermark, detect_watermark, embed_watermark
from tools.prof_prosody import gpu_info

HBM_TBS = 7.7
L2_BYTES = 126 << 20
KEY = 0x0123456789ABCDEF


def embed_time(dev, B, seconds, launches, per_graph=50):
    S = 24000 * seconds
    set_bytes = B * S * 4
    nsets = max(2, -(-2 * L2_BYTES // set_bytes) + 1)
    g = torch.Generator(device=dev).manual_seed(0)
    xs = [(torch.rand(B, S, device=dev, generator=g) * 1.6 - 0.8) for _ in range(nsets)]
    lens = torch.full((B,), S, dtype=torch.int32, device=dev)
    wm = Watermark(KEY, 1)
    s = torch.cuda.Stream(device=dev)
    s.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(s):
        for x in xs:
            ops.watermark_embed(x, lens, wm)
    torch.cuda.current_stream(dev).wait_stream(s)
    torch.cuda.synchronize(dev)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for i in range(per_graph):
            ops.watermark_embed(xs[i % nsets], lens, wm)
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
    floor_bytes = 8 * B * S
    return {"B": B, "seconds": seconds, "samples": B * S, "calls": total, "us_per_call": round(us, 3),
            "byte_floor": floor_bytes, "byte_floor_us": round(floor_bytes / (HBM_TBS * 1e6), 2),
            "share_of_byte_floor": round(floor_bytes / (HBM_TBS * 1e6) / us, 3), "buffer_sets_rotated": nsets}


def detect_scan(dev, clips, rate, enc, reps=5):
    """``clips`` marked 10 s clips delivered at ``rate`` / ``enc``; returns clips/s and the per-launch times."""
    S24 = 240000
    g = torch.Generator(device=dev).manual_seed(1)
    chunk = 128
    f = AudioFormat(rate, enc)
    y = torch.empty(clips, f.out_samples(S24), dtype=f.dtype, device=dev)
    for i in range(0, clips, chunk):                      # noise-like 24 kHz clips, marked, in the output format
        x = torch.randn(min(chunk, clips - i), S24, device=dev, generator=g) * 0.1
        y[i:i + chunk] = ops.resample_encode(embed_watermark(x, None, Watermark(KEY, 77)), None, f, y.shape[1])
    det, _, msg = detect_watermark(y, None, rate, KEY, encoding=enc)
    torch.cuda.synchronize(dev)
    ok = int((det & (msg == 77)).sum())
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        detect_watermark(y, None, rate, KEY, encoding=enc)
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / reps
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            detect_watermark(y, None, rate, KEY, encoding=enc)
        torch.cuda.synchronize(dev)
    per = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)
        if t and ev.count:
            per[ev.key[:80]] = round(t / reps / 1e3, 3)
    return {"clips": clips, "seconds_per_clip": 10, "delivered": f"{rate} Hz {enc}", "input_bytes": y.numel() *
            y.element_size(), "ms_per_call": round(ms, 3), "clips_per_s": round(clips / ms * 1e3, 1),
            "detected_with_message": ok, "device_ms_per_call_by_kernel": per}


def step_arms(dev, rounds, steps):
    model = checkpoint.build_random_artsspeech(0)
    gen = checkpoint.build_random_generator(0)
    syn = engine.Synthesizer(model, gen, device=dev, pipeline_depth=2)
    B = bench.B_PER_GPU
    sets = [bench.make_inputs(0, B, i) for i in range(bench.N_INPUT_SETS)]
    tl, ml = sets[0][1], sets[0][3]
    dev_sets = [(t.to(dev), m.to(dev), d) for t, _, m, _, d in sets]
    wm = Watermark(KEY, 0x0B0E)
    arms = {"unmarked": {}, "watermark": dict(watermark=wm),
            "watermark_loudness_8k_mulaw": dict(watermark=wm, loudness=Loudness(), audio=AudioFormat(8000, "mulaw"))}
    calls = [0]

    def step(arm):
        t, m, d = dev_sets[calls[0] % len(dev_sets)]
        calls[0] += 1
        return syn.synthesize(t, tl, m, ml, d, predict_durations=True, **arms[arm])

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
    ap.add_argument("--clips", type=int, default=1024)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("prof_watermark.py: needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res = {"gpu": gpu_info(dev)}
    res["as_watermark_embed"] = {
        "timing": "CUDA events around graph replays of back-to-back embed calls (launch gaps included); input buffer "
                  "sets rotated so that each call's input was evicted from L2 by the others",
        "runs": [embed_time(dev, B, s, args.launches) for B, s in ((16, 10), (8, 60))]}
    res["detect_watermark"] = {
        "timing": "CUDA events around whole detect_watermark calls on resident inputs (decode, resample, 2 detector "
                  "launches); per-kernel device times from a separate torch.profiler run",
        "runs": [detect_scan(dev, args.clips, 8000, "mulaw"), detect_scan(dev, args.clips, 48000, "float32")]}
    res["step"] = step_arms(dev, args.rounds, args.steps)
    text = json.dumps(res, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
