"""Cost of voice enrollment from recordings (artspeech_b200/frontend.py: ``as_audio_to_mono``, ``as_resample_encode``
to 24 kHz, ``as_trim_bounds``, ``as_log_mel_span``) on the GPU.

    python tools/prof_enroll.py [--out FILE] [--launches N] [--calls K]

For 16 recordings of 10 s in each of 8 kHz mu-law mono, 16 kHz PCM16 mono, 44.1 kHz PCM16 stereo and 48 kHz fp32
stereo (seeded tone bursts with leading and trailing silence):

1. Each stage alone: one CUDA graph of back-to-back calls, replayed to >= ``--launches`` calls between two CUDA
   events.  Consecutive calls read different input buffer sets (together more than twice the 126 MB L2).  Byte floors
   at 7.7 TB/s: downmix reads the encoded input and writes 4 bytes a sample; the resampler reads 4 bytes a sample and
   writes 4 bytes a 24 kHz sample; the trim reads 4 bytes a 24 kHz sample; the log-mel reads its span once and writes
   the mels.
2. The whole ``reference_mels`` call (decode, resample, trim, read-back, log-mel) with a host clock: the call ends in
   its own read-back and the timed loop ends in a device synchronise.
3. The style encoder (``Synthesizer.encode_voice``) on the resulting mels, for scale (CUDA events).

Writes one JSON object (with the GPU's name and power limit, read in the same run) to ``--out`` or stdout."""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from artspeech_b200 import audio, checkpoint, engine, frontend, ops
from tools.prof_prosody import gpu_info

HBM_TBS = 7.7
L2_BYTES = 126 << 20
B, SECONDS = 16, 10
CASES = [(8000, "mulaw", 1), (16000, "pcm16", 1), (44100, "pcm16", 2), (48000, "float32", 2)]


def recordings(rate, encoding, C, seed):
    """[B, S(, C)] host samples: tone bursts between 0.5-1.5 s of leading and trailing silence (with a -80 dB floor)."""
    rng = np.random.default_rng(seed)
    S = rate * SECONDS
    y = rng.standard_normal((B, S, C)) * 1e-4
    for b in range(B):
        lead, trail = (rng.uniform(0.5, 1.5, 2) * rate).astype(int)
        k = np.arange(S - lead - trail)
        for c in range(C):
            y[b, lead:S - trail, c] += 0.3 * np.sin(2 * np.pi * rng.uniform(100, 300) / rate * k) * \
                (0.6 + 0.4 * np.sin(2 * np.pi * 4 / rate * k))
    y = np.clip(y, -1, 1)
    if encoding == "float32":
        x = torch.from_numpy(y.astype(np.float32))
    else:
        s = np.clip(np.rint(32767 * y), -32768, 32767).astype(np.int64)
        if encoding == "pcm16":
            x = torch.from_numpy(s.astype(np.int16))
        else:
            from tests import audio_ref
            x = torch.from_numpy(audio_ref.ULAW[s + 32768])
    return x[..., 0].contiguous() if C == 1 else x.contiguous()


def graph_time(dev, fns, launches, per_graph=40):
    """us per call of ``fns[i % len(fns)]()`` replayed from one CUDA graph."""
    s = torch.cuda.Stream(device=dev)
    s.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(s):
        for f in fns:
            f()
    torch.cuda.current_stream(dev).wait_stream(s)
    torch.cuda.synchronize(dev)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for i in range(per_graph):
            fns[i % len(fns)]()
    graph.replay()
    torch.cuda.synchronize(dev)
    reps = -(-launches // per_graph)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        graph.replay()
    e1.record()
    torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1) * 1e3 / (reps * per_graph)


def stage(name, us, floor_bytes, launches):
    fl = floor_bytes / (HBM_TBS * 1e6)
    return {"stage": name, "launches": launches, "us_per_call": round(us, 2), "byte_floor": int(floor_bytes),
            "byte_floor_us": round(fl, 2), "share_of_byte_floor": round(fl / us, 3)}


def profile_case(dev, rate, encoding, C, args, syn):
    x0 = recordings(rate, encoding, C, rate + C)
    S = x0.shape[1]
    set_bytes = x0.numel() * x0.element_size() + B * S * 4
    nsets = max(2, -(-2 * L2_BYTES // set_bytes) + 1)
    xs = [x0.to(dev)] + [torch.roll(x0, 97 * i, 1).to(dev) for i in range(1, nsets)]
    lens = torch.full((B,), S, dtype=torch.int32, device=dev)
    fmt = audio.to_native_rate(rate)
    S24 = fmt.out_samples(S)
    monos = [ops.audio_to_mono(x, lens, encoding) for x in xs]
    n24 = torch.empty(B, dtype=torch.int32, device=dev)
    y24s = [ops.resample_encode(m, lens, fmt, S24, out_lens=n24) for m in monos]
    bounds = ops.trim_bounds(y24s[0], n24, 30.0)
    hb = bounds.cpu()
    span = (hb[:, 1] - hb[:, 0]).to(torch.int64)
    T = int(1 + span.max() // 300)
    starts, spans = hb[:, 0].contiguous().to(dev), span.to(torch.int32).to(dev)
    fe = frontend.LogMel().to(dev)
    es = x0.element_size()
    res = {"input": f"{B} x {SECONDS} s, {rate} Hz {encoding}, {C} channel(s)", "buffer_sets_rotated": nsets,
           "trimmed_seconds_mean": round(float(span.double().mean()) / 24000, 3), "stages": []}
    if encoding != "float32" or C > 1:
        us = graph_time(dev, [lambda x=x: ops.audio_to_mono(x, lens, encoding) for x in xs], args.launches)
        res["stages"].append(stage("as_audio_to_mono", us, B * S * (C * es + 4), 1))
    us = graph_time(dev, [lambda m=m: ops.resample_encode(m, lens, fmt, S24, out_lens=n24) for m in monos],
                    args.launches)
    res["stages"].append(stage("as_resample_encode to 24 kHz", us, B * (S + S24) * 4, 1))
    us = graph_time(dev, [lambda y=y: ops.trim_bounds(y, n24, 30.0) for y in y24s], args.launches)
    res["stages"].append(stage("as_trim_bounds", us, B * S24 * 4, 2))
    us = graph_time(dev, [lambda y=y: fe(y, spans, starts=starts, n_frames=T) for y in y24s], args.launches)
    res["stages"].append(stage("as_log_mel_span", us, int(span.sum()) * 4 + B * 80 * T * 4, 1))
    res["reference_mels_ms"] = {}
    for where, inp in (("device input", xs[0]), ("host input, pinned", x0.pin_memory())):
        frontend.reference_mels(inp, None, rate, encoding)
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for _ in range(args.calls):
            mels, mel_lens, _ = frontend.reference_mels(inp, None, rate, encoding)
        torch.cuda.synchronize(dev)
        res["reference_mels_ms"][where] = round((time.perf_counter() - t0) * 1e3 / args.calls, 3)
    syn.encode_voice(mels, mel_lens)
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(3):
        syn.encode_voice(mels, mel_lens)
    e1.record()
    torch.cuda.synchronize(dev)
    res["style_encoder_ms"] = round(e0.elapsed_time(e1) / 3, 3)
    res["distinct_mel_lengths"] = len(set(mel_lens.tolist()))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--launches", type=int, default=400)
    ap.add_argument("--calls", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("prof_enroll.py: needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    model = checkpoint.build_random_artsspeech(0)
    gen = checkpoint.build_random_generator(0)
    syn = engine.Synthesizer(model, gen, device=dev, use_cuda_graph=False)
    res = {"gpu": gpu_info(dev),
           "timing": "per stage: CUDA events around graph replays of back-to-back calls with rotated input sets "
                     "(launch gaps included); reference_mels: host clock over whole calls, each ending in its "
                     "read-back; style encoder: CUDA events, eager, one group per distinct mel length",
           "cases": [profile_case(dev, r, e, c, args, syn) for r, e, c in CASES]}
    text = json.dumps(res, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
