#!/usr/bin/env python
"""Benchmark of the hot path named by BASELINE.json: ArtSpeech batched synthesis (text/phonemes +
reference mel -> mel -> waveform) on B200.

    python bench.py --gpus N --steps K --warmup W            # ours (CUDA path)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU PyTorch path
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's outputs as DIR/*.npy

Workload (BASELINE.json configs[1], SURVEY.md §8d config 2): per GPU, 16 utterances x 150 phoneme
tokens, a 3 s reference mel (240 frames) each, forced integer durations summing to 400 per
utterance -> 800 mel frames = 10.0 s of 24 kHz audio per utterance, 160 audio-seconds per step per
GPU.  Synthetic seeded inputs, random-init conditioned weights (artspeech_b200.checkpoint): the
reference's checkpoints are not redistributable (SURVEY.md F2).

One JSON line on stdout (rank 0).  `value` = audio-seconds synthesised per wall-second with inputs
resident in HBM; `e2e` = the same through the public API with pinned HOST inputs (H2D of tokens /
reference mels, D2H of the waveforms inside the timed region).

`--dump-outputs DIR` (CUDA arm) writes what the last timed step of the resident-input arm returned to its
caller (rank 0): `wav.npy` float32 [B, 300 * frames], `mel.npy` float32 [B, 80, frames] and
`mel_lengths.npy` float64 [B].  That step ran on input set
`(warmup_calls(warmup, pipeline) + steps - 1) % N_INPUT_SETS` of `make_inputs(rank, ...)`.  Inputs and
weights are seeded, so two builds run with the same arguments can be compared output for output.  The
outputs are copied on the device after the timed region and written once the clock sampling has stopped;
more than 64 MB in all is cut to a seeded sample of utterances, whose indices are then written as
`utterance_index.npy`.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import warnings

warnings.filterwarnings("ignore", category=FutureWarning)
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

B_PER_GPU, TT, TR, SUM_DUR = int(os.environ.get("ASB_BENCH_B", "16")), 150, 240, 400   # env override: experiments only
FRAMES = 2 * SUM_DUR                                   # mel frames per utterance
AUDIO_S_PER_UTT = FRAMES * 300 / 24000.0               # 10.0 s
VOCODER_FLOP_PER_FRAME = 623.7e6                       # BASELINE.md §2
WORKLOAD = "libritts_batch16x10s_text2wave"
N_INPUT_SETS = 8                                       # distinct (tokens, reference mels, durations) batches cycled by the timed loop


def shared_config():
    """The workload description, IDENTICAL in both arms (the driver compares the two ``config`` objects)."""
    return {"workload": WORKLOAD, "utterances_per_gpu": B_PER_GPU, "tokens": TT, "ref_frames": TR,
            "mel_frames": FRAMES, "audio_s_per_step_per_gpu": B_PER_GPU * AUDIO_S_PER_UTT,
            "inputs": f"{N_INPUT_SETS} seeded input sets cycled: different tokens, reference mels and durations every step",
            "durations": "the duration predictor runs inside every step (models.py:360); seeded integer durations "
                         "summing to 400 per utterance drive the length regulator (north_star: durations are fed "
                         "as integers), so every utterance is 800 frames = 10 s",
            "weights": "random-init conditioned (seed 0); vocoder checkpoint g_00935000 not available"}


def make_durations(g, B, Tt, total):
    """Seeded integer durations, >= 1 per token, summing to exactly ``total`` per utterance."""
    extra = torch.multinomial(torch.ones(B, Tt), total - Tt, replacement=True, generator=g)
    dur = torch.ones(B, Tt, dtype=torch.int64)
    dur.scatter_add_(1, extra, torch.ones_like(extra))
    assert bool((dur.sum(1) == total).all()) and int(dur.min()) >= 1
    return dur


def make_inputs(rank: int, B: int = B_PER_GPU, set_index: int = 0, Tt: int = TT, Tr: int = TR, total: int = SUM_DUR):
    g = torch.Generator().manual_seed(1234 + 1000 * set_index + rank)
    tokens = torch.randint(1, 178, (B, Tt), generator=g)
    mels = (torch.randn(B, 80, Tr, generator=g) * 0.5).clamp(-2, 2)
    dur = make_durations(g, B, Tt, total)
    tok_lens = torch.full((B,), Tt, dtype=torch.int64)
    mel_lens = torch.full((B,), Tr, dtype=torch.int64)
    return tokens, tok_lens, mels, mel_lens, dur


def make_config5(n_utts: int = 512, seed: int = 0):
    """BASELINE config 5 (SURVEY.md §8d): seeded LibriTTS-like phoneme counts (lognormal through p50 = 125,
    p90 = 314, clamped to 15..594), 2 or 3 half-rate frames per token (mean 2.67 -> ~5.3 mel frames per token),
    3 s reference mels.  Same generator as round 1's tools/box_sweep.py (5 609 audio-s in total)."""
    import math
    g = torch.Generator().manual_seed(seed)
    sigma = math.log(314 / 125) / 1.2816
    tl = (125 * torch.exp(sigma * torch.randn(n_utts, generator=g))).round().clamp(15, 594).long()
    toks = [torch.randint(1, 178, (int(t),), generator=g) for t in tl]
    durs = [2 + (torch.rand(int(t), generator=g) < 0.67).long() for t in tl]
    gm = torch.Generator().manual_seed(100 + seed)
    mels = [(torch.randn(80, TR, generator=gm) * 0.5).clamp(-2, 2) for _ in range(n_utts)]
    return toks, mels, durs


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons while the timed region runs: ONE background `nvidia-smi -lms 100` process, as
    in B200_PROFILING.md (a process per sample took driver locks often enough to slow the end-to-end arm on a busy
    box).  Started early so that it is already sampling; `begin()` marks the start of the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.t0, self.proc = index, [], 0.0, None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                          str(self.index), "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL,
                                         text=True)
            for line in self.proc.stdout:
                parts = [p.strip() for p in line.strip().split(",")]
                if len(parts) >= 6:
                    self.samples.append((time.time(), parts))
        except Exception:
            pass

    def begin(self):
        self.t0 = time.time()

    def stop(self):
        t1 = time.time()
        try:
            if self.proc is not None:
                self.proc.terminate()
        except Exception:
            pass
        self.join(timeout=3)
        inside = [s for t, s in self.samples if self.t0 <= t <= t1 + 0.15]
        if not inside:                      # a very short timed region: the samples nearest to it
            inside = [s for t, s in self.samples if t >= self.t0 - 0.3]
        sm = sorted(int(s[0]) for s in inside if s[0].isdigit())
        mx = max([int(s[1]) for s in inside if s[1].isdigit()] or [0])
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for s in inside for n, v in zip(names, s[2:6]) if v.lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": reasons,
                "samples": len(inside)}


def vocoder_traffic():
    """DRAM bytes (read + write) of the vocoder's conv launches per step, from the committed ncu capture
    (profiles/r0N_vocoder_traffic.json, newest round first); None when no capture is available."""
    for name in ("r02_vocoder_traffic.json", "r01_vocoder_traffic.json"):
        path = os.path.join(ROOT, "profiles", name)
        if os.path.isfile(path):
            try:
                return json.load(open(path)).get("dram_bytes_per_step")
            except Exception:
                return None
    return None


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        p = json.load(open(path))
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"],
                "bf16_tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir: str, wav, mel_lengths, mel) -> None:
    """Write one step's (wav, mel_lengths, mel), in the order ``Synthesizer.synthesize`` returns them, as
    ``out_dir/<name>.npy`` (float32 / float64).  Above DUMP_LIMIT_BYTES a seeded sample of utterances (the same
    rows of every array) is written instead."""
    import numpy as np
    arrays = {"wav": wav.detach().float().cpu().numpy(), "mel": mel.detach().float().cpu().numpy(),
              "mel_lengths": mel_lengths.detach().cpu().numpy().astype(np.float64)}
    B = arrays["wav"].shape[0]
    row_bytes = sum(a.nbytes for a in arrays.values()) / B
    if B * row_bytes > DUMP_LIMIT_BYTES:
        keep = max(1, int(DUMP_LIMIT_BYTES // row_bytes) - 1)     # one row's worth left for the index array
        idx = np.sort(np.random.default_rng(0).choice(B, keep, replace=False))
        arrays = {k: a[idx] for k, a in arrays.items()}
        arrays["utterance_index"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))


# ------------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU PyTorch path (oracle/restate.py is its pinned restatement;
# the reference tree itself does not exist on the GPU box)
# ------------------------------------------------------------------------------------------------
_CPU_STATE = {}


def cpu_reference_sample(n_utts: int, threads: int, set_index: int = 0):
    """Time the fp32 CPU path on ``n_utts`` utterances of the bench workload (batch-1 acoustic loop incl. the
    duration predictor, as the reference's step='test' is batch-1 only; vocoder on the same utterance).
    Returns (audio_seconds, seconds)."""
    from artspeech_b200 import checkpoint
    from oracle import restate
    torch.set_num_threads(threads)
    if not _CPU_STATE:
        model = checkpoint.build_random_artsspeech(0)
        gen = checkpoint.build_random_generator(0)
        _CPU_STATE.update(sd={k: v.detach() for k, v in model.state_dict().items()},
                          gsd={k: v.detach() for k, v in gen.state_dict().items()},
                          dist={k: v.cpu() for k, v in model.distribution.items()})
        # warm-up on a short utterance (thread pools, oneDNN primitive caches)
        t, _, m, _, _ = make_inputs(0, 1)
        restate.generator_forward(_CPU_STATE["gsd"], restate.artsspeech_test(
            _CPU_STATE["sd"], t[:1, :20], m[:1, :, :100], _CPU_STATE["dist"], durations=torch.ones(20, dtype=torch.long),
            predict_durations=True))
    sd, gsd, dist = _CPU_STATE["sd"], _CPU_STATE["gsd"], _CPU_STATE["dist"]
    tokens, _, mels, _, dur = make_inputs(0, max(n_utts, 1), set_index)
    t0 = time.perf_counter()
    for i in range(n_utts):
        mel = restate.artsspeech_test(sd, tokens[i:i + 1], mels[i:i + 1], dist, durations=dur[i], predict_durations=True)
        wav = restate.generator_forward(gsd, mel)
        assert wav.shape[-1] == FRAMES * 300
    dt = time.perf_counter() - t0
    return n_utts * AUDIO_S_PER_UTT, dt


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    threads = os.cpu_count() or 1
    n_per_step = 2
    for i in range(min(args.warmup, 1)):
        cpu_reference_sample(1, threads, i)
    times = []
    audio = 0.0
    for i in range(args.steps):
        a, t = cpu_reference_sample(n_per_step, threads, i % N_INPUT_SETS)
        audio += a
        times.append(t)
    total = sum(times)
    value = audio / total
    sample = (f"{n_per_step} of the step's {B_PER_GPU} utterances per step (10 s each; the step is a batch-1 loop, so "
              f"audio-s/s does not depend on how many are run), duration predictor + acoustic + vocoder, fp32 torch "
              f"restatement of the reference pinned to it by tests/test_oracle_pinning.py")
    line = {"impl": "reference", "metric": "synthesized_audio_seconds_per_second", "value": value,
            "unit": "audio-s/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": shared_config(),
            "cpu_baseline": {"value": value, "unit": "audio-s/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)
    return 0


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def _events():
    return torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)


def warmup_calls(warmup: int, depth: int) -> int:
    """Untimed calls of each arm before its timed steps: at least 3, and two per batch in flight."""
    return max(warmup, 3, 2 * depth)


def _median(xs):
    xs = sorted(xs)
    return xs[len(xs) // 2]


def bench_vocoder_roofline(syn, mel_static, lens_static, dev, steps):
    """The dominant kernel family: the vocoder's tensor-core convolutions (fused resblock-pair launches +
    implicit-GEMM launches, nothing else), replayed from a CUDA graph (no launch gaps), CUDA events on the launch
    stream.  Timed twice: a short burst (the kernel family alone: vs the BURST bf16 peak) and a >= 2 s loop (vs the
    SUSTAINED peak, both from MEASURED_PEAKS.json)."""
    from artspeech_b200 import ops
    gen = syn.generator
    m16 = mel_static.transpose(1, 2).to(gen.compute_dtype).contiguous()
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        for _ in range(2):
            gen.forward_channels_last(m16, lens_static)
    torch.cuda.current_stream(dev).wait_stream(side)
    torch.cuda.synchronize(dev)
    vg = torch.cuda.CUDAGraph()
    before = ops.launch_count
    with torch.cuda.graph(vg):
        gen.forward_channels_last(m16, lens_static)
    launches = ops.launch_count - before
    for _ in range(3):
        vg.replay()
    torch.cuda.synchronize(dev)
    e0, e1 = _events()
    # best of 10 single replays after one idle second: how MEASURED_PEAKS.json's burst peak itself was taken (best of
    # 10 sub-millisecond GEMMs on an idle GPU); the SM clock drops within ~0.3 s of sustained load
    time.sleep(1.0)
    singles = []
    for _ in range(10):
        e0.record()
        vg.replay()
        e1.record()
        torch.cuda.synchronize(dev)
        singles.append(e0.elapsed_time(e1))
    bench_vocoder_roofline.best_ms = min(singles)
    reps = max(10, steps)
    e0.record()
    for _ in range(reps):
        vg.replay()
    e1.record()
    torch.cuda.synchronize(dev)
    burst_ms = e0.elapsed_time(e1) / reps
    long_reps = int(2200.0 / burst_ms) + 1
    e0.record()
    for _ in range(long_reps):
        vg.replay()
    e1.record()
    torch.cuda.synchronize(dev)
    long_ms = e0.elapsed_time(e1) / long_reps
    return launches, burst_ms, long_ms, long_reps


def bench_config1(model, gen, dev):
    """BASELINE config 1 on the GPU: ONE utterance (120 phonemes, 3 s reference mel), latency per call with a host
    synchronisation after each: to the mel, to the waveform (forced Σdur = 400 -> 10 s, and with predicted
    durations: two graphs + the frame-count read-back), and time to the first audio chunk of Generator.stream()."""
    from artspeech_b200 import engine
    syn = engine.Synthesizer(model, gen, device=dev, pipeline_depth=1)
    tok, tl, mel, ml, dur = make_inputs(0, 1, 0, Tt=120, total=SUM_DUR)
    tok_p, mel_p = tok.pin_memory(), mel.pin_memory()
    wav_h = torch.empty(1, FRAMES * 300).pin_memory()

    def call(durations):
        t0 = time.perf_counter()
        wav, _, _ = syn.synthesize(tok_p, tl, mel_p, ml, durations, predict_durations=True)
        n = wav.shape[1]
        wav_h[:, :n].copy_(wav, non_blocking=True)
        torch.cuda.current_stream(dev).synchronize()
        return (time.perf_counter() - t0) * 1e3, n

    for _ in range(3):
        call(dur)
        call(None)
    forced = _median([call(dur)[0] for _ in range(15)])
    pred = [call(None) for _ in range(15)]
    # the same with the reference voice's style-encoder outputs cached (engine.encode_voice, SURVEY.md §8f)
    voice = syn.encode_voice(mel.to(dev), ml)

    def call_voice():
        t0 = time.perf_counter()
        wav, _, _ = syn.synthesize(tok_p, tl, mel_p, ml, dur, voice=voice, predict_durations=True)
        wav_h[:, :wav.shape[1]].copy_(wav, non_blocking=True)
        torch.cuda.current_stream(dev).synchronize()
        return (time.perf_counter() - t0) * 1e3
    for _ in range(3):
        call_voice()
    cached = _median([call_voice() for _ in range(15)])
    # acoustic model alone (to the mel): its own graph
    tok_d, mel_d = tok.to(dev), mel.to(dev)
    tl_d, ml_d, dur_d = tl.to(dev), ml.to(dev), dur.to(dev)
    meta = {"mel_lens": [TR], "Lmax": SUM_DUR}
    run = lambda: model([tok_d, tl_d, mel_d, ml_d], step="test", durations=dur_d, host_meta=meta, predict_durations=True)
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        run()
    torch.cuda.current_stream(dev).wait_stream(side)
    torch.cuda.synchronize(dev)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        mel_out = run()
    ts = []
    for _ in range(12):
        t0 = time.perf_counter()
        g.replay()
        torch.cuda.current_stream(dev).synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    to_mel = _median(ts[2:])
    # streaming vocoder: first 64-frame chunk (+ receptive-field halo) of the mel, incl. its device->host copy
    first = []
    chunk_h = torch.empty(1, 1, 64 * 300).pin_memory()
    for _ in range(8):
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        _, w = next(iter(gen.stream(mel_out, chunk_frames=64)))
        chunk_h.copy_(w, non_blocking=True)
        torch.cuda.current_stream(dev).synchronize()
        first.append((time.perf_counter() - t0) * 1e3)
    return {"workload": "1 utterance, 120 phonemes, 3 s reference mel, 800 frames = 10 s (forced) / predicted",
            "ms_to_mel": to_mel, "ms_to_waveform": forced, "audio_s_per_s": AUDIO_S_PER_UTT / (forced / 1e3),
            "ms_to_waveform_voice_cached": cached,
            "ms_to_waveform_predicted_durations": _median([p[0] for p in pred]),
            "predicted_audio_s": pred[0][1] / 24000.0,
            "stream_first_chunk_ms_after_mel": _median(first[2:]),
            "time_to_first_audio_ms": to_mel + _median(first[2:]),
            "note": "host wall-clock per call incl. H2D of the inputs, D2H of the waveform and a stream synchronise"}


def bench_config3(gen, dev, pk):
    """BASELINE config 3: vocoder-only sweep, mel 80 x {200, 800, 3200} frames at batch 1..64, whole Generator,
    TFLOP/s at 623.7 MFLOP per frame, graph replay, vs the burst bf16 peak."""
    out = {}
    fr = []
    for T in (200, 800, 3200):
        for B in (1, 2, 4, 8, 16, 32, 64):
            g0 = torch.Generator().manual_seed(0)
            mel = torch.randn(B, T, 80, generator=g0).clamp(-2, 2).to(dev).to(gen.compute_dtype)
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                gen.forward_channels_last(mel)
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize(dev)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                gen.forward_channels_last(mel)
            g.replay()
            torch.cuda.synchronize(dev)
            e0, e1 = _events()
            reps = 3 if B * T >= 51200 else 10
            e0.record()
            for _ in range(reps):
                g.replay()
            e1.record()
            torch.cuda.synchronize(dev)
            ms = e0.elapsed_time(e1) / reps
            tf = VOCODER_FLOP_PER_FRAME * B * T / (ms / 1e3) / 1e12
            out[f"{B}x{T}"] = round(tf, 1)
            fr.append(tf / pk["bf16_tflops"])
            del g, mel
            torch.cuda.empty_cache()
    fr.sort()
    return {"tflops": out, "frac_of_burst_peak": {"min": fr[0], "median": fr[len(fr) // 2], "max": fr[-1]},
            "note": "whole Generator (51 launches) per point; small points do not fill 148 SMs"}


def bench_config4(syn, dev, steps=3):
    """BASELINE config 4: 8 utterances x 60 s (900 tokens, 4800 frames), text -> waveform."""
    sets = [make_inputs(0, 8, i, Tt=900, total=2400) for i in range(2)]
    dsets = [(t.to(dev), tl, m.to(dev), ml, d) for t, tl, m, ml, d in sets]
    torch.cuda.reset_peak_memory_stats(dev)
    for i in range(4):
        t, tl, m, ml, d = dsets[i % 2]
        syn.synthesize(t, tl, m, ml, d, predict_durations=True)
    syn.join()
    torch.cuda.synchronize(dev)
    e0, e1 = _events()
    e0.record()
    for i in range(steps):
        t, tl, m, ml, d = dsets[i % 2]
        syn.synthesize(t, tl, m, ml, d, predict_durations=True)
    syn.join()
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / steps
    return {"workload": "8 utterances x 60 s (900 tokens, 4800 mel frames each)", "ms_per_step": ms,
            "audio_s_per_s": 8 * 60.0 / (ms / 1e3), "peak_mem_GB": torch.cuda.max_memory_allocated(dev) / 1e9}


def bench_predicted(model, gen, dev, host_sets, tok_lens, mel_lens, depth, steps):
    """The same batches with NO durations given: graph A (encoders + duration predictor, round / clamp on the device)
    -> read-back of 16 frame counts -> graph B (regulator, predictors, decoder, vocoder) for the frame bucket the
    predictions land in.  Random-init weights predict ~1 half-rate frame per token, so the predictor's output bias is
    shifted by +1.67 for this measurement only (mean 2.67 frames per token, the LibriTTS ratio of the workload: ~10 s
    per utterance, but now different for every utterance and step); run last, the weights are restored afterwards."""
    from artspeech_b200 import engine
    lin = model.durationPredictor.duration_proj.linear_layer
    old = lin.bias.detach().clone()
    with torch.no_grad():
        lin.bias += 1.67
    model.invalidate_plans()
    def run(bound):
        syn = engine.Synthesizer(model, gen, device=dev, pipeline_depth=depth, max_graphs=64, duration_bound=bound)
        wav_h = [torch.empty(B_PER_GPU, 2 * FRAMES * 300, dtype=torch.float32).pin_memory() for _ in range(depth + 1)]
        len_h = [torch.zeros(B_PER_GPU, dtype=torch.int32).pin_memory() for _ in range(steps + 3 * N_INPUT_SETS)]
        frames = []

        waiting = []

        def collect(i, k, ticket):
            wav, lens, _ = syn.finish(ticket)
            with torch.cuda.stream(syn.last_stream):
                wav_h[i % len(wav_h)][:, :wav.shape[1]].copy_(wav, non_blocking=True)
                len_h[k].copy_(lens, non_blocking=True)      # frame counts travel with the waveforms

        def step(i, k):
            # one call of look-ahead: the next batch's graph A is enqueued before the host waits for this batch's frame
            # counts (engine.synthesize(defer=True) / finish), as engine.synthesize_many does
            t, m, _ = host_sets[i % N_INPUT_SETS]
            waiting.append((i, k, syn.synthesize(t, tok_lens, m, mel_lens, None, defer=True)))
            while len(waiting) > (1 if depth >= 2 else 0):
                collect(*waiting.pop(0))

        def drain():
            while waiting:
                collect(*waiting.pop(0))
        for i in range(3 * N_INPUT_SETS):                  # every input set in every pipeline slot: all buckets captured
            step(i, steps + i)
        drain()
        syn.join()
        torch.cuda.synchronize(dev)
        captured = syn.stats["captures"]
        e0, e1 = _events()
        t0 = time.perf_counter()
        e0.record()
        for i in range(steps):
            step(i, i)
        drain()
        syn.join()
        e1.record()
        torch.cuda.synchronize(dev)
        wall = time.perf_counter() - t0
        ms = e0.elapsed_time(e1)
        audio = sum(int(v) for k in range(steps) for v in len_h[k].tolist()) * 300 / 24000.0
        return {"value": audio / (ms / 1e3), "unit": "audio-s/s", "ms_per_step": ms / steps, "wall_ms_per_step": wall * 1e3 / steps,
                "mean_audio_s_per_utterance": audio / (steps * B_PER_GPU), "graphs": captured,
                "captures_in_timed_region": syn.stats["captures"] - captured}
    try:
        exact = run(None)
        exact["note"] = ("graph A (encoders + predictor) -> device->host read-back of 16 frame counts -> graph B for the frame "
                         "bucket the predictions land in")
        bounded = run(4.0)
        bounded["note"] = ("Synthesizer(duration_bound=4.0): ONE graph with the frame bucket tokens x 4 half-rate frames, no "
                           "host synchronisation; tiles beyond an utterance's predicted length are skipped by the kernels")
        return {"two_graphs_exact_bucket": exact, "one_graph_bounded_bucket": bounded,
                "note": "end to end (pinned host inputs, D2H of waveforms and frame counts), durations predicted on the device"}
    finally:
        with torch.no_grad():
            lin.bias.copy_(old)
        model.invalidate_plans()


def bench_config5(syn, dev, rank, world, dist, passes=2):
    """BASELINE config 5: 512 seeded mixed-length utterances, LPT-sharded over the run's N GPUs (strong scaling),
    each rank through engine.synthesize_many (length-bucketed micro-batches on bucketed CUDA graphs, waveforms
    copied to pinned host memory).  Warm-up passes run until no new graph is captured; timing = max over ranks."""
    from artspeech_b200 import engine
    toks, mels, durs = make_config5()
    frames = [2 * int(d.sum()) for d in durs]
    # length-contiguous shards of equal cost: every rank's micro-batches stay as homogeneous as on one GPU (LPT on
    # frame counts deals each rank the whole length distribution: 37 % padding at 8 ranks instead of 9 %)
    mine = engine.shard_by_length(frames, world)[rank]
    my_t, my_m, my_d = [toks[i] for i in mine], [mels[i] for i in mine], [durs[i] for i in mine]
    arena = engine.HostArena()
    for _ in range(4):
        before = syn.stats["captures"]
        engine.synthesize_many(syn, my_t, my_m, my_d, to_host=True, arena=arena)
        if syn.stats["captures"] == before:
            break
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    e0, e1 = _events()
    e0.record()
    for _ in range(passes):
        wavs, fr = engine.synthesize_many(syn, my_t, my_m, my_d, to_host=True, arena=arena)
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / passes
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    audio = sum(frames) * 300 / 24000.0
    nb = len(engine.bucket_utterances([frames[i] for i in mine], 16, 25600, quantum=2 * syn.frame_quantum))
    return {"workload": "512 seeded mixed-length utterances (15-594 tokens), 3 s reference mels, sharded over the N GPUs "
                        "(length-contiguous shards of equal cost, engine.shard_by_length)",
            "scaling": "strong", "n_gpus": world, "audio_s": audio, "ms_per_pass": ms,
            "audio_s_per_s": audio / (ms / 1e3), "micro_batches_rank0": nb, "graphs_rank0": syn.stats["captures"],
            "graph_replays_rank0": syn.stats["replays"], "eager_calls_rank0": syn.stats["eager"],
            "d2h": "every rank copies its own waveforms to pinned host memory inside the timed region"}


def run_ours(args):
    import torch.distributed as dist
    from artspeech_b200 import checkpoint, engine, ops

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the CUDA path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    model = checkpoint.build_random_artsspeech(0)
    gen = checkpoint.build_random_generator(0)
    depth = 1 if args.no_graph else args.pipeline
    syn = engine.Synthesizer(model, gen, device=dev, use_cuda_graph=not args.no_graph, pipeline_depth=depth)

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()                 # nvidia-smi needs a moment to come up: running well before the timed region
    sets = [make_inputs(rank, B_PER_GPU, i) for i in range(N_INPUT_SETS)]
    tok_lens, mel_lens = sets[0][1], sets[0][3]
    dev_sets = [(t.to(dev), m.to(dev), d) for t, _, m, _, d in sets]
    # pinned host staging for the end-to-end arm
    host_sets = [(t.pin_memory(), m.pin_memory(), d) for t, _, m, _, d in sets]
    wav_hs = [torch.empty(B_PER_GPU, FRAMES * 300, dtype=torch.float32).pin_memory() for _ in range(max(depth, 1) + 1)]
    calls = [0, 0]
    last_resident = [None]
    wav_lens_d = torch.full((B_PER_GPU,), FRAMES * 300, device=dev)
    gat = engine.WaveformGatherer(dev, [(B_PER_GPU, FRAMES * 300)] * world, torch.float32, dst=0) if world > 1 else None

    def step_resident():
        t, m, d = dev_sets[calls[0] % N_INPUT_SETS]
        calls[0] += 1
        last_resident[0] = syn.synthesize(t, tok_lens, m, mel_lens, d, predict_durations=True)
        return last_resident[0]

    def step_e2e():
        t, m, d = host_sets[calls[1] % N_INPUT_SETS]
        calls[1] += 1
        # pinned host tokens / mels go straight into the graph's static buffers (H2D inside the call)
        wav, _, _ = syn.synthesize(t, tok_lens, m, mel_lens, d, predict_durations=True)
        # the waveforms are produced on the engine's stream for this call: D2H (and the gather) follow on that stream
        with torch.cuda.stream(syn.last_stream):
            wav_hs[calls[1] % len(wav_hs)].copy_(wav, non_blocking=True)
        if gat is not None:
            gat.submit(wav, wav_lens_d, syn.last_stream)       # one collective, on its own stream, overlapped
        return wav

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, steps):
        barrier()
        e0, e1 = _events()
        e0.record()
        for _ in range(steps):
            fn()
        syn.join()                 # pipelined calls run on the engine's streams: the end event waits for all of them
        if gat is not None:
            gat.results()          # ... and for the last gather
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    warm = max(args.warmup, 3)
    for _ in range(warmup_calls(args.warmup, depth)):
        step_resident()
        step_e2e()
    barrier()
    captures_after_warmup = syn.stats["captures"]

    # inputs (tokens 19 KB + mels 1.2 MB) are tiny, but every step streams > 10 GB of activations
    # through HBM, far beyond the 126 MB L2: no explicit flush needed between timed iterations.
    if sampler:
        sampler.begin()
    l0 = ops.launch_count
    ms = timed(step_resident, args.steps)
    launches = ops.launch_count - l0
    dumped = None
    if args.dump_outputs and rank == 0:
        # the graphs' output buffers are reused by the next call with the same shapes: a device copy now, written to
        # disk after the clock sampling window
        dumped = [t.clone() for t in last_resident[0]]
    ms_e2e = timed(step_e2e, args.steps)
    clocks = sampler.stop() if sampler else None
    if dumped is not None:
        dump_outputs(args.dump_outputs, *dumped)
        del dumped
    assert syn.stats["captures"] == captures_after_warmup, "the timed region must replay graphs, not capture them"

    # BASELINE config 5 on every rank (strong scaling over the run's N GPUs)
    c5 = None
    if not args.no_graph and not args.skip_configs:
        syn5 = engine.Synthesizer(model, gen, device=dev, pipeline_depth=depth, max_graphs=96)
        c5 = bench_config5(syn5, dev, rank, world, dist)
        del syn5
        torch.cuda.empty_cache()

    extras = {}
    if rank == 0:
        # host link probe: the e2e arm moves 15.4 MB of waveforms per step over PCIe; on a box whose link is slow or
        # shared this copy, not the GPU, bounds e2e
        hb = torch.empty(64 << 20, dtype=torch.uint8).pin_memory()
        db = torch.empty(64 << 20, dtype=torch.uint8, device=dev)
        e0, e1 = _events()
        link = {}
        for name, (dst, src) in (("h2d_GBps", (db, hb)), ("d2h_GBps", (hb, db))):
            dst.copy_(src, non_blocking=True)
            torch.cuda.synchronize(dev)
            e0.record()
            for _ in range(4):
                dst.copy_(src, non_blocking=True)
            e1.record()
            torch.cuda.synchronize(dev)
            link[name] = 4 * hb.numel() / (e0.elapsed_time(e1) / 1e3) / 1e9
        extras["host_link"] = link
        del hb, db
    if rank == 0 and world == 1:
        pk = peaks()
        e0, e1 = _events()
        # the same step with the style-encoder outputs cached per reference voice (SURVEY.md §8f)
        tok_d, mel_d, dur = dev_sets[0]
        voice = syn.encode_voice(mel_d, mel_lens)
        step_voice = lambda: syn.synthesize(tok_d, tok_lens, mel_d, mel_lens, dur, voice=voice, predict_durations=True)
        for _ in range(2 * depth + 1):
            step_voice()
        ms_cached = timed(step_voice, args.steps)
        extras["voice_cached"] = {"value": B_PER_GPU * AUDIO_S_PER_UTT * args.steps / (ms_cached / 1e3), "unit": "audio-s/s",
                                  "ms_per_step": ms_cached / args.steps,
                                  "note": "style-encoder outputs cached per reference voice (not the BASELINE config: informational)"}

        _, lens_m, mel_out = step_resident()
        syn.join()
        torch.cuda.synchronize(dev)
        voc_launches, voc_ms, voc_long_ms, long_reps = bench_vocoder_roofline(syn, mel_out.clone(), lens_m.clone(), dev, args.steps)
        voc_flops = VOCODER_FLOP_PER_FRAME * B_PER_GPU * FRAMES
        achieved = voc_flops / (voc_ms / 1e3) / 1e12
        sustained = voc_flops / (voc_long_ms / 1e3) / 1e12
        extras["roofline"] = {
            "bound": "tensor", "kernel": f"resblock_pair + conv_igemm kernels (vocoder, {voc_launches} launches per step)",
            "achieved": achieved, "peak": pk["bf16_tflops"], "unit": "TFLOP/s", "frac": achieved / pk["bf16_tflops"],
            "traffic": vocoder_traffic(),
            "peak_source": pk["source"] + " BURST bf16 (the kernel family timed alone, graph replay, %.0f ms)" % (voc_ms * max(10, args.steps)),
            "flops_per_step": voc_flops, "vocoder_ms": voc_ms, "vocoder_share_of_step": voc_ms / (ms / args.steps),
            "best_of_10_after_idle": {"vocoder_ms": bench_vocoder_roofline.best_ms,
                                      "achieved": voc_flops / bench_vocoder_roofline.best_ms / 1e9,
                                      "frac": voc_flops / bench_vocoder_roofline.best_ms / 1e9 / pk["bf16_tflops"],
                                      "note": "single graph replays after 1 s idle, best of 10: the protocol of the burst peak "
                                              "itself; 'achieved' above is the mean over back-to-back replays on the loaded GPU"},
            "sustained": {"achieved": sustained, "peak": pk["bf16_tflops_sustained"],
                          "frac": sustained / pk["bf16_tflops_sustained"], "vocoder_ms": voc_long_ms,
                          "loop_s": voc_long_ms * long_reps / 1e3,
                          "note": "same graph replayed back to back for >= 2 s vs the sustained bf16 peak"}}

        # MAS (SURVEY.md §8 a13, BASELINE config 5): 64 x 200 tokens x 1000 frames, fp32, bit-exact path
        from artspeech_b200 import mas
        gm = torch.Generator().manual_seed(7)
        val = torch.randn(64, 200, 1000, generator=gm).to(dev)
        xl = torch.randint(100, 201, (64,), generator=gm)
        yl = torch.maximum(torch.randint(500, 1001, (64,), generator=gm), xl)
        xl[0], yl[0] = 200, 1000
        xl_d, yl_d = xl.to(dev, torch.int32), yl.to(dev, torch.int32)
        for _ in range(3):
            mas.maximum_path_lens(val, xl_d, yl_d)
        torch.cuda.synchronize(dev)
        e0.record()
        for _ in range(20):
            mas.maximum_path_lens(val, xl_d, yl_d)
        e1.record()
        torch.cuda.synchronize(dev)
        mas_ms = e0.elapsed_time(e1) / 20
        mas_bytes = 2.0 * 64 * 200 * 1000 * 4
        extras["mas"] = {"shape": "64x200x1000 fp32", "ms": mas_ms, "algorithmic_GBps": mas_bytes / mas_ms / 1e6,
                         "frac_of_hbm_peak": mas_bytes / mas_ms / 1e6 / pk["hbm_gbs"],
                         "note": "serial dependency chain over Ty: latency-bound by construction, not roofline-graded"}
        del val

        # HBM-bound kernel family: fused InstanceNorm + AdaIN + LeakyReLU (as_adain_norm_apply) at the decoder's
        # widest block, fp32 in -> f16 out.  Six rotating input sets (> 126 MB L2), launches replayed back to back
        # from a CUDA graph, algorithmic bytes = one read + one write of the tensor.
        nset, Cd = 6, 1024
        xs = [torch.randn(B_PER_GPU, FRAMES, Cd, device=dev) * 0.7 + 3.0 for _ in range(nset)]
        gbv = torch.randn(B_PER_GPU, 2 * Cd, device=dev) * 0.3
        lens_f = torch.full((B_PER_GPU,), FRAMES, dtype=torch.int32, device=dev)
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for xv in xs:
                ops.adain_norm(xv, gbv, 0.2, lens_f, torch.float16)
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        ag = torch.cuda.CUDAGraph()
        with torch.cuda.graph(ag):
            keep = [ops.adain_norm(xv, gbv, 0.2, lens_f, torch.float16) for xv in xs]
        ag.replay()
        torch.cuda.synchronize(dev)
        e0.record()
        for _ in range(5):
            ag.replay()
        e1.record()
        torch.cuda.synchronize(dev)
        ad_us = e0.elapsed_time(e1) / (5 * nset) * 1e3
        ad_bytes = B_PER_GPU * FRAMES * Cd * (4 + 2)
        extras["roofline_hbm"] = {
            "bound": "hbm", "kernel": "adain_ring_kernel (InstanceNorm + AdaIN + LeakyReLU, 16x800x1024 fp32 -> f16)",
            "achieved": ad_bytes / ad_us / 1e3, "peak": pk["hbm_gbs"], "unit": "GB/s",
            "frac": ad_bytes / ad_us / 1e3 / pk["hbm_gbs"], "us_per_launch": ad_us,
            "bytes_per_launch": ad_bytes, "l2": "6 rotating input sets (474 MB), graph replay"}
        del xs, keep, ag

        # the step before the path (SURVEY.md §8f): log-mel front-end of the 16 reference recordings (3 s each)
        from artspeech_b200 import frontend
        fe = frontend.LogMel().to(dev)
        wv = torch.randn(B_PER_GPU, TR * 300, device=dev) * 0.1
        for _ in range(3):
            fe(wv)
        torch.cuda.synchronize(dev)
        e0.record()
        for _ in range(20):
            fe(wv)
        e1.record()
        torch.cuda.synchronize(dev)
        extras["frontend"] = {"kernel": "log_mel_kernel (STFT 2048/1200/300 + 80 mel + log, fp32)", "recordings": B_PER_GPU,
                              "seconds_each": TR * 300 / 24000.0, "us": e0.elapsed_time(e1) / 20 * 1e3,
                              "note": "not part of the timed step (reference mels are the step's inputs, as in BASELINE configs)"}
        torch.cuda.empty_cache()
        if not args.skip_configs:
            extras["config1"] = bench_config1(model, gen, dev)
            extras["config3"] = bench_config3(syn.generator, dev, pk)
            torch.cuda.empty_cache()
            extras["config4"] = bench_config4(syn, dev)
            extras["predicted_durations"] = bench_predicted(model, gen, dev, host_sets, tok_lens, mel_lens, depth, args.steps)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    audio_per_step = world * B_PER_GPU * AUDIO_S_PER_UTT
    value = audio_per_step * args.steps / (ms / 1e3)
    e2e_value = audio_per_step * args.steps / (ms_e2e / 1e3)
    t0, m0, _ = host_sets[0]
    meta_bytes = 4 * (B_PER_GPU * ((TT + syn.token_quantum - 1) // syn.token_quantum * syn.token_quantum) + B_PER_GPU)
    line = {
        "metric": "synthesized_audio_seconds_per_second", "value": value, "unit": "audio-s/s", "n_gpus": world,
        "steps": args.steps, "warmup": warm, "ms_per_step": ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16 (vocoder) / f16 (acoustic) operands, f32 accumulate", "data": "synthetic",
        "config": shared_config(),
        "engine": {"cuda_graph": not args.no_graph, "batches_in_flight": depth,
                   "graph_key": "shape bucket (B, tokens/32, ref frames, frames/80); tokens, mels, lengths and durations "
                                "are graph inputs refreshed per call",
                   "graphs_captured": captures_after_warmup, "stats": dict(syn.stats),
                   "l2": "activations streamed per step >> 126 MB L2, no explicit flush",
                   "multi_gpu": None if world == 1 else "every rank D2H-copies its own waveforms; one asynchronous "
                                "NCCL gather per step to rank 0 on a communication stream (e2e arm only)"},
        "e2e": {"value": e2e_value, "unit": "audio-s/s", "ms_per_step": ms_e2e / args.steps,
                "h2d_bytes_per_step": int(t0.numel() * 8 + m0.numel() * 4 + meta_bytes),
                "d2h_bytes_per_step": int(wav_hs[0].numel() * 4)},
        "gpu_launches": int(launches),
        "clocks": clocks,
    }
    line.update(extras)
    if c5 is not None:
        line["config5"] = c5
    if world == 1 and not args.no_cpu_baseline:
        a, t = cpu_reference_sample(args.cpu_utts, os.cpu_count() or 1)
        line["cpu_baseline"] = {"value": a / t, "unit": "audio-s/s", "cores": os.cpu_count() or 1, "kind": "port",
                                "sample": f"{args.cpu_utts} utterances of the same workload (10 s each), batch-1 duration "
                                          f"predictor + acoustic + vocoder, fp32 torch restatement of the reference"}
    emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


_JSON_FD = None


def emit(line: dict) -> None:
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-graph", action="store_true", help="launch kernels eagerly instead of replaying a CUDA graph")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--pipeline", type=int, default=2,
                    help="batches in flight per GPU (2: the acoustic model of step i+1 overlaps the vocoder of step i)")
    ap.add_argument("--cpu-utts", type=int, default=16, help="utterances of the CPU baseline sample (~0.6 s each on 16 cores)")
    ap.add_argument("--skip-configs", action="store_true", help="headline + rooflines only (no config1/3/4/5 extras)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the CUDA arm's outputs (--impl ours)")
    # stdout carries exactly ONE line (the JSON): libraries that write to fd 1 (NCCL prints its version banner there
    # when NCCL_DEBUG is set) are sent to stderr for the whole run, the JSON line goes to the saved descriptor
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
