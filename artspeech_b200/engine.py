"""Batched text -> waveform synthesis (the glue of the reference's ``test.py:90-119``).

``Synthesizer`` owns an ``ArtsSpeech`` (second stage) and a vocoder ``Generator`` on one GPU and
runs ``tokens + reference mel -> mel -> waveform`` for a batch of utterances, each with batch-1
semantics.  The pass is replayed from CUDA graphs keyed on shape buckets, with tokens, reference mels, lengths and
durations as graph inputs (launch-bound otherwise: ~600 kernels per step); see ``Synthesizer``.

Multi-GPU: utterances are independent (SURVEY.md §8e); ``shard_utterances`` assigns them to ranks
longest-first (LPT) and ``gather_waveforms`` collects the results on rank 0 over NCCL — the only
collective on the path.
"""
from __future__ import annotations

import os
from collections import OrderedDict
from typing import List, Optional, Sequence

import torch

from . import _lib, nn_util, ops
from . import audio as audio_mod
from . import prosody as prosody_mod

SAMPLE_RATE = 24000
HOP = 300


def _ceil_to(v: int, q: int) -> int:
    return (int(v) + q - 1) // q * q


def _wm_kw(wm) -> dict:
    """The ``watermark`` keyword of a call that has one: calls without keep their exact signature."""
    return {} if wm is None else {"wm": wm}


class _Captured:
    """One captured CUDA graph with its static inputs / outputs (all owned by the graph's memory pool)."""
    __slots__ = ("graph", "tok", "mels", "voice", "meta", "dur", "lens_t", "mel_lens", "pin_meta", "pin_free", "out",
                 "launches", "state", "uid", "pros", "pin_pros", "ctrl", "dscale")

    def __init__(self):
        self.graph = self.tok = self.mels = self.voice = self.meta = self.dur = self.lens_t = self.mel_lens = None
        self.pin_meta = self.pin_free = self.out = self.state = None
        self.pros = self.pin_pros = self.ctrl = self.dscale = None
        self.launches = 0
        self.uid = 0


class _Ticket:
    """A call issued with ``synthesize(..., defer=True)``: with predicted durations everything up to the frame-count
    read-back is enqueued; ``Synthesizer.finish`` synchronises on it and enqueues the rest."""
    __slots__ = ("result", "last", "last_stream", "slot", "run_stream", "is_side", "ent", "got", "B", "launches", "fmt",
                 "loud", "wm")

    def __init__(self):
        self.result = self.last = self.last_stream = self.ent = self.got = self.run_stream = self.fmt = None
        self.loud = self.wm = None
        self.slot = self.B = self.launches = 0
        self.is_side = False


class Synthesizer:
    """Text -> waveform for batches of utterances on one GPU.

    **Graph replay for real traffic.**  A pass is ~600 small launches, so it is replayed from CUDA graphs.  A graph is
    keyed on a *shape bucket* only -- ``(B, tokens rounded up to token_quantum, reference frames, half-rate frames
    rounded up to frame_quantum)`` -- never on the data: tokens, reference mels, token lengths and **durations are graph
    inputs**, copied into static device buffers before each replay (one pinned staging copy carries durations and
    lengths).  Every kernel on the path takes per-utterance lengths, so a bucket serves any mix of lengths below its
    bounds with batch-1 semantics per utterance.  The cache is an LRU of at most ``max_graphs`` graphs per pipeline
    slot sharing one memory pool per slot (the default ``frame_quantum`` of 40 half-rate frames = 80 mel frames makes
    the buckets whole seconds of audio); a bucket is captured the ``capture_after``-th time it is seen and runs
    eagerly before that.

    **Durations.**  ``durations=None``: the duration predictor runs on the device (graph A: encoders + predictor +
    ``round().clamp(min=1)``), the host reads back B integers (the utterances' frame counts, the only device->host
    synchronisation of the pass; the reference does 2*Tt+1, models.py:362-366), picks the frame bucket and replays
    graph B (length regulator -> predictors -> decoder -> vocoder).  ``durations=`` given (north_star: "durations
    are fed from the reference's integer output"): one graph, no synchronisation; with ``predict_durations=True``
    the predictor still runs inside that graph (its output is returned in ``last["duration"]`` /
    ``last["pred_dur"]``) while the given durations drive the length regulator.

    ``duration_bound`` (half-rate frames per token, e.g. 4.0 = 0.1 s per phoneme) removes that hand-off as well: with
    predicted durations the WHOLE pass is then one graph whose frame bucket is ``tokens * duration_bound`` -- every
    tensor-core kernel on the path leaves out the tiles beyond an utterance's predicted length, so the generous
    bucket costs zero-fill writes, not compute -- and the frame counts come back with the waveforms
    (``last["frames"]`` is None, ``last["pred_sum"]`` / the returned ``mel_lengths`` are device tensors; an
    utterance whose prediction exceeds the bound is truncated there, ``synthesize_many`` re-runs those exactly).

    ``pipeline_depth`` > 1 keeps that many calls in flight: call ``i`` runs on side stream ``i % depth`` with its own
    graph instances and buffers, so the latency-bound acoustic model of one batch overlaps the throughput-bound
    vocoder of the previous one.  The outputs of a call are produced on ``last_stream``: consume them there (``with
    torch.cuda.stream(syn.last_stream)``) or after ``join()``.  **Aliasing:** on the graph path the returned tensors
    are views of the graph's static output buffers -- they stay valid until the next call that lands in the same
    slot *and* bucket; enqueue the copy that consumes them (on ``last_stream``) before making that call.
    ``pcm16=True`` returns int16 samples (``rint(32767 * wav)``, the on-disk format of ``soundfile.write`` at
    test.py:119) written directly by the vocoder's last kernel: half the device->host bytes per utterance.

    **Prosody.**  ``synthesize(..., prosody=[Prosody, ...])`` (one per utterance, ``artspeech_b200.prosody``) scales
    the predicted durations and edits the predicted F0 / energy / EMA tracks.  The controls are graph inputs like the
    durations (a control block and a per-token duration scale staged through one pinned buffer), so one graph serves
    controls that change on every call.  Controlled calls have graphs of their own (one extra launch); calls
    without ``prosody`` replay the same graphs as before.

    **Output formats.**  ``synthesize(..., audio=AudioFormat(rate, encoding))`` (``artspeech_b200.audio``) returns the
    waveforms resampled and encoded (e.g. 8 kHz G.711 mu-law for telephony, 16 kHz PCM for recognisers): one
    ``as_resample_encode`` launch on the call's stream after the graph replay, into a fresh stream-ordered allocation.
    It is not captured, so the format may change on every call without new graphs.  A format equal to the engine's
    native output (24 kHz fp32, or 24 kHz PCM with ``pcm16=True``) takes the unformatted path; any other format needs
    ``pcm16=False`` (the resampler reads fp32).

    **Loudness normalisation.**  ``synthesize(..., loudness=Loudness(target_lufs, max_true_peak_db))`` meters each
    utterance's 24 kHz waveform on the GPU (BS.1770 integrated loudness and 4x true peak, ``as_loudness_measure``,
    three launches) and applies one gain per utterance inside the format stage, before the encoding (with the native
    format too).  Like the format stage it is not captured; it needs ``pcm16=False``.

    **Watermark.**  ``synthesize(..., watermark=Watermark(key, message))`` adds a keyed, inaudible-by-design mark that
    ``audio.detect_watermark`` finds in any output format (``as_watermark_embed``, one launch on the call's stream
    after the graph, before the meter and the format stage, so those see the delivered samples).  It is not captured;
    with no ``audio`` and no ``loudness`` the marked 24 kHz fp32 waveform is the result.  It needs ``pcm16=False``."""

    def __init__(self, model, generator, device="cuda:0", use_cuda_graph: bool = True, pipeline_depth: int = 1,
                 pcm16: bool = False, acoustic_sms: Optional[int] = None, token_quantum: int = 32,
                 frame_quantum: int = 40, max_graphs: int = 48, capture_after: int = 1,
                 duration_bound: Optional[float] = None):
        self.device = torch.device(device)
        self.pcm16 = bool(pcm16)
        # SM split between the two phases when batches overlap: the acoustic model's persistent kernels are sized
        # for ``acoustic_sms`` SMs and the vocoder's for the rest, so that the latency-bound acoustic chain of batch
        # i+1 always finds free SMs beside the vocoder of batch i (0 / None: every kernel sizes for the whole GPU)
        env = os.environ.get("ASB_ACOUSTIC_SMS")
        self.acoustic_sms = int(env) if env is not None else (acoustic_sms or 0)
        self.pipeline_depth = max(1, int(pipeline_depth))
        self.token_quantum, self.frame_quantum = max(1, int(token_quantum)), max(1, int(frame_quantum))
        self.max_graphs, self.capture_after = max(1, int(max_graphs)), max(1, int(capture_after))
        self.duration_bound = None if duration_bound is None else float(duration_bound)
        self._slot_streams = None
        self._slot_done = {}
        self._calls = 0
        self.last_stream = None
        self.last = {}
        self.model = model.to(self.device).eval()
        self.model.distribution = {k: v.to(self.device) for k, v in self.model.distribution.items()}
        self.model.prosody_constants()          # host floats of the pitch / energy statistics: read once, here
        self.generator = generator.to(self.device).eval()
        self.use_cuda_graph = use_cuda_graph
        self._graphs = [OrderedDict() for _ in range(self.pipeline_depth)]     # per slot: key -> _Captured (LRU)
        self._pools = [None] * self.pipeline_depth
        self._seen = {}
        self._uid = 0
        self._epoch = nn_util.plan_epoch()
        self.launches_per_call = None
        self.stats = {"captures": 0, "replays": 0, "eager": 0, "evictions": 0, "drops": 0}

    @classmethod
    def from_cache(cls, path: str, device="cuda:0", expect_hash: Optional[str] = None, **kw) -> "Synthesizer":
        """Start from a converted checkpoint (``python -m artspeech_b200.convert``, SURVEY.md §8f-4): the folded,
        packed weights are read from ``path`` instead of being re-derived from the parameters in this process."""
        from . import convert
        model, gen = convert.load_cache(path, device, expect_hash)
        return cls(model, gen, device=device, **kw)

    # ---------------------------------------------------------------------------------------
    @torch.no_grad()
    def encode_voice(self, mels, mel_lens):
        """Style-encoder pass for a batch of reference recordings: ``mels`` fp32 [B,80,Tr] (device), ``mel_lens``
        int64 [B] (host) -> ``(f0, n, ema, Style)``, reusable as ``synthesize(..., voice=...)`` for every
        utterance spoken with these voices (item i of the batch uses voice i)."""
        ml = [int(v) for v in mel_lens.tolist()]
        return tuple(self.model.style_encoder(mels, mel_lens.to(self.device), "second", self.model.distribution,
                                              host_lengths=ml))

    @torch.no_grad()
    def enroll(self, x, lengths, sample_rate: int, encoding: str = "float32", top_db: Optional[float] = 30.0,
               noise_reduction_db: Optional[float] = None):
        """Voices from recordings: ``frontend.reference_mels`` (decode, downmix, resample to 24 kHz, optionally reduce
        stationary noise by up to ``noise_reduction_db``, trim silence, log-mel; semantics in
        ``artspeech_b200.frontend``) then ``encode_voice``, eagerly.  ``x`` ``[B, S]`` or ``[B, S, C]`` samples of
        ``encoding`` at ``sample_rate`` Hz, ``lengths`` host samples per channel.  Returns ``(mels, mel_lens, voice)``,
        which ``synthesize(tokens, tok_lens, mels, mel_lens, voice=voice)`` takes as they are."""
        from . import frontend
        mels, mel_lens, _ = frontend.reference_mels(x, lengths, sample_rate, encoding, top_db, device=self.device,
                                                    noise_reduction_db=noise_reduction_db)
        return mels, mel_lens, self.encode_voice(mels, mel_lens)

    # -- the two phases (models.ArtsSpeech.encode / decode + the vocoder) ---------------------------------------
    @staticmethod
    def _nvtx(name):
        """NVTX range per phase (visible in nsys / ncu --nvtx timelines) when ASB_NVTX=1; also recorded at capture
        time, so a captured graph's kernels carry the phase they belong to."""
        import contextlib
        if os.environ.get("ASB_NVTX") == "1":
            return torch.cuda.nvtx.range(name)
        return contextlib.nullcontext()

    def _sm_limit(self, n):
        if self.acoustic_sms and self.pipeline_depth > 1:
            _lib.load().as_set_sm_limit(n)

    def _phase_a(self, tok, lens_t, mels, mel_lens_dev, host_mel_lens, voice, predict, dscale=None):
        self._sm_limit(self.acoustic_sms)
        try:
            with self._nvtx("asb.encode (text / arts / style encoders, duration predictor)"):
                return self.model.encode(tok, lens_t, mels, mel_lens_dev, host_mel_lens, voice, predict, dscale)
        finally:
            self._sm_limit(0)

    def _phase_b(self, st, dur, Lmax, ctrl=None):
        total = torch.cuda.get_device_properties(self.device).multi_processor_count
        gen = self.generator
        try:
            self._sm_limit(self.acoustic_sms)
            with self._nvtx("asb.decode (length regulator, F0/N/EMA predictors, mel decoder)"):
                mel_cl, aux = self.model.decode(st, dur, Lmax, mel16_dtype=gen.compute_dtype, ctrl=ctrl)
            self._sm_limit(max(2, total - self.acoustic_sms))
            with self._nvtx("asb.vocoder (HiFi-GAN generator)"):
                wav, wav_lengths = gen.forward_channels_last(aux["mel16"], aux["mel_lengths"],
                                                             torch.int16 if self.pcm16 else torch.float32,
                                                             return_lengths=True)
        finally:
            self._sm_limit(0)
        mel = ops.to_channels_first(mel_cl, torch.float32)
        return dict(wav=wav.view(wav.shape[0], -1), mel_lengths=aux["mel_lengths"], mel=mel,
                    duration=st["duration"], pred_dur=st["pred_dur"], wav_lengths=wav_lengths)

    def _eager(self, tokens, tl, mels, ml, durations, voice, predict, pros=None):
        """No graph: ragged reference mels, ``use_cuda_graph=False`` or a bucket not captured yet."""
        dev = self.device
        self.stats["eager"] += 1
        tokens = tokens.to(dev, non_blocking=True)
        mels = mels.to(dev, non_blocking=True)
        lens_t = torch.tensor(tl, dtype=torch.int32).to(dev, non_blocking=True)
        mel_lens_dev = torch.tensor(ml, dtype=torch.int64).to(dev, non_blocking=True)
        ctrl = dscale = None
        if pros is not None:
            ctrl, dscale = (t.to(dev) for t in prosody_mod.pack(pros, tokens.shape[1]))
            if durations is not None:
                dscale = None
        st = self._phase_a(tokens, lens_t, mels, mel_lens_dev, ml, voice, predict or durations is None, dscale)
        if durations is None:
            dur = st["pred_dur"]
            sums = [int(v) for v in st["pred_sum"].tolist()]                       # the one host sync
        else:
            dur = durations.to(torch.int32).to(dev, non_blocking=True).contiguous()
            sums = [int(durations[b, :tl[b]].sum()) for b in range(len(tl))]
        out = self._phase_b(st, dur, max(sums), ctrl)
        self.last = dict(out, frames=[2 * v for v in sums], graph=False)
        return out["wav"], out["mel_lengths"], out["mel"]

    # -- graph cache --------------------------------------------------------------------------------------------
    def drop_graphs(self):
        """Forget every captured graph (they bake in the addresses of the packed weights: called when a
        ``load_state_dict`` / device move re-packed them)."""
        torch.cuda.synchronize(self.device)
        for cache in self._graphs:
            cache.clear()
        # a memory pool whose graphs are all gone cannot be captured into again: new pools for the new graphs
        self._pools = [None] * self.pipeline_depth
        self._epoch = nn_util.plan_epoch()
        self.stats["drops"] += 1

    def _lookup(self, slot, key):
        cache = self._graphs[slot]
        ent = cache.get(key)
        if ent is not None:
            cache.move_to_end(key)
        return ent

    def _insert(self, slot, key, ent):
        cache = self._graphs[slot]
        cache[key] = ent
        while len(cache) > self.max_graphs:
            # least recently used graph of this slot; its replays were issued on the slot's stream, wait for them
            (self._slot_streams[slot] if self._slot_streams else torch.cuda.current_stream(self.device)).synchronize()
            old_key, old = cache.popitem(last=False)
            self.stats["evictions"] += 1
            for k in [k for k, v in cache.items() if v.state is old]:          # B graphs reading an evicted A graph
                del cache[k]
            del old

    def _capture(self, slot, fn):
        """Warm up ``fn`` once on a side stream (weight packing, shared-memory opt-ins, allocator), then capture it
        into the slot's memory pool.  Returns (graph, outputs, launches)."""
        dev = self.device
        cur = torch.cuda.current_stream(dev)
        s = torch.cuda.Stream(device=dev)
        s.wait_stream(cur)
        with torch.cuda.stream(s):
            fn()
        cur.wait_stream(s)
        torch.cuda.synchronize(dev)
        if self._pools[slot] is None:
            self._pools[slot] = torch.cuda.graph_pool_handle()
        g = torch.cuda.CUDAGraph()
        before = ops.launch_count
        with torch.cuda.graph(g, pool=self._pools[slot]):
            out = fn()
        self.stats["captures"] += 1
        self._epoch = nn_util.plan_epoch()          # the warm-up pass may have packed weights for the first time
        return g, out, ops.launch_count - before

    def _static_inputs(self, B, Tt_b, mels, voice, controlled):
        dev = self.device
        ent = _Captured()
        self._uid += 1
        ent.uid = self._uid
        ent.tok = torch.zeros(B, Tt_b, dtype=torch.int64, device=dev)
        ent.mels = torch.zeros(tuple(mels.shape), dtype=torch.float32, device=dev)
        ent.voice = None if voice is None else tuple(torch.zeros_like(v, device=dev) for v in voice)
        ent.meta = torch.zeros(B * Tt_b + B, dtype=torch.int32, device=dev)
        ent.meta[B * Tt_b:] = 1                                                # valid lengths for the warm-up pass
        ent.dur = ent.meta[:B * Tt_b].view(B, Tt_b)
        ent.dur[:, 0] = 1
        ent.lens_t = ent.meta[B * Tt_b:]
        ent.pin_meta = torch.zeros(B * Tt_b + B, dtype=torch.int32).pin_memory()
        ent.pin_free = torch.cuda.Event()
        if controlled:
            # prosody controls: [B, 24] control block + [B, Tt_b] duration scale, identity for the warm-up pass
            W = prosody_mod.CTRL_WIDTH
            ent.pros = torch.ones(B * W + B * Tt_b, dtype=torch.float32, device=dev)
            ent.ctrl = ent.pros[:B * W].view(B, W)
            ent.ctrl.copy_(torch.tensor(prosody_mod.Prosody().ctrl_row()).expand(B, W))
            ent.dscale = ent.pros[B * W:].view(B, Tt_b)
            ent.pin_pros = torch.zeros(B * W + B * Tt_b, dtype=torch.float32).pin_memory()
        return ent

    def _stage(self, ent, tokens, tl, mels, durations, voice, run_stream, pros=None):
        """Refresh the graph's inputs (on ``run_stream``): tokens, reference mels / voice, and -- through ONE pinned
        staging buffer -- the zero-padded durations and the token lengths (and through a second one, released by the
        same event, the prosody controls of a controlled graph)."""
        B, Tt_b = ent.tok.shape
        Tt = tokens.shape[1]
        ent.pin_free.synchronize()                      # the previous replay's copy has read the staging buffer
        pm = ent.pin_meta
        pd = pm[:B * Tt_b].view(B, Tt_b)
        if durations is not None:
            pd.zero_()
            pd[:, :Tt] = durations
        pm[B * Tt_b:] = torch.as_tensor(tl, dtype=torch.int32)
        if durations is not None:
            ent.meta.copy_(pm, non_blocking=True)
        else:
            ent.lens_t.copy_(pm[B * Tt_b:], non_blocking=True)
        if ent.pros is not None:
            ctrl, dscale = prosody_mod.pack(pros, Tt_b)
            W = prosody_mod.CTRL_WIDTH
            ent.pin_pros[:B * W].view(B, W).copy_(ctrl)
            ent.pin_pros[B * W:].view(B, Tt_b).copy_(dscale)
            ent.pros.copy_(ent.pin_pros, non_blocking=True)
        ent.pin_free.record(run_stream)
        ent.tok[:, :Tt].copy_(tokens, non_blocking=True)
        if Tt < Tt_b:
            ent.tok[:, Tt:].zero_()
        if ent.voice is None:
            ent.mels.copy_(mels, non_blocking=True)
        else:
            for dst, src in zip(ent.voice, voice):
                dst.copy_(src, non_blocking=True)

    # ---------------------------------------------------------------------------------------
    @torch.no_grad()
    def synthesize(self, tokens, tok_lens, mels, mel_lens, durations=None, voice=None, predict_durations: bool = False,
                   exact_frames: bool = False, defer: bool = False, prosody=None, audio=None, loudness=None,
                   watermark=None):
        """``tokens`` int64 [B,Tt] and ``mels`` fp32 [B,80,Tr]: device tensors or (pinned) HOST tensors -- host inputs
        are copied straight into the graph's static buffers; ``tok_lens`` / ``mel_lens`` int64 [B] HOST tensors (or
        lists); ``durations`` int64 [B,Tt] HOST tensor or None (predict them, one device->host sync of B integers);
        ``voice``: cached ``encode_voice`` result (the style encoder is then skipped).
        Returns (wav [B, 300*Tm_max] fp32 or int16, mel_lengths int32 [B] (device), mel fp32 [B,80,Tm_max]) with
        ``Tm_max`` the longest utterance's frame count; per-call extras (predicted durations, frame counts) are in
        ``self.last``.  With ``duration_bound`` set and no ``durations`` the pass is sync-free: ``Tm_max`` is then the
        bound's frame bucket and the utterances' true lengths are the returned ``mel_lengths`` (``exact_frames=True``
        forces the two-graph path with the frame-count read-back).
        ``defer=True`` returns a ticket instead of the result; ``finish(ticket)`` completes the call.  With predicted
        durations the ticket is handed out BEFORE the host waits for the frame counts, so a caller can issue the next
        call's graph A first (``synthesize_many`` does): the GPU then always has work queued while the host wakes up.
        ``prosody``: one ``prosody.Prosody`` per utterance (``ValueError`` for a ``duration_scale`` other than 1 when
        ``durations`` are given); ``last["pred_dur"]`` then holds the scaled durations.
        ``audio``: an ``audio.AudioFormat``; the returned waveforms are then ``[B, audio.out_samples(300*Tm_max)]``
        of ``audio.dtype`` with silence codes beyond each utterance, and ``last["sample_lengths"]`` holds the
        utterances' sample counts at the target rate (int32, device).
        ``loudness``: an ``audio.Loudness``; each utterance is then scaled by its normalisation gain before the
        encoding (in ``audio``'s format, or the native 24 kHz fp32), and ``last["loudness"]``, ``last["true_peak"]``
        and ``last["gain_db"]`` hold the values measured before the gain (fp64 [B], device).
        ``watermark``: an ``audio.Watermark``; each utterance's 24 kHz waveform is then marked before the meter and the
        format stage (``audio.embed_watermark`` of the pass's waveform, bit for bit)."""
        dev = self.device
        cur = torch.cuda.current_stream(dev)
        self.last_stream = cur
        if torch.is_tensor(tok_lens) and tok_lens.is_cuda or torch.is_tensor(mel_lens) and mel_lens.is_cuda or \
                (durations is not None and durations.is_cuda):
            raise ValueError("synthesize: tok_lens / mel_lens / durations are host-side metadata (CPU tensors or "
                             "lists); device copies would force a synchronisation per call")
        tl = [int(v) for v in (tok_lens.tolist() if torch.is_tensor(tok_lens) else tok_lens)]
        ml = [int(v) for v in (mel_lens.tolist() if torch.is_tensor(mel_lens) else mel_lens)]
        B, Tt = tokens.shape
        Tr = mels.shape[2]
        pros = prosody_mod.check(prosody, tl, durations is not None)
        fmt = self._out_format(audio)
        loud = audio_mod.check_loudness(loudness, self.pcm16)
        wm = audio_mod.check_watermark(watermark, self.pcm16)
        if loud is not None and fmt is None:
            fmt = audio_mod.NATIVE
        controlled = pros is not None
        predict = bool(predict_durations) or durations is None
        Tt_b = _ceil_to(Tt, self.token_quantum)
        sums = None
        if durations is not None:
            sums = [int(durations[b, :tl[b]].sum()) for b in range(B)]
        graphable = self.use_cuda_graph and all(v == Tr for v in ml)
        bounded = durations is None and self.duration_bound is not None and not exact_frames
        if bounded:
            L_bound = _ceil_to(int(-(-Tt_b * self.duration_bound // 1)), self.frame_quantum)
            key_a = ("abp", voice is not None, controlled, B, Tt_b, Tr, True, L_bound)
        else:
            key_a = ("ab" if durations is not None else "a", voice is not None, controlled, B, Tt_b, Tr, predict,
                     _ceil_to(max(sums), self.frame_quantum) if sums is not None else 0)
        if graphable:
            n = self._seen.get(key_a, 0) + 1
            self._seen[key_a] = n
            graphable = n >= self.capture_after
        if not graphable:
            res = self._eager(tokens, tl, mels, ml, durations, voice, predict, pros)
            if fmt is not None or wm is not None:
                res = self._format_stage(res, fmt, loud=loud, **_wm_kw(wm))
            return self._done_ticket(res) if defer else res
        if self._epoch != nn_util.plan_epoch():
            self.drop_graphs()

        slot, run_stream = 0, cur
        if self.pipeline_depth > 1:
            if self._slot_streams is None:
                self._slot_streams = [torch.cuda.Stream(device=dev) for _ in range(self.pipeline_depth)]
            slot = self._calls % self.pipeline_depth
            run_stream = self._slot_streams[slot]
        self._calls += 1

        ent = self._lookup(slot, key_a)
        if ent is None:
            ent = self._static_inputs(B, Tt_b, mels, voice, controlled)
            mel_lens_dev = torch.full((B,), Tr, dtype=torch.int64, device=dev)
            ent.mel_lens = mel_lens_dev                 # a graph input like the others: lives as long as the graph
            if durations is not None:
                L_b = key_a[-1]

                def fn(ent=ent):
                    st = self._phase_a(ent.tok, ent.lens_t, ent.mels, mel_lens_dev, ml, ent.voice, predict)
                    return self._phase_b(st, ent.dur, L_b, ent.ctrl)
            elif bounded:
                L_b = key_a[-1]

                def fn(ent=ent):
                    st = self._phase_a(ent.tok, ent.lens_t, ent.mels, mel_lens_dev, ml, ent.voice, True, ent.dscale)
                    out = self._phase_b(st, st["pred_dur"], L_b, ent.ctrl)
                    out["pred_sum"] = st["pred_sum"]
                    return out
            else:
                def fn(ent=ent):
                    return self._phase_a(ent.tok, ent.lens_t, ent.mels, mel_lens_dev, ml, ent.voice, True, ent.dscale)
            ent.graph, ent.out, ent.launches = self._capture(slot, fn)
            if durations is None and not bounded:
                ent.state = ent.out
                ent.out = None
                ent.pin_meta = torch.zeros(B * Tt_b + B, dtype=torch.int32).pin_memory()
            self._insert(slot, key_a, ent)

        if run_stream is not cur:
            # the slot's stream picks up after whatever produced the inputs on the caller's stream;
            # the caller's stream never waits for the slot (that would serialise the pipeline)
            ready = torch.cuda.Event()
            ready.record(cur)
            run_stream.wait_event(ready)
            for t in (tokens, mels) + tuple(voice or ()):
                if t.is_cuda:
                    t.record_stream(run_stream)
        launches = ent.launches
        with torch.cuda.stream(run_stream):
            self._stage(ent, tokens, tl, mels, durations, voice, run_stream, pros)
            ent.graph.replay()
            if durations is None and not bounded:
                # the only device->host hand-off of the pass: B frame counts (the other slot keeps the GPU busy)
                pin_sum = ent.pin_meta[:B]
                pin_sum.copy_(ent.state["pred_sum"], non_blocking=True)
                t = _Ticket()
                t.got = torch.cuda.Event()
                t.got.record(run_stream)
                t.slot, t.run_stream, t.is_side, t.ent, t.B, t.launches = slot, run_stream, run_stream is not cur, ent, B, launches
                t.fmt, t.loud, t.wm = fmt, loud, wm
                if defer:
                    return t
                return self.finish(t)
            out = ent.out
            if run_stream is not cur:
                done = torch.cuda.Event()
                done.record(run_stream)
                self._slot_done[slot] = done
        self.stats["replays"] += 1
        self.last_stream = run_stream
        self.launches_per_call = launches
        ops._count(launches)
        if bounded:
            self.last = dict(out, frames=None, graph=True, frame_bound=2 * key_a[-1])
            res = (out["wav"], out["mel_lengths"], out["mel"])
        else:
            Tm = 2 * max(sums)
            self.last = dict(out, frames=[2 * v for v in sums], graph=True)
            res = (out["wav"][:, :HOP * Tm], out["mel_lengths"], out["mel"][:, :, :Tm])
        if fmt is not None or wm is not None:
            res = self._format_stage(res, fmt, slot if run_stream is not cur else None, loud, **_wm_kw(wm))
        return self._done_ticket(res) if defer else res

    def _out_format(self, audio):
        """The format stage's format, or None for the native output (``audio`` None or equal to it)."""
        if audio is None:
            return None
        if not isinstance(audio, audio_mod.AudioFormat):
            raise ValueError(f"audio: expected an AudioFormat, got {type(audio).__name__}")
        if audio == audio_mod.AudioFormat(SAMPLE_RATE, "pcm16" if self.pcm16 else "float32"):
            return None
        if self.pcm16:
            raise ValueError(f"audio={audio}: output formats resample the fp32 waveform; use Synthesizer(pcm16=False) "
                             f"(AudioFormat(24000, 'pcm16') gives the same samples as pcm16=True)")
        return audio

    def _format_stage(self, res, fmt, side_slot=None, loud=None, wm=None):
        """One ``as_resample_encode`` launch on ``last_stream`` after the pass, into a fresh stream-ordered
        allocation; not captured, so it adds no graphs.  ``side_slot``: the pipeline slot whose side stream ran the
        call (``join`` then also waits for the format stage).  ``loud``: an ``audio.Loudness``; the meter's launches
        then precede it on the same stream and its gain is applied.  ``wm``: an ``audio.Watermark``; one
        ``as_watermark_embed`` launch first marks the waveform the meter and the format read (``fmt`` None: the marked
        waveform is the result)."""
        wav, mel_lengths, mel = res
        with torch.cuda.stream(self.last_stream):
            if wm is not None:
                wav = ops.watermark_embed(wav, self.last["wav_lengths"], wm)
                if self.last.get("graph"):
                    self.launches_per_call += 1
            n = None if fmt is None else torch.empty(wav.shape[0], dtype=torch.int32, device=wav.device)
            if fmt is None:
                y = wav
            elif loud is None:
                y = ops.resample_encode(wav, self.last["wav_lengths"], fmt, fmt.out_samples(wav.shape[1]), out_lens=n)
            else:
                lufs, tp, gain_db, gain = ops.loudness_measure(wav, self.last["wav_lengths"], SAMPLE_RATE,
                                                               loud.target_lufs, loud.max_true_peak_db)
                y = ops.resample_encode(wav, self.last["wav_lengths"], fmt, fmt.out_samples(wav.shape[1]), out_lens=n,
                                        gain=gain)
                self.last.update(loudness=lufs, true_peak=tp, gain_db=gain_db)
            if side_slot is not None:
                done = torch.cuda.Event()
                done.record(self.last_stream)
                self._slot_done[side_slot] = done
        if fmt is not None:
            self.last["sample_lengths"] = n
            if self.last.get("graph"):
                self.launches_per_call += 1 + (ops.LOUDNESS_LAUNCHES if loud is not None else 0)
        return y, mel_lengths, mel

    def _done_ticket(self, res):
        t = _Ticket()
        t.result, t.last, t.last_stream = res, self.last, self.last_stream
        return t

    def finish(self, ticket: "_Ticket"):
        """Complete a deferred call: -> (wav, mel_lengths, mel) as ``synthesize`` returns them; sets ``last`` /
        ``last_stream`` for this call."""
        if ticket.result is not None:
            self.last, self.last_stream = ticket.last, ticket.last_stream
            return ticket.result
        ent, slot, B = ticket.ent, ticket.slot, ticket.B
        with torch.cuda.stream(ticket.run_stream):
            ticket.got.synchronize()
            sums = [int(v) for v in ent.pin_meta[:B].tolist()]
            L_b = _ceil_to(max(sums), self.frame_quantum)
            key_b = ("b", ent.uid, L_b)
            eb = self._lookup(slot, key_b)
            if eb is None:
                eb = _Captured()
                eb.state = ent
                st = ent.state
                # the control block of the A entry: staged with this call's graph A, in the same slot
                eb.graph, eb.out, eb.launches = self._capture(
                    slot, lambda: self._phase_b(st, st["pred_dur"], L_b, ent.ctrl))
                self._insert(slot, key_b, eb)
            eb.graph.replay()
            out = eb.out
            if ticket.is_side:
                done = torch.cuda.Event()
                done.record(ticket.run_stream)
                self._slot_done[slot] = done
        launches = ticket.launches + eb.launches
        self.stats["replays"] += 1
        self.last_stream = ticket.run_stream
        self.launches_per_call = launches
        ops._count(launches)
        Tm = 2 * max(sums)
        self.last = dict(out, frames=[2 * v for v in sums], graph=True, duration=ent.state["duration"],
                         pred_dur=ent.state["pred_dur"])
        res = (out["wav"][:, :HOP * Tm], out["mel_lengths"], out["mel"][:, :, :Tm])
        if ticket.fmt is not None or ticket.wm is not None:
            res = self._format_stage(res, ticket.fmt, slot if ticket.is_side else None, ticket.loud,
                                     **_wm_kw(ticket.wm))
        ticket.result, ticket.last, ticket.last_stream = res, self.last, self.last_stream
        return ticket.result

    def join(self):
        """Make the current stream wait for every pipelined call issued so far."""
        cur = torch.cuda.current_stream(self.device)
        for ev in self._slot_done.values():
            cur.wait_event(ev)


# -------------------------------------------------------------------------------------------
# data-parallel helpers
# -------------------------------------------------------------------------------------------
def shard_utterances(costs: Sequence[float], world_size: int) -> List[List[int]]:
    """Longest-processing-time-first assignment of utterances to ranks (cost ~ frames to synthesise)."""
    order = sorted(range(len(costs)), key=lambda i: (-costs[i], i))
    loads = [0.0] * world_size
    shards: List[List[int]] = [[] for _ in range(world_size)]
    for i in order:
        r = min(range(world_size), key=lambda k: (loads[k], k))
        shards[r].append(i)
        loads[r] += costs[i]
    return shards


def shard_by_length(frames: Sequence[int], world_size: int, utterance_cost: float = 280.0) -> List[List[int]]:
    """Length-contiguous sharding for strong scaling of a mixed-length workload (BASELINE config 5): utterances sorted
    by frame count, cut into ``world_size`` contiguous runs of equal COST, cost(u) = frames(u) + ``utterance_cost``
    (the per-utterance work that does not scale with its length -- style encoder, text encoders, duration predictor --
    in frame equivalents: ~0.27 ms per utterance against ~0.97 us per frame on B200).

    Why not LPT on frame counts (``shard_utterances``): LPT balances the frames, but it deals every rank a sample of
    the WHOLE length distribution, so the fewer utterances a rank holds the more heterogeneous its micro-batches get:
    the padded work of the 512-utterance workload grows from 1.09 x its frames on one GPU to 1.37 x on eight, and
    padding is computed (every kernel masks by length, none skips).  Contiguous runs keep every rank's micro-batches
    as homogeneous as the single-GPU ones.  Returns ``world_size`` index lists (longest utterances on rank 0); a rank
    may be empty when there are fewer utterances than ranks."""
    order = sorted(range(len(frames)), key=lambda i: (-int(frames[i]), i))
    cost = [max(int(frames[i]), 1) + float(utterance_cost) for i in order]
    total = sum(cost)
    shards: List[List[int]] = [[] for _ in range(world_size)]
    acc, r = 0.0, 0
    for pos, i in enumerate(order):
        # move on when this rank's share is used up (keeping at least one utterance per remaining rank where possible)
        while r < world_size - 1 and acc + 0.5 * cost[pos] > total * (r + 1) / world_size:
            r += 1
        shards[r].append(i)
        acc += cost[pos]
    return shards


def bucket_utterances(frames: Sequence[int], max_batch: int = 16, max_padded_frames: Optional[int] = None,
                      quantum: int = 1) -> List[List[int]]:
    """Length-bucketed micro-batches for a mixed-length shard (SURVEY.md §8e): utterances sorted by frame count,
    longest first, cut into runs of at most ``max_batch`` whose PADDED size ``len(run) * max(frames in run)`` stays
    within ``max_padded_frames`` -- neighbours in the sorted order have similar lengths, so padding stays small and
    every micro-batch costs about the same.  Every index appears exactly once; a single utterance longer than the
    budget gets a micro-batch of its own.  ``quantum`` rounds frame counts up first (the engine's shape buckets), so
    the batch size is a function of the bucket and repeated traffic maps onto a small set of graph keys."""
    order = sorted(range(len(frames)), key=lambda i: (-int(frames[i]), i))
    batches: List[List[int]] = []
    cur: List[int] = []
    cur_max = 0
    q = max(1, int(quantum))
    for i in order:
        f = (max(int(frames[i]), 1) + q - 1) // q * q
        longest = max(cur_max, f)
        over = max_padded_frames is not None and cur and (len(cur) + 1) * longest > max_padded_frames
        if cur and (len(cur) >= max_batch or over):
            batches.append(cur)
            cur, longest = [], f
        cur.append(i)
        cur_max = longest
    if cur:
        batches.append(cur)
    return batches


class HostArena:
    """Pinned host memory the waveforms of a ``synthesize_many`` call are copied into (one 2-D device->host copy
    per micro-batch).  Pinned allocations are slow, so blocks are kept and handed out again after ``reset()``;
    a request that does not fit the remaining space adds a block."""

    def __init__(self, block_bytes: int = 64 << 20):
        self.block_bytes = int(block_bytes)
        self.blocks: List[torch.Tensor] = []
        self.cur = 0
        self.off = 0

    def reset(self):
        self.cur = self.off = 0

    def take(self, n: int, dtype: torch.dtype) -> torch.Tensor:
        nbytes = (n * torch.empty((), dtype=dtype).element_size() + 255) // 256 * 256
        while True:
            if self.cur < len(self.blocks) and self.off + nbytes <= self.blocks[self.cur].numel():
                out = self.blocks[self.cur][self.off:self.off + nbytes]
                self.off += nbytes
                return out.view(dtype)[:n]
            if self.cur < len(self.blocks):
                self.cur, self.off = self.cur + 1, 0
                continue
            self.blocks.append(torch.empty(max(nbytes, self.block_bytes), dtype=torch.uint8).pin_memory())


@torch.no_grad()
def synthesize_many(syn: "Synthesizer", tokens: Sequence[torch.Tensor], ref_mels: Sequence[torch.Tensor],
                    durations: Optional[Sequence[torch.Tensor]] = None, max_batch: int = 16,
                    max_padded_frames: Optional[int] = 25600, to_host: bool = False, arena: Optional[HostArena] = None,
                    frames_per_token: float = 5.34, prosody: Optional[Sequence["prosody_mod.Prosody"]] = None,
                    audio: Optional["audio_mod.AudioFormat"] = None, loudness: Optional["audio_mod.Loudness"] = None,
                    watermark: Optional["audio_mod.Watermark"] = None):
    """Mixed-length utterances through ``syn`` in length-bucketed ragged micro-batches (BASELINE config 5).

    ``tokens[i]`` int64 [Tt_i], ``ref_mels[i]`` fp32 [80, Tr_i], ``durations[i]`` int64 [Tt_i] (host tensors) or
    ``durations=None`` to predict them (micro-batches are then formed by token count, ``frames_per_token`` being
    the planning estimate).  Micro-batch shapes are quantised to the engine's buckets, so repeated traffic replays a
    bounded set of CUDA graphs.  Returns ``(wavs, frames)``: ``wavs[i]`` holds the ``300 * frames[i]`` samples of
    utterance ``i`` (fp32, or int16 when ``syn.pcm16``), independent of what it was batched with (batch-1
    semantics) -- device tensors, or views of the pinned ``arena`` when ``to_host`` (valid after this function
    returns: it synchronises the copies).  ``prosody``: one ``prosody.Prosody`` per utterance (or None); the planning
    estimate of an utterance then grows with its mean ``duration_scale``.  ``audio``: an ``audio.AudioFormat`` (see
    ``Synthesizer.synthesize``); ``wavs[i]`` then holds the ``audio.out_samples(300 * frames[i])`` samples of
    utterance ``i`` in that format.  ``loudness``: an ``audio.Loudness`` (see ``Synthesizer.synthesize``); each
    utterance is normalised on its own waveform, so its gain does not depend on its batch-mates.  ``watermark``: an
    ``audio.Watermark`` (see ``Synthesizer.synthesize``); each utterance's mark depends only on its own samples."""
    n = len(tokens)
    pros = prosody_mod.check(prosody, [int(t.shape[0]) for t in tokens], durations is not None)
    if durations is not None:
        plan_frames = [2 * int(d.sum()) for d in durations]
    else:
        plan_frames = [int(round(frames_per_token * int(t.shape[0]) *
                                 (pros[i].mean_duration_scale(int(t.shape[0])) if pros else 1.0)))
                       for i, t in enumerate(tokens)]
    frames: List[int] = list(plan_frames)
    wavs: List[Optional[torch.Tensor]] = [None] * n
    fmt = syn._out_format(audio)
    loud_kw = {}
    if loudness is not None:
        loud_kw["loudness"] = audio_mod.check_loudness(loudness, syn.pcm16)
        fmt = fmt or audio_mod.NATIVE
    if watermark is not None:
        loud_kw["watermark"] = audio_mod.check_watermark(watermark, syn.pcm16)
    dt = fmt.dtype if fmt is not None else torch.int16 if syn.pcm16 else torch.float32

    def cut(f):
        """Samples of an utterance of ``f`` mel frames in the output format."""
        return fmt.out_samples(HOP * f) if fmt is not None else HOP * f
    arena = arena or (HostArena() if to_host else None)
    if to_host:
        arena.reset()
    pending, late = [], []

    def collect(idx, ticket):
        """Finish a deferred call and queue the copies of its waveforms (on the call's stream)."""
        wav, mel_lengths, _ = syn.finish(ticket)
        got = syn.last["frames"]
        if got is not None:
            for j, i in enumerate(idx):
                frames[i] = got[j]
        with torch.cuda.stream(syn.last_stream):
            if to_host:
                S = wav.shape[1]
                dst = arena.take(len(idx) * S, dt).view(len(idx), S)
                dst.copy_(wav, non_blocking=True)
            else:
                dst = wav.clone() if got is None else None
            if got is None:
                # sync-free pass (Synthesizer(duration_bound=...)): the frame counts come back with the waveforms
                meta = arena.take(2 * len(idx), torch.int32) if to_host else torch.empty(2 * len(idx), dtype=torch.int32).pin_memory()
                meta[:len(idx)].copy_(mel_lengths, non_blocking=True)
                meta[len(idx):].copy_(syn.last["pred_sum"], non_blocking=True)
                late.append((idx, dst, meta, syn.last["frame_bound"]))
            else:
                for j, i in enumerate(idx):
                    wavs[i] = dst[j, :cut(frames[i])] if to_host else wav[j, :cut(frames[i])].clone()

    # With predicted durations a call synchronises on its frame counts between its two graphs: issue the NEXT
    # micro-batch's first graph before finishing the current one (one call of look-ahead; needs a second pipeline slot)
    lookahead = 1 if syn.pipeline_depth >= 2 else 0
    waiting = []
    for idx in bucket_utterances(plan_frames, max_batch, max_padded_frames, quantum=2 * syn.frame_quantum):
        Tt = max(int(tokens[i].shape[0]) for i in idx)
        Tr = max(int(ref_mels[i].shape[1]) for i in idx)
        tok = torch.zeros(len(idx), Tt, dtype=torch.long).pin_memory()
        dur = torch.zeros(len(idx), Tt, dtype=torch.long) if durations is not None else None
        mel = torch.zeros(len(idx), ref_mels[idx[0]].shape[0], Tr).pin_memory()
        for j, i in enumerate(idx):
            tok[j, :tokens[i].shape[0]] = tokens[i]
            if dur is not None:
                dur[j, :durations[i].shape[0]] = durations[i]
            mel[j, :, :ref_mels[i].shape[1]] = ref_mels[i]
        tl = [int(tokens[i].shape[0]) for i in idx]
        ml = [int(ref_mels[i].shape[1]) for i in idx]
        waiting.append((idx, syn.synthesize(tok, tl, mel, ml, dur, defer=True,
                                            prosody=[pros[i] for i in idx] if pros else None, audio=fmt,
                                            **loud_kw)))
        while len(waiting) > lookahead:
            collect(*waiting.pop(0))
        pending.append((tok, mel))            # pinned inputs must outlive their asynchronous copies
    while waiting:
        collect(*waiting.pop(0))
    syn.join()
    if to_host or late:
        torch.cuda.current_stream(syn.device).synchronize()
    redo = []
    for idx, dst, meta, bound in late:
        for j, i in enumerate(idx):
            frames[i] = int(meta[j])
            wavs[i] = dst[j, :cut(frames[i])]
            if 2 * int(meta[len(idx) + j]) > bound:       # the prediction did not fit the bound: truncated there
                redo.append(i)
    for i in redo:                                         # rare: exact two-graph pass for the utterances that overflowed
        w, _, _ = syn.synthesize(tokens[i].view(1, -1).pin_memory(), [int(tokens[i].shape[0])],
                                 ref_mels[i].unsqueeze(0).pin_memory(), [int(ref_mels[i].shape[1])], None, exact_frames=True,
                                 prosody=[pros[i]] if pros else None, audio=fmt, **loud_kw)
        frames[i] = syn.last["frames"][0]
        with torch.cuda.stream(syn.last_stream):
            wavs[i] = w[0, :cut(frames[i])].clone() if not to_host else w[0, :cut(frames[i])].to("cpu")
    if redo:
        syn.join()
        torch.cuda.current_stream(syn.device).synchronize()
    return wavs, frames


def _as_bytes(t: torch.Tensor) -> torch.Tensor:
    return t.contiguous().view(-1).view(torch.uint8)


def _pack_payload(wav: torch.Tensor, lengths: torch.Tensor, Bm: int, Sm: int, out: Optional[torch.Tensor] = None):
    """One byte buffer per rank: ``Bm`` int64 sample counts (header) followed by the ``[Bm, Sm]`` samples.  int16 PCM,
    uint8 G.711 codes and fp32 all travel as bytes (the NCCL process group has no int16)."""
    es = wav.element_size()
    nbytes = 8 * Bm + Bm * Sm * es
    if out is None:
        out = torch.zeros(nbytes, dtype=torch.uint8, device=wav.device)
    head = out[:8 * Bm].view(torch.int64)
    head.zero_()
    head[:lengths.shape[0]] = lengths.to(torch.int64)
    body = out[8 * Bm:].view(wav.dtype).view(Bm, Sm)
    if tuple(wav.shape) != (Bm, Sm):
        body.zero_()
    body[:wav.shape[0], :wav.shape[1]].copy_(wav)
    return out


def _unpack_payload(buf: torch.Tensor, dtype: torch.dtype, Bm: int, Sm: int, shape):
    head = buf[:8 * Bm].view(torch.int64)
    body = buf[8 * Bm:].view(dtype).view(Bm, Sm)
    return body[:shape[0], :shape[1]], head[:shape[0]]


def gather_waveforms(wav: torch.Tensor, lengths: torch.Tensor, dst: int = 0, group=None, shapes=None):
    """Gather per-rank ``wav`` [B_r, S_r] (fp32, int16 PCM or uint8 G.711 codes) + sample ``lengths`` [B_r] on ``dst`` with ONE
    collective: each rank contributes one byte buffer (lengths header + samples, padded to the common maximum).

    Ranks may hold different batch sizes / paddings: sizes are all-gathered first unless ``shapes`` (list of
    ``(B_r, S_r)`` per rank, known on the host -- e.g. from ``shard_utterances``) is given, which skips that
    exchange and its host synchronisation.  Works with NCCL (GPU) and gloo (CPU tests).
    Returns (list of [B_r, S_r] tensors, list of lengths) on ``dst``, (None, None) elsewhere."""
    import torch.distributed as dist
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    if shapes is None:
        shape = torch.tensor([wav.shape[0], wav.shape[1]], dtype=torch.int64, device=wav.device)
        gathered = [torch.zeros_like(shape) for _ in range(world)]
        dist.all_gather(gathered, shape, group=group)
        shapes = [tuple(int(v) for v in s.tolist()) for s in gathered]
    else:
        shapes = [tuple(int(v) for v in s) for s in shapes]
        assert len(shapes) == world and shapes[rank] == tuple(wav.shape)
    Bm, Sm = max(s[0] for s in shapes), max(s[1] for s in shapes)
    mine = _pack_payload(wav, lengths, Bm, Sm)
    bufs = [torch.empty_like(mine) for _ in range(world)] if rank == dst else None
    dist.gather(mine, bufs, dst=dst, group=group)
    if rank != dst:
        return None, None
    parts = [_unpack_payload(b, wav.dtype, Bm, Sm, s) for b, s in zip(bufs, shapes)]
    return [p[0] for p in parts], [p[1] for p in parts]


class WaveformGatherer:
    """The same single-collective gather, off the critical path of a pipelined engine: ``submit`` packs the
    rank's waveforms into a ring buffer on the producer's stream (one device copy) and issues the gather on a
    dedicated communication stream, so neither the engine's streams nor the host wait for NCCL; ``results`` makes
    the caller's stream wait for the most recent gather.  Every rank also keeps (and can copy out) its own
    waveforms, so the gather is optional for serving -- it exists because north_star asks for the waveforms on one
    rank.  ``shapes``: ``(B_r, S_r)`` per rank, fixed for the gatherer's lifetime."""

    def __init__(self, device, shapes, dtype: torch.dtype, dst: int = 0, group=None, depth: int = 3):
        import torch.distributed as dist
        self.dist, self.group, self.dst = dist, group, dst
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        self.shapes = [tuple(int(v) for v in s) for s in shapes]
        assert len(self.shapes) == self.world
        self.dtype = dtype
        self.Bm, self.Sm = max(s[0] for s in self.shapes), max(s[1] for s in self.shapes)
        self.device = torch.device(device)
        self.cuda = self.device.type == "cuda"
        nbytes = 8 * self.Bm + self.Bm * self.Sm * torch.empty((), dtype=dtype).element_size()
        self.ring = [torch.zeros(nbytes, dtype=torch.uint8, device=self.device) for _ in range(depth)]
        self.recv = [[torch.empty_like(self.ring[0]) for _ in range(self.world)] if self.rank == dst else None
                     for _ in range(depth)]
        self.free = [None] * depth            # event: the gather that read ring[i] has finished
        self.comm = torch.cuda.Stream(device=self.device) if self.cuda else None
        self.n = 0
        self.last = None

    def submit(self, wav: torch.Tensor, lengths: torch.Tensor, producer_stream=None):
        i = self.n % len(self.ring)
        self.n += 1
        assert tuple(wav.shape) == self.shapes[self.rank]
        if not self.cuda:
            _pack_payload(wav, lengths, self.Bm, self.Sm, out=self.ring[i])
            self.dist.gather(self.ring[i], self.recv[i], dst=self.dst, group=self.group)
            self.last = i
            return
        ps = producer_stream or torch.cuda.current_stream(self.device)
        if self.free[i] is not None:
            ps.wait_event(self.free[i])
        with torch.cuda.stream(ps):
            _pack_payload(wav, lengths, self.Bm, self.Sm, out=self.ring[i])
            packed = torch.cuda.Event()
            packed.record(ps)
        self.comm.wait_event(packed)
        with torch.cuda.stream(self.comm):
            # the process group orders the collective after the current (= communication) stream and makes only
            # that stream wait for it
            self.dist.gather(self.ring[i], self.recv[i], dst=self.dst, group=self.group)
            done = torch.cuda.Event()
            done.record(self.comm)
        self.free[i] = done
        self.last = i

    def results(self):
        """(waveforms per rank, sample counts per rank) of the latest ``submit`` on ``dst`` (the current stream waits
        for the gather); (None, None) elsewhere."""
        if self.last is None:
            return None, None
        if self.cuda and self.free[self.last] is not None:
            torch.cuda.current_stream(self.device).wait_event(self.free[self.last])
        if self.rank != self.dst:
            return None, None
        parts = [_unpack_payload(b, self.dtype, self.Bm, self.Sm, s) for b, s in zip(self.recv[self.last], self.shapes)]
        return [p[0] for p in parts], [p[1] for p in parts]
