"""Per-utterance prosody and articulation controls for synthesis (the SSML ``<prosody>`` rate / pitch / volume
controls, plus edits of ArtSpeech's articulatory EMA track).

``Prosody`` holds one utterance's controls; every field defaults to identity.  They act where a variance-adaptor
TTS takes its controls: the duration predictor's output before the rounding (``as_round_durations_scaled``) and the
arts predictor's F0 / energy / EMA tracks before the decoder (``as_prosody_apply``, models.py:369-370).  Both are
device inputs staged like the durations, so a captured graph serves controls that change on every call.

Semantics (per utterance):

- ``duration_scale`` (a float, or one float per token): ``dur = max(1, rint(pred * scale))`` for predicted
  durations; > 1 speaks slower.  Caller-given integer durations are the caller's: a scale other than 1 is refused.
- ``pitch_shift`` (semitones) and ``pitch_range`` (``r`` >= 0): on voiced frames (``hz >= VOICING_FLOOR_HZ``,
  ``hz = f0 * pitch_std + pitch_mean``) ``hz' = exp(mu + r * (ln hz - mu) + shift * ln2 / 12)`` with ``mu`` the mean
  of ``ln hz`` over the utterance's voiced frames; ``r = 0`` is a monotone voice.  Unvoiced frames, and utterances
  without a voiced frame, keep their F0.
- ``energy_db``: a power gain, ``n' = n + energy_db * ln10 / 10 / energy_std`` (energy is ``ln ||mel power||``).
- ``articulation_scale[10]`` / ``articulation_offset[10]``: per EMA channel ``e' = m + s * (e - m) + o`` with ``m``
  the channel's mean over the utterance; the offset is in dataset-std units (the normalised track's unit).
  A scale below 1 hypo-articulates, above 1 hyper-articulates.

A track whose controls are identity is not written, so identity controls give exactly the output of no controls.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import List, Optional, Sequence, Tuple, Union

import torch

VOICING_FLOOR_HZ = 50.0          # a frame is voiced when its F0 is at least this (as_prosody_apply uses the same)
N_EMA = 10                       # EMA channels of the arts predictor
CTRL_WIDTH = 24                  # AS_PROSODY_CTRL: shift, range, dB, pad, scale[10], offset[10]


def _finite(name: str, v) -> float:
    try:
        f = float(v)
    except (TypeError, ValueError):
        raise ValueError(f"Prosody.{name}: expected a number, got {v!r}") from None
    if not math.isfinite(f):
        raise ValueError(f"Prosody.{name}: must be finite, got {f}")
    return f


def _vector(name: str, v, n: Optional[int]) -> Tuple[float, ...]:
    if torch.is_tensor(v):
        v = v.detach().cpu().reshape(-1).tolist()
    try:
        vals = tuple(_finite(name, x) for x in v)
    except TypeError:
        raise ValueError(f"Prosody.{name}: expected a sequence of numbers, got {v!r}") from None
    if n is not None and len(vals) != n:
        raise ValueError(f"Prosody.{name}: expected {n} values (one per EMA channel), got {len(vals)}")
    return vals


@dataclass(frozen=True)
class Prosody:
    """One utterance's controls (see the module docstring); validated on construction."""
    duration_scale: Union[float, Sequence[float]] = 1.0
    pitch_shift: float = 0.0
    pitch_range: float = 1.0
    energy_db: float = 0.0
    articulation_scale: Sequence[float] = field(default=(1.0,) * N_EMA)
    articulation_offset: Sequence[float] = field(default=(0.0,) * N_EMA)

    def __post_init__(self):
        ds = self.duration_scale
        if torch.is_tensor(ds) and ds.dim() == 0:
            ds = float(ds)
        if isinstance(ds, (int, float)):
            ds = _finite("duration_scale", ds)
            bad = ds <= 0
        else:
            ds = _vector("duration_scale", ds, None)
            if not ds:
                raise ValueError("Prosody.duration_scale: empty per-token vector")
            bad = min(ds) <= 0
        if bad:
            raise ValueError("Prosody.duration_scale: must be > 0")
        rng = _finite("pitch_range", self.pitch_range)
        if rng < 0:
            raise ValueError(f"Prosody.pitch_range: must be >= 0, got {rng}")
        object.__setattr__(self, "duration_scale", ds)
        object.__setattr__(self, "pitch_shift", _finite("pitch_shift", self.pitch_shift))
        object.__setattr__(self, "pitch_range", rng)
        object.__setattr__(self, "energy_db", _finite("energy_db", self.energy_db))
        object.__setattr__(self, "articulation_scale", _vector("articulation_scale", self.articulation_scale, N_EMA))
        object.__setattr__(self, "articulation_offset", _vector("articulation_offset", self.articulation_offset, N_EMA))

    @property
    def scales_durations(self) -> bool:
        """False when ``duration_scale`` is identity (1 for every token)."""
        ds = self.duration_scale
        return any(v != 1.0 for v in ds) if isinstance(ds, tuple) else ds != 1.0

    def mean_duration_scale(self, n_tokens: int) -> float:
        """Mean scale over the first ``n_tokens`` tokens (a planning estimate of the frame count's growth)."""
        ds = self.duration_scale
        if not isinstance(ds, tuple):
            return ds
        head = ds[:max(1, int(n_tokens))]
        return sum(head) / len(head)

    def ctrl_row(self) -> List[float]:
        """The utterance's row of the ``as_prosody_apply`` control block."""
        return [self.pitch_shift, self.pitch_range, self.energy_db, 0.0,
                *self.articulation_scale, *self.articulation_offset]


def check(prosody, tok_lens: Sequence[int], durations_given: bool) -> Optional[List[Prosody]]:
    """Validate the ``prosody=`` argument of a batch of ``len(tok_lens)`` utterances: ``None`` or one ``Prosody`` per
    utterance.  Raises ``ValueError`` for a wrong count, a per-token ``duration_scale`` shorter than its utterance,
    or a ``duration_scale`` other than 1 when the caller gives integer durations."""
    if prosody is None:
        return None
    if isinstance(prosody, Prosody):
        prosody = [prosody]
    prosody = list(prosody)
    if len(prosody) != len(tok_lens):
        raise ValueError(f"prosody: expected one Prosody per utterance ({len(tok_lens)}), got {len(prosody)}")
    for i, (p, n) in enumerate(zip(prosody, tok_lens)):
        if not isinstance(p, Prosody):
            raise ValueError(f"prosody[{i}]: expected a Prosody, got {type(p).__name__}")
        if durations_given and p.scales_durations:
            raise ValueError(f"prosody[{i}].duration_scale: the caller gave integer durations; scale those instead")
        if isinstance(p.duration_scale, tuple) and len(p.duration_scale) < int(n):
            raise ValueError(f"prosody[{i}].duration_scale: {len(p.duration_scale)} values for {int(n)} tokens")
    return prosody


def pack(prosody: Sequence[Prosody], Tt: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """-> (ctrl fp32 [B, CTRL_WIDTH], duration scale fp32 [B, Tt]) host tensors; a scalar ``duration_scale`` fills its
    row, a per-token one gives its first ``Tt`` values (1 beyond its length)."""
    B = len(prosody)
    ctrl = torch.tensor([p.ctrl_row() for p in prosody], dtype=torch.float32).view(B, CTRL_WIDTH)
    dscale = torch.ones(B, Tt, dtype=torch.float32)
    for b, p in enumerate(prosody):
        ds = p.duration_scale
        if isinstance(ds, tuple):
            k = min(len(ds), Tt)
            dscale[b, :k] = torch.tensor(ds[:k], dtype=torch.float32)
        else:
            dscale[b] = ds
    return ctrl, dscale


def constants(distribution) -> Tuple[float, float, float]:
    """(pitch_mean, pitch_std, energy_std) of ``Data/stats.json`` (``model.distribution``) as host floats."""
    return tuple(float(distribution[k]) for k in ("pitch_mean", "pitch_std", "energy_std"))
