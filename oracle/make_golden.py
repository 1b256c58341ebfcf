"""TEST INFRASTRUCTURE — generate the committed fixtures under tests/golden from the *unmodified*
reference (run in the build container, where /root/reference is mounted):

    python -m oracle.make_golden          # every fixture
    python -m oracle.make_golden live     # tests/golden/live_reference.pt only

Checkpoints are not stored: both sides rebuild them from a seed with
``artspeech_b200.checkpoint`` (the state-dict layout is identical to the reference's, which this
script asserts with a strict ``load_state_dict``).  Fixtures hold only inputs and reference outputs.
"""
from __future__ import annotations

import os

import numpy as np
import torch

from artspeech_b200 import checkpoint
from . import ref_loader as rl
from . import ref_runner

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def acoustic_cases():
    """(name, seed, Tt, Tr, forced durations or None)"""
    return [("a_pred_dur", 1, 30, 100, None),          # durations from the reference's own predictor
            ("b_forced_dur", 2, 41, 120, "rand1-4"),   # forced integer durations
            ("c_short", 3, 12, 90, "rand1-3")]


def make_inputs(seed, Tt, Tr, dur_spec):
    g = torch.Generator().manual_seed(seed)
    tok = torch.randint(1, 178, (1, Tt), generator=g)
    mel = torch.randn(1, 80, Tr, generator=g) * 0.5
    dur = None
    if dur_spec is not None:
        hi = int(dur_spec[-1])
        dur = torch.randint(1, hi + 1, (1, Tt), generator=g)
    return tok, mel, dur


def live_inputs():
    """Inputs of tests/test_oracle_pinning.py's live case (checkpoint seed 3)."""
    g = torch.Generator().manual_seed(11)
    tok = torch.randint(1, 178, (1, 23), generator=g)
    mel = torch.randn(1, 80, 97, generator=g) * 0.5
    return tok, mel


def live_case():
    """The reference's acoustic model on the live case's inputs (predicted durations), then the reference's vocoder
    on the mel it produced -> tests/golden/live_reference.pt."""
    os.makedirs(OUT, exist_ok=True)
    dist = rl.load_distribution()
    ours = checkpoint.build_random_artsspeech(3, dist)
    ref = rl.build_reference_artsspeech(dist)
    ref.load_state_dict(ours.state_dict(), strict=True)
    tok, mel = live_inputs()
    r = ref_runner.reference_test_step(ref, tok, mel)
    refg = rl.build_reference_generator()
    refg.remove_weight_norm()
    refg.load_state_dict(checkpoint.build_random_generator(3).state_dict(), strict=True)
    with torch.no_grad():
        wav = refg(r["mel"])
    torch.save(dict(checkpoint_seed=3, tokens=tok, ref_mel=mel, pred_dur=r["pred_dur"], mel=r["mel"], wav=wav),
               os.path.join(OUT, "live_reference.pt"))
    print("live case: mel", tuple(r["mel"].shape), "wav", tuple(wav.shape))


def main():
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(8)
    # ---- acoustic model ----
    dist = rl.load_distribution()
    ours = checkpoint.build_random_artsspeech(0, dist)
    assert {k: v.tolist() for k, v in dist.items()} == {k: v.tolist() for k, v in checkpoint.default_distribution().items()}
    ref = rl.build_reference_artsspeech(dist)
    print("acoustic:", ref.load_state_dict(ours.state_dict(), strict=True))
    cases = {}
    for name, seed, Tt, Tr, dspec in acoustic_cases():
        tok, mel, dur = make_inputs(seed, Tt, Tr, dspec)
        r = ref_runner.reference_test_step(ref, tok, mel, durations=dur)
        keep = {k: r[k] for k in ("style", "duration", "pred_dur", "F0", "N", "EMA", "mel", "f0_ext", "n_ext", "ema_ext")}
        keep["T_en_sum"] = r["T_en"].double().sum().float()
        keep["T_en"] = r["T_en"][:, :, :8].clone()          # first 8 channels: enough to catch layout bugs
        cases[name] = dict(tokens=tok, ref_mel=mel, durations=dur, out=keep)
        print(name, "mel", tuple(r["mel"].shape), "absmax %.3f" % r["mel"].abs().max().item())
    torch.save(dict(checkpoint_seed=0, cases=cases), os.path.join(OUT, "acoustic_small.pt"))

    # ---- vocoder ----
    gen = checkpoint.build_random_generator(0)
    refg = rl.build_reference_generator()
    refg.remove_weight_norm()
    print("vocoder:", refg.load_state_dict(gen.state_dict(), strict=True))
    g = torch.Generator().manual_seed(5)
    mel_in = torch.randn(2, 80, 24, generator=g).clamp(-2, 2)
    with torch.no_grad():
        wav = refg(mel_in)
    torch.save(dict(checkpoint_seed=0, mel=mel_in, wav=wav), os.path.join(OUT, "vocoder_small.pt"))
    print("vocoder wav", tuple(wav.shape), "absmax %.3f" % wav.abs().max().item())

    # ---- MAS ----
    sma = rl.reference_mas()
    rng = np.random.default_rng(0)
    mas = {}
    for name, (B, Tx, Ty) in {"small": (4, 20, 50), "mid": (6, 57, 130)}.items():
        for kind in ("randn", "ties", "softmax"):
            if kind == "randn":
                v = rng.standard_normal((B, Tx, Ty)).astype(np.float32)
            elif kind == "ties":
                v = rng.integers(0, 3, (B, Tx, Ty)).astype(np.float32)
            else:
                v = torch.softmax(torch.from_numpy(rng.standard_normal((B, Tx, Ty)).astype(np.float32) * 30), dim=1).numpy()
            xl = rng.integers(1, Tx + 1, B)
            yl = np.minimum(np.maximum(rng.integers(Ty // 2, Ty + 1, B), xl), Ty)
            xl[0], yl[0] = Tx, Ty
            mask = ((np.arange(Tx)[None, :, None] < xl[:, None, None]) &
                    (np.arange(Ty)[None, None, :] < yl[:, None, None])).astype(np.float32)
            p1 = sma.maximum_path1(torch.from_numpy(v.copy()), torch.from_numpy(mask)).numpy()
            p2 = sma.maximum_path2(torch.from_numpy(v.copy()), torch.from_numpy(mask)).numpy()
            key = f"{name}_{kind}"
            mas[key + "_value"] = v
            mas[key + "_xlen"] = xl.astype(np.int32)
            mas[key + "_ylen"] = yl.astype(np.int32)
            mas[key + "_path1"] = np.packbits(p1.astype(np.uint8), axis=None)
            mas[key + "_path2"] = np.packbits(p2.astype(np.uint8), axis=None)
    np.savez_compressed(os.path.join(OUT, "mas.npz"), **mas)
    live_case()
    print("done:", os.listdir(OUT))


if __name__ == "__main__":
    import sys
    if sys.argv[1:] == ["live"]:
        live_case()
    else:
        main()
