"""Pin oracle/restate.py (the travelling CPU restatement) to the reference: against the committed
fixtures everywhere, and against the unmodified reference modules where the original source tree is available."""
import os

import pytest
import torch

from oracle import ref_loader, restate
from tests import util


@pytest.mark.parametrize("case", ["a_pred_dur", "b_forced_dur", "c_short"])
def test_restatement_matches_reference_goldens(case):
    g = util.load_golden("acoustic_small.pt")
    model = util.acoustic_model(g["checkpoint_seed"])
    sd = {k: v.detach() for k, v in model.state_dict().items()}
    c = g["cases"][case]
    dist = {k: v.cpu() for k, v in model.distribution.items()}
    out, aux = restate.artsspeech_test(sd, c["tokens"], c["ref_mel"], dist, durations=None if c["durations"] is None
                                       else c["durations"].view(-1), want_aux=True)
    o = c["out"]
    assert torch.equal(aux["pred_dur"].view(-1), o["pred_dur"].view(-1))
    assert (aux["style"] - o["style"]).abs().max().item() < 1e-5
    for k in ("F0", "N", "EMA", "f0_ext", "n_ext", "ema_ext"):
        assert (aux[k] - o[k]).abs().max().item() < 1e-5, k
    assert (out - o["mel"]).abs().max().item() < 5e-5


LIVE_GOLDEN = os.path.join(util.GOLDEN, "live_reference.pt")


@pytest.mark.skipif(not (os.path.isfile(LIVE_GOLDEN) or ref_loader.available()),
                    reason="needs the original ArtSpeech source tree, or tests/golden/live_reference.pt generated "
                           "from it (python -m oracle.make_golden live)")
def test_restatement_matches_live_reference():
    """Checkpoint seed 3: the acoustic model, then the vocoder on the mel the reference's acoustic model produced,
    against the reference's stored outputs, and against the reference itself where its source tree is available."""
    from artspeech_b200 import checkpoint
    from oracle import make_golden
    ours = checkpoint.build_random_artsspeech(3)
    gen = checkpoint.build_random_generator(3)
    tok, mel = make_golden.live_inputs()
    want = []                                              # the reference's (pred_dur, mel, wav)
    if os.path.isfile(LIVE_GOLDEN):
        g = util.load_golden("live_reference.pt")
        assert g["checkpoint_seed"] == 3 and torch.equal(g["tokens"], tok) and torch.equal(g["ref_mel"], mel)
        want.append((g["pred_dur"], g["mel"], g["wav"]))
    if ref_loader.available():
        from oracle import ref_runner
        ref = ref_loader.build_reference_artsspeech(ref_loader.load_distribution())
        ref.load_state_dict(ours.state_dict(), strict=True)      # identical parameter tree
        r = ref_runner.reference_test_step(ref, tok, mel)
        refg = ref_loader.build_reference_generator()
        refg.remove_weight_norm()
        refg.load_state_dict(gen.state_dict(), strict=True)
        with torch.no_grad():
            want.append((r["pred_dur"], r["mel"], refg(r["mel"])))
    out, aux = restate.artsspeech_test(ours.state_dict(), tok, mel, checkpoint.default_distribution(), want_aux=True)
    for pred_dur, ref_mel_out, ref_wav in want:
        assert torch.equal(aux["pred_dur"].view(-1), pred_dur.view(-1))
        assert (out - ref_mel_out).abs().max().item() < 5e-5
        assert (restate.generator_forward(gen.state_dict(), ref_mel_out) - ref_wav).abs().max().item() < 1e-5
