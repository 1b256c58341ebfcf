"""SURVEY.md §8b: "training branches delegate to the original PyTorch code".  Running the original code needs the
original source tree (ARTSPEECH_REFERENCE); without a delegate, and when attaching one, the module is checked
everywhere."""
import random

import numpy as np
import pytest
import torch

from oracle import ref_loader


def test_training_steps_need_a_delegate_that_shares_the_parameters():
    from artspeech_b200 import checkpoint
    ours = checkpoint.build_random_artsspeech(4)
    keys_before = list(ours.state_dict().keys())
    for step in ("first", "second"):
        with pytest.raises(NotImplementedError):
            ours([None] * 7, None, None, step=step)
    # a module with the reference's parameter tree (our own class has the same state_dict layout)
    stand_in = checkpoint.build_random_artsspeech(5)
    ours.attach_training_delegate(stand_in)
    assert list(ours.state_dict().keys()) == keys_before                       # the delegate is not a sub-module
    own = dict(ours.named_parameters())
    assert all(p is own[n] for n, p in stand_in.named_parameters())             # every parameter is the same object
    own_b = dict(ours.named_buffers())
    assert all(b is own_b[n] for n, b in stand_in.named_buffers() if n in own_b)


@pytest.mark.reference
@pytest.mark.skipif(not ref_loader.available(), reason="needs the original ArtSpeech source tree")
def test_training_steps_run_the_reference_code_on_shared_parameters():
    from artspeech_b200 import checkpoint
    dist = ref_loader.load_distribution()
    ours = checkpoint.build_random_artsspeech(4, dist)
    keys_before = list(ours.state_dict().keys())
    with pytest.raises(NotImplementedError):
        ours([None] * 7, None, None, step="first")
    ref = ref_loader.build_reference_artsspeech(dist)
    ours.attach_training_delegate(ref)
    assert list(ours.state_dict().keys()) == keys_before                       # the delegate is not a sub-module
    own = dict(ours.named_parameters())
    shared = [n for n, p in ref.named_parameters() if p is own.get(n)]
    assert len(shared) == len(own) == len(list(ref.named_parameters()))         # every parameter is the same object

    g = torch.Generator().manual_seed(2)
    B, Tt, Tm = 2, 14, 192
    texts = torch.randint(1, 178, (B, Tt), generator=g)
    mels = torch.randn(B, 80, Tm, generator=g) * 0.5
    attn = torch.softmax(torch.randn(B, Tt, Tm // 2, generator=g), dim=1)
    mono = torch.zeros(B, Tt, Tm // 2)
    mono[:, torch.arange(Tm // 2) * Tt // (Tm // 2), torch.arange(Tm // 2)] = 1.0
    batch = [texts, torch.tensor([Tt, Tt]), mels, torch.tensor([Tm, Tm]), None, None, None]

    def run(module, step):
        random.seed(0); np.random.seed(0); torch.manual_seed(0)
        return module(batch, attn, mono, step, "train", 0)

    ref.train(); ours.train()
    sd0 = {k: v.clone() for k, v in ours.state_dict().items()}
    for step in ("first", "second"):
        a = run(ours, step)
        ours.load_state_dict(sd0)      # train-mode spectral norm power-iterates its (shared) u / v buffers in place
        b = run(ref, step)
        ours.load_state_dict(sd0)
        flat = lambda o: [t for x in o for t in (x if isinstance(x, (list, tuple)) else [x])]
        for x, y in zip(flat(a), flat(b)):
            assert torch.equal(x, y), step
    # gradients of the reference's training graph land on OUR parameters
    out = run(ours, "first")
    (out[0] - out[1]).abs().mean().backward()
    assert own["decoder.to_out.0.weight_v"].grad is not None and own["text_encoder.emb.weight"].grad is not None
