"""The two facts the ragged plan (csrc/ragged.cu, DESIGN.md §3.3) rests on, checked on the as-written CPU oracle (which
computes every bin of every slot, as the reference does) - no GPU, no plan involved:

  1. what lies under a pad mask cannot influence the logits as long as the region keeps one unmasked bin
     (modules.py:160-166: masked_fill(-1e9) -> softmax gives exactly 0 in FP32);
  2. with the block-form interaction mask of data.py:200-203, NOTHING of a dummy pCRE slot can influence the logits: neither its
     features nor its pad mask nor its interaction_freq entry.

Both are asserted bit-for-bit: the plan's eliminations are exact, not approximate."""
import numpy as np
import pytest
import torch

from _util import KWS, golden, import_reference, reference_available
from chromoformer_b200 import ChromoformerClassifier, ChromoformerRegressor, synthetic
from oracle import chromoformer_oracle as oracle


def _logits(sd, batch):
    with torch.no_grad():
        return oracle.chromoformer_forward(sd, *synthetic.forward_args(synthetic.expand_full_masks(batch)))


def _perturbed(batch):
    """The same genes with junk under every pad mask of a live slot and junk everywhere in the dummy slots."""
    k = batch["n_partners"]

    gen = torch.Generator().manual_seed(1)
    other = {key: ({b: t.clone() for b, t in v.items()} if isinstance(v, dict) else v.clone()) for key, v in batch.items()}
    live = torch.arange(8).view(1, 8) < k.view(-1, 1)                        # [B, 8] real pCRE slots
    for b in (2000, 500, 100):
        x, m = other["pcre_feats"][b], other["pcre_pad_masks"][b]            # [B,8,n,7], [B,8,n] (True = padded)
        junk = 5.0 * torch.rand(x.shape, generator=gen)
        # 1. live slots: anything under the pad mask
        under = (m & live.unsqueeze(2)).unsqueeze(3)
        x[:] = torch.where(under, junk, x)
        # 2. dummy slots: features everywhere, and an arbitrary pad mask
        dead = (~live).view(-1, 8, 1, 1)
        x[:] = torch.where(dead, junk, x)
        m[:] = torch.where((~live).unsqueeze(2), torch.rand(m.shape, generator=gen) < 0.5, m)
    f = other["interaction_freq"]
    dead_tok = torch.arange(9).view(1, 9) > k.view(-1, 1)                    # tokens of dummy slots
    f[:] = torch.where(dead_tok.unsqueeze(1) | dead_tok.unsqueeze(2), 3.0 * torch.rand(f.shape, generator=gen), f)
    return other


def test_masked_bins_and_dummy_slots_cannot_reach_the_logits():
    model = ChromoformerClassifier(7, 128, 128, dict(KWS[0]), dict(KWS[1]), dict(KWS[2]), seed=5)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    batch = synthetic.make_batch(6, ragged=True, seed=77)
    k = batch["n_partners"]
    assert (k < 8).any() and (k > 0).any()
    assert torch.equal(_logits(sd, _perturbed(batch)), _logits(sd, batch))


@pytest.mark.parametrize("tag", ["clf", "reg"])
def test_junk_batch_gives_the_stored_reference_logits(tag):
    """tests/golden/train_golden.npz holds the unmodified reference's logits of its seed-123 models on the seed-7 ragged
    batch (genes with dummy pCRE slots and padded bins).  The oracle fed the same genes with junk under every pad mask and
    in every dummy slot must reproduce them."""
    g = golden("train_golden.npz")
    batch = synthetic.make_batch(6, ragged=True, seed=7)
    chk = np.array([batch["pcre_feats"][100].double().sum().item(), batch["interaction_freq"].double().sum().item(),
                    float(batch["n_partners"].sum())])
    if not np.allclose(chk, g["input_checksum"], rtol=0, atol=1e-9):
        pytest.skip("torch RNG stream differs from the one the fixture was generated with")
    assert (batch["n_partners"] < 8).any()
    cls = ChromoformerClassifier if tag == "clf" else ChromoformerRegressor
    model = cls(7, 128, 128, dict(KWS[0]), dict(KWS[1]), dict(KWS[2]), seed=123)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    assert np.abs(_logits(sd, _perturbed(batch)).numpy() - g[f"{tag}_logits"]).max() < 2e-6


@pytest.mark.skipif(not reference_available(), reason="upstream chromoformer checkout not supplied ($CHROMOFORMER_REF)")
def test_same_facts_on_the_unmodified_reference():
    """The reference's own forward (imported from $CHROMOFORMER_REF, CPU) gives identical logits for the two batches."""
    net, _ = import_reference()
    ref = net.ChromoformerClassifier(7, 128, 128, dict(KWS[0]), dict(KWS[1]), dict(KWS[2]), seed=5).eval()
    batch = synthetic.make_batch(6, ragged=True, seed=77)
    assert (batch["n_partners"] < 8).any()
    with torch.no_grad():
        want = ref(*synthetic.forward_args(synthetic.expand_full_masks(batch)))
        got = ref(*synthetic.forward_args(synthetic.expand_full_masks(_perturbed(batch))))
    assert torch.equal(got, want)
