"""The facts the in-silico pCRE deletion (chromo_pcre_deletion, csrc/deletion.cu) rests on, checked on the as-written CPU
oracle - no GPU, no library involved:

  1. masking row and column i + 1 of every resolution's interaction mask gives the logits of the gene reassembled without
     pCRE i (its later slots moved up one place, a dummy slot appended, as data.py:175-203 would have built it);
  2. what the deleted slot holds then cannot reach the logits: junk in its features changes nothing, bit for bit."""
import torch

from _util import BINS, KWS
from chromoformer_b200 import ChromoformerClassifier, synthetic
from oracle import chromoformer_oracle as oracle

I, S = 8, 9


def _logits(sd, batch):
    with torch.no_grad():
        return oracle.chromoformer_forward(sd, *synthetic.forward_args(synthetic.expand_full_masks(batch)))


def _rows(batch, idx):
    idx = torch.as_tensor(idx)
    return {key: ({b: t[idx].clone() for b, t in v.items()} if isinstance(v, dict) else v[idx].clone())
            for key, v in batch.items() if key in synthetic.FORWARD_KEYS}


def _masked(batch, slots):
    """Row g of `batch` with row and column slots[g] + 1 of every interaction mask set."""
    out = _rows(batch, range(len(slots)))
    for g, i in enumerate(slots):
        for b in BINS:
            m = out["interaction_masks"][b][g, 0]
            m[i + 1, :] = True
            m[:, i + 1] = True
    return out


def _rebuilt(batch, slots):
    """Row g of `batch` rebuilt without pCRE slots[g]: the later slots move up, a dummy slot (zero features, pad mask all
    set, zero interaction frequency) comes last, the block-form interaction mask has one partner less."""
    out = _rows(batch, range(len(slots)))
    for g, i in enumerate(slots):
        keep = [j for j in range(I) if j != i]
        tok = [0] + [j + 1 for j in keep]
        for b in BINS:
            x, m = out["pcre_feats"][b], out["pcre_pad_masks"][b]
            x[g] = torch.cat([x[g, keep], torch.zeros_like(x[g, :1])])
            m[g] = torch.cat([m[g, keep], torch.ones_like(m[g, :1])])
            im = out["interaction_masks"][b][g, 0]
            k = int((~im[0, 1:]).sum()) - 1                       # partners left
            idx = torch.arange(S)
            inside = (idx.view(S, 1) <= k) & (idx.view(1, S) <= k)
            im[:] = ~inside
        f = out["interaction_freq"][g]
        f[:] = torch.nn.functional.pad(f[tok][:, tok], (0, 1, 0, 1))
    return out


def test_masking_a_slot_is_the_gene_without_that_pcre():
    model = ChromoformerClassifier(7, 128, 128, dict(KWS[0]), dict(KWS[1]), dict(KWS[2]), seed=5)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    batch = synthetic.make_batch(8, ragged=True, seed=31)
    k = batch["n_partners"].tolist()
    # every live slot of the first genes with at least two pCREs: first, middle and last slots, different counts
    pairs = [(g, i) for g in range(len(k)) if k[g] >= 2 for i in range(k[g])][:12]
    assert len({g for g, _ in pairs}) >= 2 and any(i == k[g] - 1 for g, i in pairs) and any(i == 0 for _, i in pairs)
    genes = _rows(batch, [g for g, _ in pairs])
    slots = [i for _, i in pairs]
    got = _logits(sd, _masked(genes, slots))
    want = _logits(sd, _rebuilt(genes, slots))
    assert (got - want).abs().max().item() < 2e-6
    # and deleting a pCRE does change the prediction (the check above is not vacuous)
    assert (got - _logits(sd, genes)).abs().max().item() > 1e-4


def test_deleted_slot_contents_cannot_reach_the_logits():
    model = ChromoformerClassifier(7, 128, 128, dict(KWS[0]), dict(KWS[1]), dict(KWS[2]), seed=9)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    batch = synthetic.make_batch(4, ragged=False, seed=4)
    slots = [0, 3, 5, 7]
    masked = _masked(batch, slots)
    want = _logits(sd, masked)
    gen = torch.Generator().manual_seed(2)
    for g, i in enumerate(slots):
        for b in BINS:
            x = masked["pcre_feats"][b]
            x[g, i] = 50.0 * torch.rand(x[g, i].shape, generator=gen)
        masked["interaction_freq"][g, 0, i + 1] = 1e3
    assert torch.equal(_logits(sd, masked), want)
