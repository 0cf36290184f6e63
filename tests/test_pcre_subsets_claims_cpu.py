"""The facts the pCRE subset replay (chromo_pcre_subsets, csrc/subsets.cu) rests on, checked on the as-written CPU oracle -
no GPU, no library involved:

  1. setting the rows and columns of an arbitrary set of slots in every resolution's interaction mask gives the logits of
     the gene reassembled without those pCREs (its later slots moved up, dummy slots appended, the block-form mask shrunk,
     as data.py:175-203 would have built it); the set of every pCRE gives the promoter alone;
  2. what the removed slots hold then cannot reach the logits: junk in their features and frequencies changes nothing,
     bit for bit;
  3. the token order does not matter: the variant order of subset_expand_kernel (token 0, the kept tokens, then the
     removed ones) gives the same logits."""
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


def _masked(batch, sets):
    """Row g of `batch` with the rows and columns i + 1 (i in sets[g]) of every interaction mask set."""
    out = _rows(batch, range(len(sets)))
    for g, drop in enumerate(sets):
        for b in BINS:
            m = out["interaction_masks"][b][g, 0]
            for i in drop:
                m[i + 1, :] = True
                m[:, i + 1] = True
    return out


def _rebuilt(batch, sets, k):
    """Row g of `batch` rebuilt without the pCREs of sets[g] (live slots; k[g] of them): the later slots move up, dummy
    slots (zero features, pad mask all set, zero interaction frequency) come last, the block-form interaction mask has
    len(sets[g]) partners less."""
    out = _rows(batch, range(len(sets)))
    for g, drop in enumerate(sets):
        keep = [j for j in range(I) if j not in drop]
        tok = [0] + [j + 1 for j in keep]
        kk = k[g] - len(drop)                                  # partners left
        idx = torch.arange(S)
        for b in BINS:
            x, m = out["pcre_feats"][b], out["pcre_pad_masks"][b]
            x[g] = torch.cat([x[g, keep], torch.zeros_like(x[g, :len(drop)])])
            m[g] = torch.cat([m[g, keep], torch.ones_like(m[g, :len(drop)])])
            out["interaction_masks"][b][g, 0] = ~((idx.view(S, 1) <= kk) & (idx.view(1, S) <= kk))
        f = out["interaction_freq"][g]
        f[:] = torch.nn.functional.pad(f[tok][:, tok], (0, len(drop), 0, len(drop)))
    return out


def _reordered(batch, sets):
    """_masked(batch, sets) with its tokens in the order of subset_expand_kernel: token 0, the kept tokens in their
    order, then the removed ones in their order (features, pad masks, frequencies and interaction masks permuted
    together; a removed slot's features zero)."""
    out = _masked(batch, sets)
    for g, drop in enumerate(sets):
        slots = [j for j in range(I) if j not in drop] + list(drop)
        tok = [0] + [j + 1 for j in slots]
        for b in BINS:
            x, m = out["pcre_feats"][b], out["pcre_pad_masks"][b]
            x[g] = x[g, slots]
            x[g, I - len(drop):] = 0.0
            m[g] = m[g, slots]
            im = out["interaction_masks"][b][g, 0]
            im[:] = im[tok][:, tok].clone()
        f = out["interaction_freq"][g]
        f[:] = f[tok][:, tok].clone()
    return out


def _genes_and_sets():
    batch = synthetic.make_batch(12, ragged=True, seed=31)
    k = batch["n_partners"].tolist()
    genes = [g for g in range(len(k)) if k[g] >= 4][:5]
    assert len(genes) >= 3
    kg = [k[g] for g in genes]
    sets = [
        [0, 2],                                   # non-contiguous, first slot
        [1, kg[1] - 1],                           # second and last live slots
        list(range(kg[2])),                       # every pCRE: the promoter alone
        [kg[3] - 3, kg[3] - 1] if len(genes) > 3 else [1],
        [0, 1, 3][: min(3, kg[-1])] if len(genes) > 4 else [2],
    ][:len(genes)]
    return _rows(batch, genes), sets, kg


def test_masking_a_set_of_slots_is_the_gene_without_those_pcres():
    model = ChromoformerClassifier(7, 128, 128, dict(KWS[0]), dict(KWS[1]), dict(KWS[2]), seed=5)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    genes, sets, k = _genes_and_sets()
    got = _logits(sd, _masked(genes, sets))
    want = _logits(sd, _rebuilt(genes, sets, k))
    assert (got - want).abs().max().item() < 2e-6
    # the promoter alone: every pCRE removed, or a gene built with no pCRE at all
    prom = _rows(genes, [2])
    for b in BINS:
        prom["pcre_feats"][b].zero_()
        prom["pcre_pad_masks"][b].fill_(True)
        prom["interaction_masks"][b][:] = True
        prom["interaction_masks"][b][:, 0, 0, 0] = False
    prom["interaction_freq"].zero_()
    assert (got[2] - _logits(sd, prom)[0]).abs().max().item() < 2e-6
    # and removing pCREs does change the prediction (the checks above are not vacuous)
    assert ((got - _logits(sd, genes)).abs().amax(1) > 1e-4).all()


def test_token_order_of_the_variants_changes_nothing():
    model = ChromoformerClassifier(7, 128, 128, dict(KWS[0]), dict(KWS[1]), dict(KWS[2]), seed=6)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    genes, sets, _ = _genes_and_sets()
    assert (_logits(sd, _reordered(genes, sets)) - _logits(sd, _masked(genes, sets))).abs().max().item() < 2e-6


def test_removed_slot_contents_cannot_reach_the_logits():
    model = ChromoformerClassifier(7, 128, 128, dict(KWS[0]), dict(KWS[1]), dict(KWS[2]), seed=9)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    batch = synthetic.make_batch(4, ragged=False, seed=4)
    sets = [[0, 3], [1, 2, 5, 7], [6], [0, 2, 4, 6]]
    masked = _masked(batch, sets)
    want = _logits(sd, masked)
    gen = torch.Generator().manual_seed(2)
    for g, drop in enumerate(sets):
        for i in drop:
            for b in BINS:
                x = masked["pcre_feats"][b]
                x[g, i] = 50.0 * torch.rand(x[g, i].shape, generator=gen)
            masked["interaction_freq"][g, i + 1, :] = 1e3 * torch.rand(S, generator=gen)
            masked["interaction_freq"][g, :, i + 1] = -1e3
    assert torch.equal(_logits(sd, masked), want)
