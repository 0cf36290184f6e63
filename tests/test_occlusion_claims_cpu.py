"""The facts the histone-mark occlusion replay (chromo_pcre_occlusion, csrc/occlusion.cu) rests on, checked on the
as-written CPU oracle - no GPU, no library involved:

  1. occluding bins of pCRE i changes X_in row i + 1 only, and only at the resolutions where the range is not empty: the
     Embedding row (token 0) and every other slot's Pairwise row stay bit-identical, so one Pairwise pass over the
     occluded region and the Regulation transformer over the gene's tokens give the occluded gene's logits;
  2. occluding only bins under the pad mask, or an empty set of marks, leaves the logits bit-identical;
  3. for a region without centre padding, zeroing the reads of a 2 kb-aligned interval of the raw depth and binning with
     the input path (bin_and_pad / region_representation) gives exactly the binned region with the mapped bins
     [w0 n_r / n_0, w1 n_r / n_0) zeroed at every resolution."""
import numpy as np
import torch

from _util import BINS, KWS
from chromoformer_b200 import ChromoformerClassifier, synthetic
from oracle import chromoformer_oracle as oracle

I = 8
NB = [40000 // b for b in BINS]


def _model_sd(seed=5):
    m = ChromoformerClassifier(7, 128, 128, dict(KWS[0]), dict(KWS[1]), dict(KWS[2]), seed=seed, i_max=I)
    return {k: v.detach().clone() for k, v in m.state_dict().items()}


def _x_in(sd, batch):
    """X_in per bin size, [B, S, 128]: the Embedding row, then the Pairwise row of every slot (net.py:359-376)."""
    full = synthetic.expand_full_masks(batch)
    out = {}
    with torch.no_grad():
        for b in BINS:
            emb, tss = oracle.embedding_transformer(full["promoter_feats"][b], full["promoter_pad_masks"][b], sd,
                                                    f"embed.{b}.", 2)
            pw = oracle.pairwise_interaction_transformer(emb, full["pcre_feats"][b], full["pcre_pad_masks"][b], sd,
                                                         f"pairwise_interaction.{b}.", 2)
            out[b] = torch.cat([tss, pw], 1)
    return out


def _logits(sd, batch):
    with torch.no_grad():
        return oracle.chromoformer_forward(sd, *synthetic.forward_args(synthetic.expand_full_masks(batch)))


def _copy(batch):
    return {k: ({b: t.clone() for b, t in v.items()} if isinstance(v, dict) else v.clone())
            for k, v in batch.items() if k in synthetic.FORWARD_KEYS}


def test_only_the_occluded_row_changes():
    sd = _model_sd()
    batch = synthetic.make_batch(3, ragged=False, seed=7)
    base = _x_in(sd, batch)
    for g, i, ranges, marks in ((0, 2, [(3, 9), (12, 36), (60, 180)], [1, 4]),
                                (1, 7, [(0, 0), (0, 80), (0, 0)], [0, 1, 2, 3, 4, 5, 6]),
                                (2, 0, [(19, 20), (0, 0), (399, 400)], [6])):
        occ = _copy(batch)
        for (lo, hi), b in zip(ranges, BINS):
            for m in marks:
                occ["pcre_feats"][b][g, i, lo:hi, m] = 0
        got = _x_in(sd, occ)
        for (lo, hi), b in zip(ranges, BINS):
            other = torch.ones(3, I + 1, dtype=torch.bool)
            other[g, i + 1] = False
            assert torch.equal(got[b][other], base[b][other]), (g, i, b)
            changed = not torch.equal(got[b][g, i + 1], base[b][g, i + 1])
            assert changed == (hi > lo), (g, i, b)
        # the replay's composition: the occluded region's Pairwise row spliced into the gene's X_in
        spliced = {b: base[b].clone() for b in BINS}
        for b in BINS:
            spliced[b][g, i + 1] = got[b][g, i + 1]
            assert torch.equal(spliced[b], got[b])


def test_pad_bins_and_empty_mark_sets_change_nothing():
    sd = _model_sd(seed=9)
    batch = synthetic.make_batch(6, ragged=True, seed=3, full_masks=False)
    want = _logits(sd, batch)
    occ = _copy(batch)
    for b in BINS:
        x, m = occ["pcre_feats"][b], occ["pcre_pad_masks"][b]
        pad = m.reshape(x.shape[0], I, -1, x.shape[2])
        pad = pad[:, :, pad.shape[2] // 2].bool()                 # [B, I, n]: the centre rows
        x[pad] = 0.0                                             # every mark, every padded bin of every region
    assert torch.equal(_logits(sd, occ), want)
    # an empty mark set over a whole region is no change at all (the same tensors)
    assert torch.equal(_logits(sd, _copy(batch)), want)


def test_aligned_window_equals_reads_removed_before_binning():
    rng = np.random.default_rng(11)
    raw = rng.gamma(0.6, 3.0, size=(7, 40000)).astype(np.float16)
    for w0, w1, marks in ((0, 1, [0]), (4, 9, [1, 3, 6]), (19, 20, list(range(7))), (7, 8, [2])):
        cut = raw.copy()
        cut[marks, w0 * 2000:w1 * 2000] = 0
        for b, n in zip(BINS, NB):
            full, left, n_bins, _ = oracle.region_representation(raw, b, n)
            assert left == 0 and n_bins == n                   # no centre padding
            got, _, _, _ = oracle.region_representation(cut, b, n)
            want = full.copy()
            want[np.ix_(marks, np.arange(w0 * n // NB[0], w1 * n // NB[0]))] = 0
            assert np.array_equal(got, want), (w0, w1, b)
