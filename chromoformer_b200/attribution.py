"""Input attribution: which histone-mark bins of the promoter and of each pCRE, and which pCRE-promoter interaction
frequencies, drive a prediction.

Both helpers take a batch in the ``forward_batch`` convention (the six forward arguments, dicts keyed by bin size,
as ``synthetic.make_batch`` or the reference's DataLoader produce them) and return
``{"promoter_feats": {b: ...}, "pcre_feats": {b: ...}}`` in the layouts of the inputs ([B,1,n,F] / [B,I,n,F]); with
``freq=True`` also ``"interaction_freq"`` ([B,S,S], S = I + 1).  Without it ``interaction_freq`` is held fixed, not
attributed.  The gradients come from the sm_100a backward (``chromo_backward_inputs``); the parameters are held fixed:
they do not require grad during the call, and nothing is written to ``p.grad``.  The masks are inputs held fixed.
``pcre_scores`` folds a result into one score per pCRE slot.  These are local (gradient) or path (integrated gradients)
approximations; ``pcre_deletion`` gives the exact counterfactual per pCRE: the prediction with that pCRE removed.
``pcre_subsets`` gives the prediction without any set of pCREs, and on top of it ``pcre_shapley`` (credit per pCRE that
sums to logits - promoter only) and ``pcre_interactions`` (the synergy of every pair of pCREs).  ``pcre_occlusion`` and
``occlusion_map`` give the exact counterpart of the saliency maps: the prediction with histone marks removed over a
window of bins.  ``freq_edits`` gives the exact prediction with any interaction frequencies changed, and on top of it
``contact_knockout`` (each pCRE's Hi-C contact set to 0, and every contact: the contact-blind prediction),
``contact_response`` (the prediction against contact strength) and ``contact_shapley`` (credit per contact that sums to
logits - blind): the exact counterparts of the ``freq=True`` attributions.
"""
import contextlib
import math

import numpy as np
import torch

from . import _lib
from .model import _BatchIO

__all__ = ["input_gradients", "integrated_gradients", "pcre_scores", "pcre_deletion", "pcre_subsets", "pcre_shapley",
           "pcre_interactions", "pcre_occlusion", "occlusion_map", "freq_edits", "contact_knockout", "contact_response",
           "contact_shapley"]

_FEATS = ("promoter_feats", "pcre_feats")
_MASKS = ("promoter_pad_masks", "pcre_pad_masks")
_FREQ = "interaction_freq"


def _default_target(model, target):
    # classifier: column 1 (`val_score` is softmax(logits)[:, 1], train.py:322-343); regressor: its one output
    if target is not None:
        return int(target)
    return 1 if int(model._cfg.n_out) >= 2 else 0


def _key(d, b):
    return b if b in d else str(b)


@contextlib.contextmanager
def _parameters_fixed(model):
    saved = [(p, p.requires_grad) for p in model.parameters()]
    try:
        for p, _ in saved:
            p.requires_grad_(False)
        yield
    finally:
        for p, rg in saved:
            p.requires_grad_(rg)


def _to_device(batch, model, bins):
    dev = model.flat_params.device
    out = {}
    for key in _FEATS + _MASKS + ("interaction_masks",):
        out[key] = {b: batch[key][_key(batch[key], b)].to(dev) for b in bins}
    out["interaction_freq"] = batch["interaction_freq"].to(dev)
    return out


def _grads(model, batch, target, bins, freq=False):
    """d logits[:, target].sum() / d features (and d interaction_freq with ``freq``) of a device batch keyed by int bin
    size."""
    leaves = {key: {b: batch[key][b].detach().requires_grad_(True) for b in bins} for key in _FEATS}
    if freq:
        leaves[_FREQ] = batch[_FREQ].detach().requires_grad_(True)
    with torch.enable_grad():
        logits = model.forward_batch({**batch, **leaves})
        flat = [leaves[key][b] for key in _FEATS for b in bins] + ([leaves[_FREQ]] if freq else [])
        g = torch.autograd.grad(logits[:, target].sum(), flat)
    it = iter(g)
    out = {key: {b: next(it) for b in bins} for key in _FEATS}
    if freq:
        out[_FREQ] = next(it)
    return out


def _relabel(out, batch, bins):
    res = {key: {_key(batch[key], b): out[key][b] for b in bins} for key in _FEATS}
    if _FREQ in out:
        res[_FREQ] = out[_FREQ]
    return res


def input_gradients(model, batch, target=None, freq=False):
    """Saliency: the gradient of ``logits[:, target].sum()`` with respect to every feature tensor of ``batch``, and
    with ``freq=True`` with respect to ``interaction_freq`` too.  Genes are independent, so row g of the result is the
    gradient of gene g's own logit.  ``target`` defaults to column 1 for the classifier and 0 for the regressor.  With
    the parameters held fixed and only ``interaction_freq`` asked for, the backward stops after the Regulation
    transformer; asking for the features as well costs what the features alone cost, plus one small kernel."""
    bins = list(model.binsizes)
    t = _default_target(model, target)
    with _parameters_fixed(model):
        out = _grads(model, _to_device(batch, model, bins), t, bins, freq)
    return _relabel(out, batch, bins)


def _centre_rows(m, regions):
    """A pad mask as its centre query row [B, regions, n]: the only row that can influence the logits."""
    if m.dim() == 5:                       # [B, regions, 1, n, n]
        return m[:, :, 0, m.shape[3] // 2, :]
    return m.reshape(m.shape[0], regions, m.shape[-1])


def integrated_gradients(model, batch, target=None, steps=32, baseline=None, chunk=4096, freq=False):
    """Integrated gradients, midpoint rule: with alpha_k = (k + 1/2) / steps,
        IG = (x - x0) * mean_k grad f(x0 + alpha_k (x - x0))
    where f = logits[:, target] and x is the features, or with ``freq=True`` the features and ``interaction_freq``
    moving together along one path (the feature attributions are then those of that joint path, and completeness
    holds over all of them: their sum approximates f(x) - f(x0)).  The masks and interaction masks, and without
    ``freq`` interaction_freq, stay those of ``batch``.  ``baseline`` (same layout as the result) defaults to zero
    features (ln(0 + 1), no reads) and zero interaction frequency.  The steps are stacked along the batch dimension, at
    most ``chunk`` gene evaluations per forward / backward (a training workspace is about 1.7 MB per gene); the pad
    masks are cut to their centre rows before they are replicated."""
    if steps < 1 or chunk < 1:
        raise ValueError("steps and chunk must be >= 1")
    bins = list(model.binsizes)
    t = _default_target(model, target)
    dev_batch = _to_device(batch, model, bins)
    I = int(dev_batch["pcre_feats"][bins[0]].shape[1])
    for key, regions in (("promoter_pad_masks", 1), ("pcre_pad_masks", I)):
        dev_batch[key] = {b: _centre_rows(m, regions) for b, m in dev_batch[key].items()}
    # the inputs on the path, as (key, bin) with bin None for interaction_freq
    path = [(key, b) for key in _FEATS for b in bins] + ([(_FREQ, None)] if freq else [])

    def get(d, key, b):
        return d[key] if b is None else d[key][b]

    x = [get(dev_batch, key, b).float() for key, b in path]
    if baseline is None:
        x0 = [torch.zeros_like(v) for v in x]
    else:
        x0 = [(baseline[key] if b is None else baseline[key][_key(baseline[key], b)]).to(v)
              for (key, b), v in zip(path, x)]
    delta = [v - v0 for v, v0 in zip(x, x0)]
    B = int(x[0].shape[0])
    alphas = [(k + 0.5) / steps for k in range(steps)]
    genes = min(B, chunk)                       # genes per evaluation
    per = max(1, chunk // genes)                # alpha steps per evaluation
    fixed = ("promoter_pad_masks", "pcre_pad_masks", "interaction_masks")
    out = [torch.empty_like(v) for v in x]
    with _parameters_fixed(model):
        for g0 in range(0, B, genes):
            g1 = min(B, g0 + genes)
            acc = [torch.zeros_like(v[g0:g1]) for v in x]
            for k0 in range(0, steps, per):
                ks = alphas[k0:k0 + per]
                sub = {key: {} for key in _FEATS}
                for (key, b), v0, d in zip(path, x0, delta):
                    v = torch.cat([v0[g0:g1] + a * d[g0:g1] for a in ks])
                    if b is None:
                        sub[key] = v
                    else:
                        sub[key][b] = v
                for key in fixed:
                    sub[key] = {b: dev_batch[key][b][g0:g1].repeat((len(ks),) + (1,) * (dev_batch[key][b].dim() - 1))
                                for b in bins}
                if not freq:
                    sub[_FREQ] = dev_batch[_FREQ][g0:g1].repeat(len(ks), 1, 1)
                grads = _grads(model, sub, t, bins, freq)
                n = g1 - g0
                for j, (key, b) in enumerate(path):
                    g = get(grads, key, b)
                    for i in range(len(ks)):        # the steps in order, whatever the chunking
                        acc[j] += g[i * n:(i + 1) * n]
            for j in range(len(path)):
                out[j][g0:g1] = delta[j][g0:g1] * (acc[j] / steps)
    res = {key: {} for key in _FEATS}
    for (key, b), v in zip(path, out):
        v = v.to(get(dev_batch, key, b).dtype)
        if b is None:
            res[key] = v
        else:
            res[key][b] = v
    return _relabel(res, batch, bins)


def pcre_scores(attr):
    """One score per pCRE slot, [B, I], from a result of ``input_gradients`` / ``integrated_gradients``: the sum of the
    slot's ``pcre_feats`` attribution over resolutions, bins and marks, plus, when the result has it, the
    ``interaction_freq`` attribution of its contact with the promoter, [b, 0, i + 1].  Dummy slots score exactly 0."""
    score = None
    for v in attr["pcre_feats"].values():
        s = v.float().sum(dim=(2, 3))
        score = s if score is None else score + s
    if _FREQ in attr:
        f = attr[_FREQ].float()
        score = score + f.reshape(f.shape[0], f.shape[-2], f.shape[-1])[:, 0, 1:]
    return score


def pcre_deletion(model, batch, target=None, chunk=4096, dense=False):
    """In-silico deletion of every pCRE of every gene (``chromo_pcre_deletion``): the exact logits of each gene
    reassembled without each of its pCREs, from one Embedding / Pairwise pass per gene and a batched replay of the
    Regulation transformer and the head.  Returns

        "logits"         [B, n_out]     the ordinary forward (bit-identical to ``forward_batch`` with the same ``dense``)
        "without"        [B, I, n_out]  the logits without pCRE i; on a dummy slot the logits themselves
        "promoter_only"  [B, n_out]     the logits without any pCRE
        "effect"         [B, I]         logits[:, target] - without[:, :, target]: > 0 when the pCRE raises the target
                                        logit; exactly 0.0 on dummy slots

    A slot counts as a pCRE when its token is unmasked in row 0 of some resolution's interaction mask; deleting it means
    setting row and column i + 1 of every resolution's interaction mask.  ``target`` defaults to column 1 for the
    classifier and 0 for the regressor.  At most ``chunk`` genes go to one library call (its workspace holds I + 1
    variants per gene).  ``dense`` is the hint of ``forward_batch``.  Nothing requires grad, nothing touches ``p.grad``."""
    if chunk < 1:
        raise ValueError("chunk must be >= 1")
    bins = list(model.binsizes)
    t = _default_target(model, target)
    dev_batch = _to_device(batch, model, bins)
    B = int(dev_batch["interaction_freq"].shape[0])
    flags = model._precision_flag() | (_lib.F_DENSE if dense else 0)
    parts = []
    with torch.no_grad():
        for g0 in range(0, B, chunk):
            g1 = min(B, g0 + chunk)
            lists = [[dev_batch[key][b][g0:g1] for b in bins]
                     for key in ("promoter_feats", "promoter_pad_masks", "pcre_feats", "pcre_pad_masks", "interaction_masks")]
            io = _BatchIO(model, *lists, dev_batch[_FREQ][g0:g1])
            parts.append(model._launch_deletion(io, flags))
    logits, without, promoter_only = (torch.cat(p) for p in zip(*parts))
    return {"logits": logits, "without": without, "promoter_only": promoter_only,
            "effect": logits[:, t:t + 1] - without[:, :, t]}


# ---- pCRE subsets (chromo_pcre_subsets) ----------------------------------------------------------------------------
_GENE_KEYS = ("promoter_feats", "promoter_pad_masks", "pcre_feats", "pcre_pad_masks", "interaction_masks")
_SUBSET_CHUNK = 65536           # variants per library call: about 3.8 GB of workspace in BF16, 33 GB in FP32


def _live(dev_batch, bins):
    """[B, I] bool on the device: slot i is a pCRE when token i + 1 is unmasked in row 0 of some resolution's
    interaction mask (the definition of ``pcre_deletion``)."""
    shape = dev_batch[_FREQ].shape
    im = torch.stack([dev_batch["interaction_masks"][b].reshape(shape).bool() for b in bins])
    return (~im[:, :, 0, 1:]).any(0)


def _calls(model, dev_batch, bins, var_gene, chunk, dense, launch):
    """logits [B, n_out] and var_logits [V, n_out] on the device for variants of the genes ``var_gene`` (numpy int64,
    non-decreasing, every gene with at least one variant), by library calls ``launch(io, v0, v1, vg, flags)`` over the
    variants [v0, v1), vg their genes as int32 on the device relative to the call's first gene.  One call covers whole
    genes, at most ``chunk`` variants (a gene with more gets a call of its own), so every gene's Embedding / Pairwise
    pass runs once."""
    if chunk < 1:
        raise ValueError("chunk must be >= 1")
    B = int(dev_batch[_FREQ].shape[0])
    counts = np.bincount(var_gene, minlength=B)
    if len(counts) != B or (counts == 0).any():
        raise ValueError("every gene needs at least one variant, and var_gene must lie in [0, B)")
    starts = np.concatenate([[0], np.cumsum(counts)])
    flags = model._precision_flag() | (_lib.F_DENSE if dense else 0)
    dev = model.flat_params.device
    logits, var_logits = [], []
    with torch.no_grad():
        g0 = 0
        while g0 < B:
            g1 = int(np.searchsorted(starts, starts[g0] + chunk, side="right")) - 1
            g1 = min(B, max(g1, g0 + 1))
            v0, v1 = int(starts[g0]), int(starts[g1])
            io = _BatchIO(model, *[[dev_batch[key][b][g0:g1] for b in bins] for key in _GENE_KEYS],
                          dev_batch[_FREQ][g0:g1])
            vg = torch.from_numpy((var_gene[v0:v1] - g0).astype(np.int32)).to(dev)
            lg, vl = launch(io, v0, v1, vg, flags)
            logits.append(lg)
            var_logits.append(vl)
            g0 = g1
    return torch.cat(logits), torch.cat(var_logits)


def _replay(model, dev_batch, bins, var_gene, var_drop, chunk, dense):
    """``_calls`` over ``chromo_pcre_subsets``: variant v drops the pCREs of the bit set var_drop[v] (numpy int64)."""
    dev = model.flat_params.device

    def launch(io, v0, v1, vg, flags):
        return model._launch_subsets(io, vg, torch.from_numpy(var_drop[v0:v1].astype(np.int32)).to(dev), flags)
    return _calls(model, dev_batch, bins, var_gene, chunk, dense, launch)


def pcre_subsets(model, batch, drop, target=None, chunk=_SUBSET_CHUNK, dense=False):
    """The exact logits of every gene without any set of its pCREs (``chromo_pcre_subsets``), from one Embedding /
    Pairwise pass per gene and a batched replay of the Regulation transformer and the head over the variants.

    ``drop`` is bool, [V, I] (the same V sets for every gene) or [B, V, I]: variant v of gene g is the gene without the
    pCREs of slots ``drop[g, v]``.  Dropping a dummy slot (no pCRE, see ``pcre_deletion``) changes nothing; an empty set
    gives the gene itself, the set of every pCRE the promoter alone.  Returns

        "logits"    [B, n_out]      the ordinary forward (bit-identical to ``forward_batch`` with the same ``dense``)
        "variants"  [B, V, n_out]   the logits of each variant
        "value"     [B, V]          variants[..., target], only when ``target`` is given

    At most ``chunk`` variants go to one library call, whole genes at a time (a gene with more variants than ``chunk``
    gets a call of its own).  The replay needs about 58 kB of workspace per variant in BF16 with the default
    configuration (X_in, the last Regulation layer's rows and the fused kernel's parking rows; no Embedding / Pairwise
    buffers) and about 0.5 MB in FP32.  A variant's logits do not depend on the other variants or on ``chunk`` (as for a
    forward, for chunks whose gene counts are on the same side of the 64-row threshold).  Nothing requires grad."""
    bins = list(model.binsizes)
    dev_batch = _to_device(batch, model, bins)
    B, I = (int(n) for n in dev_batch[_FREQ].shape[:2])
    I -= 1
    drop = torch.as_tensor(drop)
    if drop.dtype != torch.bool:
        raise ValueError("drop must be a bool tensor")
    if drop.dim() == 2:
        drop = drop.unsqueeze(0).expand(B, -1, -1)
    if drop.dim() != 3 or drop.shape[0] != B or drop.shape[2] != I or drop.shape[1] < 1:
        raise ValueError(f"drop must be [V, {I}] or [{B}, V, {I}] with V >= 1, got {tuple(drop.shape)}")
    V = int(drop.shape[1])
    bits = (drop.cpu().long() << torch.arange(I)).sum(-1).reshape(-1).numpy()
    logits, var_logits = _replay(model, dev_batch, bins, np.repeat(np.arange(B), V), bits, chunk, dense)
    out = {"logits": logits, "variants": var_logits.view(B, V, -1)}
    if target is not None:
        out["value"] = out["variants"][..., _default_target(model, target)]
    return out


def _shapley_exact(v, k):
    """Exact Shapley values of k players from v [G, 2^k] (float64; column s = the value of the coalition whose bit j
    is set for player j): phi_j = sum over s without j of |s|! (k - |s| - 1)! / k! (v[s + j] - v[s]), accumulated over
    s in increasing order.  [G, k]."""
    w = [math.factorial(n) * math.factorial(k - n - 1) / math.factorial(k) for n in range(k)]
    phi = torch.zeros(v.shape[0], k, dtype=torch.float64)
    for s in range(1 << k):
        js = [j for j in range(k) if not (s >> j) & 1]
        if js:
            phi[:, js] += w[bin(s).count("1")] * (v[:, [s | (1 << j) for j in js]] - v[:, s:s + 1])
    return phi


def _shapley_from_orders(v, order, k):
    """The permutation (Monte-Carlo) estimate of Shapley values from P orders per gene: v [G, P, I + 1] float64, the
    values of the prefixes of each order (entry j: the first j players of the order; entries past k[g] are not read),
    order [G, P, I] the slots in order (the k[g] players first), k [G].  Player order[g, p, j - 1] gets
    v[g, p, j] - v[g, p, j - 1]; the orders are added in turn and averaged, so per order the credits telescope to
    v(all) - v(none).  Slots that are no player get exactly 0.  [G, I]."""
    G, P, I = order.shape
    valid = torch.arange(1, I + 1).view(1, I) <= k.view(G, 1)
    phi = torch.zeros(G, I, dtype=torch.float64)
    for p in range(P):
        d = torch.where(valid, v[:, p, 1:] - v[:, p, :-1], torch.zeros((), dtype=torch.float64))
        phi.scatter_add_(1, order[:, p, :], d)
    return phi / P


def _first_variants(var_gene):
    """The index of each gene's first variant (var_gene non-decreasing, every gene present)."""
    return np.concatenate([[0], np.cumsum(np.bincount(var_gene))[:-1]])


def _shapley_descriptors(live):
    """The variants of exact Shapley values: for each gene (in order) the 2^k subsets T of its k pCREs, variant s keeping
    the pCREs whose bit is set in s (bit j: the j-th pCRE of the gene).  Returns var_gene, var_drop (numpy int64) and,
    per pCRE count k, (k, the genes [G], their pCRE slots [G, k], the variant index of each (gene, s) [G, 2^k])."""
    B, I = live.shape
    k = live.sum(1)
    live_bits = (live.long() << torch.arange(I)).sum(1).numpy()
    pos = torch.argsort((~live).to(torch.int8), dim=1, stable=True)          # the pCREs of each gene first, ascending
    n_var = (1 << k).numpy()
    starts = np.concatenate([[0], np.cumsum(n_var)])
    var_drop = np.zeros(int(starts[-1]), dtype=np.int64)
    groups = []
    for kk in sorted(set(k.tolist())):
        genes = torch.nonzero(k == kk).view(-1)
        sub = np.arange(1 << kk)
        s_bits = (sub.reshape(-1, 1) >> np.arange(kk)) & 1                     # [2^k, k]
        slots = pos[genes, :kk]
        kept = (1 << slots.numpy().astype(np.int64)) @ s_bits.T                # [G, 2^k]
        idx = starts[genes.numpy()].reshape(-1, 1) + sub.reshape(1, -1)
        var_drop[idx] = live_bits[genes.numpy()].reshape(-1, 1) & ~kept
        groups.append((kk, genes, slots, idx))
    return np.repeat(np.arange(B), n_var), var_drop, groups


def _interaction_descriptors(live):
    """The variants of pairwise interactions: for each gene (in order) the candidates () (the gene itself), (i,) and
    (i, j), i < j, whose slots are all pCREs.  Returns var_gene, var_drop (numpy int64), valid [B, n_cand] and the
    pairs in candidate order."""
    B, I = live.shape
    pairs = [(i, j) for i in range(I) for j in range(i + 1, I)]
    cand = [()] + [(i,) for i in range(I)] + pairs
    bits = torch.tensor([sum(1 << i for i in c) for c in cand])
    valid = torch.stack([live[:, list(c)].all(1) if c else torch.ones(B, dtype=torch.bool) for c in cand], 1)
    gene = torch.arange(B).view(B, 1).expand(B, len(cand))
    return gene[valid].numpy(), bits.view(1, -1).expand(B, -1)[valid].numpy(), valid, pairs


def _shapley(model, batch, target, permutations, seed, replay):
    """Shapley values of each gene's live slots, the value of a coalition T being ``logits[target]`` of
    ``replay(dev_batch, bins, var_gene, var_bits)`` (numpy int64 descriptors; bit i of var_bits: slot i is NOT in T).
    Exact over the 2^k subsets, or with ``permutations=P`` the estimate over P seeded orders; combined in FP64 in a fixed
    order.  Returns (shapley [B, I] float64 on the device, logits, the logits of the empty coalition)."""
    bins = list(model.binsizes)
    t = _default_target(model, target)
    dev_batch = _to_device(batch, model, bins)
    live = _live(dev_batch, bins).cpu()                      # (the one host read of the call)
    B, I = live.shape
    k = live.sum(1)
    live_bits = (live.long() << torch.arange(I)).sum(1)
    shapley = torch.zeros(B, I, dtype=torch.float64)
    if permutations is None:
        if int(k.max()) > 12:
            g = int(torch.argmax(k))
            raise ValueError(f"gene {g} has {int(k[g])} pCREs: exact Shapley values need 2^k variants per gene; "
                             "pass permutations= for the sampling estimate")
        var_gene, var_bits, groups = _shapley_descriptors(live)
        logits, var_logits = replay(dev_batch, bins, var_gene, var_bits)
        v = var_logits[:, t].double().cpu().numpy()
        for kk, genes, slots, idx in groups:
            if kk:
                shapley[genes.view(-1, 1), slots] = _shapley_exact(torch.from_numpy(v[idx]), kk)
        none = var_logits[torch.from_numpy(_first_variants(var_gene)).to(var_logits.device)]   # the empty coalition
    else:
        P = int(permutations)
        if P < 1:
            raise ValueError("permutations must be >= 1")
        gen = torch.Generator().manual_seed(int(seed))
        r = torch.rand(B, P, I, generator=gen, dtype=torch.float64)
        order = torch.argsort(torch.where(live.view(B, 1, I), r, torch.full((), 2.0, dtype=torch.float64)), dim=2)
        kept = torch.cat([torch.zeros(B, P, 1, dtype=torch.long), torch.cumsum(1 << order, dim=2)], 2)   # [B, P, I + 1]
        valid = (torch.arange(I + 1).view(1, 1, I + 1) <= k.view(B, 1, 1)).expand(B, P, I + 1)
        bits = live_bits.view(B, 1, 1) & ~kept
        gene = torch.arange(B).view(B, 1, 1).expand(B, P, I + 1)
        logits, var_logits = replay(dev_batch, bins, gene[valid].numpy(), bits[valid].numpy())
        v = torch.zeros(B, P, I + 1, dtype=torch.float64)
        v[valid] = var_logits[:, t].double().cpu()
        shapley = _shapley_from_orders(v, order, k)
        first = torch.nonzero(valid.reshape(-1)).view(-1)      # prefix 0 of order 0 is each gene's first variant
        none = var_logits[torch.searchsorted(first, torch.arange(B) * P * (I + 1)).to(var_logits.device)]
    return shapley.to(logits.device), logits, none


def pcre_shapley(model, batch, target=None, permutations=None, seed=0, chunk=_SUBSET_CHUNK, dense=False):
    """Shapley values of the pCREs of every gene: the players are the gene's pCREs (its live slots, as for
    ``pcre_deletion``), the value of a set T is ``logits[target]`` of the gene with only the pCREs of T kept (from
    ``pcre_subsets``).  A pCRE's value is its average marginal contribution over every order in which the pCREs could be
    added, so redundant pCREs share their credit and cooperating pCREs are not credited twice, and the values of a gene
    sum to v(all) - v(none) = logits[target] - promoter_only[target] (up to the rounding of the FP64 combination).

    Exact by default: every subset of each gene's k pCREs, 2^k variants per gene; a gene with more than 12 pCREs is a
    ValueError (use ``permutations=``).  With ``permutations=P``: the estimate over P random orders per gene (seeded by
    ``seed``), k + 1 prefix variants per order; per order the credits sum exactly to v(all) - v(none).  The values are
    combined in FP64 in a fixed order.  Returns

        "shapley"        [B, I] float64   exactly 0.0 on dummy slots
        "logits"         [B, n_out]       the ordinary forward
        "promoter_only"  [B, n_out]       the logits without any pCRE

    ``target`` defaults to column 1 for the classifier and 0 for the regressor; ``chunk`` and ``dense`` are those of
    ``pcre_subsets``.  Cost: one Embedding / Pairwise pass per gene and the Regulation transformer over the variants; a
    variant keeping m pCREs costs m + 1 tokens on the BF16 path (DESIGN.md 3.5)."""
    def replay(dev_batch, bins, var_gene, var_drop):
        return _replay(model, dev_batch, bins, var_gene, var_drop, chunk, dense)
    shapley, logits, promoter_only = _shapley(model, batch, target, permutations, seed, replay)
    return {"shapley": shapley, "logits": logits, "promoter_only": promoter_only}


def _interactions(f0, fi, fij, pairs, live):
    """Delta_ij = f(N) - f(N without i) - f(N without j) + f(N without i, j) for the live pairs: f0 [G], fi [G, I],
    fij [G, n_pairs] float64 for the pairs (i, j), i < j.  Returns (interaction [G, I, I], exactly symmetric, 0.0 on
    the diagonal and on dead rows / columns; effect [G, I] = f0 - fi, 0.0 on dead slots)."""
    G, I = live.shape
    zero = torch.zeros((), dtype=torch.float64)
    inter = torch.zeros(G, I, I, dtype=torch.float64)
    for c, (i, j) in enumerate(pairs):
        d = torch.where(live[:, i] & live[:, j], f0 - fi[:, i] - fi[:, j] + fij[:, c], zero)
        inter[:, i, j] = d
        inter[:, j, i] = d
    return inter, torch.where(live, f0.view(G, 1) - fi, zero)


def pcre_interactions(model, batch, target=None, chunk=_SUBSET_CHUNK, dense=False):
    """Pairwise interaction effects of the pCREs of every gene, from the 1 + k + k (k - 1) / 2 variants of a gene with
    k pCREs (``pcre_subsets``): with f = logits[target] and N the gene's pCREs,

        Delta_ij = f(N) - f(N without i) - f(N without j) + f(N without i and j)

    the extra effect of removing both over removing each alone: 0 when the two act independently, < 0 when each covers
    for the other (redundant), > 0 when each needs the other (synergy).  Returns

        "interaction"  [B, I, I] float64   exactly symmetric; exactly 0.0 on the diagonal and on dummy slots
        "effect"       [B, I] float64      f(N) - f(N without i) (as ``pcre_deletion``'s); 0.0 on dummy slots
        "logits"       [B, n_out]          the ordinary forward

    f(N) is the replayed gene itself.  ``target``, ``chunk`` and ``dense`` as for ``pcre_shapley``."""
    bins = list(model.binsizes)
    t = _default_target(model, target)
    dev_batch = _to_device(batch, model, bins)
    live = _live(dev_batch, bins).cpu()
    B, I = live.shape
    var_gene, var_drop, valid, pairs = _interaction_descriptors(live)
    logits, var_logits = _replay(model, dev_batch, bins, var_gene, var_drop, chunk, dense)
    v = torch.zeros(B, valid.shape[1], dtype=torch.float64)
    v[valid] = var_logits[:, t].double().cpu()
    inter, effect = _interactions(v[:, 0], v[:, 1:1 + I], v[:, 1 + I:], pairs, live)
    dev = logits.device
    return {"interaction": inter.to(dev), "effect": effect.to(dev), "logits": logits}


# ---- histone-mark occlusion (chromo_pcre_occlusion) ----------------------------------------------------------------
_OCCLUSION_CHUNK = 65536        # variants per library call: about 4.5 GB of workspace in BF16, 31 GB in FP32 (DESIGN.md 3.6)
_FORWARD_CHUNK = 8192           # genes per forward_batch call of the promoter windows
_INT32_MAX = 2 ** 31 - 1


def _int32(a, bad):
    """int64 numpy -> int32, every value outside int32 replaced by ``bad`` (so that it stays invalid on the device)."""
    a = np.asarray(a, dtype=np.int64)
    return np.where((a < -_INT32_MAX - 1) | (a > _INT32_MAX), bad, a).astype(np.int32)


def _mark_bits(marks, V, F):
    """Mark sets as uint32 bit patterns in int32 [V]: from bool [V, F] or from integers (bit m: mark m)."""
    m = torch.as_tensor(marks)
    if m.dtype == torch.bool:
        if m.dim() != 2 or m.shape != (V, F):
            raise ValueError(f"bool marks must be [{V}, {F}], got {tuple(m.shape)}")
        bits = (m.cpu().long() << torch.arange(F)).sum(-1).numpy()
    else:
        bits = m.cpu().long().reshape(-1).numpy()
        if bits.shape[0] != V:
            raise ValueError(f"marks must hold {V} mark sets, got {bits.shape[0]}")
        bits = np.where((bits < 0) | (bits > 0xFFFFFFFF), 0xFFFFFFFF, bits)     # (out of range: invalid on the device)
    return bits.astype(np.uint32).view(np.int32)


def _occlude(model, dev_batch, bins, gene, slot, var_bins, marks, chunk, dense):
    """logits [B, n_out] and var_logits [V, n_out] (descriptor order) on the device from numpy descriptors (gene, slot
    int64 [V], var_bins int64 [V, n_res, 2], marks int32 [V]).  One library call covers whole genes, at most ``chunk``
    variants (a gene with more gets a call of its own), so every gene's Embedding / Pairwise pass runs once.  Descriptors
    of a gene outside [0, B) stay invalid (NaN rows): they go to calls of their own, at most ``chunk`` per call, each over
    gene 0 alone (whose logits there are discarded)."""
    if chunk < 1:
        raise ValueError("chunk must be >= 1")
    B = int(dev_batch[_FREQ].shape[0])
    V = int(gene.shape[0])
    ok = (gene >= 0) & (gene < B)
    bad = np.nonzero(~ok)[0]
    good = np.nonzero(ok)[0]
    order = good[np.argsort(gene[good], kind="stable")]       # the valid descriptors by gene, stable
    starts = np.concatenate([[0], np.cumsum(np.bincount(gene[good], minlength=B))])
    flags = model._precision_flag() | (_lib.F_DENSE if dense else 0)
    dev = model.flat_params.device
    n_out = int(model._cfg.n_out)
    logits, var_logits = [], torch.empty(V, n_out, dtype=torch.float32, device=dev)

    def call(g0, g1, idx, vg):
        io = _BatchIO(model, *[[dev_batch[k][b][g0:g1] for b in bins] for k in _GENE_KEYS], dev_batch[_FREQ][g0:g1])
        if idx.size:
            vs, vb, vm = slot[idx], var_bins[idx], marks[idx]
        else:                                                   # genes without variants: one invalid one, discarded
            vg, vs = np.full(1, -1), np.zeros(1, dtype=np.int64)
            vb, vm = np.zeros((1,) + var_bins.shape[1:], dtype=np.int64), np.zeros(1, dtype=np.int32)
        desc = [torch.from_numpy(a).to(dev) for a in (_int32(vg, -1), _int32(vs, -1), _int32(vb, -1), vm)]
        lg, vl = model._launch_occlusion(io, *desc, flags)
        if idx.size:
            var_logits[torch.from_numpy(idx).to(dev)] = vl
        return lg

    with torch.no_grad():
        for v0 in range(0, len(bad), chunk):
            idx = bad[v0:v0 + chunk]
            call(0, 1, idx, np.full(len(idx), -1))
        g0 = 0
        while g0 < B:
            g1 = int(np.searchsorted(starts, starts[g0] + chunk, side="right")) - 1
            g1 = min(B, max(g1, g0 + 1))
            idx = order[starts[g0]:starts[g1]]
            logits.append(call(g0, g1, idx, gene[idx] - g0))
            g0 = g1
    return torch.cat(logits), var_logits


def pcre_occlusion(model, batch, gene, slot, bins, marks, target=None, chunk=_OCCLUSION_CHUNK, dense=False):
    """The exact logits of genes with histone marks removed over bin ranges of one pCRE (``chromo_pcre_occlusion``).
    Variant v is gene ``gene[v]`` with

        pcre_feats[r][gene[v], slot[v], bins[v, r, 0]:bins[v, r, 1], m] = 0     for every resolution r, every m in marks[v]

    (r in the order of ``model.binsizes``); the masks and interaction_freq stay as they are.  Zero is what the input
    path writes where no read fell (ln(0 + 1)), so a variant is the gene as if those marks had no reads there.  An empty
    range leaves that resolution alone.  ``gene``, ``slot``: ints [V]; ``bins``: ints [V, n_res, 2]; ``marks``: bool
    [V, n_feats] or integer bit sets [V] (bit m: mark m).  A dead slot (no pCRE, see ``pcre_deletion``) gives the gene's
    logits exactly; an invalid descriptor (gene or slot out of range, a range with lo < 0, lo > hi or hi > n_r, a mark
    at or above n_feats) gives a NaN row and leaves the others alone.  Returns

        "logits"    [B, n_out]   the ordinary forward (bit-identical to ``forward_batch`` with the same ``dense``)
        "variants"  [V, n_out]   the logits of each variant, in descriptor order
        "value"     [V]          variants[:, target], only when ``target`` is given

    One Embedding / Pairwise pass per gene, one Pairwise pass over the occluded region per variant, and the Regulation
    transformer and the head over the variants.  At most ``chunk`` variants go to one library call, whole genes at a
    time; descriptors of a gene out of range go to calls of their own.  A variant's logits do not depend on the other
    variants of its call (every occluded region is computed on its own, on the GEMM paths of its gene's pass), nor on
    ``chunk`` as long as every call's gene count B keeps B, B * I and B * (I + 1) on the same side of 64 and, in BF16
    without ``dense``, B * I on the same side of the 897 rows (113 genes at I = 8) from which the gene pass builds its
    ragged plan (a forward's results depend on the same thresholds).  With that plan the gene's own rows come from
    shared key windows, so an empty occlusion matches ``logits`` to BF16 rounding, not bit for bit.  Nothing requires
    grad, nothing touches ``p.grad``."""
    binsizes = list(model.binsizes)
    dev_batch = _to_device(batch, model, binsizes)
    F, NR = int(model._cfg.n_feats), len(binsizes)
    gene = np.asarray(torch.as_tensor(gene).cpu().long().reshape(-1).numpy())
    V = int(gene.shape[0])
    if V < 1:
        raise ValueError("at least one variant is needed")
    slot = torch.as_tensor(slot).cpu().long().reshape(-1).numpy()
    var_bins = torch.as_tensor(bins).cpu().long().numpy()
    if slot.shape[0] != V or var_bins.shape != (V, NR, 2):
        raise ValueError(f"slot must be [{V}] and bins [{V}, {NR}, 2], got {slot.shape} and {var_bins.shape}")
    logits, var_logits = _occlude(model, dev_batch, binsizes, gene, slot, var_bins, _mark_bits(marks, V, F), chunk, dense)
    out = {"logits": logits, "variants": var_logits}
    if target is not None:
        out["value"] = var_logits[:, _default_target(model, target)]
    return out


def _mark_sets(marks, F):
    """bool [M, F] mark sets from "all", "each" or a bool [M, F] list."""
    if isinstance(marks, str):
        if marks == "all":
            return torch.ones(1, F, dtype=torch.bool)
        if marks == "each":
            return torch.eye(F, dtype=torch.bool)
        raise ValueError('marks must be "all", "each" or a bool [M, n_feats] list of mark sets')
    m = torch.as_tensor(marks)
    if m.dtype != torch.bool or m.dim() != 2 or m.shape[1] != F or m.shape[0] < 1:
        raise ValueError(f"mark sets must be bool [M, {F}], got {tuple(m.shape)} {m.dtype}")
    return m.cpu()


def occlusion_map(model, batch, window=1, stride=None, marks="all", target=None, chunk=_OCCLUSION_CHUNK, dense=False):
    """Occlusion map of every region of every gene: the logits with the marks of each mark set removed over each genomic
    window, for the promoter and for every pCRE slot.

    Windows are ``[w0, w0 + window)`` for w0 = 0, stride, 2 stride, ... (``stride`` defaults to ``window``) in units of the
    coarsest bin (n_0 bins per region, the smallest n_r); at resolution r the window covers the bins
    ``[w0 n_r / n_0, (w0 + window) n_r / n_0)``, which needs n_0 to divide every n_r (20 / 80 / 400 for 2 kb / 500 bp /
    100 bp bins).  For a region without centre padding that is exactly the gene with the reads of that genomic interval
    removed before binning; for a padded region (shorter than the window of w_max, centred by data.py) it is a window in
    bin space, and bins under the pad mask carry no information, so occluding only those changes nothing.
    ``marks``: "all" (one set of every mark), "each" (one set per mark) or bool [M, n_feats].  Returns

        "pcre"             [B, I, W, M, n_out]  logits with pCRE slot i occluded (``pcre_occlusion``); on a dummy slot
                                                the logits themselves
        "promoter"         [B, W, M, n_out]     logits with the promoter occluded
        "effect_pcre"      [B, I, W, M]         logits[:, target] - pcre[..., target]; exactly 0.0 on dummy slots
        "effect_promoter"  [B, W, M]            logits[:, target] - promoter[..., target]
        "logits"           [B, n_out]           the ordinary forward
        "windows"          [W, 2]               the windows, in coarsest-bin units

    The pCRE variants replay one Pairwise region each plus the Regulation transformer (``pcre_occlusion``; dummy slots
    are not replayed).  Promoter windows cannot take that route: the promoter's Embedding row is the query of every
    Pairwise layer of its resolution, so occluding promoter bins changes every token of the gene, and such a variant is
    a full forward: those genes are built on the device, occluded, and run through ``forward_batch``, a window and
    mark set at a time.  Occlusion is not additive: the single-mark maps of "each" need not sum to the map of "all".
    ``target`` defaults to column 1 for the classifier and 0 for the regressor.  Nothing requires grad."""
    binsizes = list(model.binsizes)
    t = _default_target(model, target)
    dev_batch = _to_device(batch, model, binsizes)
    F = int(model._cfg.n_feats)
    n = [int(dev_batch["pcre_feats"][b].shape[2]) for b in binsizes]
    n0 = min(n)
    if any(nr % n0 for nr in n):
        raise ValueError(f"the coarsest resolution's {n0} bins must divide every resolution's bins {n}")
    window = int(window)
    stride = window if stride is None else int(stride)
    if window < 1 or stride < 1 or window > n0:
        raise ValueError(f"window must be in [1, {n0}] and stride >= 1")
    w0 = np.arange(0, n0 - window + 1, stride)
    windows = np.stack([w0, w0 + window], 1)                             # [W, 2]
    sets = _mark_sets(marks, F)                                         # [M, F]
    W, M = len(w0), int(sets.shape[0])
    bits = (sets.long() << torch.arange(F)).sum(-1).numpy()             # [M]
    B, S = (int(x) for x in dev_batch[_FREQ].shape[:2])
    I = S - 1
    live = _live(dev_batch, binsizes).cpu().numpy()                     # (the host read of the call)
    rb = np.stack([windows * (nr // n0) for nr in n], 1)                # [W, n_res, 2]
    g, i = np.nonzero(live)                                             # live slots, gene-major
    K = len(g)
    gene = np.repeat(g, W * M)
    slot = np.repeat(i, W * M)
    var_bins = np.tile(np.repeat(rb, M, axis=0), (K, 1, 1))             # [(K W M), n_res, 2]
    vmarks = np.tile(bits, K * W).astype(np.uint32).view(np.int32)
    if K:
        logits, vl = _occlude(model, dev_batch, binsizes, gene, slot, var_bins, vmarks, chunk, dense)
    else:
        logits, vl = _occlude(model, dev_batch, binsizes, np.full(1, -1), np.zeros(1, dtype=np.int64),
                              np.zeros((1, len(n), 2), dtype=np.int64), np.zeros(1, dtype=np.int32), chunk, dense)
        vl = vl[:0]
    n_out = logits.shape[1]
    pcre = logits.view(B, 1, 1, 1, n_out).expand(B, I, W, M, n_out).clone()
    live_t = torch.from_numpy(live).to(logits.device)
    pcre[live_t] = vl.view(K, W, M, n_out)
    promoter = torch.empty(B, W, M, n_out, dtype=torch.float32, device=logits.device)
    with torch.no_grad():
        for w in range(W):
            for m in range(M):
                feats = {}
                for r, b in enumerate(binsizes):
                    x = dev_batch["promoter_feats"][b].clone()
                    lo, hi = (int(v) for v in rb[w, r])
                    x[..., lo:hi, sets[m].to(x.device)] = 0
                    feats[b] = x
                for g0 in range(0, B, _FORWARD_CHUNK):
                    g1 = min(B, g0 + _FORWARD_CHUNK)
                    sub = {k: {b: dev_batch[k][b][g0:g1] for b in binsizes} for k in _GENE_KEYS}
                    sub["promoter_feats"] = {b: feats[b][g0:g1] for b in binsizes}
                    sub[_FREQ] = dev_batch[_FREQ][g0:g1]
                    promoter[g0:g1, w, m] = model.forward_batch(sub, dense=dense)
    return {"pcre": pcre, "promoter": promoter,
            "effect_pcre": logits[:, t].view(B, 1, 1, 1) - pcre[..., t],
            "effect_promoter": logits[:, t].view(B, 1, 1) - promoter[..., t],
            "logits": logits, "windows": torch.from_numpy(windows)}


# ---- interaction-frequency edits (chromo_freq_edits) ---------------------------------------------------------------
def _freq_replay(model, dev_batch, bins, var_gene, var_freq, chunk, dense):
    """``_calls`` over ``chromo_freq_edits``: ``var_freq(v0, v1)`` gives the edits of variants [v0, v1) as float32
    [v1 - v0, S, S] on the device (NaN = keep), built for that call only."""
    def launch(io, v0, v1, vg, flags):
        return model._launch_freq_edits(io, vg, var_freq(v0, v1), flags)
    return _calls(model, dev_batch, bins, var_gene, chunk, dense, launch)


def freq_edits(model, batch, freq, target=None, chunk=_SUBSET_CHUNK, dense=False):
    """The exact logits of every gene with its pCRE-promoter interaction frequencies changed (``chromo_freq_edits``),
    from one Embedding / Pairwise pass per gene and a batched replay of the Regulation transformer and the head over the
    variants (interaction_freq enters only the Regulation attention, as the bias gamma_f * freq).

    ``freq`` is float, [V, S, S] (the same V edits for every gene) or [B, V, S, S], S = I + 1: variant v of gene g is
    the gene with ``interaction_freq[g]`` replaced entry by entry by the entries of ``freq[g, v]`` that are not NaN (NaN
    keeps the gene's value, so an all-NaN edit gives the gene itself).  The contact of pCRE i with the promoter is entry
    (0, i + 1); see ``contact_knockout``, ``contact_response`` and ``contact_shapley``.  An edit with a +-inf entry gives
    a NaN row.  Returns

        "logits"    [B, n_out]      the ordinary forward (bit-identical to ``forward_batch`` with the same ``dense``)
        "variants"  [B, V, n_out]   the logits of each variant
        "value"     [B, V]          variants[..., target], only when ``target`` is given

    ``chunk`` and ``dense`` are those of ``pcre_subsets``; each call's edits are moved to the device for that call only.
    Nothing requires grad."""
    bins = list(model.binsizes)
    dev_batch = _to_device(batch, model, bins)
    B, S = (int(n) for n in dev_batch[_FREQ].shape[:2])
    freq = torch.as_tensor(freq)
    if not freq.is_floating_point():
        raise ValueError("freq must be a float tensor")
    if freq.dim() not in (3, 4) or tuple(freq.shape[-2:]) != (S, S) or freq.shape[-3] < 1 or \
            (freq.dim() == 4 and freq.shape[0] != B):
        raise ValueError(f"freq must be [V, {S}, {S}] or [{B}, V, {S}, {S}] with V >= 1, got {tuple(freq.shape)}")
    V = int(freq.shape[-3])
    dev = model.flat_params.device
    if freq.dim() == 3:
        shared = freq.to(device=dev, dtype=torch.float32)

        def var_freq(v0, v1):
            return shared[torch.arange(v0, v1, device=dev) % V]
    else:
        flat = freq.reshape(B * V, S, S)

        def var_freq(v0, v1):
            return flat[v0:v1].to(device=dev, dtype=torch.float32)
    logits, var_logits = _freq_replay(model, dev_batch, bins, np.repeat(np.arange(B), V), var_freq, chunk, dense)
    out = {"logits": logits, "variants": var_logits.view(B, V, -1)}
    if target is not None:
        out["value"] = out["variants"][..., _default_target(model, target)]
    return out


def _contact_replay(model, dev_batch, bins, var_gene, var_bits, var_value, chunk, dense, relative=False):
    """``_freq_replay`` of contact edits: variant v sets the contact [0, i + 1] of every slot i of the bit set
    var_bits[v] to var_value[v], or with ``relative`` to var_value[v] times the gene's own contact; nothing else
    changes (numpy descriptors)."""
    dev = model.flat_params.device
    freq = dev_batch[_FREQ]
    S = int(freq.shape[1])
    slot_bits = torch.arange(S - 1, device=dev)
    gene_t = torch.from_numpy(np.asarray(var_gene, dtype=np.int64)).to(dev)
    bits_t = torch.from_numpy(np.asarray(var_bits, dtype=np.int64)).to(dev)
    value_t = torch.from_numpy(np.asarray(var_value, dtype=np.float32)).to(dev)

    def var_freq(v0, v1):
        sel = ((bits_t[v0:v1].view(-1, 1) >> slot_bits) & 1).bool()
        value = value_t[v0:v1].view(-1, 1)
        contact = value * freq[gene_t[v0:v1], 0, 1:].float() if relative else value.expand(v1 - v0, S - 1)
        out = torch.full((v1 - v0, S, S), float("nan"), dtype=torch.float32, device=dev)
        out[:, 0, 1:] = torch.where(sel, contact, torch.full((), float("nan"), device=dev))
        return out
    return _freq_replay(model, dev_batch, bins, var_gene, var_freq, chunk, dense)


def contact_knockout(model, batch, target=None, chunk=_SUBSET_CHUNK, dense=False):
    """The exact logits of every gene with the Hi-C contact of each pCRE with the promoter (interaction_freq[g, 0, i + 1],
    the only entry the dataset writes) set to 0, the pCRE's marks kept, and with every contact set to 0 ("contact-blind":
    the prediction without the Hi-C information).  Returns

        "without"       [B, I, n_out]  the logits with the contact of pCRE i set to 0; on a dummy slot the logits
        "blind"         [B, n_out]     the logits with every contact set to 0
        "effect"        [B, I]         logits[:, target] - without[:, :, target]; exactly 0.0 on dummy slots
        "blind_effect"  [B]            logits[:, target] - blind[:, target]
        "logits"        [B, n_out]     the ordinary forward

    ``pcre_deletion``'s effect removes the marks and the contact together; the difference of the two effects is what
    the pCRE contributes beyond its contact.  Dummy slots (no pCRE, see ``pcre_deletion``) run no variant.  ``target``
    defaults to column 1 for the classifier and 0 for the regressor; ``chunk`` and ``dense`` as for ``pcre_subsets``."""
    bins = list(model.binsizes)
    t = _default_target(model, target)
    dev_batch = _to_device(batch, model, bins)
    live = _live(dev_batch, bins).cpu()
    B, I = live.shape
    g, i = (x.numpy() for x in torch.nonzero(live, as_tuple=True))
    live_bits = (live.long() << torch.arange(I)).sum(1).numpy()
    # per gene: one variant per pCRE (slot order), then the blind one
    gene = np.concatenate([g, np.arange(B)])
    bits = np.concatenate([np.int64(1) << i, live_bits])
    blind_row = np.concatenate([np.zeros(len(g), dtype=bool), np.ones(B, dtype=bool)])
    order = np.argsort(gene, kind="stable")
    gene, bits, blind_row = gene[order], bits[order], blind_row[order]
    logits, var_logits = _contact_replay(model, dev_batch, bins, gene, bits, np.zeros(len(gene)), chunk, dense)
    n_out = logits.shape[1]
    blind_t = torch.from_numpy(blind_row).to(logits.device)
    without = logits.view(B, 1, n_out).expand(B, I, n_out).clone()
    without[live.to(logits.device)] = var_logits[~blind_t]
    blind = var_logits[blind_t]
    return {"without": without, "blind": blind, "effect": logits[:, t:t + 1] - without[:, :, t],
            "blind_effect": logits[:, t] - blind[:, t], "logits": logits}


def contact_response(model, batch, values, relative=False, target=None, chunk=_SUBSET_CHUNK, dense=False):
    """Response curves of the prediction against contact strength: for every pCRE i of every gene and every grid value
    ``values[j]``, the exact logits with the contact interaction_freq[g, 0, i + 1] set to ``values[j]``, or with
    ``relative=True`` to ``values[j]`` times the gene's own contact (1.0 gives the gene itself); everything else
    unchanged.  Returns

        "response"  [B, I, G, n_out]   on a dummy slot the logits themselves (no variant is run for it)
        "value"     [B, I, G]          response[..., target]
        "logits"    [B, n_out]         the ordinary forward

    ``target`` defaults to column 1 for the classifier and 0 for the regressor; ``chunk`` and ``dense`` as for
    ``pcre_subsets``."""
    bins = list(model.binsizes)
    t = _default_target(model, target)
    dev_batch = _to_device(batch, model, bins)
    values = np.asarray(torch.as_tensor(values, dtype=torch.float32).reshape(-1).numpy())
    G = len(values)
    if G < 1:
        raise ValueError("values must hold at least one value")
    live = _live(dev_batch, bins).cpu()
    B, I = live.shape
    g, i = (x.numpy() for x in torch.nonzero(live, as_tuple=True))
    # genes without a pCRE get one empty variant (the gene itself, discarded): every gene needs one
    empty = np.nonzero(~live.any(1).numpy())[0]
    gene = np.concatenate([np.repeat(g, G), empty])
    bits = np.concatenate([np.repeat(np.int64(1) << i, G), np.zeros(len(empty), dtype=np.int64)])
    value = np.concatenate([np.tile(values, len(g)), np.zeros(len(empty), dtype=np.float32)])
    order = np.argsort(gene, kind="stable")
    gene, bits, value = gene[order], bits[order], value[order]
    logits, var_logits = _contact_replay(model, dev_batch, bins, gene, bits, value, chunk, dense, relative)
    n_out = logits.shape[1]
    response = logits.view(B, 1, 1, n_out).expand(B, I, G, n_out).clone()
    response[live.to(logits.device)] = var_logits[torch.from_numpy(bits != 0).to(logits.device)].view(len(g), G, n_out)
    return {"response": response, "value": response[..., t], "logits": logits}


def contact_shapley(model, batch, target=None, permutations=None, seed=0, chunk=_SUBSET_CHUNK, dense=False):
    """Shapley values of the Hi-C contacts of every gene: the players are the contacts interaction_freq[g, 0, i + 1] of
    the gene's pCREs (its live slots, as for ``pcre_deletion``), and the value of a set T is ``logits[target]`` with the
    contacts outside T set to 0 (the marks of every pCRE kept).  The values of a gene sum to
    v(all) - v(none) = logits[target] - blind[target] (``contact_knockout``), up to the rounding of the FP64 combination:
    the exact counterpart of ``integrated_gradients(freq=True)`` restricted to the contacts.  Exact by default (2^k
    variants per gene; more than 12 pCREs is a ValueError); ``permutations=P`` gives the seeded estimate over P orders
    per gene, as for ``pcre_shapley``.  Returns

        "shapley"  [B, I] float64   exactly 0.0 on dummy slots
        "logits"   [B, n_out]       the ordinary forward
        "blind"    [B, n_out]       the logits with every contact set to 0

    ``target``, ``chunk`` and ``dense`` as for ``pcre_shapley``."""
    def replay(dev_batch, bins, var_gene, var_bits):
        return _contact_replay(model, dev_batch, bins, var_gene, var_bits, np.zeros(len(var_gene)), chunk, dense)
    shapley, logits, blind = _shapley(model, batch, target, permutations, seed, replay)
    return {"shapley": shapley, "logits": logits, "blind": blind}
