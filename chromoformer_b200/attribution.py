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
"""
import contextlib

import torch

from . import _lib
from .model import _BatchIO

__all__ = ["input_gradients", "integrated_gradients", "pcre_scores", "pcre_deletion"]

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
