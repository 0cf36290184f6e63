"""Feature attribution: which histone-mark bins of the promoter and of each pCRE drive a prediction.

Both helpers take a batch in the ``forward_batch`` convention (the six forward arguments, dicts keyed by bin size,
as ``synthetic.make_batch`` or the reference's DataLoader produce them) and return
``{"promoter_feats": {b: ...}, "pcre_feats": {b: ...}}`` in the layouts of the inputs ([B,1,n,F] / [B,I,n,F]).
The gradients come from the sm_100a backward (``chromo_backward_inputs``); the parameters are held fixed: they do not
require grad during the call, and nothing is written to ``p.grad``.  The masks and ``interaction_freq`` are inputs
held fixed, not attributed.
"""
import contextlib

import torch

__all__ = ["input_gradients", "integrated_gradients"]

_FEATS = ("promoter_feats", "pcre_feats")
_MASKS = ("promoter_pad_masks", "pcre_pad_masks")


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


def _grads(model, batch, target, bins):
    """d logits[:, target].sum() / d features of a device batch keyed by int bin size."""
    leaves = {key: {b: batch[key][b].detach().requires_grad_(True) for b in bins} for key in _FEATS}
    with torch.enable_grad():
        logits = model.forward_batch({**batch, **leaves})
        flat = [leaves[key][b] for key in _FEATS for b in bins]
        g = torch.autograd.grad(logits[:, target].sum(), flat)
    it = iter(g)
    return {key: {b: next(it) for b in bins} for key in _FEATS}


def _relabel(out, batch, bins):
    return {key: {_key(batch[key], b): out[key][b] for b in bins} for key in _FEATS}


def input_gradients(model, batch, target=None):
    """Saliency: the gradient of ``logits[:, target].sum()`` with respect to every feature tensor of ``batch``.  Genes
    are independent, so row g of the result is the gradient of gene g's own logit.  ``target`` defaults to column 1
    for the classifier and 0 for the regressor."""
    bins = list(model.binsizes)
    t = _default_target(model, target)
    with _parameters_fixed(model):
        out = _grads(model, _to_device(batch, model, bins), t, bins)
    return _relabel(out, batch, bins)


def _centre_rows(m, regions):
    """A pad mask as its centre query row [B, regions, n]: the only row that can influence the logits."""
    if m.dim() == 5:                       # [B, regions, 1, n, n]
        return m[:, :, 0, m.shape[3] // 2, :]
    return m.reshape(m.shape[0], regions, m.shape[-1])


def integrated_gradients(model, batch, target=None, steps=32, baseline=None, chunk=4096):
    """Integrated gradients over the features, midpoint rule: with alpha_k = (k + 1/2) / steps,
        IG = (x - x0) * mean_k grad f(x0 + alpha_k (x - x0))
    where f = logits[:, target] and the masks, interaction masks and interaction_freq stay those of ``batch``.
    ``baseline`` (same layout as the result) defaults to zero features: ln(0 + 1), no reads.  The steps are stacked
    along the batch dimension, at most ``chunk`` gene evaluations per forward / backward (a training workspace is
    about 1.7 MB per gene); the pad masks are cut to their centre rows before they are replicated."""
    if steps < 1 or chunk < 1:
        raise ValueError("steps and chunk must be >= 1")
    bins = list(model.binsizes)
    t = _default_target(model, target)
    dev_batch = _to_device(batch, model, bins)
    I = int(dev_batch["pcre_feats"][bins[0]].shape[1])
    for key, regions in (("promoter_pad_masks", 1), ("pcre_pad_masks", I)):
        dev_batch[key] = {b: _centre_rows(m, regions) for b, m in dev_batch[key].items()}
    x = {key: {b: dev_batch[key][b].float() for b in bins} for key in _FEATS}
    if baseline is None:
        x0 = {key: {b: torch.zeros_like(x[key][b]) for b in bins} for key in _FEATS}
    else:
        x0 = {key: {b: baseline[key][_key(baseline[key], b)].to(x[key][b]) for b in bins} for key in _FEATS}
    delta = {key: {b: x[key][b] - x0[key][b] for b in bins} for key in _FEATS}
    B = int(x["promoter_feats"][bins[0]].shape[0])
    alphas = [(k + 0.5) / steps for k in range(steps)]
    genes = min(B, chunk)                       # genes per evaluation
    per = max(1, chunk // genes)                # alpha steps per evaluation
    fixed = ("promoter_pad_masks", "pcre_pad_masks", "interaction_masks")
    out = {key: {b: torch.empty_like(x[key][b]) for b in bins} for key in _FEATS}
    with _parameters_fixed(model):
        for g0 in range(0, B, genes):
            g1 = min(B, g0 + genes)
            acc = {key: {b: torch.zeros_like(x[key][b][g0:g1]) for b in bins} for key in _FEATS}
            for k0 in range(0, steps, per):
                ks = alphas[k0:k0 + per]
                sub = {key: {b: torch.cat([x0[key][b][g0:g1] + a * delta[key][b][g0:g1] for a in ks]) for b in bins}
                       for key in _FEATS}
                for key in fixed:
                    sub[key] = {b: dev_batch[key][b][g0:g1].repeat((len(ks),) + (1,) * (dev_batch[key][b].dim() - 1))
                                for b in bins}
                sub["interaction_freq"] = dev_batch["interaction_freq"][g0:g1].repeat(len(ks), 1, 1)
                grads = _grads(model, sub, t, bins)
                n = g1 - g0
                for key in _FEATS:
                    for b in bins:
                        for i in range(len(ks)):        # the steps in order, whatever the chunking
                            acc[key][b] += grads[key][b][i * n:(i + 1) * n]
            for key in _FEATS:
                for b in bins:
                    out[key][b][g0:g1] = delta[key][b][g0:g1] * (acc[key][b] / steps)
    dtype = {key: {b: dev_batch[key][b].dtype for b in bins} for key in _FEATS}
    out = {key: {b: out[key][b].to(dtype[key][b]) for b in bins} for key in _FEATS}
    return _relabel(out, batch, bins)
