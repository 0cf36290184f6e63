"""Gradients with respect to the input features (chromo_backward_inputs through _ChromoFunction) and the attribution
helpers, against autograd over the oracle with the feature tensors as leaves.  FP32 tolerance: per-tensor max-abs error
<= 2e-4 of that tensor's max-abs oracle gradient (the parameter yardstick of test_training_gpu.py)."""
import pytest
import torch

from _util import KWS
from chromoformer_b200 import Chromoformer, ChromoformerClassifier, ChromoformerRegressor, _lib, synthetic
from chromoformer_b200.attribution import input_gradients, integrated_gradients
from oracle import chromoformer_oracle as oracle

pytestmark = pytest.mark.gpu
REL = 2e-4
BINS = (2000, 500, 100)
FEATS = ("promoter_feats", "pcre_feats")


def _mk(cls, seed=11):
    return cls(7, 128, 128, dict(KWS[0]), dict(KWS[1]), dict(KWS[2]), seed=seed)


def _sd(model):
    return {k: v.detach().clone() for k, v in model.named_parameters()}


def _oracle_feature_grads(sd, batch, objective):
    """autograd.grad(objective(logits), features) over the oracle; returns (logits, {key: {b: grad}})."""
    args = synthetic.forward_args(batch)
    leaves = {key: {b: t.detach().clone().requires_grad_(True) for b, t in batch[key].items()} for key in FEATS}
    args[0], args[2] = leaves["promoter_feats"], leaves["pcre_feats"]
    logits = oracle.chromoformer_forward(sd, *args)
    flat = [leaves[key][b] for key in FEATS for b in BINS]
    g = iter(torch.autograd.grad(objective(logits), flat))
    return logits.detach(), {key: {b: next(g) for b in BINS} for key in FEATS}


def _leaves(batch, dev="cuda"):
    args = synthetic.forward_args(batch, dev)
    leaves = {key: {b: args[i][b].clone().requires_grad_(True) for b in BINS} for i, key in ((0, FEATS[0]), (2, FEATS[1]))}
    args[0], args[2] = leaves["promoter_feats"], leaves["pcre_feats"]
    return args, leaves


def _flat_list(leaves):
    return [leaves[key][b] for key in FEATS for b in BINS]


def _max_rel(got, want):
    return (got.detach().cpu().float() - want).abs().max().item() / max(want.abs().max().item(), 1e-12)


@pytest.mark.parametrize("tag,ragged,i_max,n", [("reg", True, 8, 6), ("clf", False, 8, 3), ("reg", True, 16, 2)])
def test_feature_gradients_vs_oracle(tag, ragged, i_max, n):
    """loss.backward() with the features requiring grad: feature and parameter gradients in one pass."""
    cls = ChromoformerRegressor if tag == "reg" else ChromoformerClassifier
    model = _mk(cls)
    sd = _sd(model)
    batch = synthetic.make_batch(n, i_max=i_max, ragged=ragged, full_masks=True, seed=21, stress=True)
    target = batch["labels_reg"].view(-1, 1) if tag == "reg" else batch["labels_clf"]
    crit = torch.nn.MSELoss() if tag == "reg" else torch.nn.CrossEntropyLoss()
    logits_o, dx_o = _oracle_feature_grads(sd, batch, lambda lg: crit(lg, target))
    _, _, grads_o = oracle.forward_backward(sd, synthetic.forward_args(batch), target, tag == "reg")
    model.cuda().train()
    plain = model(*synthetic.forward_args(batch, "cuda")).detach()
    model.zero_grad(set_to_none=True)
    args, leaves = _leaves(batch)
    out = model(*args)
    crit(out, target.cuda()).backward()
    assert torch.equal(out.detach(), plain)
    assert (out.detach().cpu() - logits_o).abs().max().item() < 5e-5
    for key in FEATS:
        for b in BINS:
            g = leaves[key][b].grad
            assert g is not None and g.shape == leaves[key][b].shape and g.dtype == torch.float32
            err = _max_rel(g, dx_o[key][b])
            assert err < REL, (key, b, err)
    for name, p in model.named_parameters():
        if grads_o[name] is None:
            assert p.grad is None, name
            continue
        assert _max_rel(p.grad, grads_o[name]) < REL, name


@pytest.mark.parametrize("tag,n", [("reg", 64), ("clf", 70)])
def test_bf16_feature_gradients_vs_oracle(tag, n):
    """CHROMO_F_BF16 training workspace: the yardstick of test_bf16_training_step_gradients_vs_oracle (cosine with the
    FP32 oracle >= 0.99, relative L2 within 2 x what BF16 operands do to the oracle + 0.02)."""
    cls = ChromoformerRegressor if tag == "reg" else ChromoformerClassifier
    model = _mk(cls)
    sd = _sd(model)
    batch = synthetic.make_batch(n, ragged=True, full_masks=False, seed=21)
    full = synthetic.expand_full_masks(batch)
    target = batch["labels_reg"].view(-1, 1) if tag == "reg" else batch["labels_clf"]
    crit = torch.nn.MSELoss() if tag == "reg" else torch.nn.CrossEntropyLoss()
    _, dx_o = _oracle_feature_grads(sd, full, lambda lg: crit(lg, target))
    with oracle.bf16_operands():
        _, dx_e = _oracle_feature_grads(sd, full, lambda lg: crit(lg, target))
    model.cuda().train()
    model.precision = "bf16"
    args, leaves = _leaves(batch)
    out = model(*args)
    dx = torch.autograd.grad(crit(out, target.cuda()), _flat_list(leaves))
    g0 = torch.cat([dx_o[key][b].flatten().double() for key in FEATS for b in BINS])
    ge = torch.cat([dx_e[key][b].flatten().double() for key in FEATS for b in BINS])
    g2 = torch.cat([g.detach().cpu().flatten().double() for g in dx])
    cos = torch.nn.functional.cosine_similarity(g2, g0, dim=0).item()
    rel_e, rel_2 = ((ge - g0).norm() / g0.norm()).item(), ((g2 - g0).norm() / g0.norm()).item()
    print(f"BF16 feature gradients: cosine {cos:.5f}, rel L2 {rel_2:.4f} (BF16 operands alone {rel_e:.4f})")
    assert cos >= 0.99, cos
    assert rel_2 <= 2.0 * rel_e + 0.02, (rel_2, rel_e)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_exact_zeros_on_padded_bins_and_dummy_slots(precision):
    """DESIGN.md §3.3: padded bins of a region with a valid bin and every dummy pCRE slot cannot move the logits; their
    gradient is exactly 0.0, here and in the oracle."""
    model = _mk(ChromoformerClassifier)
    sd = _sd(model)
    batch = synthetic.make_batch(12, ragged=True, full_masks=True, seed=5, stress=True)
    _, dx_o = _oracle_feature_grads(sd, batch, lambda lg: lg[:, 1].sum())
    model.cuda()
    model.precision = precision
    got = input_gradients(model, batch)
    k = batch["n_partners"]
    dummy = torch.arange(8).view(1, 8) >= k.view(-1, 1)                          # [B, I]
    assert dummy.any() and (~dummy).any()
    for b in BINS:
        n = 40000 // b
        pad = batch["pcre_pad_masks"][b][:, :, 0, n // 2, :]                     # [B, I, n], True = padded
        live_region = ~dummy & (~pad).any(-1)
        padded_bin = (pad & live_region.unsqueeze(-1)).unsqueeze(-1).expand(-1, -1, -1, 7)
        assert padded_bin.any()
        for g in (got["pcre_feats"][b].cpu(), dx_o["pcre_feats"][b]):
            assert (g[padded_bin] == 0).all()
            assert (g[dummy] == 0).all()
            assert (g[~padded_bin & ~dummy.view(12, 8, 1, 1)] != 0).any()


def test_parameter_gradients_unchanged_by_feature_gradients():
    """The parameter gradients of a pass that also returns feature gradients are those of the ordinary pass: the same
    launches, plus one input_grad_rows_kernel per (Pairwise layer, resolution) and one per resolution for the promoter."""
    lib = _lib.load()
    model = _mk(ChromoformerRegressor).cuda().train()
    batch = synthetic.make_batch(4, ragged=True, seed=8)
    target = batch["labels_reg"].view(-1, 1).cuda()
    runs = []
    for with_feats in (False, True, False):
        model.zero_grad(set_to_none=True)
        args, leaves = _leaves(batch) if with_feats else (synthetic.forward_args(batch, "cuda"), None)
        out = model(*args)
        loss = torch.nn.functional.mse_loss(out, target)
        c0 = lib.chromo_launch_counter(0)
        loss.backward()
        torch.cuda.synchronize()
        runs.append((model.flat_grads.clone(), lib.chromo_launch_counter(0) - c0))
    (plain, n_plain), (feat, n_feat), (again, _) = runs
    assert n_feat == n_plain + 3 * 2 + 3
    if torch.equal(plain, again):       # the ordinary pass reproduces itself bit for bit: so must this one
        print("parameter gradients: ordinary pass reproducible; with feature gradients bit-identical:",
              torch.equal(feat, plain))
        assert torch.equal(feat, plain)
    else:                               # FP32 atomics summed in another order: the same noise and no more
        noise = (plain - again).abs().max().item()
        print(f"parameter gradients: ordinary pass differs from itself by {noise:.3e} (atomics order)")
        assert (feat - plain).abs().max().item() <= 4 * noise + 1e-6 * plain.abs().max().item()


def test_no_parameter_mode():
    """model.requires_grad_(False): feature gradients only, no weight contraction, p.grad untouched."""
    lib = _lib.load()
    batch = synthetic.make_batch(5, ragged=True, full_masks=True, seed=13, stress=True)
    model = _mk(ChromoformerClassifier)
    _, dx_o = _oracle_feature_grads(_sd(model), batch, lambda lg: lg.sum())
    model.cuda()
    counts = []
    for frozen in (False, True):
        model.zero_grad(set_to_none=True)
        model.requires_grad_(not frozen)
        args, leaves = _leaves(batch)
        out = model(*args)
        c0 = lib.chromo_launch_counter(0)
        dx = torch.autograd.grad(out.sum(), _flat_list(leaves))
        counts.append(lib.chromo_launch_counter(0) - c0)
        if frozen:
            assert all(p.grad is None for p in model.parameters())
            for g, (key, b) in zip(dx, [(key, b) for key in FEATS for b in BINS]):
                assert _max_rel(g, dx_o[key][b]) < REL, (key, b)
    assert counts[1] < counts[0], counts
    model.requires_grad_(True)


def test_shapes_and_dtypes_float16_and_legacy_api():
    batch = synthetic.make_batch(3, ragged=True, seed=17)
    half = {key: {b: t.half() for b, t in batch[key].items()} for key in FEATS}
    rounded = dict(batch, **{key: {b: t.float() for b, t in half[key].items()} for key in FEATS})
    model = _mk(ChromoformerClassifier, seed=3).cuda()
    model.requires_grad_(False)
    ref = input_gradients(model, rounded)
    args, leaves = _leaves(dict(batch, **half))
    out = model(*args)
    dx = torch.autograd.grad(out[:, 1].sum(), _flat_list(leaves))
    for g, (key, b) in zip(dx, [(key, b) for key in FEATS for b in BINS]):
        assert g.dtype == torch.float16 and g.shape == half[key][b].shape
        assert _max_rel(g.float(), ref[key][b].cpu()) < 1e-3, (key, b)
    # the legacy flat API (net.py:228-270) with the same weights
    legacy = Chromoformer(seed=3, i_max=8).cuda()
    legacy.requires_grad_(False)
    a = synthetic.forward_args(batch, "cuda")
    flat_args, feats = [], []
    for b in BINS:
        xp, xc = a[0][b].clone().requires_grad_(True), a[2][b].clone().requires_grad_(True)
        feats += [xp, xc]
        flat_args += [xp, a[1][b], xc, a[3][b], a[4][b]]
    out = legacy(*flat_args, a[5])
    g = torch.autograd.grad(out[:, 1].sum(), feats)
    want = input_gradients(model, batch)
    for i, b in enumerate(BINS):
        for gg, key in ((g[2 * i], "promoter_feats"), (g[2 * i + 1], "pcre_feats")):
            assert gg.shape == batch[key][b].shape and gg.dtype == torch.float32
            assert _max_rel(gg, want[key][b].cpu()) < REL, (key, b)


def test_integrated_gradients_vs_oracle_and_chunking():
    steps, B = 4, 3
    batch = synthetic.make_batch(B, ragged=True, full_masks=True, seed=29, stress=True)
    model = _mk(ChromoformerClassifier)
    sd = _sd(model)
    acc = {key: {b: torch.zeros_like(batch[key][b]) for b in BINS} for key in FEATS}
    for k in range(steps):
        alpha = (k + 0.5) / steps
        scaled = dict(batch, **{key: {b: alpha * batch[key][b] for b in BINS} for key in FEATS})
        _, g = _oracle_feature_grads(sd, scaled, lambda lg: lg[:, 1].sum())
        for key in FEATS:
            for b in BINS:
                acc[key][b] += g[key][b]
    ig_o = {key: {b: batch[key][b] * acc[key][b] / steps for b in BINS} for key in FEATS}
    model.cuda()
    was = [p.requires_grad for p in model.parameters()]
    whole = integrated_gradients(model, batch, steps=steps)
    assert [p.requires_grad for p in model.parameters()] == was
    assert all(p.grad is None for p in model.parameters())
    for key in FEATS:
        for b in BINS:
            assert whole[key][b].shape == batch[key][b].shape
            assert _max_rel(whole[key][b], ig_o[key][b]) < REL, (key, b)
    for chunk in (2 * B, 2):        # steps split in two; genes split too
        part = integrated_gradients(model, batch, steps=steps, chunk=chunk)
        for key in FEATS:
            for b in BINS:
                assert _max_rel(part[key][b], whole[key][b].cpu()) < REL, (chunk, key, b)
