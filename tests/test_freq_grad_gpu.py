"""Gradients with respect to interaction_freq (chromo_backward_inputs with CHROMO_F_FREQ_GRAD through _ChromoFunction)
and the attribution helpers' freq option, against autograd over the oracle with interaction_freq (and the features) as
leaves.  FP32 tolerance: per-tensor max-abs error <= 2e-4 of that tensor's max-abs oracle gradient, the yardstick of
test_input_grad_gpu.py."""
import pytest
import torch

from _util import KWS
from chromoformer_b200 import Chromoformer, ChromoformerClassifier, ChromoformerRegressor, _lib, synthetic
from chromoformer_b200.attribution import input_gradients, integrated_gradients, pcre_scores
from oracle import chromoformer_oracle as oracle

pytestmark = pytest.mark.gpu
REL = 2e-4
BINS = (2000, 500, 100)
FEATS = ("promoter_feats", "pcre_feats")
FREQ = "interaction_freq"
REG4 = {"n_layers": 2, "n_heads": 4, "d_model": 128, "d_ff": 256}     # reg_heads != 8: the one-warp-per-head kernel


def _mk(cls, seed=11, reg=None):
    return cls(7, 128, 128, dict(KWS[0]), dict(KWS[1]), dict(reg or KWS[2]), seed=seed)


def _sd(model):
    return {k: v.detach().clone() for k, v in model.named_parameters()}


def _oracle_grads(sd, batch, objective, heads=None):
    """autograd.grad(objective(logits), features + interaction_freq) over the oracle."""
    args = synthetic.forward_args(batch)
    leaves = {key: {b: t.detach().clone().requires_grad_(True) for b, t in batch[key].items()} for key in FEATS}
    fq = batch[FREQ].detach().clone().requires_grad_(True)
    args[0], args[2], args[5] = leaves["promoter_feats"], leaves["pcre_feats"], fq
    logits = oracle.chromoformer_forward(sd, *args, heads=heads)
    flat = [leaves[key][b] for key in FEATS for b in BINS] + [fq]
    g = list(torch.autograd.grad(objective(logits), flat))
    dfreq = g.pop()
    it = iter(g)
    return logits.detach(), {key: {b: next(it) for b in BINS} for key in FEATS}, dfreq


def _leaves(batch, feats=True, freq=True, dev="cuda"):
    """Forward arguments on the device with the chosen inputs as leaves; returns (args, [leaves in order])."""
    args = synthetic.forward_args(batch, dev)
    flat = []
    if feats:
        for i in (0, 2):
            args[i] = {b: args[i][b].clone().requires_grad_(True) for b in BINS}
            flat += list(args[i].values())
    if freq:
        args[5] = args[5].clone().requires_grad_(True)
        flat.append(args[5])
    return args, flat


def _max_rel(got, want):
    return (got.detach().cpu().float() - want).abs().max().item() / max(want.abs().max().item(), 1e-12)


def _check_params(model, grads_o):
    for name, p in model.named_parameters():
        if grads_o[name] is None:
            assert p.grad is None, name
            continue
        assert _max_rel(p.grad, grads_o[name]) < REL, name


@pytest.mark.parametrize("tag,ragged,i_max,n", [("reg", True, 8, 6), ("clf", False, 8, 3), ("reg", True, 16, 2),
                                                ("clf", False, 16, 2)])
def test_freq_gradient_vs_oracle(tag, ragged, i_max, n):
    """loss.backward() with the features and interaction_freq requiring grad: every input gradient and the parameter
    gradients in one pass (gene kernel: <9> for i_max 8, <17> for i_max 16)."""
    cls = ChromoformerRegressor if tag == "reg" else ChromoformerClassifier
    model = _mk(cls)
    sd = _sd(model)
    batch = synthetic.make_batch(n, i_max=i_max, ragged=ragged, full_masks=True, seed=21, stress=True)
    target = batch["labels_reg"].view(-1, 1) if tag == "reg" else batch["labels_clf"]
    crit = torch.nn.MSELoss() if tag == "reg" else torch.nn.CrossEntropyLoss()
    logits_o, dx_o, dfreq_o = _oracle_grads(sd, batch, lambda lg: crit(lg, target))
    _, _, grads_o = oracle.forward_backward(sd, synthetic.forward_args(batch), target, tag == "reg")
    model.cuda().train()
    plain = model(*synthetic.forward_args(batch, "cuda")).detach()
    model.zero_grad(set_to_none=True)
    args, flat = _leaves(batch)
    out = model(*args)
    crit(out, target.cuda()).backward()
    assert torch.equal(out.detach(), plain)
    assert (out.detach().cpu() - logits_o).abs().max().item() < 5e-5
    g = args[5].grad
    assert g is not None and g.shape == args[5].shape and g.dtype == torch.float32
    assert dfreq_o.abs().max().item() > 0
    err = _max_rel(g, dfreq_o)
    print(f"dfreq max rel error {err:.2e}")
    assert err < REL, err
    for i, key in ((0, "promoter_feats"), (2, "pcre_feats")):
        for b in BINS:
            assert _max_rel(args[i][b].grad, dx_o[key][b]) < REL, (key, b)
    _check_params(model, grads_o)


def test_freq_gradient_warp_kernel_vs_oracle():
    """reg_heads = 4 (d_model 128): the backward runs reg_attention_bwd_kernel (one warp per (gene, head)) and sums
    the per-head partials in freq_grad_sum_kernel."""
    model = _mk(ChromoformerRegressor, reg=REG4)
    sd = _sd(model)
    heads = {"embed": 2, "pairwise_interaction": 2, "regulation": 4}
    for i_max in (8, 16):
        batch = synthetic.make_batch(5, i_max=i_max, ragged=True, full_masks=True, seed=23, stress=True)
        target = batch["labels_reg"].view(-1, 1)
        crit = torch.nn.MSELoss()
        logits_o, dx_o, dfreq_o = _oracle_grads(sd, batch, lambda lg: crit(lg, target), heads=heads)
        model.cuda().train()
        model.zero_grad(set_to_none=True)
        args, flat = _leaves(batch)
        out = model(*args)
        assert (out.detach().cpu() - logits_o).abs().max().item() < 5e-5
        crit(out, target.cuda()).backward()
        err = _max_rel(args[5].grad, dfreq_o)
        print(f"warp kernel, i_max {i_max}: dfreq max rel error {err:.2e}")
        assert err < REL, (i_max, err)
        for i, key in ((0, "promoter_feats"), (2, "pcre_feats")):
            for b in BINS:
                assert _max_rel(args[i][b].grad, dx_o[key][b]) < REL, (i_max, key, b)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_exact_zeros_on_masked_pairs(precision):
    """dS is 0 wherever the interaction mask is set (dummy slots), so d interaction_freq is exactly 0.0 there, here and
    in the oracle; inside the live block it is not."""
    model = _mk(ChromoformerClassifier)
    sd = _sd(model)
    batch = synthetic.make_batch(12, ragged=True, full_masks=True, seed=5, stress=True)
    _, _, dfreq_o = _oracle_grads(sd, batch, lambda lg: lg[:, 1].sum())
    model.cuda()
    model.precision = precision
    got = input_gradients(model, batch, freq=True)[FREQ].cpu()
    masked = batch["interaction_masks"][BINS[0]][:, 0]                           # [B, S, S], True = masked
    for b in BINS:
        assert torch.equal(batch["interaction_masks"][b][:, 0], masked)
    assert masked.any() and (~masked).any()
    for g in (got, dfreq_o):
        assert (g[masked] == 0).all()
        assert (g[~masked] != 0).any()


@pytest.mark.parametrize("tag,n", [("reg", 64), ("clf", 70)])
def test_bf16_freq_gradient_vs_oracle(tag, n):
    """CHROMO_F_BF16 training workspace: cosine with the FP32 oracle >= 0.99, relative L2 within 2 x what BF16
    operands do to the oracle + 0.02 (the yardstick of test_bf16_feature_gradients_vs_oracle)."""
    cls = ChromoformerRegressor if tag == "reg" else ChromoformerClassifier
    model = _mk(cls)
    sd = _sd(model)
    batch = synthetic.make_batch(n, ragged=True, full_masks=False, seed=21)
    full = synthetic.expand_full_masks(batch)
    target = batch["labels_reg"].view(-1, 1) if tag == "reg" else batch["labels_clf"]
    crit = torch.nn.MSELoss() if tag == "reg" else torch.nn.CrossEntropyLoss()
    _, _, g0 = _oracle_grads(sd, full, lambda lg: crit(lg, target))
    with oracle.bf16_operands():
        _, _, ge = _oracle_grads(sd, full, lambda lg: crit(lg, target))
    model.cuda().train()
    model.precision = "bf16"
    args, flat = _leaves(batch, feats=False)
    out = model(*args)
    (g2,) = torch.autograd.grad(crit(out, target.cuda()), flat)
    g0, ge, g2 = g0.flatten().double(), ge.flatten().double(), g2.cpu().flatten().double()
    cos = torch.nn.functional.cosine_similarity(g2, g0, dim=0).item()
    rel_e, rel_2 = ((ge - g0).norm() / g0.norm()).item(), ((g2 - g0).norm() / g0.norm()).item()
    print(f"BF16 interaction_freq gradient: cosine {cos:.5f}, rel L2 {rel_2:.4f} (BF16 operands alone {rel_e:.4f})")
    assert cos >= 0.99, cos
    assert rel_2 <= 2.0 * rel_e + 0.02, (rel_2, rel_e)


def _same_or_noise(got, plain, again, what):
    """Bit-identical when the ordinary pass reproduces itself; otherwise within the noise of its FP32 atomics."""
    if torch.equal(plain, again):
        assert torch.equal(got, plain), what
        return 0.0
    noise = (plain - again).abs().max().item()
    assert (got - plain).abs().max().item() <= 4 * noise + 1e-6 * plain.abs().max().item(), what
    return noise


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_other_gradients_unchanged_and_deterministic(precision):
    """Asking for d interaction_freq as well leaves the parameter and feature gradients of the pass as they were, adds
    exactly one launch (freq_grad_sum_kernel), and two such passes give bit-identical d interaction_freq (the kernels
    sum it in a fixed order, without atomics) whenever the gradient arriving at the Regulation stage is itself
    reproduced bit for bit."""
    lib = _lib.load()
    model = _mk(ChromoformerRegressor).cuda().train()
    model.precision = precision
    batch = synthetic.make_batch(4, ragged=True, seed=8)
    target = batch["labels_reg"].view(-1, 1).cuda()
    runs = []
    for with_freq in (False, True, False, True):
        model.zero_grad(set_to_none=True)
        args, flat = _leaves(batch, freq=with_freq)
        out = model(*args)
        loss = torch.nn.functional.mse_loss(out, target)
        c0 = lib.chromo_launch_counter(0)
        loss.backward()
        torch.cuda.synchronize()
        runs.append((model.flat_grads.clone(), torch.cat([t.grad.flatten() for t in flat[:6]]),
                     args[5].grad.clone() if with_freq else None, lib.chromo_launch_counter(0) - c0))
    (p0, f0, _, n0), (p1, f1, d1, n1), (p2, f2, _, n2), (p3, f3, d3, n3) = runs
    assert n1 == n3 == n0 + 1 and n2 == n0, (n0, n1, n2, n3)
    noise_p = _same_or_noise(p1, p0, p2, "parameter gradients")
    noise_f = _same_or_noise(f1, f0, f2, "feature gradients")
    print(f"{precision}: ordinary pass self-noise: parameters {noise_p:.3e}, features {noise_f:.3e}; "
          f"dfreq bit-identical across passes: {torch.equal(d1, d3)}")
    if torch.equal(f1, f3):             # the same gradient arrived at the inputs: the same dfreq, bit for bit
        assert torch.equal(d1, d3)
    else:
        assert (d1 - d3).abs().max().item() <= 1e-4 * d1.abs().max().item()


def test_freq_only_pass():
    """model.requires_grad_(False) and only interaction_freq requiring grad: the pass stops after the Regulation stage
    (fewer launches than a feature-gradient pass), p.grad stays None, and d interaction_freq meets the FP32 bound."""
    lib = _lib.load()
    batch = synthetic.make_batch(5, ragged=True, full_masks=True, seed=13, stress=True)
    model = _mk(ChromoformerClassifier)
    _, _, dfreq_o = _oracle_grads(_sd(model), batch, lambda lg: lg.sum())
    model.cuda()
    model.requires_grad_(False)
    counts = []
    for feats, freq in ((True, False), (False, True)):
        args, flat = _leaves(batch, feats=feats, freq=freq)
        out = model(*args)
        c0 = lib.chromo_launch_counter(0)
        g = torch.autograd.grad(out.sum(), flat)
        counts.append(lib.chromo_launch_counter(0) - c0)
    assert all(p.grad is None for p in model.parameters())
    assert counts[1] < counts[0], counts
    print("launches: feature gradients", counts[0], "interaction_freq only", counts[1])
    assert _max_rel(g[0], dfreq_o) < REL
    model.requires_grad_(True)


def test_shapes_and_dtypes_float16_and_legacy_api():
    batch = synthetic.make_batch(3, ragged=True, seed=17)
    half = batch[FREQ].half()
    rounded = dict(batch, **{FREQ: half.float()})
    model = _mk(ChromoformerClassifier, seed=3).cuda()
    model.requires_grad_(False)
    ref = input_gradients(model, rounded, freq=True)[FREQ]
    args = synthetic.forward_args(batch, "cuda")
    args[5] = half.cuda().requires_grad_(True)
    (g,) = torch.autograd.grad(model(*args)[:, 1].sum(), [args[5]])
    assert g.dtype == torch.float16 and g.shape == half.shape
    assert _max_rel(g.float(), ref.cpu()) < 1e-3
    # forward_batch, as the attribution helpers call it
    dev = {k: ({b: t.cuda() for b, t in v.items()} if isinstance(v, dict) else v.cuda()) for k, v in batch.items()}
    fq = dev[FREQ].clone().requires_grad_(True)
    (g,) = torch.autograd.grad(model.forward_batch(dict(dev, **{FREQ: fq}))[:, 1].sum(), [fq])
    assert _max_rel(g, input_gradients(model, batch, freq=True)[FREQ].cpu()) < REL
    # the legacy flat API (net.py:228-270) with the same weights
    legacy = Chromoformer(seed=3, i_max=8).cuda()
    legacy.requires_grad_(False)
    a = synthetic.forward_args(batch, "cuda")
    flat_args = []
    for b in BINS:
        flat_args += [a[0][b], a[1][b], a[2][b], a[3][b], a[4][b]]
    fq = a[5].clone().requires_grad_(True)
    (g,) = torch.autograd.grad(legacy(*flat_args, fq)[:, 1].sum(), [fq])
    want = input_gradients(model, batch, freq=True)[FREQ]
    assert g.shape == batch[FREQ].shape and g.dtype == torch.float32
    assert _max_rel(g, want.cpu()) < REL


def _ig_oracle(sd, batch, steps):
    """The oracle's midpoint sum over the joint path (features and interaction_freq from zero), target column 1."""
    acc = {key: {b: torch.zeros_like(batch[key][b]) for b in BINS} for key in FEATS}
    acc_f = torch.zeros_like(batch[FREQ])
    for k in range(steps):
        alpha = (k + 0.5) / steps
        scaled = dict(batch, **{key: {b: alpha * batch[key][b] for b in BINS} for key in FEATS})
        scaled[FREQ] = alpha * batch[FREQ]
        _, g, gf = _oracle_grads(sd, scaled, lambda lg: lg[:, 1].sum())
        for key in FEATS:
            for b in BINS:
                acc[key][b] += g[key][b]
        acc_f += gf
    out = {key: {b: batch[key][b] * acc[key][b] / steps for b in BINS} for key in FEATS}
    out[FREQ] = batch[FREQ] * acc_f / steps
    return out


def _total(attr):
    """Per-gene sum of every attribution of a result."""
    t = attr[FREQ].double().cpu().sum(dim=(1, 2)) if FREQ in attr else 0.0
    for key in FEATS:
        for v in attr[key].values():
            t = t + v.double().cpu().flatten(1).sum(1)
    return t


def test_integrated_gradients_with_freq_vs_oracle_chunking_and_scores():
    steps, B = 4, 3
    batch = synthetic.make_batch(B, ragged=True, full_masks=True, seed=29, stress=True)
    model = _mk(ChromoformerClassifier)
    ig_o = _ig_oracle(_sd(model), batch, steps)
    model.cuda()
    was = [p.requires_grad for p in model.parameters()]
    whole = integrated_gradients(model, batch, steps=steps, freq=True)
    assert [p.requires_grad for p in model.parameters()] == was
    assert all(p.grad is None for p in model.parameters())
    assert set(whole) == set(FEATS) | {FREQ}
    assert whole[FREQ].shape == batch[FREQ].shape
    assert _max_rel(whole[FREQ], ig_o[FREQ]) < REL
    for key in FEATS:
        for b in BINS:
            assert _max_rel(whole[key][b], ig_o[key][b]) < REL, (key, b)
    for chunk in (2 * B, 2):        # steps split in two; genes split too
        part = integrated_gradients(model, batch, steps=steps, chunk=chunk, freq=True)
        for key in FEATS:
            for b in BINS:
                assert _max_rel(part[key][b], whole[key][b].cpu()) < REL, (chunk, key, b)
        assert _max_rel(part[FREQ], whole[FREQ].cpu()) < REL, chunk
    # freq=False: the result of the call without the keyword, with the keys it always had - bit for bit when that call
    # reproduces itself, else within its own run-to-run noise (the FP32 backward's split contractions add with atomics)
    plain = integrated_gradients(model, batch, steps=steps)
    again = integrated_gradients(model, batch, steps=steps)
    off = integrated_gradients(model, batch, steps=steps, freq=False)
    assert set(off) == set(plain) == set(FEATS)
    for key in FEATS:
        for b in BINS:
            _same_or_noise(off[key][b], plain[key][b], again[key][b], (key, b))
    assert set(input_gradients(model, batch, freq=False)) == set(FEATS)
    # pcre_scores: slot sums of the pcre_feats attribution plus the promoter-contact frequency attribution
    sc = pcre_scores(whole).cpu()
    want = sum(whole["pcre_feats"][b].cpu().sum(dim=(2, 3)) for b in BINS) + whole[FREQ].cpu()[:, 0, 1:]
    assert sc.shape == (B, 8) and torch.allclose(sc, want, rtol=1e-6, atol=1e-7)
    dummy = torch.arange(8).view(1, 8) >= batch["n_partners"].view(-1, 1)
    assert dummy.any() and (sc[dummy] == 0).all() and (sc[~dummy] != 0).all()
    assert (pcre_scores(input_gradients(model, batch)).cpu()[dummy] == 0).all()


def test_integrated_gradients_completeness():
    """Sum of all attributions of the joint path ~ f(x) - f(x0).  The gap is the midpoint rule's quadrature error: it
    must shrink as the steps grow (8 -> 64), and at 64 steps stay within 1 % of max |f(x) - f(x0)| over the genes.
    (The midpoint error of a smooth path integral falls as 1 / steps^2, so 64 steps leave about 1/64 of the 8-step gap;
    the ReLU kinks on the path make it fall more slowly, hence the 1 % margin rather than the FP32 bound.)"""
    batch = synthetic.make_batch(6, ragged=True, seed=31)
    model = _mk(ChromoformerClassifier).cuda()
    model.requires_grad_(False)
    dev = synthetic.forward_args(batch, "cuda")
    with torch.no_grad():
        fx = model(*dev)[:, 1].double().cpu()
        zero = list(dev)
        zero[0] = {b: torch.zeros_like(t) for b, t in dev[0].items()}
        zero[2] = {b: torch.zeros_like(t) for b, t in dev[2].items()}
        zero[5] = torch.zeros_like(dev[5])
        fx0 = model(*zero)[:, 1].double().cpu()
    model.requires_grad_(True)
    want = fx - fx0
    gaps = {s: (_total(integrated_gradients(model, batch, steps=s, freq=True)) - want).abs().max().item()
            for s in (8, 64)}
    scale = want.abs().max().item()
    print(f"completeness: max |f(x) - f(x0)| {scale:.4e}, gap at 8 steps {gaps[8]:.3e}, at 64 steps {gaps[64]:.3e}")
    assert gaps[64] <= gaps[8]
    assert gaps[64] <= 0.01 * scale, (gaps, scale)
