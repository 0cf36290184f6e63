"""Ragged plan of the BF16 inference path (csrc/ragged.cu): dead pCRE slots and padded bins are not computed.

The plan only uses what the masks themselves guarantee (data.py:156-203: centred valid spans, dummy slots behind a
block-form interaction mask), so its results must agree with the CPU oracle - which computes every slot and every bin as
the reference does - within the BF16 tolerance, and with the same kernels run without the plan (the CHROMO_F_DENSE hint)
to rounding noise.  The adversarial cases are the ones where an elimination would be WRONG if the plan trusted the data
layout instead of the masks."""
import pytest
import torch

from _util import KWS
from chromoformer_b200 import ChromoformerClassifier, synthetic
from chromoformer_b200.engine import InferenceEngine
from oracle import chromoformer_oracle as oracle

pytestmark = pytest.mark.gpu
BF16_TOL = 1e-2


def _mk(seed=123):
    return ChromoformerClassifier(7, 128, 128, dict(KWS[0]), dict(KWS[1]), dict(KWS[2]), seed=seed)


def _oracle_logits(sd, batch, idx):
    part = {}
    for key, v in batch.items():
        part[key] = {b: t[idx] for b, t in v.items()} if isinstance(v, dict) else v[idx]
    part = synthetic.expand_full_masks(part)
    with torch.no_grad():
        return oracle.chromoformer_forward(sd, *synthetic.forward_args(part))


def _run(model, batch, ragged):
    eng = InferenceEngine(model, chunk=batch["interaction_freq"].size(0))
    dev = eng.to_device(batch)
    dev["dense"] = not ragged          # the CHROMO_F_DENSE hint: the plan is not built
    return eng.predict_device(dev).cpu()


def test_ragged_batch_with_and_without_plan():
    """configs[3]: pCRE counts of the demo histogram, log-normal pCRE lengths.  1200 genes = 75 tiles of 128 rows."""
    n = 1200
    model = _mk()
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    batch = synthetic.make_batch(n, ragged=True, seed=5)
    model.cuda().eval()
    model.precision = "bf16"
    got = _run(model, batch, True)
    ref = _run(model, batch, False)
    assert torch.isfinite(got).all()
    # same kernels, other tile composition and key windows: the online softmax rounds P against another running maximum
    assert (got - ref).abs().max().item() < 5e-3
    idx = torch.cat([torch.arange(0, 48), torch.arange(n - 48, n)])
    want = _oracle_logits(sd, batch, idx)
    assert (got[idx] - want).abs().max().item() < BF16_TOL
    # every pCRE count of the histogram is in the checked genes
    assert set(batch["n_partners"][idx].tolist()) >= {0, 1, 8}
    # the reference DataLoader's own collation ([B,I,1,n,n] masks: the plan reads the centre rows through the stride)
    sub = synthetic.slice_batch(batch, 0, 256)
    full = synthetic.expand_full_masks(sub)
    assert torch.equal(_run(model, full, True), _run(model, sub, True))


def test_dense_batch_same_with_and_without_plan():
    """All slots live, all spans full: the stable sort keeps the order and every window is the whole table - bit-identical
    to the run without the plan, so the hint never changes the results of a batch it is derived for."""
    n = 256
    model = _mk(seed=3)
    batch = synthetic.make_batch(n, ragged=False, seed=2)
    model.cuda().eval()
    model.precision = "bf16"
    assert torch.equal(_run(model, batch, True), _run(model, batch, False))
    # the engine recognises such a batch on the host and passes the hint
    eng = InferenceEngine(model, chunk=n)
    assert eng.to_device(batch)["dense"] is True
    rag = synthetic.make_batch(n, ragged=True, seed=2)
    assert eng.to_device(rag)["dense"] is False


def test_masks_decide_not_the_layout():
    """Batches the reference's Dataset never produces but its forward accepts."""
    n = 320
    model = _mk(seed=11)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    batch = synthetic.make_batch(n, ragged=True, seed=9)
    gen = torch.Generator().manual_seed(1)
    k = batch["n_partners"]
    S = 9
    for b in (2000, 500, 100):
        nb = 40000 // b
        mc = batch["pcre_pad_masks"][b]                      # [B, 8, n] centre rows, True = padded
        xc = batch["pcre_feats"][b]
        im = batch["interaction_masks"][b]                   # [B, 1, S, S]
        # (a) genes 0..15: arbitrary interaction masks (not block form): every slot stays live
        im[:16, 0] = torch.rand(16, S, S, generator=gen) < 0.4
        im[:16, 0, :, 0] = False
        # (b) genes 16..31: a LIVE slot whose pad row is fully masked (uniform softmax over all bins in the reference)
        mc[16:32, 0] = True
        # (c) genes 32..47: holes inside the valid span, and a second island far from the centre
        mc[32:48, 0, ::3] = True
        mc[32:48, 1, :2] = False
        mc[32:48, 1, nb - 1] = False
        # (d) genes 48..63: dead slots (behind the block mask) with unmasked bins and data in them
        mc[48:64, 7] = False
        xc[48:64, 7] = torch.rand(16, nb, 7, generator=gen)
        # (e) genes 64..79: the pad mask says "valid" over zero-feature bins beyond the span of live slots
        mc[64:80, 0] = False
    model.cuda().eval()
    model.precision = "bf16"
    got = _run(model, batch, True)
    ref = _run(model, batch, False)
    assert torch.isfinite(got).all()
    assert (got - ref).abs().max().item() < 5e-3
    idx = torch.arange(0, 80)
    want = _oracle_logits(sd, batch, idx)
    assert (got[idx] - want).abs().max().item() < BF16_TOL
    assert (k[idx] < 8).any()


def test_ragged_imax16_token_classes():
    """i_max = 16: 17-token Regulation tiles, token classes 17 / 9 / 5 / 3 / 2 / 1."""
    n = 700
    model = ChromoformerClassifier(7, 128, 128, dict(KWS[0]), dict(KWS[1]), dict(KWS[2]), seed=21, i_max=16)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    batch = synthetic.make_batch(n, i_max=16, ragged=True, seed=13)
    # spread the pCRE counts over every class (the synthetic histogram only knows 0..8 and 16)
    gen = torch.Generator().manual_seed(2)
    k = torch.randint(0, 17, (n,), generator=gen)
    idx = torch.arange(17)
    inside = (idx.view(1, 17, 1) <= k.view(n, 1, 1)) & (idx.view(1, 1, 17) <= k.view(n, 1, 1))
    for b in (2000, 500, 100):
        batch["interaction_masks"][b] = (~inside).unsqueeze(1)
        live = (torch.arange(16).view(1, 16) < k.view(n, 1))
        batch["pcre_pad_masks"][b] = batch["pcre_pad_masks"][b] | ~live.unsqueeze(2)
    batch["n_partners"] = k
    model.cuda().eval()
    model.precision = "bf16"
    got = _run(model, batch, True)
    ref = _run(model, batch, False)
    assert torch.isfinite(got).all()
    assert (got - ref).abs().max().item() < 5e-3
    sel = torch.arange(0, 40)
    want = _oracle_logits(sd, batch, sel)
    assert (got[sel] - want).abs().max().item() < BF16_TOL
    assert len(set(k[sel].tolist())) >= 10


def test_plan_is_capturable_into_a_cuda_graph():
    """The plan is built on a library-owned side stream (fork / join by events) with a cub sort and a memset in it: all of
    that must be legal inside a stream capture, and a replay must rebuild the plan from the CURRENT contents of the inputs."""
    n = 512
    model = _mk(seed=17).cuda().eval()
    model.precision = "bf16"
    eng = InferenceEngine(model, chunk=n)
    a = eng.to_device(synthetic.make_batch(n, ragged=True, seed=51))
    b = eng.to_device(synthetic.make_batch(n, ragged=True, seed=52))
    a["dense"] = b["dense"] = False
    keys = [k for k in a if k != "dense"]
    with torch.no_grad():
        want_a = model.forward_batch(a).clone()
        want_b = model.forward_batch(b).clone()
        static = {k: ({bb: t.clone() for bb, t in a[k].items()} if isinstance(a[k], dict) else a[k].clone()) for k in keys}
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            model.forward_batch(static)
        torch.cuda.current_stream().wait_stream(s)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            out = model.forward_batch(static)
        g.replay()
        assert torch.equal(out, want_a)
        for k in keys:                                   # other genes, other plan, same graph
            if isinstance(static[k], dict):
                for bb in static[k]:
                    static[k][bb].copy_(b[k][bb])
            else:
                static[k].copy_(b[k])
        g.replay()
        assert torch.equal(out, want_b)
