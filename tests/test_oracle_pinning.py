"""Pin the CPU oracle (oracle/chromoformer_oracle.py) against the reference's own known answers
and against outputs of the unmodified reference committed under tests/golden/ (SURVEY §8c)."""
import numpy as np
import pytest
import torch

from _util import BINS, KWS, as_dict, demo_batch, golden, import_reference, reference_available, smoke_inputs
from chromoformer_b200 import Chromoformer, ChromoformerClassifier, ChromoformerRegressor, synthetic
from oracle import chromoformer_oracle as oracle


def _sd(model):
    return {k: v.detach().clone() for k, v in model.state_dict().items()}


def test_known_answers_of_net_main():
    """net.py:558-568: -3.1917 / -3.1917 / -0.1900 on the seeded __main__ inputs."""
    g = golden("smoke_main.npz")
    m0, m1, m2 = Chromoformer(), ChromoformerClassifier(), ChromoformerRegressor()
    x_p, m_p, x_c, m_c, i_m, freq = smoke_inputs()
    chk = np.array([x_p[2].double().sum().item(), x_c[2].double().sum().item(), freq.double().sum().item(),
                    float(sum(int(m.sum()) for m in m_c))])
    if not np.allclose(chk, g["input_checksum"], rtol=0, atol=1e-9):
        pytest.skip("torch RNG stream differs from the one the fixture was generated with")
    args = (as_dict(x_p), as_dict(m_p), as_dict(x_c), as_dict(m_c), as_dict(i_m), freq)
    o0 = oracle.chromoformer_forward(oracle.legacy_to_dict_layout(_sd(m0)), *args)
    o1 = oracle.chromoformer_forward(_sd(m1), *args)
    o2 = oracle.chromoformer_forward(_sd(m2), *args)
    assert abs(o0.sum().item() + 3.1917) < 5e-5
    assert abs(o1.sum().item() + 3.1917) < 5e-5
    assert abs(o2.sum().item() + 0.1900) < 5e-5
    assert np.abs(o0.numpy() - g["legacy"]).max() < 2e-6
    assert np.abs(o1.numpy() - g["classifier"]).max() < 2e-6
    assert np.abs(o2.numpy() - g["regressor"]).max() < 2e-6


def test_demo_untrained_golden():
    """demo/random_prediction.out: 100 demo genes, ChromoformerClassifier(seed=123), sigmoid(logit[1])."""
    from sklearn import metrics
    g = golden("demo_logits.npz")
    sd = _sd(ChromoformerClassifier(7, 128, 128, dict(KWS[0]), dict(KWS[1]), dict(KWS[2]), seed=123))
    logits = []
    for lo in range(0, 100, 25):
        b = demo_batch(lo, lo + 25)
        logits.append(oracle.chromoformer_forward(sd, *synthetic.forward_args(b)))
    logits = torch.cat(logits).numpy()
    assert np.abs(logits - g["logits"]).max() < 2e-6
    pred = 1.0 / (1.0 + np.exp(-logits[:, 1].astype(np.float64)))
    assert np.abs(pred - g["random_prediction"]).max() < 1e-6
    labels = demo_batch(0, 100)["labels"].numpy()
    assert abs(metrics.roc_auc_score(labels, pred) - 0.5720594138900041) < 1e-12
    assert abs(metrics.average_precision_score(labels, pred) - 0.5902055587970536) < 1e-12
    assert metrics.accuracy_score(labels, (pred > 0.5).astype(int)) == 0.49


@pytest.mark.parametrize("tag", ["reg", "clf"])
def test_training_golden(tag):
    """Loss, gradients and three AdamW steps of the reference on a seeded synthetic batch."""
    g = golden("train_golden.npz")
    batch = synthetic.make_batch(6, ragged=True, full_masks=True, seed=7)
    chk = np.array([batch["pcre_feats"][100].double().sum().item(), batch["interaction_freq"].double().sum().item(),
                    float(batch["n_partners"].sum())])
    if not np.allclose(chk, g["input_checksum"], rtol=0, atol=1e-9):
        pytest.skip("torch RNG stream differs from the one the fixture was generated with")
    cls = ChromoformerRegressor if tag == "reg" else ChromoformerClassifier
    model = cls(7, 128, 128, dict(KWS[0]), dict(KWS[1]), dict(KWS[2]), seed=123)
    names = [n for n, _ in model.named_parameters()]
    assert names == list(g["param_names"])
    sd = {k: v.detach().clone() for k, v in model.named_parameters()}
    target = batch["labels_reg"].view(-1, 1) if tag == "reg" else batch["labels_clf"]
    args = synthetic.forward_args(batch)
    m = {k: torch.zeros_like(v) for k, v in sd.items()}
    v = {k: torch.zeros_like(t) for k, t in sd.items()}
    for step in range(3):
        loss, logits, grads = oracle.forward_backward(sd, args, target, regression=(tag == "reg"))
        assert abs(loss.item() - g[f"{tag}_losses"][step]) < 2e-6
        if step == 0:
            assert np.abs(logits.numpy() - g[f"{tag}_logits"]).max() < 2e-6
            has = np.array([grads[n] is not None for n in names])
            assert (has == g[f"{tag}_has_grad"]).all() and (~has).sum() == 36
            gn = np.array([0.0 if grads[n] is None else grads[n].double().norm().item() for n in names])
            assert np.allclose(gn, g[f"{tag}_grad_norm"], rtol=2e-4, atol=1e-9)
            for key in g.files:
                if key.startswith(f"{tag}_grad::"):
                    ref = g[key]
                    got = grads[key.split("::")[1]].numpy()
                    assert np.abs(got - ref).max() <= 1e-5 * max(1e-3, np.abs(ref).max())
        for n in names:
            if grads[n] is None:
                continue
            sd[n], m[n], v[n] = oracle.adamw_step(sd[n], grads[n], m[n], v[n], step + 1)
    ps = np.array([sd[n].double().sum().item() for n in names])
    assert np.allclose(ps, g[f"{tag}_param_sum_after3"], rtol=0, atol=2e-5)
    for key in ("fc_head.0.bias", "embed.100.lin_proj.weight"):
        assert np.abs(sd[key].numpy() - g[f"{tag}_param_after3::{key}"]).max() < 1e-7


def test_input_path_golden():
    """oracle.build_item on raw FP16 regions == ChromoformerDataset items of the reference."""
    raw = golden("raw_regions.npz")
    items = golden("demo_items.npz")
    for gi, idx in enumerate(raw["index"]):
        pcres = []
        while f"g{gi}_pcre{len(pcres)}" in raw.files:
            pcres.append(raw[f"g{gi}_pcre{len(pcres)}"])
        it = oracle.build_item(raw[f"g{gi}_promoter"], str(raw["strands"][gi]), pcres, raw[f"g{gi}_scores"])
        ref = demo_batch(int(idx), int(idx) + 1)
        for b in BINS:
            assert np.abs(it["promoter_feats"][b] - ref["promoter_feats"][b][0].numpy()).max() < 2e-6
            assert np.abs(it["pcre_feats"][b] - ref["pcre_feats"][b][0].numpy()).max() < 2e-6
            assert (it["promoter_pad_masks"][b] == ref["promoter_pad_masks"][b][0].numpy()).all()
            assert (it["pcre_pad_masks"][b] == ref["pcre_pad_masks"][b][0].numpy()).all()
            assert (it["interaction_masks"][b] == ref["interaction_masks"][b][0].numpy()).all()
        assert np.abs(it["interaction_freq"] - items["freq"][idx]).max() < 1e-6


@pytest.mark.skipif(not reference_available(), reason="upstream chromoformer checkout not supplied ($CHROMOFORMER_REF)")
def test_oracle_equals_live_reference():
    """Direct comparison with the unmodified reference imported from $CHROMOFORMER_REF."""
    net, _ = import_reference()
    ref = net.ChromoformerRegressor(7, 128, 128, dict(KWS[0]), dict(KWS[1]), dict(KWS[2]), seed=5)
    batch = synthetic.make_batch(3, i_max=8, ragged=True, full_masks=True, seed=11, stress=True)
    args = synthetic.forward_args(batch)
    with torch.no_grad():
        want = ref(*args)
    got = oracle.chromoformer_forward(_sd(ref), *args)
    assert (got - want).abs().max().item() < 2e-6
    mine = ChromoformerRegressor(7, 128, 128, dict(KWS[0]), dict(KWS[1]), dict(KWS[2]), seed=5)
    for (k1, v1), (k2, v2) in zip(ref.state_dict().items(), mine.state_dict().items()):
        assert k1 == k2 and torch.equal(v1, v2)
