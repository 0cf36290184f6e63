"""SURVEY §8c: the pretrained-checkpoint goldens (`demo/prediction.out`, `demo/prediction.reg.out`, AUC 0.9330 /
AP 0.9417 / ACC 0.83 of demo/img/demo_result.png; R2 0.6224 / r 0.7944) pin the path as soon as the two `.pt` files of
the reference's `.MISSING_LARGE_BLOBS` are supplied.  This test switches on automatically when either file is found under
$CHROMOFORMER_PT_DIR, $CHROMOFORMER_REF/demo or baseline/_ref/demo, and is skipped otherwise
(the published predictions themselves are committed: tests/golden/demo_pretrained_predictions.npz).

Tolerances: FP32 path 2e-5 on the published predictions (as for random_prediction.out); BF16 path logits within 1e-2,
AUROC / Pearson r equal to 3 decimals, >= 99 of 100 labels equal (north_star)."""
import os

import numpy as np
import pytest
import torch

from _util import ROOT, demo_batch, golden
from chromoformer_b200 import ChromoformerClassifier, ChromoformerRegressor, synthetic

CLF_PT = "chromoformer-reproduction-E003-conf1-fold1.pt"
REG_PT = "chromoformer-reg-reproduction-E003-conf1-fold1.pt"


def _find(name):
    dirs = [os.environ.get("CHROMOFORMER_PT_DIR"), os.path.join(os.environ.get("CHROMOFORMER_REF", ""), "demo"),
            os.path.join(ROOT, "baseline", "_ref", "demo")]
    for d in dirs:
        if d and os.path.exists(os.path.join(d, name)):
            return os.path.join(d, name)
    return None


def _predict(cls, path, precision):
    model = cls(seed=123)
    ckpt = torch.load(path, map_location="cpu", weights_only=False)
    model.load_state_dict(ckpt["net"] if "net" in ckpt else ckpt)        # any key generation (misc/convert_weight.py)
    model.cuda().eval()
    model.precision = precision
    with torch.no_grad():
        return model(*synthetic.forward_args(demo_batch(0, 100), "cuda")).double().cpu().numpy()


@pytest.mark.gpu
@pytest.mark.skipif(_find(CLF_PT) is None, reason="pretrained classifier checkpoint not supplied (.MISSING_LARGE_BLOBS)")
def test_pretrained_classifier_predictions():
    from sklearn import metrics
    g = golden("demo_pretrained_predictions.npz")
    want, y = g["prediction_clf"], g["label"]
    sig = lambda z: 1.0 / (1.0 + np.exp(-z[:, 1]))                        # run_demo.py:116
    fp32 = _predict(ChromoformerClassifier, _find(CLF_PT), "fp32")
    assert np.abs(sig(fp32) - want).max() < 2e-4          # published with TF32-era GPUs: demo/test.out differs by 1.3e-4
    assert round(metrics.roc_auc_score(y, sig(fp32)), 3) == 0.933
    assert round(metrics.average_precision_score(y, sig(fp32)), 3) == 0.942
    assert metrics.accuracy_score(y, (sig(fp32) > 0.5).astype(int)) == 0.83
    bf16 = _predict(ChromoformerClassifier, _find(CLF_PT), "bf16")
    assert np.abs(bf16 - fp32).max() < 1e-2
    assert round(metrics.roc_auc_score(y, sig(bf16)), 3) == 0.933
    assert ((sig(bf16) > 0.5) == (sig(fp32) > 0.5)).mean() >= 0.99


@pytest.mark.gpu
@pytest.mark.skipif(_find(REG_PT) is None, reason="pretrained regressor checkpoint not supplied (.MISSING_LARGE_BLOBS)")
def test_pretrained_regressor_predictions():
    from scipy import stats
    g = golden("demo_pretrained_predictions.npz")
    want, y = g["prediction_reg"], np.log2(g["expression"] + 1)
    fp32 = _predict(ChromoformerRegressor, _find(REG_PT), "fp32").ravel()
    assert np.abs(fp32 - want).max() < 2e-3
    assert round(stats.pearsonr(y, fp32)[0], 3) == 0.794
    bf16 = _predict(ChromoformerRegressor, _find(REG_PT), "bf16").ravel()
    assert np.abs(bf16 - fp32).max() < 1e-2
    assert round(stats.pearsonr(y, bf16)[0], 3) == round(stats.pearsonr(y, fp32)[0], 3)


def test_published_pretrained_metrics_are_recomputable():
    """Keeps the fixture honest without the weights: demo/img/demo_result.png's numbers follow from prediction.out."""
    from scipy import stats
    from sklearn import metrics
    g = golden("demo_pretrained_predictions.npz")
    assert abs(metrics.roc_auc_score(g["label"], g["prediction_clf"]) - 0.9329586511441188) < 1e-12
    assert abs(metrics.average_precision_score(g["label"], g["prediction_clf"]) - 0.9416600059601521) < 1e-12
    assert metrics.accuracy_score(g["label"], (g["prediction_clf"] > 0.5).astype(int)) == 0.83
    y = np.log2(g["expression"] + 1)
    assert round(metrics.r2_score(y, g["prediction_reg"]), 4) == 0.6224
    assert round(stats.pearsonr(y, g["prediction_reg"])[0], 4) == 0.7944
