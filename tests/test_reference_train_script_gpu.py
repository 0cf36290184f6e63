"""The reference's OWN training script (chromoformer/train.py, unmodified text) run against this package: the file is copied
at test time from the staged reference (baseline/_ref, or an upstream checkout named by $CHROMOFORMER_REF) into a temporary package
whose `data` / `net` / `util` modules are this repo's drop-in names, and executed as `python -m <pkg>.train` with the
reference's command line (train.py:26-37) on a tiny dataset - stock torch.optim.AdamW + StepLR on the flat-buffer
parameters, `loss.backward()` through the C ABI, sklearn / scipy metrics on `out.cpu()`, checkpoint keys of train.py:322-343.
Nothing of the script is edited; only `wandb` is replaced by a no-op stub (no network on the box)."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import yaml

from _util import ROOT
from test_train_cli_gpu import _make_dataset

pytestmark = pytest.mark.gpu

WANDB_STUB = '''
class _Cfg(dict):
    def update(self, *a, **k):
        pass
config = _Cfg()
summary = _Cfg()
def init(*a, **k):
    return None
def log(*a, **k):
    return None
'''


def _reference_train_py():
    for base in (os.path.join(ROOT, "baseline", "_ref"), os.environ.get("CHROMOFORMER_REF", "")):
        p = os.path.join(base, "chromoformer", "train.py")
        if base and os.path.exists(p):
            return p
    return None


@pytest.mark.parametrize("regression,precision", [(False, "fp32"), (True, "bf16")])
def test_unmodified_reference_train_script(tmp_path, regression, precision):
    src = _reference_train_py()
    if src is None:
        pytest.skip("no staged reference (baseline/_ref) on this machine")
    pkg = tmp_path / "refscript"
    pkg.mkdir()
    (pkg / "__init__.py").write_text("")
    (pkg / "train.py").write_text(open(src).read())                      # the reference's text, byte for byte
    (pkg / "data.py").write_text("from chromoformer.data import ChromoformerDataset\n")
    (pkg / "net.py").write_text("from chromoformer.net import ChromoformerClassifier, ChromoformerRegressor\n")
    (pkg / "util.py").write_text("from chromoformer.util import seed_everything\n")
    (tmp_path / "wandb.py").write_text(WANDB_STUB)
    data = tmp_path / "data"
    data.mkdir()
    meta = _make_dataset(data)
    cfg = yaml.safe_load(open(os.path.join(ROOT, "chromoformer", "configs", "default.yaml")))
    cfg.update(num_epoch=3, bsz=4)                                        # range(1, 3): two epochs
    cfg_path = tmp_path / "config.yaml"
    yaml.safe_dump(cfg, open(cfg_path, "w"))
    out = tmp_path / "ckpt.pt"
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([str(tmp_path), ROOT]), WANDB_MODE="disabled", CHROMO_PRECISION=precision)
    cmd = [sys.executable, "-m", "refscript.train", "-o", str(out), "-c", str(cfg_path), "--exp-id", "t", "-m", str(meta),
           "-d", str(data), "--fold", "1"] + (["--regression"] if regression else [])
    r = subprocess.run(cmd, cwd=str(tmp_path), env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert "Validation loss=" in r.stdout
    ckpt = torch.load(out, map_location="cpu", weights_only=False)
    assert set(ckpt) == {"net", "optimizer", "epoch", "last_val_loss", "val_score", "val_label",
                         "last_val_r2" if regression else "last_val_auc"}
    assert ckpt["epoch"] == 2 and np.isfinite(float(ckpt["last_val_loss"]))
    assert len(ckpt["net"]) == 370 and len(ckpt["optimizer"]["state"]) == 334        # stock AdamW state, 334 trained tensors
