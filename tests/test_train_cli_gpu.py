"""`python -m chromoformer.train` (reference CLI, train.py:26-37) end to end on a tiny synthetic dataset:
same arguments and config schema, checkpoint written with the reference's keys (train.py:322-343) and
loadable into a fresh model through the reference's inference path (run_demo.py:86-92)."""
import os

import numpy as np
import pandas as pd
import pytest
import torch
import yaml

from _util import ROOT

pytestmark = pytest.mark.gpu


def _make_dataset(root, n_genes=24, seed=0):
    rng = np.random.default_rng(seed)
    rows = []
    for g in range(n_genes):
        tss = 1_000_000 + 100_000 * g
        depth = (rng.random((7, 40000)) < 0.3) * rng.exponential(1.0, (7, 40000))
        np.save(root / f"chr1:{tss - 20000}-{tss + 20000}.npy", depth.astype(np.float16))
        k = int(rng.integers(0, 4))
        names, scores = [], []
        for c in range(k):
            length = int(rng.integers(1800, 9000))
            s0 = 50_000_000 + 1_000_000 * g + 20_000 * c
            names.append(f"chr1:{s0}-{s0 + length}")
            scores.append(f"{1.5 + rng.random():.4f}")
            d = (rng.random((7, length)) < 0.3) * rng.exponential(1.0, (7, length))
            np.save(root / f"{names[-1]}.npy", d.astype(np.float16))
        rows.append(dict(gene_id=f"ENSG{g:011d}", expression=float(rng.exponential(3.0)), eid="E003",
                         label=(g // 4) % 2, chrom="chr1", start=tss, end=tss + 1,
                         strand="+-"[g % 2], split=1 + g % 4, neighbors=";".join(names), scores=";".join(scores)))
    meta = root / "train.csv"
    pd.DataFrame(rows).to_csv(meta, index=False)
    return meta


@pytest.mark.parametrize("regression", [False, True])
def test_train_cli_writes_reference_checkpoint(tmp_path, regression):
    import chromoformer.train as train_cli
    from chromoformer import ChromoformerClassifier, ChromoformerDataset, ChromoformerRegressor
    meta = _make_dataset(tmp_path)
    cfg = yaml.safe_load(open(os.path.join(ROOT, "chromoformer", "configs", "default.yaml")))
    cfg.update(num_epoch=3, bsz=4)                      # range(1, 3): two epochs
    cfg_path = tmp_path / "config.yaml"
    yaml.safe_dump(cfg, open(cfg_path, "w"))
    out = tmp_path / "ckpt.pt"
    argv = ["-o", str(out), "-c", str(cfg_path), "--exp-id", "test", "-m", str(meta), "-d", str(tmp_path),
            "--fold", "1", "--num-workers", "0"] + (["--regression"] if regression else [])
    train_cli.main(argv)
    ckpt = torch.load(out, map_location="cpu", weights_only=False)
    want = {"net", "optimizer", "epoch", "last_val_loss", "val_score", "val_label",
            "last_val_r2" if regression else "last_val_auc"}
    assert set(ckpt) == want and ckpt["epoch"] == 2
    assert len(ckpt["optimizer"]["state"]) == 334 and np.isfinite(float(ckpt["last_val_loss"]))
    # inference path of run_demo.py: fresh model, load_state_dict(ckpt['net']), forward
    cls = ChromoformerRegressor if regression else ChromoformerClassifier
    model = cls(cfg["n_feats"], cfg["embed"]["d_model"], cfg["d_head"], cfg["embed"], cfg["pairwise_interaction"],
                cfg["regulation"], seed=123)
    init = {k: v.clone() for k, v in model.state_dict().items()}
    model.load_state_dict(ckpt["net"])
    changed = sum(not torch.equal(init[k], v) for k, v in model.state_dict().items())
    assert changed >= 300                               # trained tensors differ from a fresh init
    model.cuda().eval()
    genes = pd.read_csv(meta).gene_id.tolist()[:6]
    ds = ChromoformerDataset(str(meta), str(tmp_path), genes, regression=regression)
    loader = torch.utils.data.DataLoader(ds, batch_size=6)
    d = next(iter(loader))
    mv = lambda v: {b: t.cuda() for b, t in v.items()}
    with torch.no_grad():
        y = model(mv(d["promoter_feats"]), mv(d["promoter_pad_masks"]), mv(d["pcre_feats"]), mv(d["pcre_pad_masks"]),
                  mv(d["interaction_masks"]), d["interaction_freq"].cuda())
    assert y.shape == (6, 1 if regression else 2) and torch.isfinite(y).all()
