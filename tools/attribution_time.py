"""Time the feature-attribution helpers on seeded synthetic genes.

    python tools/attribution_time.py [--genes 4096] [--steps 32] [--reps 3]

For FP32 and BF16 training workspaces, dense and ragged genes (synthetic.make_batch), it times
`attribution.input_gradients` (saliency over the features), the same with `freq=True` (features and
interaction_freq), saliency over interaction_freq alone (autograd with only interaction_freq requiring grad: the
backward stops after the Regulation transformer), and `attribution.integrated_gradients(steps)` without and with
`freq=True` (the joint path).  It prints genes/s (genes attributed per second, host clock around work that ends in a
device synchronise, after one warm-up call), plus the library launches of one forward + backward with and without
parameter gradients and of an interaction_freq-only one (chromo_launch_counter).  The card's name and power limit are
printed in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from chromoformer_b200 import ChromoformerClassifier, _lib, synthetic  # noqa: E402
from chromoformer_b200.attribution import input_gradients, integrated_gradients  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except (OSError, subprocess.SubprocessError, IndexError):
        q = torch.cuda.get_device_name(0) + ", power limit unknown"
    return q


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / reps


def freq_saliency(model, dev):
    """d logits[:, 1].sum() / d interaction_freq with the parameters and the features held fixed."""
    model.requires_grad_(False)
    fq = dev["interaction_freq"].clone().requires_grad_(True)
    g = torch.autograd.grad(model.forward_batch(dict(dev, interaction_freq=fq))[:, 1].sum(), [fq])
    model.requires_grad_(True)
    return g


def launches(model, batch, with_params, feats=True, freq=False):
    """Library launches of one forward + backward that returns the chosen input gradients."""
    lib = _lib.load()
    model.requires_grad_(with_params)
    args = synthetic.forward_args(batch, "cuda")
    leaves = []
    if feats:
        for i in (0, 2):
            args[i] = {b: t.clone().requires_grad_(True) for b, t in args[i].items()}
            leaves += list(args[i].values())
    if freq:
        args[5] = args[5].clone().requires_grad_(True)
        leaves.append(args[5])
    c0 = lib.chromo_launch_counter(0)
    out = model(*args)
    torch.autograd.grad(out[:, 1].sum(), leaves)
    torch.cuda.synchronize()
    n = lib.chromo_launch_counter(0) - c0
    model.zero_grad(set_to_none=True)
    model.requires_grad_(True)
    return n


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--genes", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=32)
    ap.add_argument("--chunk", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--json", default=None, help="also write the rows to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("attribution_time.py needs a CUDA device")
    print("card:", card(), flush=True)
    model = ChromoformerClassifier(seed=42).cuda()
    rows = []
    for ragged in (False, True):
        batch = synthetic.make_batch(a.genes, ragged=ragged, seed=1)
        small = synthetic.slice_batch(batch, 0, 64)
        dev = {k: ({b: t.cuda() for b, t in v.items()} if isinstance(v, dict) else v.cuda()) for k, v in batch.items()}
        for precision in ("fp32", "bf16"):
            model.precision = precision
            t_sal = timed(lambda: input_gradients(model, dev), a.reps)
            t_salf = timed(lambda: input_gradients(model, dev, freq=True), a.reps)
            t_fq = timed(lambda: freq_saliency(model, dev), a.reps)
            t_ig = timed(lambda: integrated_gradients(model, dev, steps=a.steps, chunk=a.chunk), max(1, a.reps - 2))
            t_igf = timed(lambda: integrated_gradients(model, dev, steps=a.steps, chunk=a.chunk, freq=True),
                          max(1, a.reps - 2))
            row = {"genes": a.genes, "ragged": ragged, "precision": precision,
                   "saliency_genes_per_s": a.genes / t_sal, "saliency_s": t_sal,
                   "saliency_feats_and_freq_s": t_salf, "saliency_freq_only_s": t_fq,
                   "saliency_freq_only_genes_per_s": a.genes / t_fq,
                   f"ig{a.steps}_genes_per_s": a.genes / t_ig, f"ig{a.steps}_s": t_ig,
                   f"ig{a.steps}_joint_freq_genes_per_s": a.genes / t_igf, f"ig{a.steps}_joint_freq_s": t_igf,
                   "launches_64_genes_feature_grads_only": launches(model, small, False),
                   "launches_64_genes_with_param_grads": launches(model, small, True),
                   "launches_64_genes_freq_grad_only": launches(model, small, False, feats=False, freq=True)}
            print(json.dumps(row), flush=True)
            rows.append(row)
    model.precision = "fp32"
    if a.json:
        with open(a.json, "w") as f:
            json.dump({"card": card(), "rows": rows}, f, indent=1)


if __name__ == "__main__":
    main()
