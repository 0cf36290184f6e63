"""BF16-path deviation from the FP32 reference on the 100 demo genes and on synthetic genes, per kernel variant.

Prints one markdown table (committed under profiles/).  Needs a GPU; reads only tests/golden fixtures.
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402
from sklearn import metrics  # noqa: E402

from _util import demo_batch, golden  # noqa: E402
from chromoformer_b200 import ChromoformerClassifier, synthetic  # noqa: E402

VARIANTS = [
    ("this library, bf16 (default kernels)", {}),
    ("bf16, unfused single-query attention (CHROMO_NO_SQA_FUSED=1)", {"CHROMO_NO_SQA_FUSED": "1"}),
]


if __name__ == "__main__":
    import subprocess
    if len(sys.argv) > 1 and sys.argv[1] == "--child":
        g = golden("demo_logits.npz")
        batch = demo_batch(0, 100)
        syn = synthetic.make_batch(2048, ragged=True, seed=3)
        model = ChromoformerClassifier(seed=123).cuda().eval()
        with torch.no_grad():
            model.precision = "fp32"
            want_syn = model(*synthetic.forward_args(syn, "cuda")).cpu().numpy()
            model.precision = sys.argv[2]
            got = model(*synthetic.forward_args(batch, "cuda")).cpu().numpy()
            got_syn = model(*synthetic.forward_args(syn, "cuda")).cpu().numpy()
        np.savez(sys.argv[3], logits=got, syn_err=np.abs(got_syn - want_syn).max())
        sys.exit(0)
    g = golden("demo_logits.npz")
    amp = golden("demo_autocast.npz")
    labels = demo_batch(0, 100)["labels"].numpy()
    ref = g["logits"]
    sig = lambda z: 1.0 / (1.0 + np.exp(-z[:, 1].astype(np.float64)))
    a_ref, p_ref = metrics.roc_auc_score(labels, sig(ref)), metrics.average_precision_score(labels, sig(ref))
    print("| variant | max abs logit error (demo) | AUROC shift (demo) | AP shift (demo) | label agreement | max abs logit error (2048 synthetic genes) |")
    print("|---|---:|---:|---:|---:|---:|")

    def line(name, logits, syn_err):
        print("| %s | %.2e | %.2e | %.2e | %.3f | %s |" % (
            name, np.abs(logits - ref).max(), abs(metrics.roc_auc_score(labels, sig(logits)) - a_ref),
            abs(metrics.average_precision_score(labels, sig(logits)) - p_ref),
            np.mean((logits[:, 1] > logits[:, 0]) == (ref[:, 1] > ref[:, 0])), syn_err))

    line("reference under its own torch.autocast(bfloat16), CPU", amp["logits_autocast"], "n/a")
    runs = [("this library, fp32", "fp32", {})] + [(n, "bf16", e) for n, e in VARIANTS]
    for name, prec, env in runs:
        out = "/tmp/precision_%d.npz" % os.getpid()
        e = dict(os.environ); e.update(env)
        subprocess.run([sys.executable, os.path.abspath(__file__), "--child", prec, out], env=e, check=True,
                       stdout=subprocess.DEVNULL)
        r = np.load(out)
        line(name, r["logits"], "%.2e" % float(r["syn_err"]))
