"""Does a gene's BF16 result depend on where it sits in a chunk?  Prints max |diff| per shift."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from chromoformer_b200 import ChromoformerClassifier, synthetic
from chromoformer_b200.engine import InferenceEngine

model = ChromoformerClassifier(seed=123).cuda().eval()
model.precision = sys.argv[1] if len(sys.argv) > 1 else "bf16"
batch = synthetic.make_batch(600, ragged=False, seed=0)
eng = InferenceEngine(model, chunk=4096)
dev = eng.to_device(batch)
base = eng.predict_device(dev).cpu()
again = eng.predict_device(dev).cpu()
print("run-to-run:", (base - again).abs().max().item())
for shift in (1, 3, 7, 14, 64, 100):
    sub = eng.to_device(synthetic.slice_batch(batch, shift, 600))
    got = eng.predict_device(sub).cpu()
    d = (got - base[shift:]).abs()
    print(f"shift {shift}: max {d.max().item():.3e}, genes differing {(d.max(1).values > 0).sum().item()} / {d.size(0)}")
