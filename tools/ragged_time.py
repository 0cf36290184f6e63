"""genes/s of the device-resident 18,955-gene sweep (BF16), dense and ragged genes, with and without the ragged plan
(csrc/ragged.cu; the CHROMO_F_DENSE hint switches it off)."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from chromoformer_b200 import ChromoformerClassifier, synthetic, _lib  # noqa: E402
from chromoformer_b200.engine import InferenceEngine  # noqa: E402

N = int(sys.argv[1]) if len(sys.argv) > 1 else 18955
model = ChromoformerClassifier(seed=123).cuda().eval()
model.precision = "bf16"
lib = _lib.load()
for name, ragged in (("dense", False), ("ragged", True)):
    host = synthetic.make_batch(N, ragged=ragged, seed=1000)
    eng = InferenceEngine(model, chunk=N)
    res = eng.to_device(host)
    out = torch.empty(N, 2, device="cuda")
    outs = {}
    for plan in (True, False):
        res["dense"] = not plan                  # (CHROMO_F_DENSE hint only for the plan-off leg: the plan is built otherwise)
        for _ in range(3):
            eng.predict_device(res, out)
        torch.cuda.synchronize()
        lib.chromo_launch_counter(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(30):
            eng.predict_device(res, out)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 30
        outs[plan] = out.clone()
        print(f"{name:6s} plan={'on ' if plan else 'off'}: {ms:.3f} ms/sweep = {N / ms * 1e3 / 1e6:.3f} M genes/s, "
              f"{lib.chromo_launch_counter(0) // 30} launches", flush=True)
    print(f"{name:6s} max |dlogit| plan on/off = {(outs[True] - outs[False]).abs().max().item():.2e}")
    del res
    model._ws_cache.clear()
