"""Time histone-mark occlusion maps on seeded synthetic genes.

    python tools/occlusion_time.py [--genes 18955] [--reps 3] [--chunk 65536]

BF16, one dense set and one ragged set of the demo's shape (synthetic.make_batch(ragged=True)); the map of
attribution.occlusion_map(window=1, marks="all"): every mark removed over each 2 kb window (20 per region) of every pCRE
and of the promoter.  For each set it times, with CUDA events, `reps` times each, alternating:
  (a) the pCRE part of the map as attribution.occlusion_map runs it: attribution.pcre_occlusion over the (gene, live slot,
      window) variants - one Embedding / Pairwise pass per gene, one Pairwise pass over the occluded region per variant,
      the Regulation transformer and the head replayed over the variants (chromo_pcre_occlusion);
  (b) the same variants as a user builds them today: for each (slot, window) the genes whose slot is a pCRE, their
      features copied on the device with the window zeroed, run through forward_batch;
  (m) the whole occlusion_map call, which adds the promoter windows (20 forward_batch sweeps over occluded copies).
Printed per set: the median and range of each arm, the library launches of one sweep (chromo_launch_counter), the
workspace bytes per variant of (a), the max |(a) - (b)| over the target logit of every variant, and the card's name and
power limit, all from the same run.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from chromoformer_b200 import ChromoformerClassifier, _lib, synthetic  # noqa: E402
from chromoformer_b200 import attribution  # noqa: E402

BINS = (2000, 500, 100)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except (OSError, subprocess.SubprocessError, IndexError):
        q = torch.cuda.get_device_name(0) + ", power limit unknown"
    return q


def descriptors(live, n):
    """The pCRE variants of occlusion_map(window=1, marks="all"), in its order: (gene, live slot) gene-major, then the
    windows.  n: bins per resolution."""
    W = n[0]
    rb = np.stack([np.stack([np.arange(W), np.arange(1, W + 1)], 1) * (nr // W) for nr in n], 1)     # [W, n_res, 2]
    g, i = np.nonzero(live.numpy())
    return np.repeat(g, W), np.repeat(i, W), np.tile(rb, (len(g), 1, 1)), np.full(len(g) * W, 127)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--genes", type=int, default=18955)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--chunk", type=int, default=65536)
    args = ap.parse_args()
    lib = _lib.load()
    print(f"card: {card()}", flush=True)
    model = ChromoformerClassifier(seed=7).cuda().eval()
    model.precision = "bf16"
    t = 1
    n = args.genes
    nb = [40000 // b for b in BINS]
    W = nb[0]
    for ragged in (False, True):
        batch = synthetic.make_batch(n, ragged=ragged, seed=11)
        dev = {key: ({b: x.cuda() for b, x in v.items()} if isinstance(v, dict) else v.cuda())
               for key, v in batch.items() if key in synthetic.FORWARD_KEYS}
        live = attribution._live(dev, list(BINS)).cpu()
        I = live.shape[1]
        gene, slot, var_bins, marks = descriptors(live, nb)
        V = len(gene)
        # (b): per slot, the genes whose slot is a pCRE and their inputs, gathered once
        per_slot = []
        for i in range(I):
            idx = torch.nonzero(live[:, i]).view(-1).cuda()
            if idx.numel():
                per_slot.append((i, idx, {key: ({b: x[idx] for b, x in v.items()} if isinstance(v, dict) else v[idx])
                                          for key, v in dev.items()}))

        def arm_a():
            return attribution.pcre_occlusion(model, dev, gene, slot, var_bins, marks, chunk=args.chunk)

        def arm_b():
            out = []
            with torch.no_grad():
                for i, idx, sub in per_slot:
                    for w in range(W):
                        x = {}
                        for b, nr in zip(BINS, nb):
                            k = nr // W
                            x[b] = sub["pcre_feats"][b].clone()
                            x[b][:, i, w * k:(w + 1) * k, :] = 0
                        out.append(model.forward_batch({**sub, "pcre_feats": x}))
            return out

        def arm_m():
            return attribution.occlusion_map(model, dev, window=1, marks="all", chunk=args.chunk)

        # the variant values of (a) against (b), both in occlusion_map's [B, I, W] layout
        a = arm_a()["variants"][:, t]
        pa = torch.full((n, I, W), float("nan"), device="cuda")
        pa[torch.from_numpy(gene).cuda(), torch.from_numpy(slot).cuda(), torch.from_numpy(np.tile(np.arange(W), V // W)).cuda()] = a
        pb = torch.full((n, I, W), float("nan"), device="cuda")
        outs = iter(arm_b())
        for i, idx, _ in per_slot:
            for w in range(W):
                pb[idx, i, w] = next(outs)[:, t]
        lv = live.cuda()
        err = (pa[lv] - pb[lv]).abs().max().item()
        torch.cuda.synchronize()
        counts = []
        for fn in (arm_a, arm_b, arm_m):
            lib.chromo_launch_counter(1)
            fn()
            counts.append(int(lib.chromo_launch_counter(1)))
        times = {"a": [], "b": [], "m": []}
        for _ in range(args.reps):
            for key, fn in (("a", arm_a), ("b", arm_b), ("m", arm_m)):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                fn()
                e1.record()
                torch.cuda.synchronize()
                times[key].append(e0.elapsed_time(e1))
        cfg = _lib.Config.from_buffer_copy(model._cfg)
        genes_call = max(1, min(n, args.chunk // (I * W)))
        ws = lib.chromo_pcre_occlusion_workspace_floats(ctypes.byref(cfg), genes_call, args.chunk, _lib.F_BF16) * 4
        ws_small = lib.chromo_pcre_occlusion_workspace_floats(ctypes.byref(cfg), genes_call, args.chunk // 2, _lib.F_BF16) * 4
        med = {k: statistics.median(v) for k, v in times.items()}
        res = {"set": "ragged" if ragged else "dense", "genes": n, "pcre_variants": V, "live_slots": int(live.sum()),
               "windows": W}
        for k in ("a", "b", "m"):
            res[f"{k}_ms"] = round(med[k], 1)
            res[f"{k}_ms_range"] = [round(min(times[k]), 1), round(max(times[k]), 1)]
        res.update({"speedup_a_over_b": round(med["b"] / med["a"], 2), "a_launches": counts[0], "b_launches": counts[1],
                    "m_launches": counts[2],
                    "a_workspace_bytes_per_variant": round((ws - ws_small) / (args.chunk - args.chunk // 2)),
                    "a_workspace_bytes": ws, "max_abs_a_minus_b": err})
        print(json.dumps(res), flush=True)
        del dev, per_slot, pa, pb, a
        model._ws_cache.clear()
        model.mark_parameters_changed()      # (a new workspace may reuse a freed address: repack the BF16 weights)
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
