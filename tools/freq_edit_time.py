"""Time the contact analyses (interaction-frequency edits) on seeded synthetic genes.

    python tools/freq_edit_time.py [--genes 18955] [--reps 3] [--chunk 65536]

BF16, one dense set and one ragged set of the demo's shape (synthetic.make_batch(ragged=True)).  For each set and each
analysis (attribution.contact_knockout; attribution.contact_response with 8 values; exact attribution.contact_shapley)
it times
  (a) the analysis: one Embedding / Pairwise pass per gene, the Regulation transformer and the head replayed over the
      frequency variants (chromo_freq_edits);
  (b) the baseline: the same variants as forward_batch calls with the edited interaction_freq, built on the device
      beforehand: call s runs variant s of every gene that has one, over the genes' shared feature tensors.
Both arms are warmed up once, then timed `reps` times each, alternating, with CUDA events; the median and the range are
printed, with the library launches of one sweep (chromo_launch_counter), the workspace bytes per variant of (a), the max
|(a) - (b)| over the variant values of the target logit, and the card's name and power limit, all from the same run.
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
VALUES = [0.0, 0.25, 0.5, 1.0, 1.5, 2.0, 3.0, 4.0]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except (OSError, subprocess.SubprocessError, IndexError):
        q = torch.cuda.get_device_name(0) + ", power limit unknown"
    return q


def recorded(fn):
    """Run fn with attribution._freq_replay wrapped: (var_gene, the device edits of every variant, var_logits)."""
    orig, rec = attribution._freq_replay, {}

    def spy(model, dev_batch, bins, var_gene, var_freq, chunk, dense):
        out = orig(model, dev_batch, bins, var_gene, var_freq, chunk, dense)
        rec.update(gene=var_gene, freq=var_freq(0, len(var_gene)), var_logits=out[1])
        return out
    attribution._freq_replay = spy
    try:
        fn()
    finally:
        attribution._freq_replay = orig
    return rec["gene"], rec["freq"], rec["var_logits"]


def edited_batches(dev, var_gene, var_freq):
    """The variants as ordinary batches, built on the device: batch s holds variant s of every gene that has one, with
    its edited interaction_freq.  The genes are sorted by their variant count once, so the genes of batch s are a prefix
    of the sorted genes and every batch shares their feature tensors.  Returns the batches and, for each variant, its
    row in the concatenated outputs."""
    B = dev["interaction_freq"].shape[0]
    counts = np.bincount(var_gene, minlength=B)
    starts = np.concatenate([[0], np.cumsum(counts)])
    order = np.argsort(-counts, kind="stable")
    rank = np.empty(B, dtype=np.int64)
    rank[order] = np.arange(B)
    o = torch.from_numpy(order).cuda()
    srt = {key: {bb: dev[key][bb][o].contiguous() for bb in BINS} for key in attribution._GENE_KEYS}
    g = torch.from_numpy(np.asarray(var_gene)).cuda()
    freq = torch.where(torch.isnan(var_freq), dev["interaction_freq"][g], var_freq)
    sizes = [int((counts > s).sum()) for s in range(int(counts.max()))]
    out = []
    for s, m in enumerate(sizes):
        b = {key: {bb: srt[key][bb][:m] for bb in BINS} for key in attribution._GENE_KEYS}
        b["interaction_freq"] = freq[torch.from_numpy(starts[order[:m]] + s).cuda()]
        out.append(b)
    offsets = np.concatenate([[0], np.cumsum(sizes)])
    row = offsets[np.arange(len(var_gene)) - starts[var_gene]] + rank[var_gene]
    return out, torch.from_numpy(row).cuda()


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
    analyses = {"knockout": lambda dev: attribution.contact_knockout(model, dev, chunk=args.chunk),
                "response8": lambda dev: attribution.contact_response(model, dev, VALUES, chunk=args.chunk),
                "shapley": lambda dev: attribution.contact_shapley(model, dev, chunk=args.chunk)}
    for ragged in (False, True):
        batch = synthetic.make_batch(n, ragged=ragged, seed=11)
        dev = {key: ({b: x.cuda() for b, x in v.items()} if isinstance(v, dict) else v.cuda())
               for key, v in batch.items() if key in synthetic.FORWARD_KEYS}
        live = attribution._live(dev, list(model.binsizes)).cpu()
        for mode, analysis in analyses.items():
            var_gene, var_freq, vl = recorded(lambda: analysis(dev))
            V = len(var_gene)
            base, row = edited_batches(dev, var_gene, var_freq)
            del var_freq

            def arm_a():
                return analysis(dev)

            def arm_b():
                with torch.no_grad():
                    return torch.cat([model.forward_batch(b) for b in base])

            fwd = arm_b()
            err = (vl[:, t] - fwd[row, t]).abs().max().item()
            torch.cuda.synchronize()
            counts = []
            for fn in (arm_a, arm_b):
                lib.chromo_launch_counter(1)
                fn()
                counts.append(int(lib.chromo_launch_counter(1)))
            times = {"a": [], "b": []}
            for _ in range(args.reps):
                for key, fn in (("a", arm_a), ("b", arm_b)):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    fn()
                    e1.record()
                    torch.cuda.synchronize()
                    times[key].append(e0.elapsed_time(e1))
            cfg = _lib.Config.from_buffer_copy(model._cfg)
            per_gene = int(np.bincount(var_gene).max())
            genes_call = max(1, min(n, args.chunk // max(1, per_gene)))
            ws = lib.chromo_freq_edits_workspace_floats(ctypes.byref(cfg), genes_call, args.chunk, _lib.F_BF16) * 4
            ws_small = lib.chromo_freq_edits_workspace_floats(ctypes.byref(cfg), genes_call, args.chunk // 2,
                                                              _lib.F_BF16) * 4
            ta, tb = statistics.median(times["a"]), statistics.median(times["b"])
            res = {"set": "ragged" if ragged else "dense", "analysis": mode, "genes": n, "variants": V,
                   "live_slots": int(live.sum()),
                   "a_ms": round(ta, 1), "a_ms_range": [round(min(times["a"]), 1), round(max(times["a"]), 1)],
                   "b_ms": round(tb, 1), "b_ms_range": [round(min(times["b"]), 1), round(max(times["b"]), 1)],
                   "speedup_a_over_b": round(tb / ta, 2), "a_launches": counts[0], "b_launches": counts[1],
                   "a_workspace_bytes_per_variant": round((ws - ws_small) / (args.chunk - args.chunk // 2)),
                   "a_workspace_bytes": ws, "max_abs_a_minus_b": err}
            print(json.dumps(res), flush=True)
            del base, fwd, vl, row
            model._ws_cache.clear()
            model.mark_parameters_changed()      # (a new workspace may reuse a freed address: repack the BF16 weights)
            torch.cuda.empty_cache()
        del dev


if __name__ == "__main__":
    main()
