"""Time the in-silico pCRE deletion on seeded synthetic genes.

    python tools/deletion_time.py [--genes 18955] [--reps 3] [--chunk 4096]

BF16, one dense set and one ragged set of the demo's shape (synthetic.make_batch(ragged=True)).  For each set it times
  (a) attribution.pcre_deletion: one Embedding / Pairwise pass per gene, the Regulation transformer and the head
      replayed over the I + 1 variants of each gene (chromo_pcre_deletion);
  (b) the baseline: I + 1 forward_batch calls, one per deleted slot and one for the promoter alone, on reassembled batches
      built on the device beforehand (later slots moved up, a dummy slot appended, as data.py:175-203 would build them).
Each sweep covers every deletion of every gene.  Both arms are warmed up once, then timed `reps` times each, alternating,
with CUDA events; the median and the range are printed.  Also printed: genes/s, the speed-up of (a) over (b), the
library launches of one sweep (chromo_launch_counter), the workspace bytes per gene of (a) and of a forward, and the
max |(a) - (b)| over live slots and promoter-only.  The card's name and power limit are printed in the same run.
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

import torch  # noqa: E402

from chromoformer_b200 import ChromoformerClassifier, _lib, synthetic  # noqa: E402
from chromoformer_b200.attribution import pcre_deletion  # noqa: E402

KEYS = ("promoter_feats", "promoter_pad_masks", "pcre_feats", "pcre_pad_masks", "interaction_masks")


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except (OSError, subprocess.SubprocessError, IndexError):
        q = torch.cuda.get_device_name(0) + ", power limit unknown"
    return q


def reassembled(dev, k, i):
    """The batch with pCRE slot i removed from every gene that has it (i None: every pCRE removed), on the device."""
    B, I = dev["interaction_freq"].shape[0], dev["pcre_feats"][100].shape[1]
    S = I + 1
    slot = torch.arange(I, device=k.device).view(1, I)
    if i is None:
        src, k_new = torch.full((B, I), I, device=k.device), torch.zeros_like(k)
    else:
        has = (i < k).view(B, 1)
        shifted = torch.where(slot < i, slot, slot + 1)                       # slot I: the appended dummy
        src = torch.where(has, shifted, slot.expand(B, I))
        k_new = k - has.view(B).long()
    out = {"promoter_feats": dev["promoter_feats"], "promoter_pad_masks": dev["promoter_pad_masks"],
           "pcre_feats": {}, "pcre_pad_masks": {}, "interaction_masks": {}}
    idx = torch.arange(S, device=k.device)
    inside = (idx.view(1, S, 1) <= k_new.view(B, 1, 1)) & (idx.view(1, 1, S) <= k_new.view(B, 1, 1))
    for b, x in dev["pcre_feats"].items():
        m = dev["pcre_pad_masks"][b]
        xd = torch.cat([x, torch.zeros_like(x[:, :1])], 1)
        md = torch.cat([m, torch.ones_like(m[:, :1])], 1)
        out["pcre_feats"][b] = torch.gather(xd, 1, src.view(B, I, 1, 1).expand(B, I, *x.shape[2:])).contiguous()
        out["pcre_pad_masks"][b] = torch.gather(md, 1, src.view(B, I, 1).expand(B, I, m.shape[2])).contiguous()
        out["interaction_masks"][b] = (~inside).unsqueeze(1)
    tok = torch.cat([torch.zeros(B, 1, dtype=torch.long, device=k.device), src + 1], 1)      # token S: the dummy
    f = torch.nn.functional.pad(dev["interaction_freq"], (0, 1, 0, 1))
    f = torch.gather(f, 1, tok.view(B, S, 1).expand(B, S, S + 1))
    out["interaction_freq"] = torch.gather(f, 2, tok.view(B, 1, S).expand(B, S, S)).contiguous()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--genes", type=int, default=18955)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--chunk", type=int, default=4096)
    args = ap.parse_args()
    lib = _lib.load()
    print(f"card: {card()}")
    model = ChromoformerClassifier(seed=7).cuda().eval()
    model.precision = "bf16"
    n = args.genes
    for ragged in (False, True):
        batch = synthetic.make_batch(n, ragged=ragged, seed=11)
        dev = {key: ({b: t.cuda() for b, t in v.items()} if isinstance(v, dict) else v.cuda())
               for key, v in batch.items() if key in synthetic.FORWARD_KEYS}
        k = batch["n_partners"].cuda()
        I = dev["pcre_feats"][100].shape[1]
        variants = [reassembled(dev, k, i) for i in range(I)] + [reassembled(dev, k, None)]

        def arm_a():
            return pcre_deletion(model, dev, chunk=args.chunk)

        def arm_b():
            with torch.no_grad():
                return [model.forward_batch(v) for v in variants]

        d, fwd = arm_a(), arm_b()
        torch.cuda.synchronize()
        live = torch.arange(I, device=k.device).view(1, I) < k.view(-1, 1)
        err = max((d["without"] - torch.stack(fwd[:I], 1))[live].abs().max().item() if live.any() else 0.0,
                  (d["promoter_only"] - fwd[I]).abs().max().item())
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
        io_cfg = _lib.Config.from_buffer_copy(model._cfg)
        chunk = min(n, args.chunk)
        ws_del = lib.chromo_pcre_deletion_workspace_floats(ctypes.byref(io_cfg), chunk, _lib.F_BF16) * 4 / chunk
        ws_fwd = lib.chromo_workspace_floats(ctypes.byref(io_cfg), chunk, _lib.F_BF16) * 4 / chunk
        ta, tb = statistics.median(times["a"]), statistics.median(times["b"])
        res = {"set": "ragged" if ragged else "dense", "genes": n, "live_slots": int(live.sum()),
               "a_ms_per_sweep": round(ta, 2), "a_ms_range": [round(min(times["a"]), 2), round(max(times["a"]), 2)],
               "b_ms_per_sweep": round(tb, 2), "b_ms_range": [round(min(times["b"]), 2), round(max(times["b"]), 2)],
               "a_genes_per_s": round(n / ta * 1e3), "b_genes_per_s": round(n / tb * 1e3),
               "speedup_a_over_b": round(tb / ta, 2), "a_launches_per_sweep": counts[0],
               "b_launches_per_sweep": counts[1], "a_calls_per_sweep": (n + args.chunk - 1) // args.chunk,
               "a_workspace_bytes_per_gene": round(ws_del), "forward_workspace_bytes_per_gene": round(ws_fwd),
               "max_abs_a_minus_b": err}
        print(json.dumps(res), flush=True)
        del variants, dev, d, fwd
        model._ws_cache.clear()
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
