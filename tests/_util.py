"""Shared helpers for the test-suite (fixtures under tests/golden/)."""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLDEN = os.path.join(HERE, "golden")
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
BINS = (2000, 500, 100)
KWS = ({"n_layers": 1, "n_heads": 2, "d_model": 128, "d_ff": 128},
       {"n_layers": 2, "n_heads": 2, "d_model": 128, "d_ff": 256},
       {"n_layers": 6, "n_heads": 8, "d_model": 256, "d_ff": 256})


def golden(name):
    return np.load(os.path.join(GOLDEN, name), allow_pickle=False)


def demo_batch(lo=0, hi=100, full_masks=True):
    """The reference's collated demo items [lo, hi) rebuilt from tests/golden/demo_items.npz."""
    g = golden("demo_items.npz")
    B = hi - lo
    out = {"promoter_feats": {}, "promoter_pad_masks": {}, "pcre_feats": {}, "pcre_pad_masks": {},
           "interaction_masks": {}}
    k = torch.from_numpy(g["n_partners"][lo:hi]).long()
    for b in BINS:
        n = 40000 // b
        out["promoter_feats"][b] = torch.from_numpy(g[f"xp_{b}"][lo:hi])
        out["pcre_feats"][b] = torch.from_numpy(g[f"xc_{b}"][lo:hi])
        sp = torch.from_numpy(g[f"span_p_{b}"][lo:hi]).long()          # [B,2]
        sc = torch.from_numpy(g[f"span_c_{b}"][lo:hi]).long()          # [B,8,2]
        pos = torch.arange(n)
        vp = (pos.view(1, n) >= sp[:, :1]) & (pos.view(1, n) < (sp[:, :1] + sp[:, 1:2]))      # [B,n]
        vc = (pos.view(1, 1, n) >= sc[:, :, :1]) & (pos.view(1, 1, n) < (sc[:, :, :1] + sc[:, :, 1:2]))
        if full_masks:
            mp = ~(vp.view(B, 1, 1, n, 1) & vp.view(B, 1, 1, 1, n))
            mc = ~(vp.view(B, 1, 1, n, 1) & vc.view(B, 8, 1, 1, n))
        else:
            mp = (~vp).view(B, 1, n)        # centre row: the promoter is never padded in the demo
            mc = ~vc
        out["promoter_pad_masks"][b] = mp.contiguous()
        out["pcre_pad_masks"][b] = mc.contiguous()
        idx = torch.arange(9)
        inside = (idx.view(1, 9, 1) <= k.view(B, 1, 1)) & (idx.view(1, 1, 9) <= k.view(B, 1, 1))
        out["interaction_masks"][b] = (~inside).unsqueeze(1)
    out["interaction_freq"] = torch.from_numpy(g["freq"][lo:hi])
    out["labels"] = torch.from_numpy(g["labels"][lo:hi])
    out["n_partners"] = k
    return out


def smoke_inputs():
    """RNG draw sequence of net.py:437-466; call right after building the three models."""
    bsz, i_max = 8, 8
    ns = (20, 80, 400)
    x_p = [torch.randn([bsz, 1, n, 7]) for n in ns]
    x_c = [torch.randn([bsz, i_max, n, 7]) for n in ns]
    m_p = [torch.randn([bsz, 1, 1, n, n]).bool() for n in ns]
    m_c = [torch.randn([bsz, i_max, 1, n, n]).bool() for n in ns]
    i_m = [torch.randn([bsz, 1, 1 + i_max, 1 + i_max]).bool() for _ in ns]
    freq = torch.randn([bsz, 1 + i_max, 1 + i_max])
    return x_p, m_p, x_c, m_c, i_m, freq


def as_dict(lst):
    return {b: t for b, t in zip(BINS, lst)}


def reference_available():
    """True when $CHROMOFORMER_REF names a checkout of the upstream chromoformer repository."""
    return os.path.isdir(os.environ.get("CHROMOFORMER_REF", ""))


def import_reference():
    ref = os.environ["CHROMOFORMER_REF"]
    if not getattr(torch.Tensor.cuda, "_patched_identity", False) and not torch.cuda.is_available():
        ident_t = lambda self, *a, **k: self
        ident_t._patched_identity = True
        torch.Tensor.cuda = ident_t
        torch.nn.Module.cuda = lambda self, *a, **k: self
    # the repo ships its own `chromoformer` shim package: load the reference under another name
    import importlib.util
    import types
    pkg = types.ModuleType("chromoformer_reference")
    pkg.__path__ = [os.path.join(ref, "chromoformer")]
    sys.modules.setdefault("chromoformer_reference", pkg)
    mods = {}
    for name in ("modules", "net", "data"):
        full = f"chromoformer_reference.{name}"
        if full in sys.modules:
            mods[name] = sys.modules[full]
            continue
        spec = importlib.util.spec_from_file_location(full, os.path.join(ref, "chromoformer", f"{name}.py"))
        mod = importlib.util.module_from_spec(spec)
        sys.modules[full] = mod
        spec.loader.exec_module(mod)
        mods[name] = mod
    return mods["net"], mods["data"]
