"""Histone-mark occlusion (chromo_pcre_occlusion, csrc/occlusion.cu; attribution.pcre_occlusion / occlusion_map) against
the CPU oracle of the occluded genes rebuilt on the host, against the library's own forward of those genes, and for the
exact cases: dead slots, invalid descriptors, independence from the other variants, CUDA-graph capture."""
import ctypes

import numpy as np
import pytest
import torch

from _util import BINS, KWS
from chromoformer_b200 import ChromoformerClassifier, ChromoformerRegressor, _lib, synthetic
from chromoformer_b200.attribution import occlusion_map, pcre_occlusion
from chromoformer_b200.model import _BatchIO
from oracle import chromoformer_oracle as oracle

pytestmark = pytest.mark.gpu
REL32 = 2e-4           # FP32: of the max-abs oracle logit
TOL16 = 5e-3           # BF16, absolute
REG4 = {"n_layers": 2, "n_heads": 4, "d_model": 128, "d_ff": 256}     # reg_heads != 8: no fused Regulation kernel
NB = [40000 // b for b in BINS]      # bins per resolution: 20, 80, 400


def _mk(cls=ChromoformerClassifier, seed=11, i_max=8, reg=None):
    return cls(7, 128, 128, dict(KWS[0]), dict(KWS[1]), dict(reg or KWS[2]), seed=seed, i_max=i_max)


def _copy(batch, idx=None):
    def pick(t):
        return (t if idx is None else t[torch.as_tensor(idx, device=t.device)]).clone()
    return {key: ({b: pick(t) for b, t in v.items()} if isinstance(v, dict) else pick(v))
            for key, v in batch.items() if key in synthetic.FORWARD_KEYS}


def _cuda(batch):
    return {k: ({b: t.cuda() for b, t in v.items()} if isinstance(v, dict) else v.cuda()) for k, v in _copy(batch).items()}


def _live(batch):
    im = torch.stack([batch["interaction_masks"][b].reshape(batch["interaction_freq"].shape) for b in BINS])
    return (~im[:, :, 0, 1:].bool()).any(0).cpu()


def _occluded(batch, gene, slot, bins, marks):
    """One gene per variant, rebuilt with pcre_feats[r][g, slot, lo:hi, m] = 0 for the marks m of the bit set."""
    out = _copy(batch, list(gene))
    for v in range(len(gene)):
        ms = [m for m in range(7) if (int(marks[v]) >> m) & 1]
        for r, b in enumerate(BINS):
            lo, hi = int(bins[v][r][0]), int(bins[v][r][1])
            x = out["pcre_feats"][b]
            for m in ms:
                x[v, int(slot[v]), lo:hi, m] = 0
    return out


def _oracle(sd, batch, rows=8, reg_heads=8):
    heads = {"embed": 2, "pairwise_interaction": 2, "regulation": reg_heads}
    outs = []
    B = batch["interaction_freq"].shape[0]
    for lo in range(0, B, rows):
        part = synthetic.expand_full_masks(synthetic.slice_batch(_copy(batch), lo, min(B, lo + rows)))
        with torch.no_grad():
            outs.append(oracle.chromoformer_forward(sd, *synthetic.forward_args(part), heads=heads))
    return torch.cat(outs)


def _variants(B, I, V, seed, live=None):
    """Random windows with random mark sets, single marks, every mark, and ranges at one resolution only; on live slots
    when `live` is given."""
    gen = np.random.default_rng(seed)
    gene, slot, bins, marks = [], [], [], []
    for v in range(V):
        g = int(gen.integers(B))
        cand = np.nonzero(live[g].numpy())[0] if live is not None and live[g].any() else np.arange(I)
        kind = v % 4
        rb = []
        w0 = int(gen.integers(NB[0]))
        w1 = int(gen.integers(w0 + 1, NB[0] + 1))
        only = int(gen.integers(len(NB)))
        for r, n in enumerate(NB):
            if kind == 3 and r != only:
                rb.append((3, 3))                              # empty: this resolution untouched
            elif kind == 3:
                lo = int(gen.integers(n))
                rb.append((lo, int(gen.integers(lo, n + 1))))
            else:
                rb.append((w0 * n // NB[0], w1 * n // NB[0]))
        m = [int(gen.integers(1, 128)), 1 << int(gen.integers(7)), 127, int(gen.integers(1, 128))][kind]
        gene.append(g), slot.append(int(gen.choice(cand))), bins.append(rb), marks.append(m)
    return np.array(gene), np.array(slot), np.array(bins), np.array(marks)


@pytest.mark.parametrize("tag,ragged,i_max,n,reg", [("clf", True, 8, 3, None), ("reg", False, 8, 2, None),
                                                    ("reg", True, 16, 2, None), ("clf", False, 16, 2, None),
                                                    ("clf", True, 8, 2, REG4)])
def test_against_the_oracle_of_the_occluded_gene(tag, ragged, i_max, n, reg):
    cls = ChromoformerRegressor if tag == "reg" else ChromoformerClassifier
    model = _mk(cls, i_max=i_max, reg=reg)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    batch = synthetic.make_batch(n, i_max=i_max, ragged=ragged, seed=41, stress=True)
    gene, slot, bins, marks = _variants(n, i_max, 12, seed=n + i_max, live=_live(batch))
    want = _oracle(sd, _occluded(batch, gene, slot, bins, marks), reg_heads=(reg or KWS[2])["n_heads"])
    scale = want.abs().max().item()
    model.cuda().eval()
    for precision in ("fp32", "bf16"):
        model.precision = precision
        d = pcre_occlusion(model, batch, gene, slot, bins, marks)
        err = (d["variants"].cpu() - want).abs().max().item()
        print(f"{precision}: max |error| {err:.3e} (max |logit| {scale:.3f})")
        assert err <= (REL32 * scale if precision == "fp32" else TOL16), err


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_against_the_forward_of_the_occluded_genes(precision):
    n, I = 96, 8
    model = _mk(seed=3).cuda().eval()
    model.precision = precision
    dev = _cuda(synthetic.make_batch(n, ragged=True, seed=6, stress=True))
    live = _live(dev)
    tol = 1e-6 if precision == "fp32" else TOL16
    gene, slot, bins, marks = _variants(n, I, 200, seed=5, live=live)
    for dense in (True, False):
        d = pcre_occlusion(model, dev, gene, slot, bins, marks, dense=dense)
        with torch.no_grad():
            plain = model.forward_batch(dev, dense=dense)
            want = model.forward_batch(_occluded(dev, gene, slot, bins, marks))
        assert torch.equal(d["logits"], plain)
        err = (d["variants"] - want).abs().max().item()
        print(f"{precision} dense={dense}: max |variant - forward of the occluded gene| {err:.3e}")
        assert err <= tol
    # no change at all: empty mark set, empty ranges, ranges under the pad mask only
    V = 60
    gene = np.nonzero(live.any(1).numpy())[0][np.arange(V) % int(live.any(1).sum())]
    slot = np.array([int(np.nonzero(live[g].numpy())[0][-1]) for g in gene])
    bins = np.tile(np.array([[0, n_r] for n_r in NB]), (V, 1, 1))
    marks = np.full(V, 127)
    marks[:20] = 0
    bins[20:40] = 5
    pad = {}
    for r, b in enumerate(BINS):
        m = dev["pcre_pad_masks"][b].reshape(n, I, -1, NB[r])
        pad[b] = m[:, :, m.shape[2] // 2].cpu().bool()        # the centre row: the only one the logits see
    for v in range(40, V):
        for r, b in enumerate(BINS):
            row = pad[b][gene[v], slot[v]]                 # the pad-mask row of the region: bins before its valid span
            lo = int(torch.nonzero(~row)[0]) if (~row).any() else 0
            bins[v, r] = (0, lo)
    d = pcre_occlusion(model, dev, gene, slot, bins, marks)
    err = (d["variants"] - d["logits"][torch.from_numpy(gene).cuda()]).abs().max().item()
    print(f"{precision}: max |no-op variant - gene| {err:.3e}")
    assert err <= tol


def test_exact_cases_dead_slots_and_invalid_descriptors():
    n, I = 32, 8
    model = _mk(seed=13).cuda().eval()
    batch = synthetic.make_batch(n, ragged=True, seed=2)
    live = _live(batch)
    for precision in ("bf16", "fp32"):
        model.precision = precision
        gene, slot, bins, marks = _variants(n, I, 64, seed=9)
        dead = ~live[torch.from_numpy(gene), torch.from_numpy(slot)].numpy()
        assert dead.any() and (~dead).any()
        ref = pcre_occlusion(model, batch, gene, slot, bins, marks)
        with torch.no_grad():
            assert torch.equal(ref["logits"], model.forward_batch(_cuda(batch)))
        assert torch.equal(ref["variants"][torch.from_numpy(dead).cuda()],
                           ref["logits"][torch.from_numpy(gene[dead]).cuda()])
        # invalid descriptors: NaN rows, the others bit-identical to the call without them
        bad_g, bad_s, bad_b, bad_m = gene.copy(), slot.copy(), bins.copy(), marks.copy()
        bad = [3, 11, 20, 27, 35, 44, 50, 63]
        bad_g[3], bad_g[11] = -1, n
        bad_s[20], bad_s[27] = -1, I
        bad_b[35, 1] = (5, 4)                                  # lo > hi
        bad_b[44, 2] = (0, NB[2] + 1)                          # hi > n
        bad_b[50, 0] = (-1, 3)
        bad_m[63] = 1 << 7                                     # mark 7 of 7 marks
        got = pcre_occlusion(model, batch, bad_g, bad_s, bad_b, bad_m)
        assert torch.isnan(got["variants"][bad]).all()
        keep = torch.tensor([v for v in range(64) if v not in bad])
        alone = pcre_occlusion(model, batch, gene[keep], slot[keep], bins[keep], marks[keep])
        assert torch.equal(got["variants"][keep.cuda()], alone["variants"])
        assert torch.equal(got["variants"][keep.cuda()], ref["variants"][keep.cuda()])
        assert torch.equal(got["logits"], ref["logits"])
    # many descriptors of genes out of range and a small chunk: no library call holds more than `chunk` variants
    V0 = 64
    many_g = np.concatenate([gene, np.full(40, -7), np.full(10, n + 3)])
    pad = lambda a, fill: np.concatenate([a, np.broadcast_to(fill, (50,) + a.shape[1:])])
    sizes, launch = [], model._launch_occlusion

    def counted(io, vg, *rest):
        sizes.append(int(vg.numel()))
        return launch(io, vg, *rest)
    model._launch_occlusion = counted
    try:
        small = pcre_occlusion(model, batch, many_g, pad(slot, 0), pad(bins, bins[0]), pad(marks, 1), chunk=16)
    finally:
        del model._launch_occlusion
    assert max(sizes) <= 16, sizes
    assert torch.isnan(small["variants"][V0:]).all()
    assert torch.equal(small["variants"][:V0], ref["variants"])        # (FP32: every path is the same at any chunk)
    assert torch.equal(small["logits"], ref["logits"])
    assert all(p.grad is None for p in model.parameters())


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_independence_of_the_other_variants_chunks_and_calls(precision):
    n, I = 256, 8
    model = _mk(seed=29).cuda().eval()
    model.precision = precision
    batch = _cuda(synthetic.make_batch(n, ragged=True, seed=31))
    gene, slot, bins, marks = _variants(n, I, 10000, seed=7)
    ref = pcre_occlusion(model, batch, gene, slot, bins, marks)
    for v in (0, 1234, 9999):                                  # alone against among 10^4 others
        one = pcre_occlusion(model, batch, gene[v:v + 1], slot[v:v + 1], bins[v:v + 1], marks[v:v + 1])
        assert torch.equal(one["variants"][0], ref["variants"][v]), v
    # across chunks: 48 genes with 200 variants each, chunks that split them into calls of 8, 16 and 24 genes, against
    # one call of all 48.  Every call then keeps the gene pass's paths: B < 64 for the PP / Embedding / head GEMMs,
    # B * I >= 64 for the Pairwise GEMMs, B * S >= 64 for the Regulation replay, and no call has the 113 genes the
    # ragged plan's persistent query GEMM needs, so no key window depends on the call
    small = _copy(batch, list(range(48)))
    _, slot, bins, marks = _variants(48, I, 48 * 200, seed=8)
    gene = np.repeat(np.arange(48), 200)
    ref = pcre_occlusion(model, small, gene, slot, bins, marks)
    for chunk in (1600, 3200, 4800):
        got = pcre_occlusion(model, small, gene, slot, bins, marks, chunk=chunk)
        assert torch.equal(got["variants"], ref["variants"]), chunk
        assert torch.equal(got["logits"], ref["logits"]), chunk
    again = pcre_occlusion(model, small, gene, slot, bins, marks)
    assert torch.equal(again["variants"], ref["variants"])
    assert not any(t.requires_grad for t in ref.values())


def _io(model, batch):
    args = synthetic.forward_args(batch, "cuda")
    return _BatchIO(model, *[[d[b] for b in BINS] for d in args[:5]], args[5])


def _call(lib, model, io, desc, logits, vl, ws, flags):
    g, s, b, m = desc
    return lib.chromo_pcre_occlusion(ctypes.byref(io.cfg), model.flat_params.data_ptr(), ctypes.byref(io.struct),
                                     g.numel(), g.data_ptr(), s.data_ptr(), b.data_ptr(), m.data_ptr(),
                                     logits.data_ptr(), vl.data_ptr(), ws.data_ptr(), ws.numel(), flags,
                                     torch.cuda.current_stream().cuda_stream)


def test_capturable_into_a_cuda_graph():
    n, V = 128, 2048
    lib = _lib.load()
    model = _mk(seed=37).cuda().eval()
    a = _copy(synthetic.make_batch(n, ragged=True, seed=61))
    b = _copy(synthetic.make_batch(n, ragged=True, seed=62))
    desc_b = [torch.from_numpy(x.astype(np.int32)).cuda() for x in _variants(n, 8, V, seed=3)]
    io_b = _io(model, b)
    no = int(model._cfg.n_out)
    need = lib.chromo_pcre_occlusion_workspace_floats(ctypes.byref(io_b.cfg), n, V, _lib.F_BF16)
    ws = torch.empty(need, device="cuda")
    want_l, want_v = torch.empty(n, no, device="cuda"), torch.empty(V, no, device="cuda")
    assert _call(lib, model, io_b, desc_b, want_l, want_v, ws, _lib.F_BF16) == 0
    io = _io(model, a)
    desc = [torch.zeros_like(t) for t in desc_b]
    logits, vl = torch.empty(n, no, device="cuda"), torch.empty(V, no, device="cuda")
    ws2 = torch.empty(need, device="cuda")
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        assert _call(lib, model, io, desc, logits, vl, ws2, _lib.F_BF16) == 0       # (packs the weights outside the graph)
    torch.cuda.current_stream().wait_stream(s)
    with torch.cuda.graph(g):
        rc = _call(lib, model, io, desc, logits, vl, ws2, _lib.F_BF16 | _lib.F_PACKED)
    assert rc == 0
    for dst, src in zip(io.keep, io_b.keep):
        dst.copy_(src)
    for dst, src in zip(desc, desc_b):
        dst.copy_(src)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(logits, want_l)
    assert torch.equal(vl, want_v)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_occlusion_map(precision):
    n, I = 16, 8
    model = _mk(seed=17).cuda().eval()
    model.precision = precision
    batch = _cuda(synthetic.make_batch(n, ragged=True, seed=19))
    live = _live(batch).cuda()
    tol = 1e-6 if precision == "fp32" else TOL16
    r = occlusion_map(model, batch, window=4, marks="all")
    W = 5
    assert r["pcre"].shape == (n, I, W, 1, 2) and r["promoter"].shape == (n, W, 1, 2)
    assert r["effect_pcre"].shape == (n, I, W, 1) and r["effect_promoter"].shape == (n, W, 1)
    assert torch.equal(r["windows"], torch.tensor([[0, 4], [4, 8], [8, 12], [12, 16], [16, 20]]))
    assert torch.equal(r["effect_pcre"][~live], torch.zeros_like(r["effect_pcre"][~live]))
    with torch.no_grad():
        assert torch.equal(r["logits"], model.forward_batch(batch))
    # the pCRE entries against pcre_occlusion of the same descriptors, the promoter entries against the forward
    g, i = (x.cpu().numpy() for x in torch.nonzero(live, as_tuple=True))
    w = 2
    d = pcre_occlusion(model, batch, g, i, np.tile(np.array([[8 * k, 12 * k] for k in (1, 4, 20)]), (len(g), 1, 1)),
                       np.full(len(g), 127))
    assert torch.equal(r["pcre"][live][:, w, 0], d["variants"])
    x = _copy(batch)
    for k, b in zip((1, 4, 20), BINS):
        x["promoter_feats"][b][..., 8 * k:12 * k, :] = 0
    with torch.no_grad():
        want = model.forward_batch(x)
    assert (r["promoter"][:, w, 0] - want).abs().max().item() <= tol
    each = occlusion_map(model, batch, window=10, stride=5, marks="each", target=0)
    assert each["pcre"].shape == (n, I, 3, 7, 2) and each["promoter"].shape == (n, 3, 7, 2)
    assert torch.equal(each["effect_pcre"][~live], torch.zeros_like(each["effect_pcre"][~live]))
    assert torch.equal(each["effect_pcre"], each["logits"][:, 0].view(n, 1, 1, 1) - each["pcre"][..., 0])
