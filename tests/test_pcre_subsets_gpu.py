"""pCRE subsets (chromo_pcre_subsets, csrc/subsets.cu; attribution.pcre_subsets / pcre_shapley / pcre_interactions)
against the CPU oracle of the genes reassembled without each set of pCREs, against the library's own forward with the
removed slots' rows and columns of every interaction mask set, and against pcre_deletion."""
import ctypes
import itertools
import math

import pytest
import torch

from _util import BINS, KWS
from chromoformer_b200 import ChromoformerClassifier, ChromoformerRegressor, _lib, synthetic
from chromoformer_b200.attribution import pcre_deletion, pcre_interactions, pcre_shapley, pcre_subsets
from chromoformer_b200.model import _BatchIO
from oracle import chromoformer_oracle as oracle

pytestmark = pytest.mark.gpu
REL32 = 2e-4           # FP32: of the max-abs oracle logit
TOL16 = 5e-3           # BF16, absolute (test_ragged_gpu.py)
REG4 = {"n_layers": 2, "n_heads": 4, "d_model": 128, "d_ff": 256}     # reg_heads != 8: no fused Regulation kernel


def _mk(cls=ChromoformerClassifier, seed=11, i_max=8, reg=None):
    return cls(7, 128, 128, dict(KWS[0]), dict(KWS[1]), dict(reg or KWS[2]), seed=seed, i_max=i_max)


def _sd(model):
    return {k: v.detach().clone() for k, v in model.state_dict().items()}


def _copy(batch, idx=None):
    def pick(t):
        return (t if idx is None else t[torch.as_tensor(idx)]).clone()
    return {key: ({b: pick(t) for b, t in v.items()} if isinstance(v, dict) else pick(v))
            for key, v in batch.items() if key in synthetic.FORWARD_KEYS}


def _cuda(batch):
    return {k: ({b: t.cuda() for b, t in v.items()} if isinstance(v, dict) else v.cuda()) for k, v in _copy(batch).items()}


def _live(batch):
    im = torch.stack([batch["interaction_masks"][b].reshape(batch["interaction_freq"].shape) for b in BINS])
    return (~im[:, :, 0, 1:].bool()).any(0).cpu()


def _rebuilt(batch, items):
    """Gene g reassembled without the pCREs of `drop` for each (g, drop): the kept slots move up in their order, dummy
    slots (zero features, pad mask all set, zero frequency) come last, the block-form interaction mask keeps the
    partners left.  Only live slots are removed (a dead slot is no pCRE)."""
    I = batch["pcre_feats"][BINS[0]].shape[1]
    S = I + 1
    live = _live(batch)
    out = _copy(batch, [g for g, _ in items])
    for r, (g, drop) in enumerate(items):
        drop = [i for i in drop if live[g, i]]
        keep = [j for j in range(I) if j not in drop]
        tok = [0] + [j + 1 for j in keep]
        kk = int(live[g].sum()) - len(drop)
        idx = torch.arange(S)
        for b in BINS:
            x, m = out["pcre_feats"][b], out["pcre_pad_masks"][b]
            x[r] = torch.cat([x[r, keep], torch.zeros_like(x[r, :len(drop)])])
            m[r] = torch.cat([m[r, keep], torch.ones_like(m[r, :len(drop)])])
            out["interaction_masks"][b][r, 0] = ~((idx.view(S, 1) <= kk) & (idx.view(1, S) <= kk))
        f = out["interaction_freq"][r]
        f[:] = torch.nn.functional.pad(f[tok][:, tok], (0, S - len(tok), 0, S - len(tok)))
    return out


def _oracle(sd, batch, rows=8):
    outs = []
    B = batch["interaction_freq"].shape[0]
    for lo in range(0, B, rows):
        part = synthetic.expand_full_masks(synthetic.slice_batch(batch, lo, min(B, lo + rows)))
        with torch.no_grad():
            outs.append(oracle.chromoformer_forward(sd, *synthetic.forward_args(part)))
    return torch.cat(outs)


def _masked(batch, drop):
    """Gene g of `batch` once per variant v of drop [B, V, I], with the rows and columns of the live slots of drop[g, v]
    set in every interaction mask (the forward's view of the variant)."""
    B, V, I = drop.shape
    live = _live(batch)
    d = (drop & live.view(B, 1, I)).reshape(B * V, I)
    out = _copy(batch, torch.arange(B).repeat_interleave(V))
    tok = torch.cat([torch.zeros(B * V, 1, dtype=torch.bool), d], 1).to(out["interaction_freq"].device)
    for b in BINS:
        m = out["interaction_masks"][b]
        m[:, 0] |= tok.view(-1, I + 1, 1) | tok.view(-1, 1, I + 1)
    return out


def _random_drop(B, V, I, seed, p=0.4):
    gen = torch.Generator().manual_seed(seed)
    return torch.rand(B, V, I, generator=gen) < p


def _tol(precision, scale):
    return REL32 * scale if precision == "fp32" else TOL16


@pytest.mark.parametrize("tag,ragged,i_max,n", [("clf", True, 8, 4), ("reg", False, 8, 2), ("reg", True, 16, 3),
                                                ("clf", False, 16, 2)])
def test_against_the_oracle_of_the_reassembled_gene(tag, ragged, i_max, n):
    cls = ChromoformerRegressor if tag == "reg" else ChromoformerClassifier
    model = _mk(cls, i_max=i_max)
    sd = _sd(model)
    batch = synthetic.make_batch(n, i_max=i_max, ragged=ragged, seed=41, stress=True)
    V = 6
    drop = _random_drop(n, V, i_max, seed=n + i_max)
    drop[:, 0] = False                                        # the gene itself
    drop[:, 1] = True                                         # the promoter alone
    want = _oracle(sd, _rebuilt(batch, [(g, torch.nonzero(drop[g, v]).view(-1).tolist())
                                        for g in range(n) for v in range(V)])).view(n, V, -1)
    scale = want.abs().max().item()
    model.cuda().eval()
    for precision in ("fp32", "bf16"):
        model.precision = precision
        d = pcre_subsets(model, batch, drop)
        err = (d["variants"].cpu() - want).abs().max().item()
        print(f"{precision}: max |error| {err:.3e} (max |logit| {scale:.3f})")
        assert err <= _tol(precision, scale), err


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_against_the_masked_forward_deletion_and_the_plain_forward(precision):
    n, I, V = 96, 8, 5
    model = _mk(seed=3).cuda().eval()
    model.precision = precision
    dev = _cuda(synthetic.make_batch(n, ragged=True, seed=6, stress=True))
    drop = _random_drop(n, V, I, seed=2)
    drop[:, 0] = False
    for dense in (True, False):
        d = pcre_subsets(model, dev, drop, dense=dense)
        with torch.no_grad():
            plain = model.forward_batch(dev, dense=dense)
        assert torch.equal(d["logits"], plain)
    with torch.no_grad():
        want = model.forward_batch(_masked(dev, drop)).view(n, V, -1)
    tol = 1e-6 if precision == "fp32" else TOL16
    err = (d["variants"] - want).abs().max().item()
    empty = (d["variants"][:, 0] - d["logits"]).abs().max().item()
    print(f"{precision}: max |variant - masked forward| {err:.3e}; empty drop vs logits {empty:.3e}")
    assert err <= tol and empty <= tol
    # single-slot drops: pcre_deletion's `without`
    single = torch.eye(I, dtype=torch.bool).unsqueeze(0).expand(n, I, I)
    s = pcre_subsets(model, dev, single)
    dl = pcre_deletion(model, dev)
    live = _live(dev)
    err = (s["variants"] - dl["without"])[live.cuda()].abs().max().item()
    print(f"{precision}: max |single-slot variant - pcre_deletion without| {err:.3e}")
    assert err <= tol
    # a dead slot dropped changes nothing: its variant is the gene itself
    dead = ~live.cuda()
    assert dead.any()
    err = (s["variants"] - s["logits"].unsqueeze(1))[dead].abs().max().item()
    assert err <= tol, err


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_arbitrary_interaction_masks(precision):
    n, I, S, V = 48, 8, 9, 4
    model = _mk(seed=19).cuda().eval()
    model.precision = precision
    batch = synthetic.make_batch(n, ragged=True, seed=23)
    gen = torch.Generator().manual_seed(5)
    for b in BINS:
        im = batch["interaction_masks"][b]
        im[:24, 0] = torch.rand(24, S, S, generator=gen) < 0.4
        im[:24, 0, :, 0] = False
    dev = _cuda(batch)
    drop = _random_drop(n, V, I, seed=9)
    d = pcre_subsets(model, dev, drop)
    with torch.no_grad():
        want = model.forward_batch(_masked(dev, drop)).view(n, V, -1)
    err = (d["variants"] - want).abs().max().item()
    print(f"{precision}: max |variant - masked forward| {err:.3e}")
    assert err <= (1e-6 if precision == "fp32" else TOL16)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_non_fused_regulation_path(precision):
    n, I, V = 40, 8, 4
    model = _mk(ChromoformerRegressor, seed=13, reg=REG4).cuda().eval()
    model.precision = precision
    dev = _cuda(synthetic.make_batch(n, ragged=True, seed=17))
    drop = _random_drop(n, V, I, seed=4)
    d = pcre_subsets(model, dev, drop)
    with torch.no_grad():
        assert torch.equal(d["logits"], model.forward_batch(dev))
        want = model.forward_batch(_masked(dev, drop)).view(n, V, -1)
    err = (d["variants"] - want).abs().max().item()
    print(f"{precision}: max |variant - masked forward| {err:.3e}")
    assert err <= (1e-6 if precision == "fp32" else TOL16)


def _brute_shapley(sd, batch, genes, t):
    """Shapley values of target column t from oracle forwards of every reassembled subset of each gene's pCREs."""
    live = _live(batch)
    out = []
    for g in genes:
        players = torch.nonzero(live[g]).view(-1).tolist()
        k = len(players)
        subsets = list(range(1 << k))
        items = [(g, [players[j] for j in range(k) if not (s >> j) & 1]) for s in subsets]
        v = _oracle(sd, _rebuilt(batch, items))[:, t].double()
        phi = torch.zeros(batch["pcre_feats"][BINS[0]].shape[1], dtype=torch.float64)
        for j in range(k):
            for s in subsets:
                if not (s >> j) & 1:
                    n = bin(s).count("1")
                    w = math.factorial(n) * math.factorial(k - n - 1) / math.factorial(k)
                    phi[players[j]] += w * (v[s | (1 << j)] - v[s])
        out.append(phi)
    return torch.stack(out)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_shapley_against_brute_force(precision):
    n = 24
    model = _mk(seed=21)
    sd = _sd(model)
    batch = synthetic.make_batch(n, ragged=True, seed=33)
    k = _live(batch).sum(1)
    genes = [g for g in range(n) if 1 <= k[g] <= 4][:3]
    assert len(genes) >= 2
    want = _brute_shapley(sd, batch, genes, 1)
    scale = _oracle(sd, _copy(batch, genes)).abs().max().item()
    model.cuda().eval()
    model.precision = precision
    r = pcre_shapley(model, batch)
    got = r["shapley"].cpu()[genes]
    err = (got - want).abs().max().item()
    print(f"{precision}: max |shapley - brute force| {err:.3e} (max |logit| {scale:.3f})")
    assert err <= 4 * _tol(precision, scale)
    live = _live(batch)
    assert torch.equal(r["shapley"].cpu()[~live], torch.zeros(int((~live).sum()), dtype=torch.float64))
    eff = (r["shapley"].sum(1) - (r["logits"][:, 1] - r["promoter_only"][:, 1]).double()).abs().max().item()
    print(f"{precision}: max |sum shapley - (logit - promoter_only)| {eff:.3e}")
    assert eff <= (1e-5 if precision == "fp32" else TOL16)
    with torch.no_grad():
        prom = model.forward_batch(_masked(_cuda(batch), torch.ones(n, 1, 8, dtype=torch.bool)))
    assert (r["promoter_only"] - prom).abs().max().item() <= (1e-6 if precision == "fp32" else TOL16)


@pytest.mark.parametrize("i_max,permutations", [(8, None), (16, 6)])
def test_shapley_efficiency(i_max, permutations):
    n = 40
    model = _mk(seed=27, i_max=i_max).cuda().eval()
    model.precision = "bf16"
    batch = synthetic.make_batch(n, i_max=i_max, ragged=True, seed=35)
    r = pcre_shapley(model, batch, permutations=permutations)
    live = _live(batch)
    assert torch.equal(r["shapley"].cpu()[~live], torch.zeros(int((~live).sum()), dtype=torch.float64))
    with torch.no_grad():
        logits = model.forward_batch(_cuda(batch))
    assert torch.equal(r["logits"], logits)
    eff = (r["shapley"].sum(1) - (r["logits"][:, 1] - r["promoter_only"][:, 1]).double()).abs().max().item()
    print(f"i_max {i_max}: max |sum shapley - (logit - promoter_only)| {eff:.3e}")
    assert eff <= TOL16
    again = pcre_shapley(model, batch, permutations=permutations)
    assert torch.equal(again["shapley"], r["shapley"])
    if i_max == 16:
        with pytest.raises(ValueError, match="permutations="):
            pcre_shapley(model, synthetic.make_batch(4, i_max=16, ragged=False, seed=1))


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_interactions(precision):
    n, I = 24, 8
    model = _mk(seed=23)
    sd = _sd(model)
    batch = synthetic.make_batch(n, ragged=True, seed=37)
    live = _live(batch)
    model.cuda().eval()
    model.precision = precision
    r = pcre_interactions(model, batch)
    inter = r["interaction"].cpu()
    assert torch.equal(inter, inter.transpose(1, 2))
    assert torch.equal(torch.diagonal(inter, dim1=1, dim2=2), torch.zeros(n, I, dtype=torch.float64))
    assert torch.equal(inter[~live], torch.zeros(int((~live).sum()), I, dtype=torch.float64))
    assert torch.equal(r["effect"].cpu()[~live], torch.zeros(int((~live).sum()), dtype=torch.float64))
    # the oracle, for the pairs of a few genes
    genes = [g for g in range(n) if live[g].sum() >= 3][:2]
    items, pairs = [], []
    for g in genes:
        pl = torch.nonzero(live[g]).view(-1).tolist()
        for i, j in itertools.combinations(pl[:4], 2):
            pairs.append((g, i, j))
            items += [(g, []), (g, [i]), (g, [j]), (g, [i, j])]
    v = _oracle(sd, _rebuilt(batch, items))[:, 1].double().view(-1, 4)
    want = v[:, 0] - v[:, 1] - v[:, 2] + v[:, 3]
    got = torch.stack([inter[g, i, j] for g, i, j in pairs])
    scale = v.abs().max().item()
    err = (got - want).abs().max().item()
    print(f"{precision}: max |interaction - oracle| {err:.3e} (max |logit| {scale:.3f})")
    assert err <= 4 * _tol(precision, scale)
    dl = pcre_deletion(model, batch)
    assert (r["effect"] - dl["effect"].double())[live.cuda()].abs().max().item() <= 2 * _tol(precision, scale)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_chunking_and_repeat_are_bit_identical(precision):
    n, V, I = 24, 4, 8            # every call holds 8 to 24 genes: the gene pass's paths are the same in each
    model = _mk(seed=29).cuda().eval()
    model.precision = precision
    batch = synthetic.make_batch(n, ragged=True, seed=31)
    drop = _random_drop(n, V, I, seed=8)
    ref = pcre_subsets(model, batch, drop)
    for chunk in (32, 48, n * V):
        got = pcre_subsets(model, batch, drop, chunk=chunk)
        for key in ref:
            assert torch.equal(got[key], ref[key]), (chunk, key)
    again = pcre_subsets(model, batch, drop)
    for key in ref:
        assert torch.equal(again[key], ref[key]), key
    assert not any(v.requires_grad for v in ref.values())
    assert all(p.grad is None for p in model.parameters())


def _io(model, batch):
    args = synthetic.forward_args(batch, "cuda")
    return _BatchIO(model, *[[d[b] for b in BINS] for d in args[:5]], args[5])


def _call(lib, model, io, vg, vd, logits, vl, ws, n=None, flags=_lib.F_BF16, V=None):
    return lib.chromo_pcre_subsets(ctypes.byref(io.cfg), model.flat_params.data_ptr(), ctypes.byref(io.struct),
                                   vg.data_ptr() if vg is not None else None, vd.data_ptr() if vd is not None else None,
                                   (vg if vg is not None else vd).numel() if V is None else V, logits.data_ptr(),
                                   vl.data_ptr() if vl is not None else None, ws.data_ptr(),
                                   ws.numel() if n is None else n, flags, torch.cuda.current_stream().cuda_stream)


def test_capturable_into_a_cuda_graph():
    n, V = 256, 1024
    lib = _lib.load()
    model = _mk(seed=37).cuda().eval()
    a = _copy(synthetic.make_batch(n, ragged=True, seed=61))
    b = _copy(synthetic.make_batch(n, ragged=True, seed=62))
    gen = torch.Generator().manual_seed(3)
    vg_b = torch.randint(0, n, (V,), generator=gen, dtype=torch.int32).cuda()
    vd_b = torch.randint(0, 256, (V,), generator=gen, dtype=torch.int32).cuda()
    io_b = _io(model, b)
    no = int(model._cfg.n_out)
    need = lib.chromo_pcre_subsets_workspace_floats(ctypes.byref(io_b.cfg), n, V, _lib.F_BF16)
    ws = torch.empty(need, device="cuda")
    want_l, want_v = torch.empty(n, no, device="cuda"), torch.empty(V, no, device="cuda")
    assert _call(lib, model, io_b, vg_b, vd_b, want_l, want_v, ws) == 0
    io = _io(model, a)
    vg, vd = torch.zeros_like(vg_b), torch.zeros_like(vd_b)
    logits, vl = torch.empty(n, no, device="cuda"), torch.empty(V, no, device="cuda")
    ws2 = torch.empty(need, device="cuda")
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        assert _call(lib, model, io, vg, vd, logits, vl, ws2) == 0          # (packs the weights outside the graph)
    torch.cuda.current_stream().wait_stream(s)
    with torch.cuda.graph(g):
        rc = _call(lib, model, io, vg, vd, logits, vl, ws2, flags=_lib.F_BF16 | _lib.F_PACKED)
    assert rc == 0
    for dst, src in zip(io.keep, io_b.keep):
        dst.copy_(src)
    vg.copy_(vg_b)
    vd.copy_(vd_b)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(logits, want_l)
    assert torch.equal(vl, want_v)


def test_errors_and_descriptor_guard():
    lib = _lib.load()
    model = _mk(seed=43).cuda().eval()
    n = 16
    batch = synthetic.make_batch(n, ragged=True, seed=2)
    io = _io(model, batch)
    I, no = int(io.cfg.i_max), int(model._cfg.n_out)
    gen = torch.Generator().manual_seed(4)
    V = 64
    vg = torch.randint(0, n, (V,), generator=gen, dtype=torch.int32)
    vd = torch.randint(0, 1 << I, (V,), generator=gen, dtype=torch.int32)
    bad = [5, 17, 30, 41, 63]
    vg_bad, vd_bad = vg.clone(), vd.clone()
    vg_bad[5], vg_bad[17], vg_bad[30] = -1, n, 2 ** 31 - 1
    vd_bad[41], vd_bad[63] = 1 << I, -2 ** 31                                # bit I; bit 31
    for flags in (_lib.F_BF16, 0):
        need = lib.chromo_pcre_subsets_workspace_floats(ctypes.byref(io.cfg), n, V, flags)
        ws = torch.empty(need, device="cuda")
        logits, vl = torch.empty(n, no, device="cuda"), torch.empty(V, no, device="cuda")
        good = [v for v in range(V) if v not in bad]
        sel = torch.tensor(good)
        vl_good = torch.empty(len(good), no, device="cuda")
        assert _call(lib, model, io, vg[sel].cuda(), vd[sel].cuda(), logits, vl_good, ws, flags=flags) == 0
        assert _call(lib, model, io, vg_bad.cuda(), vd_bad.cuda(), logits, vl, ws, flags=flags) == 0
        torch.cuda.synchronize()
        assert torch.isnan(vl[bad]).all()
        assert torch.equal(vl[sel.cuda()], vl_good), flags
    ws = torch.empty(lib.chromo_pcre_subsets_workspace_floats(ctypes.byref(io.cfg), n, V, _lib.F_BF16), device="cuda")
    vgc, vdc = vg.cuda(), vd.cuda()
    assert _call(lib, model, io, vgc, vdc, logits, vl, ws, n=ws.numel() - 1) == -2
    assert str(ws.numel()) in lib.chromo_last_error().decode()
    assert _call(lib, model, io, vgc, vdc, logits, None, ws) == -1
    assert _call(lib, model, io, None, vdc, logits, vl, ws) == -1
    assert _call(lib, model, io, vgc, None, logits, vl, ws) == -1
    assert _call(lib, model, io, vgc, vdc, logits, vl, ws, V=0) == -1
    for badf in (_lib.F_TRAINING, _lib.F_BWD_HEAD_REG, _lib.F_BWD_REST, _lib.F_FREQ_GRAD, 8):
        assert _call(lib, model, io, vgc, vdc, logits, vl, ws, flags=_lib.F_BF16 | badf) == -1, badf
    with pytest.raises(ValueError):
        pcre_subsets(model, batch, torch.zeros(3, I + 1, dtype=torch.bool))
    with pytest.raises(ValueError):
        pcre_subsets(model, batch, torch.zeros(3, I, dtype=torch.int32))
