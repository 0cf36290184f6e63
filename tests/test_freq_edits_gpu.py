"""Interaction-frequency edits (chromo_freq_edits, csrc/freq_edits.cu; attribution.freq_edits / contact_knockout /
contact_response / contact_shapley) against the CPU oracle of each gene with its interaction_freq replaced, against the
library's own forward with the edited interaction_freq, against pcre_subsets and against the interaction_freq
integrated gradients."""
import ctypes
import math

import pytest
import torch

from _util import BINS, KWS
from chromoformer_b200 import ChromoformerClassifier, ChromoformerRegressor, _lib, synthetic
from chromoformer_b200.attribution import (contact_knockout, contact_response, contact_shapley, freq_edits,
                                           integrated_gradients, pcre_subsets)
from chromoformer_b200.model import _BatchIO
from oracle import chromoformer_oracle as oracle

pytestmark = pytest.mark.gpu
REL32 = 2e-4           # FP32: of the max-abs oracle logit
TOL16 = 5e-3           # BF16, absolute (test_ragged_gpu.py)
REG4 = {"n_layers": 2, "n_heads": 4, "d_model": 128, "d_ff": 256}     # reg_heads != 8: no fused Regulation kernel
NAN = float("nan")


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


def _edited(batch, edits):
    """Gene g once per variant v of edits [B, V, S, S] (NaN = keep), with interaction_freq replaced."""
    B, V = edits.shape[:2]
    out = _copy(batch, torch.arange(B).repeat_interleave(V))
    f = out["interaction_freq"]
    e = edits.reshape(B * V, *edits.shape[2:]).to(f.device)
    out["interaction_freq"] = torch.where(torch.isnan(e), f, e)
    return out


def _oracle(sd, batch, rows=8):
    outs = []
    B = batch["interaction_freq"].shape[0]
    for lo in range(0, B, rows):
        part = synthetic.expand_full_masks(synthetic.slice_batch(batch, lo, min(B, lo + rows)))
        with torch.no_grad():
            outs.append(oracle.chromoformer_forward(sd, *synthetic.forward_args(part)))
    return torch.cat(outs)


def _edits(B, S, seed):
    """[B, 5, S, S]: row 0, column 0, pCRE-pCRE entries, values of +-10, and a mix with NaNs in between."""
    gen = torch.Generator().manual_seed(seed)
    e = torch.full((B, 5, S, S), NAN)
    e[:, 0, 0, :] = torch.rand(B, S, generator=gen) * 3
    e[:, 1, :, 0] = torch.randn(B, S, generator=gen)
    e[:, 2, 1:, 1:] = torch.rand(B, S - 1, S - 1, generator=gen) * 2
    e[:, 3, 0, 1:] = torch.where(torch.rand(B, S - 1, generator=gen) < 0.5, 10.0, -10.0)
    pick = torch.rand(B, S, S, generator=gen) < 0.4
    e[:, 4] = torch.where(pick, torch.randn(B, S, S, generator=gen) * 4, torch.full((), NAN))
    return e


def _tol(precision, scale):
    return REL32 * scale if precision == "fp32" else TOL16


@pytest.mark.parametrize("tag,ragged,i_max,n", [("clf", True, 8, 4), ("reg", False, 8, 2), ("reg", True, 16, 3),
                                                ("clf", False, 16, 2)])
def test_against_the_oracle_of_the_edited_gene(tag, ragged, i_max, n):
    cls = ChromoformerRegressor if tag == "reg" else ChromoformerClassifier
    model = _mk(cls, i_max=i_max)
    sd = _sd(model)
    batch = synthetic.make_batch(n, i_max=i_max, ragged=ragged, seed=41, stress=True)
    edits = _edits(n, i_max + 1, seed=n + i_max)
    want = _oracle(sd, _edited(batch, edits)).view(n, edits.shape[1], -1)
    scale = want.abs().max().item()
    model.cuda().eval()
    for precision in ("fp32", "bf16"):
        model.precision = precision
        d = freq_edits(model, batch, edits)
        err = (d["variants"].cpu() - want).abs().max().item()
        print(f"{precision}: max |error| {err:.3e} (max |logit| {scale:.3f})")
        assert err <= _tol(precision, scale), err


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_against_the_edited_forward_and_the_plain_forward(precision):
    n, S = 96, 9
    model = _mk(seed=3).cuda().eval()
    model.precision = precision
    dev = _cuda(synthetic.make_batch(n, ragged=True, seed=6, stress=True))
    edits = _edits(n, S, seed=2)
    for dense in (True, False):
        d = freq_edits(model, dev, edits, dense=dense)
        with torch.no_grad():
            plain = model.forward_batch(dev, dense=dense)
        assert torch.equal(d["logits"], plain)
    with torch.no_grad():
        want = model.forward_batch(_edited(dev, edits)).view(n, edits.shape[1], -1)
    tol = 1e-6 if precision == "fp32" else TOL16
    err = (d["variants"] - want).abs().max().item()
    print(f"{precision}: max |variant - edited forward| {err:.3e}")
    assert err <= tol
    # the same V edits for every gene ([V, S, S]) give what the per-gene form gives
    shared = freq_edits(model, dev, edits[0], target=1)
    per_gene = freq_edits(model, dev, edits[0].expand(n, -1, -1, -1).clone())
    assert torch.equal(shared["variants"], per_gene["variants"])
    assert torch.equal(shared["value"], shared["variants"][..., 1])


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_unedited_variants_are_the_empty_drop_set_of_pcre_subsets(precision):
    n, S = 40, 9
    model = _mk(seed=5).cuda().eval()
    model.precision = precision
    batch = synthetic.make_batch(n, ragged=True, seed=9)
    edits = torch.full((n, 2, S, S), NAN)
    edits[:, 1] = batch["interaction_freq"]                   # the gene's own freq, written
    d = freq_edits(model, batch, edits)
    s = pcre_subsets(model, batch, torch.zeros(1, S - 1, dtype=torch.bool))
    assert torch.equal(d["variants"][:, 0], s["variants"][:, 0])
    assert torch.equal(d["variants"][:, 1], s["variants"][:, 0])
    assert torch.equal(d["logits"], s["logits"])


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_non_fused_regulation_path(precision):
    n, S = 40, 9
    model = _mk(ChromoformerRegressor, seed=13, reg=REG4).cuda().eval()
    model.precision = precision
    dev = _cuda(synthetic.make_batch(n, ragged=True, seed=17))
    edits = _edits(n, S, seed=4)
    d = freq_edits(model, dev, edits)
    with torch.no_grad():
        assert torch.equal(d["logits"], model.forward_batch(dev))
        want = model.forward_batch(_edited(dev, edits)).view(n, edits.shape[1], -1)
    err = (d["variants"] - want).abs().max().item()
    print(f"{precision}: max |variant - edited forward| {err:.3e}")
    assert err <= (1e-6 if precision == "fp32" else TOL16)


def _contacts_zeroed(batch, keep=None):
    """batch with every contact [0, i + 1] set to 0 (except where keep [B, I] is True)."""
    out = _copy(batch)
    f = out["interaction_freq"]
    keep = torch.zeros(f.shape[0], f.shape[1] - 1, dtype=torch.bool) if keep is None else keep
    f[:, 0, 1:] = torch.where(keep.to(f.device), f[:, 0, 1:], torch.zeros((), device=f.device))
    return out


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_contact_knockout(precision):
    n, I = 48, 8
    model = _mk(seed=7).cuda().eval()
    model.precision = precision
    dev = _cuda(synthetic.make_batch(n, ragged=True, seed=12))
    live = _live(dev)
    k = contact_knockout(model, dev)
    tol = 1e-6 if precision == "fp32" else TOL16
    dead = ~live.cuda()
    assert dead.any()
    assert torch.equal(k["effect"][dead], torch.zeros(int(dead.sum()), device="cuda"))
    assert torch.equal(k["without"][dead], k["logits"].unsqueeze(1).expand(n, I, -1)[dead])
    with torch.no_grad():
        blind = model.forward_batch(_contacts_zeroed(dev))
        assert torch.equal(k["logits"], model.forward_batch(dev))
    err = (k["blind"] - blind).abs().max().item()
    print(f"{precision}: max |blind - forward with row 0 zeroed| {err:.3e}")
    assert err <= tol
    assert torch.equal(k["blind_effect"], k["logits"][:, 1] - k["blind"][:, 1])
    # each knockout against the forward of its gene with that contact zeroed
    g, i = torch.nonzero(live, as_tuple=True)
    keep = torch.ones(len(g), I, dtype=torch.bool)
    keep[torch.arange(len(g)), i] = False
    with torch.no_grad():
        want = model.forward_batch(_contacts_zeroed(_copy(dev, g.cuda()), keep))
    err = (k["without"][g.cuda(), i.cuda()] - want).abs().max().item()
    print(f"{precision}: max |without - forward with the contact zeroed| {err:.3e}")
    assert err <= tol


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_contact_response_identities(precision):
    n, I = 32, 8
    model = _mk(seed=17).cuda().eval()
    model.precision = precision
    batch = synthetic.make_batch(n, ragged=True, seed=14)
    live = _live(batch)
    same = freq_edits(model, batch, torch.full((1, I + 1, I + 1), NAN))["variants"][:, 0]     # the replayed gene
    r = contact_response(model, batch, [0.0, 1.0, 2.5], relative=True)
    assert r["response"].shape == (n, I, 3, int(model._cfg.n_out))
    lv = live.cuda()
    assert torch.equal(r["response"][:, :, 1][lv], same.unsqueeze(1).expand(n, I, -1)[lv])
    assert torch.equal(r["response"][~lv], r["logits"].view(n, 1, 1, -1).expand(n, I, 3, -1)[~lv])
    # the relative value 0 is the knockout
    k = contact_knockout(model, batch)
    assert torch.equal(r["response"][:, :, 0][lv], k["without"][lv])
    # an absolute value equal to the gene's own contact: every live contact of the batch set to 0.75 first
    batch["interaction_freq"][:, 0, 1:] = torch.where(live, torch.full((), 0.75), torch.zeros(()))
    same = freq_edits(model, batch, torch.full((1, I + 1, I + 1), NAN))["variants"][:, 0]
    r = contact_response(model, batch, [0.75, -3.0], target=0)
    assert torch.equal(r["response"][:, :, 0][lv], same.unsqueeze(1).expand(n, I, -1)[lv])
    assert torch.equal(r["value"], r["response"][..., 0])
    with torch.no_grad():
        want = model.forward_batch(_cuda(batch))
    assert (r["response"][:, :, 0][lv] - want.unsqueeze(1).expand(n, I, -1)[lv]).abs().max().item() <= \
        (1e-6 if precision == "fp32" else TOL16)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_contact_shapley_against_brute_force(precision):
    n, I = 24, 8
    model = _mk(seed=21).cuda().eval()
    model.precision = precision
    batch = synthetic.make_batch(n, ragged=True, seed=33)
    live = _live(batch)
    k = live.sum(1)
    genes = [g for g in range(n) if 1 <= k[g] <= 4][:4]
    assert len(genes) >= 2
    r = contact_shapley(model, batch)
    dev = _cuda(batch)
    for g in genes:
        players = torch.nonzero(live[g]).view(-1).tolist()
        kk = len(players)
        keep = torch.zeros(1 << kk, I, dtype=torch.bool)
        for s in range(1 << kk):
            for j in range(kk):
                keep[s, players[j]] = bool((s >> j) & 1)
        with torch.no_grad():
            v = model.forward_batch(_contacts_zeroed(_copy(dev, [g] * (1 << kk)), keep))[:, 1].double().cpu()
        phi = torch.zeros(I, dtype=torch.float64)
        for j in range(kk):
            for s in range(1 << kk):
                if not (s >> j) & 1:
                    m = bin(s).count("1")
                    phi[players[j]] += math.factorial(m) * math.factorial(kk - m - 1) / math.factorial(kk) * \
                        (v[s | (1 << j)] - v[s])
        err = (r["shapley"][g].cpu() - phi).abs().max().item()
        print(f"{precision}: gene {g} ({kk} contacts): max |shapley - brute force| {err:.3e}")
        assert err <= (1e-5 if precision == "fp32" else 4 * TOL16)
    for P in (None, 6):
        s = r if P is None else contact_shapley(model, batch, permutations=P, seed=3)
        assert torch.equal(s["shapley"].cpu()[~live], torch.zeros(int((~live).sum()), dtype=torch.float64))
        eff = (s["shapley"].sum(1) - (s["logits"][:, 1].double() - s["blind"][:, 1].double())).abs().max().item()
        print(f"{precision}, permutations {P}: max |sum shapley - (logit - blind)| {eff:.3e}")
        assert eff <= (1e-5 if precision == "fp32" else TOL16)


def test_contact_completeness_against_freq_integrated_gradients():
    """Freq-only integrated gradients from the contact-blind gene (features equal to the features, the contacts
    zeroed) sum to logits - blind.  In FP32 the gap is the midpoint rule's error, which falls about 4x per doubling of
    the steps, plus a floor set by the gradients themselves (the FP32 backward is held to 2e-4 of the largest gradient,
    test_freq_grad_gpu.py): measured about 1e-4 per gene, so the first doubling shows the rule's rate and the last
    stays under that floor's bound."""
    n = 32
    model = _mk(seed=31).cuda().eval()
    batch = synthetic.make_batch(n, ragged=True, seed=8)
    k = contact_knockout(model, batch)
    target = (k["logits"][:, 1] - k["blind"][:, 1]).double()
    base = _copy(batch)
    baseline = {key: base[key] for key in ("promoter_feats", "pcre_feats")}
    baseline["interaction_freq"] = _contacts_zeroed(batch)["interaction_freq"]
    gaps = []
    for steps in (4, 8, 16):
        ig = integrated_gradients(model, batch, steps=steps, baseline=baseline, freq=True)
        total = ig["interaction_freq"].double().sum((1, 2))
        for key in ("promoter_feats", "pcre_feats"):
            for v in ig[key].values():
                assert (v == 0).all()
        gaps.append((total - target).abs().sum().item())
    print("sum over genes of |sum IG - (logit - blind)|, steps 4 / 8 / 16:", gaps)
    assert 2.5 < gaps[0] / gaps[1] < 6.5, gaps
    assert gaps[2] < gaps[1] and gaps[2] / n < 2e-4, gaps


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_determinism_alone_among_many_and_across_chunks(precision):
    n, S = 24, 9
    model = _mk(seed=29).cuda().eval()
    model.precision = precision
    batch = synthetic.make_batch(n, ragged=True, seed=31)
    many = _edits(n, S, seed=5).repeat(1, 84, 1, 1)[:, :417]                # 24 * 417 = 10,008 variants
    many[:, 5:] += torch.randn(many[:, 5:].shape, generator=torch.Generator().manual_seed(1)) * 0.01
    big = freq_edits(model, batch, many)
    for v in (0, 3, 200, 416):
        alone = freq_edits(model, batch, many[:, v:v + 1])
        assert torch.equal(alone["variants"][:, 0], big["variants"][:, v]), v
    again = freq_edits(model, batch, many)
    assert torch.equal(again["variants"], big["variants"])
    # every call holds 8 to 24 genes: the gene pass's paths are the same in each
    edits = _edits(n, S, seed=8)[:, :4]
    ref = freq_edits(model, batch, edits)
    for chunk in (32, 48, n * 4):
        got = freq_edits(model, batch, edits, chunk=chunk)
        for key in ref:
            assert torch.equal(got[key], ref[key]), (chunk, key)
    assert not any(v.requires_grad for v in ref.values())
    assert all(p.grad is None for p in model.parameters())


def _io(model, batch):
    args = synthetic.forward_args(batch, "cuda")
    return _BatchIO(model, *[[d[b] for b in BINS] for d in args[:5]], args[5])


def _call(lib, model, io, vg, vf, logits, vl, ws, flags=_lib.F_BF16):
    return lib.chromo_freq_edits(ctypes.byref(io.cfg), model.flat_params.data_ptr(), ctypes.byref(io.struct),
                                 vg.data_ptr(), vf.data_ptr(), vg.numel(), logits.data_ptr(), vl.data_ptr(),
                                 ws.data_ptr(), ws.numel(), flags, torch.cuda.current_stream().cuda_stream)


def test_capturable_into_a_cuda_graph():
    n, V, S = 256, 1024, 9
    lib = _lib.load()
    model = _mk(seed=37).cuda().eval()
    a = _copy(synthetic.make_batch(n, ragged=True, seed=61))
    b = _copy(synthetic.make_batch(n, ragged=True, seed=62))
    gen = torch.Generator().manual_seed(3)
    vg_b = torch.randint(0, n, (V,), generator=gen, dtype=torch.int32).cuda()
    vf_b = torch.where(torch.rand(V, S, S, generator=gen) < 0.3, torch.randn(V, S, S, generator=gen),
                       torch.full((), NAN)).cuda()
    io_b = _io(model, b)
    no = int(model._cfg.n_out)
    need = lib.chromo_freq_edits_workspace_floats(ctypes.byref(io_b.cfg), n, V, _lib.F_BF16)
    ws = torch.empty(need, device="cuda")
    want_l, want_v = torch.empty(n, no, device="cuda"), torch.empty(V, no, device="cuda")
    assert _call(lib, model, io_b, vg_b, vf_b, want_l, want_v, ws) == 0
    io = _io(model, a)
    vg, vf = torch.zeros_like(vg_b), torch.zeros_like(vf_b)
    logits, vl = torch.empty(n, no, device="cuda"), torch.empty(V, no, device="cuda")
    ws2 = torch.empty(need, device="cuda")
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        assert _call(lib, model, io, vg, vf, logits, vl, ws2) == 0          # (packs the weights outside the graph)
    torch.cuda.current_stream().wait_stream(s)
    with torch.cuda.graph(g):
        rc = _call(lib, model, io, vg, vf, logits, vl, ws2, flags=_lib.F_BF16 | _lib.F_PACKED)
    assert rc == 0
    for dst, src in zip(io.keep, io_b.keep):
        dst.copy_(src)
    vg.copy_(vg_b)
    vf.copy_(vf_b)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(logits, want_l)
    assert torch.equal(vl, want_v)


def test_descriptor_guard_and_errors():
    lib = _lib.load()
    model = _mk(seed=43).cuda().eval()
    n, S, V = 16, 9, 64
    batch = synthetic.make_batch(n, ragged=True, seed=2)
    io = _io(model, batch)
    no = int(model._cfg.n_out)
    gen = torch.Generator().manual_seed(4)
    vg = torch.randint(0, n, (V,), generator=gen, dtype=torch.int32)
    vf = torch.where(torch.rand(V, S, S, generator=gen) < 0.3, torch.randn(V, S, S, generator=gen) * 3,
                     torch.full((), NAN))
    vf[7] = NAN                                                              # all NaN: valid, the gene itself
    bad = [5, 17, 30, 41, 50, 63]
    vg_bad, vf_bad = vg.clone(), vf.clone()
    vg_bad[5], vg_bad[17], vg_bad[30] = -1, n, 2 ** 31 - 1
    vf_bad[41, 0, 3] = float("inf")
    vf_bad[50, 4, 2] = -float("inf")
    vf_bad[63, 8, 8] = float("inf")
    vf_bad[63, 0, 1] = NAN
    for flags in (_lib.F_BF16, 0):
        need = lib.chromo_freq_edits_workspace_floats(ctypes.byref(io.cfg), n, V, flags)
        ws = torch.empty(need, device="cuda")
        logits, vl = torch.empty(n, no, device="cuda"), torch.empty(V, no, device="cuda")
        good = [v for v in range(V) if v not in bad]
        sel = torch.tensor(good)
        vl_good = torch.empty(len(good), no, device="cuda")
        assert _call(lib, model, io, vg[sel].cuda(), vf[sel].cuda(), logits, vl_good, ws, flags=flags) == 0
        assert _call(lib, model, io, vg_bad.cuda(), vf_bad.cuda(), logits, vl, ws, flags=flags) == 0
        torch.cuda.synchronize()
        assert torch.isnan(vl[bad]).all()
        assert torch.isfinite(vl_good).all()
        assert torch.equal(vl[sel.cuda()], vl_good), flags
    with pytest.raises(ValueError):
        freq_edits(model, batch, torch.zeros(3, S + 1, S + 1))
    with pytest.raises(ValueError):
        freq_edits(model, batch, torch.zeros(3, S, S, dtype=torch.int32))
    with pytest.raises(ValueError):
        freq_edits(model, batch, torch.zeros(n + 1, 2, S, S))
    with pytest.raises(ValueError, match="permutations="):
        contact_shapley(model, synthetic.make_batch(4, i_max=16, ragged=False, seed=1))

