"""In-silico pCRE deletion (chromo_pcre_deletion, csrc/deletion.cu; attribution.pcre_deletion) against the CPU oracle of
the genes reassembled without each pCRE, and against the library's own forward with the deleted slot's row and column
of every interaction mask set."""
import ctypes

import pytest
import torch

from _util import BINS, KWS
from chromoformer_b200 import ChromoformerClassifier, ChromoformerRegressor, _lib, synthetic
from chromoformer_b200.attribution import pcre_deletion
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


def _live(batch):
    """[B, I]: slot i is live when token i + 1 is unmasked in row 0 of some resolution's interaction mask."""
    im = torch.stack([batch["interaction_masks"][b].reshape(batch["interaction_freq"].shape) for b in BINS])
    return (~im[:, :, 0, 1:].bool()).any(0)


def _masked(batch, slot):
    """Every gene with row and column slot + 1 of every interaction mask set (slot None: tokens 1..I)."""
    out = _copy(batch)
    for b in BINS:
        m = out["interaction_masks"][b]
        sel = slice(1, None) if slot is None else slice(slot + 1, slot + 2)
        m[:, 0, sel, :] = True
        m[:, 0, :, sel] = True
    return out


def _rebuilt(batch, pairs):
    """Gene g reassembled without pCRE i for each (g, i): later slots move up, a dummy slot (zero features, pad mask all
    set, zero frequency) comes last, the block-form interaction mask has one partner less.  i None: no pCRE at all."""
    I = batch["pcre_feats"][BINS[0]].shape[1]
    S = I + 1
    out = _copy(batch, [g for g, _ in pairs])
    for r, (g, i) in enumerate(pairs):
        k = int(_live(_copy(batch, [g]))[0].sum())
        drop = list(range(I)) if i is None else [i]
        keep = [j for j in range(I) if j not in drop]
        tok = [0] + [j + 1 for j in keep]
        for b in BINS:
            x, m = out["pcre_feats"][b], out["pcre_pad_masks"][b]
            x[r] = torch.cat([x[r, keep], torch.zeros_like(x[r, :len(drop)])])
            m[r] = torch.cat([m[r, keep], torch.ones_like(m[r, :len(drop)])])
            kk = 0 if i is None else k - 1                       # partners left
            idx = torch.arange(S)
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


def _run(model, batch, precision, **kw):
    model.precision = precision
    d = pcre_deletion(model, batch, **kw)
    return {k: v.cpu() for k, v in d.items()}


@pytest.mark.parametrize("tag,ragged,i_max,n", [("clf", True, 8, 4), ("reg", False, 8, 2), ("reg", True, 16, 3),
                                                ("clf", False, 16, 1)])
def test_against_the_oracle_of_the_reassembled_gene(tag, ragged, i_max, n):
    cls = ChromoformerRegressor if tag == "reg" else ChromoformerClassifier
    model = _mk(cls, i_max=i_max)
    sd = _sd(model)
    batch = synthetic.make_batch(n, i_max=i_max, ragged=ragged, seed=41, stress=True)
    live = _live(batch)
    pairs = [(g, i) for g in range(n) for i in range(i_max) if live[g, i]]
    assert pairs
    want = _oracle(sd, _rebuilt(batch, pairs + [(g, None) for g in range(n)]))
    want_without, want_prom = want[:len(pairs)], want[len(pairs):]
    scale = want.abs().max().item()
    model.cuda().eval()
    for precision in ("fp32", "bf16"):
        d = _run(model, batch, precision)
        got_without = torch.stack([d["without"][g, i] for g, i in pairs])
        err = max((got_without - want_without).abs().max().item(), (d["promoter_only"] - want_prom).abs().max().item())
        print(f"{precision}: max |error| {err:.3e} (max |logit| {scale:.3f})")
        if precision == "fp32":
            assert err <= REL32 * scale, err
        else:
            assert err < TOL16, err


def _masked_forwards(model, batch, I, **kw):
    with torch.no_grad():
        return torch.stack([model.forward_batch(_masked(batch, i), **kw).cpu() for i in range(I)], 1)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_against_the_masked_forward_and_the_plain_forward(precision):
    n, I = 96, 8
    model = _mk(seed=3).cuda().eval()
    batch = synthetic.make_batch(n, ragged=True, seed=6, stress=True)
    dev = {k: ({b: t.cuda() for b, t in v.items()} if isinstance(v, dict) else v.cuda()) for k, v in _copy(batch).items()}
    model.precision = precision
    live = _live(batch)
    assert live.any() and (~live).any()
    for dense in (True, False):
        d = _run(model, dev, precision, dense=dense)
        with torch.no_grad():
            plain = model.forward_batch(dev, dense=dense).cpu()
        assert torch.equal(d["logits"], plain)
    want = _masked_forwards(model, dev, I)
    err = (d["without"] - want)[live].abs().max().item()
    prom = (d["promoter_only"] - model.forward_batch(_masked(dev, None)).cpu()).abs().max().item()
    print(f"{precision}: max |without - masked forward| {err:.3e}, promoter_only {prom:.3e}")
    tol = 1e-6 if precision == "fp32" else TOL16
    assert err <= tol and prom <= tol
    # dead slots: the logits themselves, bit for bit, and an effect of exactly zero
    dead = ~live
    assert torch.equal(d["without"][dead], d["logits"].unsqueeze(1).expand_as(d["without"])[dead])
    assert torch.equal(d["effect"][dead], torch.zeros(int(dead.sum())))
    t = 1
    assert torch.equal(d["effect"], d["logits"][:, t:t + 1] - d["without"][:, :, t])


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_junk_in_dead_slots_changes_nothing(precision):
    n = 64
    model = _mk(seed=8).cuda().eval()
    batch = synthetic.make_batch(n, ragged=True, seed=12)
    live = _live(batch)
    other = _copy(batch)
    gen = torch.Generator().manual_seed(3)
    for b in BINS:
        x = other["pcre_feats"][b]
        x[:] = torch.where((~live).view(n, -1, 1, 1), 9.0 * torch.rand(x.shape, generator=gen), x)
    a, b_ = _run(model, batch, precision), _run(model, other, precision)
    for key in a:
        assert torch.equal(a[key], b_[key]), key


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_arbitrary_interaction_masks(precision):
    """Masks the reference's Dataset never produces: no block form, so the variants keep every slot (the plan's
    fallback to the full token class), and a slot can be live in one resolution only."""
    n, I, S = 48, 8, 9
    model = _mk(seed=19).cuda().eval()
    batch = synthetic.make_batch(n, ragged=True, seed=23)
    gen = torch.Generator().manual_seed(5)
    for b in BINS:
        im = batch["interaction_masks"][b]
        im[:24, 0] = torch.rand(24, S, S, generator=gen) < 0.4
        im[:24, 0, :, 0] = False
    live = _live(batch)
    d = _run(model, batch, precision)
    want = _masked_forwards(model, {k: ({b: t.cuda() for b, t in v.items()} if isinstance(v, dict) else v.cuda())
                                    for k, v in _copy(batch).items()}, I)
    err = (d["without"] - want)[live].abs().max().item()
    print(f"{precision}: max |without - masked forward| {err:.3e}")
    assert err <= (1e-6 if precision == "fp32" else TOL16)
    assert torch.equal(d["without"][~live], d["logits"].unsqueeze(1).expand_as(d["without"])[~live])


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_non_fused_regulation_path(precision):
    n, I = 40, 8
    model = _mk(ChromoformerRegressor, seed=13, reg=REG4).cuda().eval()
    batch = synthetic.make_batch(n, ragged=True, seed=17)
    dev = {k: ({b: t.cuda() for b, t in v.items()} if isinstance(v, dict) else v.cuda()) for k, v in _copy(batch).items()}
    live = _live(batch)
    d = _run(model, dev, precision)
    with torch.no_grad():
        assert torch.equal(d["logits"], model.forward_batch(dev).cpu())
    want = _masked_forwards(model, dev, I)
    err = (d["without"] - want)[live].abs().max().item()
    print(f"{precision}: max |without - masked forward| {err:.3e}")
    assert err <= (1e-6 if precision == "fp32" else TOL16)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_chunking_and_repeat_are_bit_identical(precision):
    n = 23
    model = _mk(seed=29).cuda().eval()
    batch = synthetic.make_batch(n, ragged=True, seed=31)
    ref = _run(model, batch, precision)
    again = _run(model, batch, precision)
    for chunk in (1, 5, n, 4096):
        got = _run(model, batch, precision, chunk=chunk)
        for key in ref:
            assert torch.equal(got[key], ref[key]), (chunk, key)
    for key in ref:
        assert torch.equal(again[key], ref[key]), key
    assert not any(v.requires_grad for v in ref.values())
    assert all(p.grad is None for p in model.parameters())


def test_capturable_into_a_cuda_graph():
    n = 256
    model = _mk(seed=37).cuda().eval()
    model.precision = "bf16"
    a = _copy(synthetic.make_batch(n, ragged=True, seed=61))
    b = _copy(synthetic.make_batch(n, ragged=True, seed=62))
    to_dev = lambda x: {k: ({bb: t.cuda() for bb, t in v.items()} if isinstance(v, dict) else v.cuda()) for k, v in x.items()}
    a, b = to_dev(a), to_dev(b)
    want_b = pcre_deletion(model, b)
    static = to_dev(a)
    with torch.no_grad():
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            pcre_deletion(model, static)
        torch.cuda.current_stream().wait_stream(s)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            out = pcre_deletion(model, static)
        for k in static:
            if isinstance(static[k], dict):
                for bb in static[k]:
                    static[k][bb].copy_(b[k][bb])
            else:
                static[k].copy_(b[k])
        g.replay()
        torch.cuda.synchronize()
    for key in want_b:
        assert torch.equal(out[key], want_b[key]), key


def test_errors():
    lib = _lib.load()
    model = _mk(seed=43).cuda().eval()
    batch = synthetic.make_batch(4, ragged=True, seed=2)
    args = synthetic.forward_args(batch, "cuda")
    io = _BatchIO(model, *[[d[b] for b in BINS] for d in args[:5]], args[5])
    dev = torch.device("cuda")
    I, no = int(io.cfg.i_max), int(model._cfg.n_out)
    logits, without, prom = (torch.empty(4, no, device=dev), torch.empty(4, I, no, device=dev), torch.empty(4, no, device=dev))
    flags = _lib.F_BF16
    need = lib.chromo_pcre_deletion_workspace_floats(ctypes.byref(io.cfg), 4, flags)
    assert need > lib.chromo_workspace_floats(ctypes.byref(io.cfg), 4 * (I + 1), flags)
    ws = torch.empty(need, device=dev)
    stream = torch.cuda.current_stream().cuda_stream

    def call(flags=flags, n=need, w=without):
        return lib.chromo_pcre_deletion(ctypes.byref(io.cfg), model.flat_params.data_ptr(), ctypes.byref(io.struct),
                                        logits.data_ptr(), w.data_ptr() if w is not None else None, prom.data_ptr(),
                                        ws.data_ptr(), n, flags, stream)

    assert call() == 0
    torch.cuda.synchronize()
    assert call(n=need - 1) == -2 and str(need) in lib.chromo_last_error().decode()
    assert call(w=None) == -1
    for bad in (_lib.F_TRAINING, _lib.F_BWD_HEAD_REG, _lib.F_BWD_REST, _lib.F_FREQ_GRAD, 8):
        assert call(flags=flags | bad) == -1, bad
    with pytest.raises(_lib.ChromoLibError):
        model._launch_deletion(io, _lib.F_TRAINING)
