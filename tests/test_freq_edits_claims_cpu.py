"""The facts the interaction-frequency edits (chromo_freq_edits, csrc/freq_edits.cu) rest on, checked on the as-written
CPU oracle - no GPU, no library involved:

  1. interaction_freq reaches neither the Embedding nor the Pairwise stage: X_in is bit-identical under any
     interaction_freq, junk (NaN, inf, huge values) included, so one Embedding / Pairwise pass per gene serves every
     frequency variant of that gene;
  2. an edit of a pair that is masked at every resolution leaves the logits bit-identical, so a dummy slot's contact
     has no effect;
and the wiring of contact_shapley / contact_knockout / contact_response with a game in place of the replay: the players
are the live contacts, an absent contact is 0, the values sum to v(all) - v(none)."""
import numpy as np
import torch

from _util import BINS, KWS
from chromoformer_b200 import ChromoformerClassifier, attribution, synthetic
from oracle import chromoformer_oracle as oracle

I = 8
S = I + 1


def _model_sd(seed=5):
    m = ChromoformerClassifier(7, 128, 128, dict(KWS[0]), dict(KWS[1]), dict(KWS[2]), seed=seed, i_max=I)
    return {k: v.detach().clone() for k, v in m.state_dict().items()}


def _forward(sd, batch, monkeypatch=None):
    """The oracle's logits and, through the Regulation transformer's input, X_in per bin size."""
    seen = {}
    orig = oracle.regulation_transformer

    def spy(x, mask, bias, sd_, pre, n_heads):
        seen[pre] = x.clone()
        return orig(x, mask, bias, sd_, pre, n_heads)
    monkeypatch.setattr(oracle, "regulation_transformer", spy)
    with torch.no_grad():
        logits = oracle.chromoformer_forward(sd, *synthetic.forward_args(synthetic.expand_full_masks(batch)))
    return logits, [seen[f"regulation.{b}."] for b in BINS]


def _copy(batch):
    return {k: ({b: t.clone() for b, t in v.items()} if isinstance(v, dict) else v.clone())
            for k, v in batch.items() if k in synthetic.FORWARD_KEYS}


def test_x_in_does_not_read_interaction_freq(monkeypatch):
    sd = _model_sd()
    batch = synthetic.make_batch(4, ragged=True, seed=7)
    _, base = _forward(sd, batch, monkeypatch)
    gen = torch.Generator().manual_seed(1)
    for junk in (torch.randn(4, S, S, generator=gen) * 10, torch.full((4, S, S), float("nan")),
                 torch.full((4, S, S), float("inf")), torch.full((4, S, S), -3e38), torch.zeros(4, S, S)):
        edited = _copy(batch)
        edited["interaction_freq"] = junk
        _, got = _forward(sd, edited, monkeypatch)
        for a, b in zip(got, base):
            assert torch.equal(a, b)


def test_edits_of_pairs_masked_at_every_resolution_change_nothing(monkeypatch):
    sd = _model_sd(seed=9)
    batch = synthetic.make_batch(6, ragged=True, seed=3)
    want, _ = _forward(sd, batch, monkeypatch)
    shape = batch["interaction_freq"].shape
    masked = torch.stack([batch["interaction_masks"][b].reshape(shape).bool() for b in BINS]).all(0)   # [B, S, S]
    live = attribution._live(batch, BINS)
    assert (~live).any() and masked.any()
    gen = torch.Generator().manual_seed(2)
    for values in (torch.randn(shape, generator=gen) * 10, torch.full(shape, 1e6), torch.full(shape, -10.0)):
        edited = _copy(batch)
        edited["interaction_freq"] = torch.where(masked, values, batch["interaction_freq"])
        got, _ = _forward(sd, edited, monkeypatch)
        assert torch.equal(got, want)
    # a dummy slot's contact [0, i + 1] in particular
    edited = _copy(batch)
    g, i = torch.nonzero(~live, as_tuple=True)
    edited["interaction_freq"][g, 0, i + 1] = 7.5
    got, _ = _forward(sd, edited, monkeypatch)
    assert torch.equal(got, want)


def test_descriptors_and_wiring_with_a_game_in_place_of_the_replay(monkeypatch):
    """contact_shapley / contact_knockout / contact_response / freq_edits end to end, with the library replay replaced
    by a quadratic game over the contacts each variant's freq edit leaves (value column 1), on genes of the synthetic
    ragged set."""
    model = ChromoformerClassifier(seed=1)
    batch = synthetic.make_batch(10, ragged=True, seed=3)
    B = 10
    bins = list(model.binsizes)
    live = attribution._live(attribution._to_device(batch, model, bins), bins)
    freq = batch["interaction_freq"].clone()
    contact = freq[:, 0, 1:].double()
    gen = torch.Generator().manual_seed(0)
    a = torch.randn(B, I, generator=gen, dtype=torch.float64)
    b = torch.randn(B, I, I, generator=gen, dtype=torch.float64).triu(1)
    b = b + b.transpose(1, 2)

    def game(g, c):
        """value of genes g [V] at contacts c [V, I] (only live contacts count)."""
        c = c * live[g]
        return (a[g] * c).sum(1) + torch.einsum("vi,vij,vj->v", c, b[g], c) / 2

    calls = []

    def fake_freq_replay(model_, dev_batch, bins_, var_gene, var_freq, chunk, dense):
        assert (np.diff(var_gene) >= 0).all()
        V = len(var_gene)
        f = var_freq(0, V)
        assert f.shape == (V, S, S) and f.dtype == torch.float32
        g = torch.from_numpy(np.asarray(var_gene))
        edited = torch.where(torch.isnan(f), dev_batch["interaction_freq"][g].float(), f)
        calls.append((g, f))
        val = game(g, edited[:, 0, 1:].double())
        full = game(torch.arange(B), contact)
        return torch.stack([full, full], 1).float(), torch.stack([val, val], 1).float()

    monkeypatch.setattr(attribution, "_freq_replay", fake_freq_replay)
    # Shapley values of a quadratic game in the contacts x_i (absent: 0): a_i x_i + 1/2 sum_j b_ij x_i x_j
    lc = contact * live
    truth = torch.where(live, a * lc + (b * lc.view(B, 1, I)).sum(2) * lc / 2, torch.zeros((), dtype=torch.float64))
    r = attribution.contact_shapley(model, batch)
    g, f = calls[-1]
    rest = torch.ones(S, S, dtype=torch.bool)
    rest[0, 1:] = False
    assert torch.isnan(f[:, rest]).all()                                  # only the contacts are edited ...
    edited_contacts = ~torch.isnan(f[:, 0, 1:])
    assert not (edited_contacts & ~live[g]).any()                         # ... and only live ones, to 0
    assert (f[:, 0, 1:][edited_contacts] == 0).all()
    assert (r["shapley"] - truth).abs().max().item() < 1e-4
    assert torch.equal(r["shapley"][~live], torch.zeros(int((~live).sum()), dtype=torch.float64))
    assert (r["blind"] == 0).all()                                        # v(none): every contact 0
    eff = r["shapley"].sum(1) - (r["logits"][:, 1] - r["blind"][:, 1]).double()
    assert eff.abs().max().item() < 1e-4
    p = attribution.contact_shapley(model, batch, permutations=5, seed=4)
    assert (p["shapley"].sum(1) - r["logits"][:, 1].double()).abs().max().item() < 1e-4
    assert torch.equal(p["shapley"], attribution.contact_shapley(model, batch, permutations=5, seed=4)["shapley"])
    # knockout: without[g, i] is the game with contact i set to 0; blind with every contact 0
    k = attribution.contact_knockout(model, batch)
    full = game(torch.arange(B), contact).float()
    for gg in range(B):
        for i in range(I):
            c = contact[gg:gg + 1].clone()
            c[0, i] = 0
            want = game(torch.tensor([gg]), c).float() if live[gg, i] else full[gg:gg + 1]
            assert torch.allclose(k["without"][gg, i, 1], want[0], atol=1e-5)
    assert torch.equal(k["effect"][~live], torch.zeros(int((~live).sum())))
    assert (k["blind"] == 0).all() and torch.equal(k["blind_effect"], full)
    # response: absolute and relative grids
    vals = [0.0, 0.5, 2.0]
    for relative in (False, True):
        resp = attribution.contact_response(model, batch, vals, relative=relative)
        assert resp["response"].shape == (B, I, 3, 2) and resp["value"].shape == (B, I, 3)
        for gg, i in zip(*torch.nonzero(live, as_tuple=True)):
            for j, v in enumerate(vals):
                c = contact[gg:gg + 1].clone()
                c[0, i] = v * c[0, i] if relative else v
                assert torch.allclose(resp["value"][gg, i, j], game(gg.view(1), c).float()[0], atol=1e-5)
        assert torch.equal(resp["value"][~live], full.view(B, 1, 1).expand(B, I, 3)[~live])
    # freq_edits: shared [V, S, S] and per-gene [B, V, S, S] edits give the same variants
    edits = torch.full((2, S, S), float("nan"))
    edits[1, 0, 1:] = 0.25
    shared = attribution.freq_edits(model, batch, edits, target=1)
    per_gene = attribution.freq_edits(model, batch, edits.expand(B, 2, S, S).clone(), target=1)
    assert torch.equal(shared["variants"], per_gene["variants"])
    assert torch.allclose(shared["value"][:, 0], full)
