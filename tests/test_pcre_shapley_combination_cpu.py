"""The FP64 combination code of pcre_shapley / pcre_interactions (chromoformer_b200/attribution.py) on a quadratic game
with known answers, no GPU:  v(T) = sum_{i in T} a_i + sum_{i < j in T} b_ij  has Shapley values a_i + 1/2 sum_j b_ij and
pairwise interactions Delta_ij = b_ij."""
import itertools

import numpy as np
import torch

from chromoformer_b200.attribution import _interactions, _shapley_exact, _shapley_from_orders

I = 6


def _game(k, seed):
    gen = torch.Generator().manual_seed(seed)
    a = torch.randn(k, generator=gen, dtype=torch.float64)
    b = torch.randn(k, k, generator=gen, dtype=torch.float64).triu(1)
    b = b + b.T
    return a, b


def _value(a, b, members):
    m = list(members)
    return a[m].sum() + b[m][:, m].sum() / 2


def _shapley_truth(a, b):
    return a + b.sum(1) / 2


def test_exact_shapley_of_a_quadratic_game():
    for k in (1, 2, 5):
        games = [_game(k, seed) for seed in range(3)]
        v = torch.stack([torch.stack([_value(a, b, [j for j in range(k) if (s >> j) & 1]) for s in range(1 << k)])
                         for a, b in games])
        phi = _shapley_exact(v, k)
        want = torch.stack([_shapley_truth(a, b) for a, b in games])
        assert (phi - want).abs().max().item() < 1e-12
        assert (phi.sum(1) - (v[:, -1] - v[:, 0])).abs().max().item() < 1e-12      # efficiency


def _genes():
    """Three genes of I slots: k players on scattered slots (the others are dummy slots)."""
    slots = [[0, 2, 3, 5], [1, 4, 5], [0, 1, 2, 3, 4]]
    live = torch.zeros(len(slots), I, dtype=torch.bool)
    for g, s in enumerate(slots):
        live[g, s] = True
    return slots, live


def test_permutation_estimate_telescopes_and_is_exact_over_every_order():
    slots, live = _genes()
    G = len(slots)
    games = [_game(len(s), 10 + g) for g, s in enumerate(slots)]
    k = live.sum(1)

    def prefix_values(orders_per_gene):
        P = len(orders_per_gene[0])
        order = torch.zeros(G, P, I, dtype=torch.long)
        v = torch.zeros(G, P, I + 1, dtype=torch.float64)
        for g, (s, (a, b)) in enumerate(zip(slots, games)):
            dead = [j for j in range(I) if j not in s]
            for p, players in enumerate(orders_per_gene[g]):
                order[g, p] = torch.tensor([s[q] for q in players] + dead)
                for j in range(len(s) + 1):
                    v[g, p, j] = _value(a, b, players[:j])
                v[g, p, len(s) + 1:] = 7.0                         # past k: never read
        return v, order

    # a few random orders: per order the credits sum to v(all) - v(none)
    gen = torch.Generator().manual_seed(1)
    rand_orders = [[torch.randperm(len(s), generator=gen).tolist() for _ in range(3)] for s in slots]
    v, order = prefix_values(rand_orders)
    phi = _shapley_from_orders(v, order, k)
    full = torch.stack([_value(a, b, range(len(s))) - _value(a, b, []) for s, (a, b) in zip(slots, games)])
    assert (phi.sum(1) - full).abs().max().item() < 1e-12
    assert torch.equal(phi[~live], torch.zeros(int((~live).sum()), dtype=torch.float64))
    # every order once (the k! orders of each gene, padded to the same count by repeating the list): exact Shapley
    n = max(len(s) for s in slots)
    all_orders = []
    for s in slots:
        perms = list(itertools.permutations(range(len(s))))
        all_orders.append([list(p) for p in perms] * (len(list(itertools.permutations(range(n)))) // len(perms)))
    v, order = prefix_values(all_orders)
    phi = _shapley_from_orders(v, order, k)
    for g, (s, (a, b)) in enumerate(zip(slots, games)):
        assert (phi[g, s] - _shapley_truth(a, b)).abs().max().item() < 1e-12
    assert torch.equal(phi[~live], torch.zeros(int((~live).sum()), dtype=torch.float64))


def test_interactions_of_a_quadratic_game():
    slots, live = _genes()
    G = len(slots)
    pairs = [(i, j) for i in range(I) for j in range(i + 1, I)]
    f0 = torch.zeros(G, dtype=torch.float64)
    fi = torch.zeros(G, I, dtype=torch.float64)
    fij = torch.zeros(G, len(pairs), dtype=torch.float64)
    truth = torch.zeros(G, I, I, dtype=torch.float64)
    for g, s in enumerate(slots):
        a, b = _game(len(s), 20 + g)
        player = {slot: q for q, slot in enumerate(s)}
        everyone = set(range(len(s)))
        f0[g] = _value(a, b, everyone)
        for i in s:
            fi[g, i] = _value(a, b, everyone - {player[i]})
        for c, (i, j) in enumerate(pairs):
            if i in player and j in player:
                fij[g, c] = _value(a, b, everyone - {player[i], player[j]})
                truth[g, i, j] = truth[g, j, i] = b[player[i], player[j]]
            else:
                fij[g, c] = 3.0                                     # a variant that was not run: never read
        for i in range(I):
            if i not in player:
                fi[g, i] = -5.0
    inter, effect = _interactions(f0, fi, fij, pairs, live)
    assert (inter - truth).abs().max().item() < 1e-12
    assert torch.equal(inter, inter.transpose(1, 2))
    assert torch.equal(torch.diagonal(inter, dim1=1, dim2=2), torch.zeros(G, I, dtype=torch.float64))
    dead = ~live
    assert torch.equal(inter[dead], torch.zeros(int(dead.sum()), I, dtype=torch.float64))
    assert torch.equal(inter.transpose(1, 2)[dead], torch.zeros(int(dead.sum()), I, dtype=torch.float64))
    assert torch.equal(effect[dead], torch.zeros(int(dead.sum()), dtype=torch.float64))
    assert (effect[live] - (f0.view(G, 1) - fi)[live]).abs().max().item() == 0.0


def test_descriptors_and_wiring_with_a_game_in_place_of_the_replay(monkeypatch):
    """pcre_shapley / pcre_interactions / pcre_subsets end to end, with the library replay replaced by a quadratic game
    over the kept pCREs (value column 1), on genes of the synthetic ragged set."""
    from chromoformer_b200 import ChromoformerClassifier, attribution, synthetic

    model = ChromoformerClassifier(seed=1)
    batch = synthetic.make_batch(10, ragged=True, seed=3)
    B, I = 10, 8
    live = attribution._live(attribution._to_device(batch, model, list(model.binsizes)), list(model.binsizes))
    gen = torch.Generator().manual_seed(0)
    a = torch.randn(B, I, generator=gen, dtype=torch.float64)
    b = torch.randn(B, I, I, generator=gen, dtype=torch.float64).triu(1)
    b = b + b.transpose(1, 2)

    def fake_replay(model_, dev_batch, bins, var_gene, var_drop, chunk, dense):
        assert (np.diff(var_gene) >= 0).all()
        kept = live[torch.from_numpy(var_gene)] & ~((torch.from_numpy(var_drop).view(-1, 1) >> torch.arange(I)) & 1).bool()
        kf = kept.double()
        g = torch.from_numpy(var_gene)
        val = (a[g] * kf).sum(1) + torch.einsum("vi,vij,vj->v", kf, b[g], kf) / 2
        full = (a * live).sum(1) + torch.einsum("gi,gij,gj->g", live.double(), b, live.double()) / 2
        return (torch.stack([full, full], 1).float(), torch.stack([val, val], 1).float())

    monkeypatch.setattr(attribution, "_replay", fake_replay)
    bl = b * live.view(B, 1, I) * live.view(B, I, 1)
    truth = torch.where(live, a + bl.sum(2) / 2, torch.zeros((), dtype=torch.float64))
    r = attribution.pcre_shapley(model, batch)
    assert (r["shapley"] - truth).abs().max().item() < 1e-5
    assert torch.equal(r["shapley"][~live], torch.zeros(int((~live).sum()), dtype=torch.float64))
    assert (r["promoter_only"] == 0).all()
    p = attribution.pcre_shapley(model, batch, permutations=5, seed=4)
    eff = p["shapley"].sum(1) - r["logits"][:, 1].double()
    assert eff.abs().max().item() < 1e-5
    assert torch.equal(p["shapley"], attribution.pcre_shapley(model, batch, permutations=5, seed=4)["shapley"])
    it = attribution.pcre_interactions(model, batch)
    assert (it["interaction"] - bl).abs().max().item() < 1e-5
    assert torch.equal(it["interaction"], it["interaction"].transpose(1, 2))
    drop = torch.zeros(3, I, dtype=torch.bool)
    drop[1, 0] = drop[2] = True
    sub = attribution.pcre_subsets(model, batch, drop, target=1)
    assert sub["variants"].shape == (B, 3, 2) and sub["value"].shape == (B, 3)
    assert (sub["value"][:, 2] == 0).all()
