"""The CPU restatement of the balanced minimum-evolution rules (oracle/bme_oracle.py) against the definitions it rests on:
every formula gain is the brute-force change of Pauplin's length under that interchange, the balanced lengths sum to
that length, and on an additive matrix they are the generating branch lengths.  No GPU involved."""
import numpy as np
import pytest

from oracle import bme_oracle, nj_oracle
from test_gpu_nj import additive_tree_matrix


def random_tree(n, rng):
    """A random binary tree in the NJ node numbering: n - 3 random joins of two live slots, then the trifurcation."""
    live = list(range(n))
    joins = []
    while len(live) > 3:
        a, b = sorted(rng.choice(len(live), 2, replace=False))
        i, j = live[a], live[b]
        joins.append((i, j, 0.0, 0.0))
        live.pop(b)
    return bme_oracle.from_joins(n, joins)


def random_matrix(n, rng):
    D = rng.rand(n, n)
    D = D + D.T
    np.fill_diagonal(D, 0)
    return D


@pytest.mark.parametrize("n", [5, 6, 9, 17, 40])
def test_formula_gains_are_the_brute_force_change_of_the_pauplin_length(n):
    rng = np.random.RandomState(100 + n)
    for _ in range(3):
        t = random_tree(n, rng)
        D = random_matrix(n, rng)
        L = bme_oracle.pauplin_length(t, D)
        brute = bme_oracle.all_nni_gains(t, D)
        formula = bme_oracle.formula_gains(t, D)
        assert len(formula) == len(brute) == 2 * (n - 3)
        for v, variant, g, split in formula:
            assert abs(g - brute[split]) <= 1e-12 * L, (v, variant)
        # ... and the same through the Newick the tree is written as
        nw = bme_oracle.newick(t, bme_oracle.balanced_lengths(t, D))
        assert bme_oracle.all_nni_gains(nw, D).keys() == brute.keys()
        assert bme_oracle.pauplin_length(nw, D) == pytest.approx(L, rel=1e-14)


@pytest.mark.parametrize("n", [3, 4, 5, 12, 40])
def test_balanced_lengths_sum_to_the_pauplin_length(n):
    rng = np.random.RandomState(200 + n)
    for _ in range(3):
        t = random_tree(n, rng)
        D = random_matrix(n, rng)
        lens = bme_oracle.balanced_lengths(t, D)
        assert len(lens) == 2 * n - 3
        assert abs(sum(lens.values()) - bme_oracle.pauplin_length(t, D)) <= 1e-12 * bme_oracle.pauplin_length(t, D)


def generating_lengths(n, seed):
    """additive_tree_matrix's tree again (same draws): {bipartition side without leaf 0 (or a leaf index): length}."""
    rng = np.random.RandomState(seed)
    edges = [(0, n, rng.uniform(0.05, 0.3)), (1, n, rng.uniform(0.05, 0.3)), (2, n, rng.uniform(0.05, 0.3))]
    nxt = n + 1
    for leaf in range(3, n):
        u, v, L = edges.pop(int(rng.randint(len(edges))))
        x = rng.uniform(0.2, 0.8) * L
        edges += [(u, nxt, x), (nxt, v, L - x), (leaf, nxt, rng.uniform(0.05, 0.3))]
        nxt += 1
    adj = {}
    for u, v, L in edges:
        adj.setdefault(u, []).append(v)
        adj.setdefault(v, []).append(u)
    out = {}
    for u, v, L in edges:
        seen, stack = {v}, [v]                    # the side of v once edge (u, v) is cut
        while stack:
            w = stack.pop()
            for y in adj[w]:
                if y not in seen and not (w == v and y == u):
                    seen.add(y)
                    stack.append(y)
        side = frozenset(k for k in seen if k < n)
        if 0 in side:
            side = frozenset(range(n)) - side
        out[side] = L
    return out


def test_balanced_lengths_of_the_generating_tree_of_an_additive_matrix():
    n = 40
    D, true_splits = additive_tree_matrix(n, 5)
    gen = generating_lengths(n, 5)
    _, joins, _ = nj_oracle.nj(D)
    t = bme_oracle.from_joins(n, joins)
    assert {frozenset("Ind_%d" % k for k in s) for s in t.splits()} == true_splits
    lens = bme_oracle.balanced_lengths(t, D)
    for w, length in lens.items():
        side = frozenset(t.leaves_below(w))
        if 0 in side:
            side = frozenset(range(n)) - side
        assert abs(length - gen[side]) <= 1e-12, w
    # no interchange improves the generating tree
    L = bme_oracle.pauplin_length(t, D)
    assert max(g for _, _, g, _ in bme_oracle.formula_gains(t, D)) <= 1e-12 * L


def test_bme_refinement_is_a_local_optimum_below_the_nj_length():
    rng = np.random.RandomState(7)
    n = 30
    D = random_matrix(n, rng)
    nw, n_nni, rounds, L = bme_oracle.bme(D)
    assert n_nni >= 1 and len(rounds) == n_nni + 1
    assert all(r[2] for r in rounds[:-1]) and not rounds[-1][2]
    assert L <= bme_oracle.pauplin_length(nj_oracle.nj(D)[0], D)
    assert max(bme_oracle.all_nni_gains(nw, D).values()) <= 1e-12 * L
    assert bme_oracle.pauplin_length(nw, D) == pytest.approx(L, rel=1e-14)
    _, lens = nj_oracle.newick_lengths(nw)
    assert sum(lens) == pytest.approx(L, rel=1e-9)


def test_bme_refinement_ends_on_matrices_with_negative_entries():
    """The acceptance scale is the Pauplin length of |d|: an all-equal negative matrix (every gain exactly 0, L < 0) takes
    no interchange, and on mixed signs every applied interchange lowers L."""
    n = 6
    nw, n_nni, rounds, L = bme_oracle.bme(-(np.ones((n, n)) - np.eye(n)))
    assert n_nni == 0 and len(rounds) == 1 and rounds[0][:3] == (0.0, 0.0, False) and L < 0
    rng = np.random.RandomState(3)
    D = rng.rand(40, 40) - 0.5
    D = (D + D.T) / 2
    np.fill_diagonal(D, 0)
    nw, n_nni, rounds, L = bme_oracle.bme(D)
    assert n_nni >= 1 and L < 0
    assert all(r[0] > 0 for r in rounds[:-1])
    assert L < bme_oracle.pauplin_length(nj_oracle.nj(D)[0], D)
