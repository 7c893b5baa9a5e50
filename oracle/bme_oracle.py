"""CPU restatement of the balanced minimum-evolution rules of ngsdist_b200/csrc/bme.cu -- TEST INFRASTRUCTURE ONLY.

FastME, which the reference's workflow (README.md:83-98) runs on the .dist file, is an external program, so parity with
it is unpinned.  This restates the published criterion (Desper & Gascuel 2002; Pauplin 2000) with the tie rules of
DESIGN §3 N4:
    tau_ij  edges between leaves i and j,  P_ij = 2^-tau_ij d_ij,  S_XY = sum_{i in X, j in Y} P_ij
    L(T) = sum_{i<j} 2^(1 - tau_ij) d_ij
The tree is rooted at individual 0; internal node ids follow the NJ join order (join t makes node n + t, the final
trifurcation centre is 2n - 3).  For every internal edge (u, v), v an internal child of u: A = everything not below u,
B = v's sibling, C and D = v's children (C holds the smaller individual index), and
    gain(B<->C) = S_AB + S_CD - 2 (S_AC + S_BD),  gain(B<->D) = S_AB + S_CD - 2 (S_AD + S_BC)
    length(u, v) = 2 (S_AC + S_AD + S_BC + S_BD) - 2 (S_AB + S_CD)
    pendant edge of leaf i (X, Y the other two subtrees at its neighbour): 2 (S_iX + S_iY - S_XY)
Greedy: the largest gain (ties: smallest (v, variant), B<->C is variant 0) is applied while it exceeds 1e-12 M,
    M = sum_{i<j} 2^(1 - tau_ij) |d_ij|   (= L when no distance is negative).

pauplin_length() and all_nni_gains() are the brute-force definitions: path lengths from the tree, every NNI applied."""
import re

import numpy as np

from . import nj_oracle


class Tree:
    """Unrooted binary tree on leaves 0..n-1 (internal nodes n..2n-3), rooted at leaf 0: u0 is leaf 0's neighbour,
    kids[w] the two children of internal node w."""

    def __init__(self, n, adj):
        self.n = n
        self.u0 = adj[0][0]
        self.parent = {self.u0: 0}
        self.kids = {}
        stack = [self.u0]
        while stack:
            w = stack.pop()
            ks = [x for x in adj[w] if x != self.parent[w]]
            self.kids[w] = ks
            for x in ks:
                self.parent[x] = w
                if x >= n:
                    stack.append(x)
        self.order()

    def leaves_below(self, w):
        if w < self.n:
            return [w]
        return self.leaves_below(self.kids[w][0]) + self.leaves_below(self.kids[w][1])

    def order(self):
        """Children by smallest individual index; DFS leaf positions (leaf 0 first); lo/hi position ranges."""
        def minleaf(w):
            if w < self.n:
                return w
            m = [minleaf(k) for k in self.kids[w]]
            if m[1] < m[0]:
                self.kids[w].reverse()
            return min(m)
        minleaf(self.u0)
        self.perm, self.lo, self.hi = [0], {0: 0}, {0: 1}

        def visit(w):
            if w < self.n:
                self.lo[w] = len(self.perm)
                self.perm.append(w)
                self.hi[w] = len(self.perm)
                return
            for k in self.kids[w]:
                visit(k)
            self.lo[w], self.hi[w] = self.lo[self.kids[w][0]], self.hi[self.kids[w][1]]
        visit(self.u0)

    def internal_nodes(self):
        """The v of every internal edge (u, v), in increasing id."""
        return [v for v in sorted(self.kids) if v != self.u0]

    def nni(self, v, variant):
        u = self.parent[v]
        bi = 1 if self.kids[u][0] == v else 0
        B, C = self.kids[u][bi], self.kids[v][variant]
        self.kids[u][bi], self.parent[C] = C, u
        self.kids[v][variant], self.parent[B] = B, v
        self.order()

    def tau(self):
        """Edges between every pair of leaves (indexed by leaf): all pairs split by internal node w meet at w."""
        n = self.n
        depth = {0: 0, self.u0: 1}
        stack = [self.u0]
        while stack:
            w = stack.pop()
            for k in self.kids[w]:
                depth[k] = depth[w] + 1
                if k >= n:
                    stack.append(k)
        lca = np.zeros((n, n), dtype=np.int64)              # in positions; pairs with leaf 0 meet at leaf 0 (depth 0)
        for w, (a, b) in self.kids.items():
            lca[self.lo[a]:self.hi[a], self.lo[b]:self.hi[b]] = depth[w]
            lca[self.lo[b]:self.hi[b], self.lo[a]:self.hi[a]] = depth[w]
        dl = np.array([depth[k] for k in self.perm], dtype=np.int64)
        tp = dl[:, None] + dl[None, :] - 2 * lca
        np.fill_diagonal(tp, 0)
        T = np.empty_like(tp)
        T[np.ix_(self.perm, self.perm)] = tp
        return T

    def splits(self):
        """Non-trivial bipartitions as frozensets of leaf indices (the side without leaf 0)."""
        out = set()
        for w in self.kids:
            if w != self.u0:
                side = frozenset(self.leaves_below(w))
                if 1 < len(side) < self.n - 1:
                    out.add(side)
        return out


def from_joins(n, joins):
    """The NJ tree of nj_oracle.nj's join list: join t makes node n + t, the three slots left meet at node 2n - 3."""
    adj = {k: [] for k in range(2 * n - 2)}
    slot = list(range(n))

    def link(a, b):
        adj[a].append(b)
        adj[b].append(a)
    retired = set()
    for t, (i, j, _, _) in enumerate(joins):
        link(n + t, slot[i])
        link(n + t, slot[j])
        slot[i] = n + t
        retired.add(j)
    for k in range(n):
        if k not in retired:
            link(2 * n - 3, slot[k])
    return Tree(n, adj)


def from_newick(newick, labels=None):
    """Parse a binary Newick (trifurcating or bifurcating root; lengths and internal labels ignored) into a Tree; leaves
    are numbered by `labels` or by their "Ind_<i>" names."""
    toks = re.findall(r"[(),;]|[^(),;:]+|:[^(),;]+", newick)
    index = {l: k for k, l in enumerate(labels)} if labels is not None else None
    n = sum(1 for k, t in enumerate(toks) if t not in "(),;" and t[0] != ":" and toks[k - 1] != ")")
    adj = {}

    def link(a, b):
        adj.setdefault(a, []).append(b)
        adj.setdefault(b, []).append(a)
    stack, nxt, prev = [], n, None
    for t in toks:
        if t == "(":
            if stack:
                link(stack[-1], nxt)
            stack.append(nxt)
            nxt += 1
        elif t == ")":
            stack.pop()
        elif t not in ",;" and t[0] != ":" and prev != ")":
            link(stack[-1], index[t] if index is not None else int(t[len("Ind_"):]))
        prev = t
    root = n
    if len(adj[root]) == 2:                          # a bifurcating root is not a node of the unrooted tree
        a, b = adj.pop(root)
        adj[a] = [b if x == root else x for x in adj[a]]
        adj[b] = [a if x == root else x for x in adj[b]]
        last = nxt - 1                               # keep the internal ids n .. 2n - 3
        if last != root:
            adj[root] = adj.pop(last)
            for x in adj[root]:
                adj[x] = [root if y == last else y for y in adj[x]]
    return Tree(n, adj)


def edge_lengths(newick, labels=None):
    """{side of the edge without leaf 0: length} of every edge of a Newick tree written by newick() / ngsd_bme_tree."""
    toks = re.findall(r"[(),;]|[^(),;:]+|:[^(),;]+", newick)
    index = {l: k for k, l in enumerate(labels)} if labels is not None else None
    stack, last, out, allv = [], None, {}, set()
    for t in toks:
        if t == "(":
            stack.append(set())
        elif t == ")":
            last = stack.pop()
            if stack:
                stack[-1] |= last
        elif t[0] == ":":
            out[frozenset(last)] = float(t[1:])
        elif t not in ",;":
            last = {index[t] if index is not None else int(t[len("Ind_"):])}
            allv |= last
            stack[-1] |= last
    return {(frozenset(allv) - s if 0 in s else s): length for s, length in out.items()}


def pauplin_length(newick, d, labels=None):
    """L(T) = sum_{i<j} 2^(1 - tau_ij) d_ij of a Newick tree, from its path lengths."""
    t = newick if isinstance(newick, Tree) else from_newick(newick, labels)
    d = np.asarray(d, dtype=np.float64)
    T = t.tau()
    iu = np.triu_indices(t.n, 1)
    return float(np.sum(np.ldexp(d[iu], 1 - T[iu])))


def all_nni_gains(newick, d, labels=None):
    """Brute force: {new bipartition (side without leaf 0): L(T) - L(T')} over both NNIs of every internal edge, each
    applied to a copy of the tree and L(T') recomputed from path lengths."""
    import copy
    t = newick if isinstance(newick, Tree) else from_newick(newick, labels)
    L0 = pauplin_length(t, d)
    base = t.splits()
    out = {}
    for v in t.internal_nodes():
        for variant in (0, 1):
            t2 = copy.deepcopy(t)
            t2.nni(v, variant)
            new = t2.splits() - base
            assert len(new) == 1
            out[next(iter(new))] = L0 - pauplin_length(t2, d)
    return out


def _S(t, d):
    """S(X, Y) of position ranges X, Y (lists of (lo, hi)), with P[p, q] = 2^-tau d of the leaves at positions p, q."""
    perm = np.array(t.perm)
    P = np.ldexp(np.asarray(d, dtype=np.float64)[np.ix_(perm, perm)], -t.tau()[np.ix_(perm, perm)])
    np.fill_diagonal(P, 0.0)
    return lambda X, Y: sum(float(P[a:b, c:e].sum()) for a, b in X for c, e in Y)


def _ranges(t, v, u):
    """A, B, C, D of internal edge (u, v) as position ranges."""
    r = lambda w: [(t.lo[w], t.hi[w])]
    B = [k for k in t.kids[u] if k != v][0]
    C, D = t.kids[v]
    return [(0, t.lo[u]), (t.hi[u], t.n)], r(B), r(C), r(D)


def formula_gains(t, d):
    """[(v, variant, gain, new bipartition)] from the S-sums of the rules above, in increasing (v, variant); the new
    bipartition is the side without leaf 0 of edge (u, v) after the swap."""
    S = _S(t, d)
    out = []
    for v in t.internal_nodes():
        A, B, C, D = _ranges(t, v, t.parent[v])
        sAB, sCD, sAC, sBD, sAD, sBC = S(B, A), S(C, D), S(C, A), S(B, D), S(D, A), S(B, C)
        for variant, g in ((0, sAB + sCD - 2 * (sAC + sBD)), (1, sAB + sCD - 2 * (sAD + sBC))):
            below = B + (D if variant == 0 else C)    # v's children after the swap
            out.append((v, variant, g, frozenset(t.perm[p] for a, b in below for p in range(a, b))))
    return out


def balanced_lengths(t, d):
    """{node: length of the edge above it} (leaf 0: its pendant edge)."""
    S = _S(t, d)
    out = {}
    for v in t.internal_nodes():
        A, B, C, D = _ranges(t, v, t.parent[v])
        out[v] = 2 * (S(C, A) + S(B, D) + S(D, A) + S(B, C)) - 2 * (S(B, A) + S(C, D))
    for i in range(t.n):
        if i == 0:
            (a, b) = t.kids[t.u0]
            X, Y = [(t.lo[a], t.hi[a])], [(t.lo[b], t.hi[b])]
        else:
            u = t.parent[i]
            x = [k for k in t.kids[u] if k != i][0]
            X, Y = [(t.lo[x], t.hi[x])], [(0, t.lo[u]), (t.hi[u], t.n)]
        p = [(t.lo[i], t.hi[i])]
        out[i] = 2 * (S(p, X) + S(p, Y) - S(X, Y))
    return out


def newick(t, lengths, labels=None):
    """"(Ind_0:l,(...):l,(...):l);", every node's children in order of their smallest individual index."""
    lab = lambda k: labels[k] if labels is not None else "Ind_%d" % k

    def sub(w):
        if w < t.n:
            return "%s:%.10f" % (lab(w), lengths[w])
        a, b = t.kids[w]
        return "(%s,%s):%.10f" % (sub(a), sub(b), lengths[w])
    a, b = t.kids[t.u0]
    return "(%s:%.10f,%s,%s);" % (lab(0), lengths[0], sub(a), sub(b))


def bme(dist, labels=None):
    """BME NNI refinement of nj_oracle.nj's tree.  Returns (newick, n_nni, rounds, L): rounds[k] = (best gain, second
    best gain, applied?, M) of every round evaluated, L the Pauplin length of the final tree.  A gain is applied when it
    exceeds 1e-12 M, M = sum_{i<j} 2^(1 - tau_ij) |d_ij| (the Pauplin length of |d|, which is L when no distance is
    negative): every applied NNI lowers L, so the loop ends for any finite matrix."""
    d = np.array(dist, dtype=np.float64)
    n = d.shape[0]
    _, joins, _ = nj_oracle.nj(d, labels)
    t = from_joins(n, joins)
    rounds, n_nni = [], 0
    while n > 3:
        gs = formula_gains(t, d)
        M = pauplin_length(t, np.abs(d))
        best = min(gs, key=lambda x: (-x[2], x[0], x[1]))
        second = max([g for g in gs if g is not best], key=lambda x: x[2], default=None)
        apply = best[2] > 1e-12 * M
        rounds.append((best[2], second[2] if second else -np.inf, apply, M))
        if not apply:
            break
        t.nni(best[0], best[1])
        n_nni += 1
    return newick(t, balanced_lengths(t, d), labels), n_nni, rounds, pauplin_length(t, d)
