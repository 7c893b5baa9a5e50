"""--pairwise_del on two FP64 planes (pdel two-plane mode, ngsd_internal.h): with V = Z^T S Z and the shifts l, r,
    p_i^T S p_j = q_i^T V q_j + kappa m_i m_j,   q_i = m_i (p_i0 + l0, p_i1 + l1),  q_j = m_j (p_j0 + r0, p_j1 + r1)
for triples that sum to one (present) or are zero (missing), so the contraction needs K = 2 per site and the mask term
is kappa times the exact shared-site count.  The CPU test restates the rewrite against the oracle; the GPU tests check
that the mode is taken exactly where it should be (well-conditioned scores, matrices of at least 2^30 pair-sites), its
values, and that it agrees with the three-plane contraction."""
import numpy as np
import pytest

import oracle
from test_gpu_parity import nb
from test_gpu_score import ASYM, AVG, DEFAULT, GRID, INT, NEG, SEVEN_HALF, boot_counts, check, path_of, site_map
from util import load_bin

Z = np.array([[1.0, 0.0], [0.0, 1.0], [-1.0, -1.0]])
C = np.array([0.0, 0.0, 1.0])
SCORES = {"default": DEFAULT, "int": INT, "seven_half": SEVEN_HALF, "asym": ASYM, "negative": NEG}
NAN_SCORE = [0, .5, 1, .5, float("nan"), .5, 1, .5, 0]
NEAR_SINGULAR = [2, 2, 1, 1, 1.001, 0, 0, 0, 0]         # V = [[1, 1], [1, 1.001]], r ~ 1000


def coefficients(score):
    """V, l, r, kappa by Cramer's rule (api.cu pdel2_coefficients)."""
    S = np.asarray(score, dtype=np.float64).reshape(3, 3)
    V = Z.T @ S @ Z
    det = V[0, 0] * V[1, 1] - V[0, 1] * V[1, 0]
    adj = np.array([[V[1, 1], -V[0, 1]], [-V[1, 0], V[0, 0]]])
    with np.errstate(divide="ignore", invalid="ignore"):
        r = adj @ (Z.T @ S @ C) / det
        l = adj.T @ (Z.T @ S.T @ C) / det
    kappa = C @ S @ C - l @ V @ r
    return V, l, r, kappa


def taken(score):
    V, l, r, kappa = coefficients(score)
    vals = np.concatenate([V.ravel(), l, r, [kappa]])
    return bool(np.isfinite(vals).all() and max(np.abs(l).max(), np.abs(r).max()) <= 4
                and abs(kappa) <= 4 * np.nanmax(np.abs(score)))


def soft_raw(seed, n_ind, n_sites, miss=0.1):
    rng = np.random.RandomState(seed)
    raw = rng.gamma(0.5, size=(n_sites, n_ind, 3)) + 1e-300
    raw[rng.rand(n_sites, n_ind) < miss] = 1.0 / 3.0
    return raw


def test_coefficients_of_the_dyadic_scores():
    """Exact coefficients where they are dyadic: one-hot posteriors then give exact sums (bit-exact vs the int path)."""
    want = {"default": ((-.5, 0), (-.5, 0), .5), "int": ((0, 0), (-1, 0), 0), "seven_half": ((-.5, 3.25), (-3.75, 3.25), 2.125)}
    for name, (l, r, kappa) in want.items():
        V, gl, gr, gk = coefficients(SCORES[name])
        assert tuple(gl) == l and tuple(gr) == r and gk == kappa, name
        assert V[0, 0] * V[1, 1] - V[0, 1] * V[1, 0] == 1.0
    assert all(taken(s) for s in SCORES.values())
    assert not taken(AVG) and not taken(NAN_SCORE) and not taken(NEAR_SINGULAR)


@pytest.mark.parametrize("name", sorted(SCORES))
def test_rewrite_equals_oracle(name):
    """NumPy restatement of the two-plane operands + kappa * cnt against oracle.distances on soft data, 10 % missing."""
    S = SCORES[name]
    n, n_sites = 40, 300
    P = oracle.frontend(soft_raw(3, n, n_sites))
    m = oracle.miss_mask(P).astype(np.float64)                       # [ind][site] presence (1 = data)
    V, l, r, kappa = coefficients(S)
    A = m[..., None] * (P[..., :2] + l)
    B = m[..., None] * ((P[..., :2] + r) @ V.T)
    cnt = m @ m.T
    num = np.einsum("isg,jsg->ij", A, B) + kappa * cnt
    o = oracle.distances(P, score=S, indep=True, pairwise_del=True, evol_model=0)
    iu = np.triu_indices(n, 1)
    assert np.array_equal(cnt[iu].astype(np.uint64), o["cnt"][iu])
    floor = 1e-15 * n_sites * np.abs(S).max()
    assert np.all(np.abs(num[iu] - o["num"][iu]) <= 1e-12 * np.abs(o["num"][iu]) + floor), name


# ------------------------------------------------------------------------------------------------------------ GPU --

N, S = 300, 25_600        # 44 850 pairs x 25 600 sites >= 2^30 pair-sites: the mode applies; 3 row blocks (edge + diagonal tiles)
MIN_PAIR_SITES = 1 << 30


def k4_of(g, n, n_sites):
    """K4 steps per chunk of the last unweighted, unsharded contraction of an n = 300 context (1 full, 2 edge, 3 diagonal
    tiles: 256 + 16 * 6 * 2 + 136 * 3 DMMAs per K4 step)."""
    assert n == 300 and path_of(g) == "fp64"
    step = 256 + 16 * 6 * 2 + 136 * 3
    k4, rem = divmod(g.timing().dist_dmma, -(-n_sites // 8) * step)
    assert rem == 0
    return k4


def mode_k4(score, n_sites, keep_planes=False):
    with nb().NgsDistB200(nb().Params(n_ind=N, n_sites=n_sites, in_probs=True, indep_geno=True, pairwise_del=True,
                                      score=score, keep_planes=keep_planes)) as g:
        g.push_sites(soft_raw(5, N, n_sites))
        g.frontend()
        g.distances()
        return k4_of(g, N, n_sites)


@pytest.mark.gpu
def test_mode_taken():
    """4 K4 steps per chunk exactly where the coefficients qualify and the matrix has at least 2^30 pair-sites; 6 otherwise."""
    for name, sc in list(SCORES.items()) + [("avg", AVG), ("nan", NAN_SCORE), ("near_singular", NEAR_SINGULAR)]:
        assert mode_k4(sc, S) == (4 if taken(sc) else 6), name
    assert mode_k4(DEFAULT, S, keep_planes=True) == 6
    pairs = N * (N - 1) // 2
    below = MIN_PAIR_SITES // pairs // 8 * 8                     # the largest whole-chunk site count under the threshold
    assert pairs * below < MIN_PAIR_SITES <= pairs * (below + 8)
    assert mode_k4(DEFAULT, below) == 6 and mode_k4(DEFAULT, below + 8) == 4


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(SCORES))
def test_values_against_oracle(name):
    """Replicate 0, per-site weights (block 7), the uniform-scale path (block 40), and the block cache built and reused."""
    sc = SCORES[name]
    model = 0 if name == "negative" else 1
    raw = soft_raw(7, N, S)
    pk = dict(n_ind=N, n_sites=S, in_probs=True, indep_geno=True, pairwise_del=True, evol_model=model, score=sc)
    c7, cu, cu2 = boot_counts(1, S // 7), boot_counts(2, S // 40), boot_counts(3, S // 40)
    got = {}
    with nb().NgsDistB200(nb().Params(no_block_cache=True, **pk)) as g:
        g.push_sites(raw)
        g.frontend()
        got["rep0"] = g.distances(want_num=True, want_cnt=True)
        assert k4_of(g, N, S) == 4
        got["weights"] = g.distances(c7, 7, want_num=True, want_cnt=True)
        got["uniform"] = g.distances(cu, 40, want_num=True, want_cnt=True)
    with nb().NgsDistB200(nb().Params(**pk)) as g:
        g.push_sites(raw)
        g.frontend()
        got["cache build"] = g.distances(cu, 40, want_num=True, want_cnt=True)
        assert g.timing().block_cache == 1
        got["cache reuse"] = g.distances(cu2, 40, want_num=True, want_cnt=True)
        assert g.timing().block_cache == 2
    P = oracle.frontend(raw)
    ora = {}
    for label, (c, bs) in {"rep0": (None, 1), "weights": (c7, 7), "uniform": (cu, 40), "cache build": (cu, 40),
                           "cache reuse": (cu2, 40)}.items():
        sm = None if c is None else site_map(c, bs)
        key = None if c is None else (bs, c.tobytes())
        if key not in ora:
            ora[key] = oracle.distances(P, score=sc, indep=True, pairwise_del=True, evol_model=model, site_map=sm)
        check(got[label], ora[key], sc, S if sm is None else len(sm), model, "%s %s" % (name, label))


@pytest.mark.gpu
def test_knife_edge_patch_with_asymmetric_score():
    """The boundary grid (triples the host decides, written back by k_patch) in the corner of soft data: k_patch writes the
    two-plane operands with the asymmetric score in the reference's orientation."""
    grid = load_bin(GRID["input"], GRID["n_ind"], GRID["n_sites"])
    raw = soft_raw(13, N, S)
    raw[:grid.shape[0], :grid.shape[1]] = grid
    p = nb().Params(n_ind=N, n_sites=S, in_probs=True, indep_geno=True, pairwise_del=True, evol_model=0, score=ASYM)
    with nb().NgsDistB200(p) as g:
        g.push_sites(raw)
        g.frontend()
        assert g.deferred_stats() > 50, "the grid sits on the boundaries: the host must have decided triples"
        r = g.distances(want_num=True, want_cnt=True)
        assert k4_of(g, N, S) == 4
    o = oracle.distances(oracle.frontend(raw), score=ASYM, indep=True, pairwise_del=True, evol_model=0)
    check(r, o, ASYM, S, 0, "knife asym")


@pytest.mark.gpu
def test_against_three_planes_at_scale():
    """2000 x 100 000, 16 replicates of distances_batch at block 1000: the same matrices as the three-plane contraction."""
    n, n_sites, bs, R = 2000, 100_000, 1000, 16
    raw = oracle.synth_raw(20261022, 0.1, n, n_sites)
    counts = np.stack([boot_counts(100 + k, n_sites // bs) for k in range(R)])
    res = {}
    for keep in (False, True):
        with nb().NgsDistB200(nb().Params(n_ind=n, n_sites=n_sites, in_probs=True, indep_geno=True, pairwise_del=True,
                                          no_block_cache=True, keep_planes=keep)) as g:
            g.push_sites(raw)
            g.frontend()
            batch = np.array(g.distances_batch(counts, bs))
            one = g.distances(counts[0], bs, want_num=True, want_cnt=True)
            res[keep] = (batch, one, g.timing().dist_dmma)
    (b2, o2, d2), (b3, o3, d3) = res[False], res[True]
    assert 3 * d2 == 2 * d3
    assert np.array_equal(o2["cnt"], o3["cnt"])
    floor = 1e-15 * R * n_sites
    assert np.all(np.abs(o2["num"] - o3["num"]) <= 1e-12 * np.abs(o3["num"]) + 1e-15 * n_sites)
    assert np.isfinite(b2).all() and np.isfinite(b3).all()
    assert np.all(np.abs(b2 - b3) <= 1e-11 * np.abs(b3) + floor / n_sites), np.abs(b2 - b3).max()


@pytest.mark.gpu
def test_non_finite_pattern():
    """Present triples with a non-finite posterior component (text input: not fatal) give the NaN / Inf pattern of the
    three planes, including (0, 0, NaN), whose NaN sits in the plane the two-plane form drops."""
    n, n_sites = N, S
    raw = soft_raw(9, n, n_sites)
    raw[10, 3] = (0.0, 0.0, np.inf)         # -> (0, 0, NaN)
    raw[50, 77] = (np.inf, 1.0, 0.0)        # -> (NaN, 0, 0)
    raw[120, 140] = (np.nan, 0.2, 0.3)
    out = {}
    for keep in (False, True):
        with nb().NgsDistB200(nb().Params(n_ind=n, n_sites=n_sites, in_probs=True, in_text=True, indep_geno=True,
                                          pairwise_del=True, keep_planes=keep)) as g:
            g.push_sites(raw)
            g.frontend()
            out[keep] = g.distances(want_num=True, want_cnt=True)
            assert k4_of(g, n, n_sites) == (6 if keep else 4)
    a, b = out[False], out[True]
    assert np.array_equal(a["cnt"], b["cnt"])
    for k in ("num", "dist"):
        assert np.array_equal(np.isnan(a[k]), np.isnan(b[k])), k
        assert np.array_equal(np.isinf(a[k]), np.isinf(b[k])), k
    assert np.isnan(a["dist"][3, 4]) and np.isnan(a["dist"][77, 0]) and np.isnan(a["dist"][0, 140])
    fin = np.isfinite(b["num"])
    assert np.allclose(a["num"][fin], b["num"][fin], rtol=1e-12, atol=1e-15 * n_sites)
