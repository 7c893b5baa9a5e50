"""Score matrices other than the two the command line can select, through every contraction that reads ngsd_cfg.score.

The default score and --avg_nuc_dist are both symmetric, so a transposed score in the front end or the knife-edge patch,
a swapped pair of terms in the fold of the per pair-site EM (dist_em.cu), row and column sums swapped in the integer
path's table (ngsd_int_lut), or a row/column role swapped in a diagonal, edge, shard or cached tile would all go
unnoticed with them.  Here the score is asymmetric (and non-integral, negative or integral), and the reference's
orientation is the one checked: score[g1][g2], g1 the genotype of the lower-index individual (ngsDist.cpp:351-353).

The integer path is taken only for an exactly integral S * score; anything else, however close, must take the FP64
planes and give the reference's sums."""
import functools

import numpy as np
import pytest

import oracle
from ngsdist_b200 import multi
from test_gpu_parity import RTOL, nb
from util import load_bin, manifest

pytestmark = pytest.mark.gpu

DEFAULT = [0, .5, 1, .5, 0, .5, 1, .5, 0]
AVG = [0, .5, 1, .5, .5, .5, 1, .5, 0]
# D1 != D3, D2 != D6, D5 != D7 and every term of the EM fold (dist_em.cu K[0..8]) non-zero
ASYM = [.1, .7, 1.3, .2, .05, .9, 1.1, .4, .3]
NEG = [.3, -.6, 1.0, .5, .1, .8, 1.4, .2, -.25]
INT = [0, 1, 2, 0, 0, 1, 0, 0, 0]                      # S * score is integral for S = 2 and S = 18
SCORES = {"asym": ASYM, "negative": NEG}


def transposed(score):
    return list(np.asarray(score, dtype=np.float64).reshape(3, 3).T.ravel())


def path_of(g):
    """Which contraction the last ngsd_distances ran: int8 tensor cores, FP64 GEMM, or (neither counter) the EM kernel."""
    t = g.timing()
    return "int" if t.dist_imma > 0 else "fp64" if t.dist_dmma > 0 else "em"


def site_map(counts, bs):
    return np.concatenate([np.arange(b * bs, (b + 1) * bs) for b in range(len(counts)) for _ in range(int(counts[b]))])


def boot_counts(seed, n_blocks):
    rng = np.random.default_rng(seed)
    return np.bincount(rng.integers(0, n_blocks, n_blocks), minlength=n_blocks).astype(np.uint32)


def close(got, want, floor, what):
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    assert got.shape == want.shape
    both_nan = np.isnan(got) & np.isnan(want)
    both_inf = np.isinf(got) & np.isinf(want) & (np.sign(got) == np.sign(want))
    with np.errstate(invalid="ignore"):
        ok = both_nan | both_inf | (np.abs(got - want) <= RTOL * np.abs(want) + floor)
    if not ok.all():
        with np.errstate(invalid="ignore", divide="ignore"):
            rel = np.abs(got - want)[~ok] / np.abs(want[~ok])
        idx = np.argwhere(~ok)[:3].tolist()
        raise AssertionError("%s: %d mismatches, worst rel %.3e, first at %s: got %r want %r" % (
            what, (~ok).sum(), np.nanmax(rel) if rel.size else np.nan, idx, got[~ok][:3].tolist(), want[~ok][:3].tolist()))


def check(r, o, score, n_sites, model, what, exact=False):
    """cnt bit-exact; num and dist within 1e-9 relative plus test_gpu_edges' absolute floor of 1e-15 per site, scaled by
    the largest |score| entry (a site term is at most that), by 1 / cnt and by the condition number of the model for dist.
    exact: num and dist bit for bit."""
    assert np.array_equal(r["cnt"], o["cnt"]), "%s: %d counts differ" % (what, (r["cnt"] != o["cnt"]).sum())
    if exact:
        assert np.array_equal(r["num"], o["num"]), "%s: num must be bit-exact (%d differ)" % (what, (r["num"] != o["num"]).sum())
        assert np.array_equal(r["dist"], o["dist"], equal_nan=True), "%s: dist must be bit-exact" % what
        return
    floor = 1e-15 * max(n_sites, 1) * np.nanmax(np.abs(score))
    close(r["num"], o["num"], floor, what + " num")
    with np.errstate(divide="ignore", invalid="ignore"):
        c = np.maximum(o["cnt"].astype(np.float64), 1.0)
        x = o["num"] / c
        cond = 1.0 if model == 0 else 1.0 / np.maximum(np.abs(1.0 - (x if model == 1 else 4.0 * x / 3.0)), 1e-300)
    close(r["dist"], o["dist"], floor / c * cond, what + " dist")


def with_zero_triples(raw, seed, whole_site=True):
    """All-zero binary triples (exp(-1.125) x 3 after the reader, sum 0.974) at 2 % of the individual-sites, and a whole
    site of them: the two-plane contraction assumes a sum of one and corrects these rows afterwards (k_deficit_fix)."""
    raw = raw.copy()
    rng = np.random.RandomState(seed)
    n_sites, n_ind, _ = raw.shape
    for _ in range(max(1, n_sites * n_ind // 50)):
        raw[rng.randint(n_sites), rng.randint(n_ind)] = 0.0
    if whole_site:
        raw[n_sites // 3, :] = 0.0
    return raw


# ------------------------------------------------------------------------------------------------------ FP64 GEMM --

FP64_MODES = {
    "two_plane": dict(indep_geno=True),
    "three_plane": dict(indep_geno=True, keep_planes=True),
    "pdel": dict(indep_geno=True, pairwise_del=True),
}


@pytest.mark.parametrize("mode", sorted(FP64_MODES))
@pytest.mark.parametrize("name", sorted(SCORES))
def test_fp64_gemm_against_oracle(name, mode):
    """300 individuals: two full row blocks and a last one of 44 (edge tiles), a diagonal tile per row block.  Replicate 0,
    per-site weights (block 7), whole-chunk blocks on the uniform-scale path, then the block cache built and reused."""
    S = SCORES[name]
    n, n_sites = 300, 600
    model = 0 if name == "negative" else 1
    bs_u = 48 if mode == "two_plane" else 40               # whole 12- or 8-site chunks of the contraction
    raw = with_zero_triples(oracle.synth_raw(71, 0.1, n, n_sites), 5)
    pk = dict(n_ind=n, n_sites=n_sites, in_probs=True, evol_model=model, score=S, **FP64_MODES[mode])
    c7, cu, cu2 = boot_counts(1, n_sites // 7), boot_counts(2, n_sites // bs_u), boot_counts(3, n_sites // bs_u)
    got = {}
    with nb().NgsDistB200(nb().Params(no_block_cache=True, **pk)) as g:
        g.push_sites(raw)
        g.frontend()
        got["rep0"] = g.distances(want_num=True, want_cnt=True)
        assert path_of(g) == "fp64"
        got["weights"] = g.distances(c7, 7, want_num=True, want_cnt=True)
        got["uniform"] = g.distances(cu, bs_u, want_num=True, want_cnt=True)
        assert path_of(g) == "fp64" and g.timing().block_cache == 0
        if mode == "pdel":
            acc = {"num": 0.0, "cnt": 0}
            covered = np.zeros((n, n), dtype=int)
            for rank in range(3):
                g.set_tile_shard(rank, 3)
                r = g.distances(want_num=True, want_cnt=True)
                own = multi.tile_owner_mask(n, rank, 3)
                assert not r["num"][~own].any() and not r["cnt"][~own].any(), "entries outside the shard of rank %d" % rank
                acc = {k: acc[k] + r[k] for k in acc}
                covered += own
            g.set_tile_shard(0, 1)
            assert (covered[~np.eye(n, dtype=bool)] == 1).all()
            assert np.array_equal(acc["cnt"], got["rep0"]["cnt"])
            assert np.allclose(acc["num"], got["rep0"]["num"], rtol=1e-12, atol=0)   # K splits are planned per shard
    with nb().NgsDistB200(nb().Params(**pk)) as g:
        g.push_sites(raw)
        g.frontend()
        got["cache build"] = g.distances(cu, bs_u, want_num=True, want_cnt=True)
        assert g.timing().block_cache == 1
        got["cache reuse"] = g.distances(cu2, bs_u, want_num=True, want_cnt=True)
        assert g.timing().block_cache == 2
    P = oracle.frontend(raw)
    draws = {"rep0": (None, 1), "weights": (c7, 7), "uniform": (cu, bs_u), "cache build": (cu, bs_u), "cache reuse": (cu2, bs_u)}
    ora = {}
    for label, (c, bs) in draws.items():
        sm = None if c is None else site_map(c, bs)
        key = None if c is None else (bs, c.tobytes())
        if key not in ora:
            ora[key] = oracle.distances(P, score=S, indep=True, pairwise_del=mode == "pdel", evol_model=model, site_map=sm)
        check(got[label], ora[key], S, n_sites if sm is None else len(sm), model, "%s %s %s" % (name, mode, label))


# ------------------------------------------------------------------------------------------------ per pair-site EM --

def dirichlet_raw(seed, n_ind, n_sites, alpha=0.5, miss=0.1):
    rng = np.random.RandomState(seed)
    raw = rng.gamma(alpha, size=(n_sites, n_ind, 3)) + 1e-300
    raw[rng.rand(n_sites, n_ind) < miss] = 1.0 / 3.0
    return raw


@pytest.mark.parametrize("pdel", [False, True])
@pytest.mark.parametrize("name", sorted(SCORES))
def test_em_against_oracle(name, pdel):
    """Soft (Dirichlet 0.5) posteriors through k_dist_em3: replicate 0, bootstrap replicates direct and from the block
    cache, and 3-rank tile shards of replicate 0."""
    S = SCORES[name]
    n, n_sites, bs = 270, 192, 16
    model = 0 if name == "negative" else 1
    raw = dirichlet_raw(11 + pdel, n, n_sites)
    reps = [boot_counts(5 + k, n_sites // bs) for k in range(2)]
    pk = dict(n_ind=n, n_sites=n_sites, in_probs=True, indep_geno=False, pairwise_del=pdel, evol_model=model, score=S)
    with nb().NgsDistB200(nb().Params(no_block_cache=True, **pk)) as g:
        g.push_sites(raw)
        g.frontend()
        r0 = g.distances(want_num=True, want_cnt=True)
        assert path_of(g) == "em"
        direct = [g.distances(c, bs, want_num=True, want_cnt=True) for c in reps]
        acc = {"num": 0.0, "cnt": 0}
        for rank in range(3):
            g.set_tile_shard(rank, 3)
            r = g.distances(want_num=True, want_cnt=True)
            own = multi.tile_owner_mask(n, rank, 3)
            assert not r["num"][~own].any() and not r["cnt"][~own].any()
            acc = {k: acc[k] + r[k] for k in acc}
        g.set_tile_shard(0, 1)
    assert np.array_equal(acc["cnt"], r0["cnt"])
    assert np.allclose(acc["num"], r0["num"], rtol=1e-12, atol=0)
    with nb().NgsDistB200(nb().Params(**pk)) as g:
        g.push_sites(raw)
        g.frontend()
        cached = []
        for k, c in enumerate(reps):
            cached.append(g.distances(c, bs, want_num=True, want_cnt=True))
            assert g.timing().block_cache == 1 + k
    P = oracle.frontend(raw)
    check(r0, oracle.distances(P, score=S, indep=False, pairwise_del=pdel, evol_model=model), S, n_sites, model, "%s em rep0" % name)
    for k, c in enumerate(reps):
        sm = site_map(c, bs)
        o = oracle.distances(P, score=S, indep=False, pairwise_del=pdel, evol_model=model, site_map=sm)
        check(direct[k], o, S, len(sm), model, "%s em rep %d direct" % (name, k + 1))
        check(cached[k], o, S, len(sm), model, "%s em rep %d cached" % (name, k + 1))


# ------------------------------------------------------------------------------------------------ called genotypes --

NEAR_HALF = [0, .5 + 3e-11, 1, .5, 0, .5, 1, .5, 0]
TINY = [1e-12 * v for v in DEFAULT]
SEVEN_HALF = [0, .5, 7.5, .5, 0, .5, 1, .5, 0]       # S * 7.5 = 15 with --pairwise_del, 135 > 127 without
NAN_SCORE = [0, float("nan"), 1, .5, 0, .5, 1, .5, 0]   # every sum that reads it is NaN, as in the reference

# (score name, score, pairwise_del) -> the contraction ngsd_int_lut must choose for hard calls
CALLED_PATHS = [
    ("default", DEFAULT, False, "int"), ("default", DEFAULT, True, "int"),
    ("avg_nuc_dist", AVG, False, "int"), ("avg_nuc_dist", AVG, True, "int"),
    ("integral", INT, False, "int"), ("integral", INT, True, "int"),
    ("seven_half", SEVEN_HALF, False, "fp64"), ("seven_half", SEVEN_HALF, True, "int"),
    ("asym", ASYM, False, "fp64"), ("asym", ASYM, True, "fp64"),
    ("negative", NEG, False, "fp64"), ("negative", NEG, True, "fp64"),
    ("near_half", NEAR_HALF, False, "fp64"), ("near_half", NEAR_HALF, True, "fp64"),
    ("tiny", TINY, False, "fp64"), ("tiny", TINY, True, "fp64"),
    ("nan", NAN_SCORE, False, "fp64"), ("nan", NAN_SCORE, True, "fp64"),
]
N_CALLED, SITES_CALLED, BS_CALLED = 130, 640, 37


@functools.lru_cache(maxsize=None)
def called_inputs():
    raw = oracle.synth_raw(97, 0.1, N_CALLED, SITES_CALLED)
    geno = np.random.RandomState(98).randint(-1, 3, size=(SITES_CALLED, N_CALLED)).astype(np.int8)
    return raw, geno


@functools.lru_cache(maxsize=None)
def called_oracle(from_likelihoods, score, pdel):
    raw, geno = called_inputs()
    P = oracle.frontend(raw, call_geno=True) if from_likelihoods else oracle.frontend_geno(geno)
    rng = oracle.Taus(9)
    maps = [None, rng.boot_map(SITES_CALLED // BS_CALLED, BS_CALLED)]
    return [oracle.distances(P, score=np.array(score), indep=True, pairwise_del=pdel, evol_model=0, site_map=sm) for sm in maps]


def run_called(feed, score, pdel, force_fp64=False):
    raw, geno = called_inputs()
    p = nb().Params(n_ind=N_CALLED, n_sites=SITES_CALLED, in_probs=feed == "call_geno", call_geno=feed == "call_geno",
                    pairwise_del=pdel, evol_model=0, score=list(score), n_boot_rep=1, boot_block_size=BS_CALLED, seed=9,
                    force_fp64=force_fp64)
    with nb().NgsDistB200(p) as g:
        if feed == "call_geno":
            g.push_sites(raw)
        elif feed == "genotypes":
            g.push_genotypes(geno)
        else:
            g.push_packed_genotypes(nb().pack_genotypes(geno))
        g.frontend()
        res = [g.distances(want_num=True, want_cnt=True)]
        path = path_of(g)
        c, bs = g.next_boot_counts()
        res.append(g.distances(c, bs, want_num=True, want_cnt=True))
    return path, res


@pytest.mark.parametrize("feed", ["call_geno", "genotypes", "packed"])
@pytest.mark.parametrize("name,score,pdel,want", [pytest.param(*c, id="%s-%s" % (c[0], "pdel" if c[2] else "nopdel")) for c in CALLED_PATHS])
def test_called_genotypes_path_and_values(name, score, pdel, want, feed):
    """Hard calls from likelihoods (--call_geno), genotype codes and 2-bit packed codes: the path the score selects, and
    the reference's sums on it.  Integer path with --pairwise_del: num and model-0 distances bit-exact against the oracle
    and against the same data forced through the FP64 contraction; every other case within 1e-9."""
    path, res = run_called(feed, tuple(score), pdel)
    ora = called_oracle(feed == "call_geno", tuple(score), pdel)       # codes and packed codes are the same input
    exact = want == "int" and pdel
    for rep, (r, o) in enumerate(zip(res, ora)):
        check(r, o, score, SITES_CALLED, 0, "%s pdel=%d %s rep %d" % (name, pdel, feed, rep), exact=exact)
    assert path == want, "score %s, pairwise_del %d: %s path taken, %s expected" % (name, pdel, path, want)
    if want == "int":
        path64, res64 = run_called(feed, tuple(score), pdel, force_fp64=True)
        assert path64 == "fp64"
        for rep, (r, r64) in enumerate(zip(res, res64)):
            check(r, r64, score, SITES_CALLED, 0, "%s pdel=%d %s rep %d int vs fp64" % (name, pdel, feed, rep), exact=exact)


# ------------------------------------------------------------------------------------------------ single-site terms --

PATHS = {   # name -> (score, params, expected path)
    "two_plane": (ASYM, dict(indep_geno=True), "fp64"),
    "three_plane": (ASYM, dict(indep_geno=True, keep_planes=True), "fp64"),
    "pdel": (ASYM, dict(indep_geno=True, pairwise_del=True), "fp64"),
    "em": (ASYM, dict(indep_geno=False), "em"),
    "em_pdel": (ASYM, dict(indep_geno=False, pairwise_del=True), "em"),
    "called": (INT, dict(call_geno=True), "int"),
    "called_pdel": (INT, dict(call_geno=True, pairwise_del=True), "int"),
}


def oracle_kw(pk):
    return dict(indep=pk.get("indep_geno", False) or pk.get("call_geno", False), pairwise_del=pk.get("pairwise_del", False))


@pytest.mark.parametrize("n_sites", [1, 3])
@pytest.mark.parametrize("path", sorted(PATHS))
def test_single_site_terms(path, n_sites):
    """num(i, j) is one or three site terms, so a transposed score is not diluted by a long sum; the asymmetric score on
    the FP64 planes and the EM, the integral one on the integer path."""
    S, pk, want = PATHS[path]
    n = 200
    raw = oracle.synth_raw(300 + n_sites, 0.1, n, n_sites)
    if "call_geno" not in pk:
        raw = with_zero_triples(raw, n_sites, whole_site=False)
    with nb().NgsDistB200(nb().Params(n_ind=n, n_sites=n_sites, in_probs=True, evol_model=0, score=S, **pk)) as g:
        g.push_sites(raw)
        g.frontend()
        r = g.distances(want_num=True, want_cnt=True)
        assert path_of(g) == want
    P = oracle.frontend(raw, call_geno=pk.get("call_geno", False))
    o = oracle.distances(P, score=S, evol_model=0, **oracle_kw(pk))
    check(r, o, S, n_sites, 0, "%s %d sites" % (path, n_sites), exact=path == "called_pdel")


# ------------------------------------------------------------------------------- transposed score, reversed order --

def synth_run(n_ind, n_sites, score, reverse, **pk):
    """Device-generated input (as test_gpu_configs.gpu_ctx_synth), individuals in reverse order when `reverse`."""
    import torch
    p = nb().Params(n_ind=n_ind, n_sites=n_sites, in_probs=True, evol_model=0, score=score, **pk)
    with nb().NgsDistB200(p) as g:
        buf = torch.empty((n_sites, n_ind, 3), dtype=torch.float64, device="cuda")
        g.synth_raw_device(buf.data_ptr(), 20251021, 0.1, 0, n_sites)      # synchronises the context's stream
        if reverse:
            buf = torch.flip(buf, dims=[1]).contiguous()
        torch.cuda.synchronize()
        g.push_sites_device(buf.data_ptr(), 0, n_sites)
        g.frontend()
        r = g.distances(want_num=True, want_cnt=True)
        path = path_of(g)
        del buf
    return path, r


@pytest.mark.parametrize("path", sorted(PATHS))
def test_transposed_score_on_reversed_individuals(path):
    """num(i, j) with score S equals num(n-1-j, n-1-i) with S^T on the individuals in reverse order: g1 is always the
    lower-index individual.  No oracle needed, so at C2 scale (500 x 20 000); reversal also moves which individuals sit
    in the edge tiles.  1e-12 relative (summation order differs), exact on the integer path."""
    S, pk, want = PATHS[path]
    n, n_sites = 500, 20000
    pa, a = synth_run(n, n_sites, S, False, **pk)
    pb, b = synth_run(n, n_sites, transposed(S), True, **pk)
    assert pa == pb == want
    num_b, cnt_b = b["num"][::-1, ::-1], b["cnt"][::-1, ::-1]
    assert np.array_equal(a["cnt"], cnt_b)
    if want == "int":
        assert np.array_equal(a["num"], num_b)
    else:
        bad = np.abs(a["num"] - num_b) > 1e-12 * np.abs(a["num"])
        assert not bad.any(), "%d entries differ, worst rel %.3e" % (bad.sum(), (np.abs(a["num"] - num_b)[bad] / np.abs(a["num"][bad])).max())
    # and the asymmetric score really is asymmetric on this data: S^T on the same order gives other sums
    if want != "int" or path == "called":
        pc, c = synth_run(n, n_sites, transposed(S), False, **pk)
        assert not np.allclose(a["num"], c["num"], rtol=1e-6, atol=0)


# -------------------------------------------------------------------------------------------- knife-edge patch --

GRID = [c for c in manifest()["binary"] if c["input"] == "grid12x96.bin"][0]


@pytest.mark.parametrize("in_text", [False, True])
@pytest.mark.parametrize("mode", ["two_plane", "indep_pdel", "em_pdel"])
def test_knife_edge_patch_with_asymmetric_score(mode, in_text):
    """Triples on the reference's comparison boundaries are decided by the host and written back by k_patch, which
    recomputes B = score . p for them: the asymmetric score must be applied there in the same orientation."""
    raw = load_bin(GRID["input"], GRID["n_ind"], GRID["n_sites"])
    n_sites, n_ind, _ = raw.shape
    pdel = mode != "two_plane"
    indep = mode != "em_pdel"
    p = nb().Params(n_ind=n_ind, n_sites=n_sites, in_probs=True, in_text=in_text, indep_geno=indep, pairwise_del=pdel,
                    evol_model=0, score=ASYM, n_boot_rep=2, boot_block_size=8, seed=12345)
    with nb().NgsDistB200(p) as g:
        g.push_sites(raw)
        res = g.run(want_num=True, want_cnt=True)
        n_host = g.deferred_stats()
    assert n_host > 50, "the grid sits on the boundaries: the host must have decided triples (%d)" % n_host
    ora = oracle.run_job(raw, kind=1 if in_text else 0, indep=indep, pairwise_del=pdel, evol_model=0, n_boot_rep=2,
                         boot_block_size=8, seed=12345, score=ASYM)
    for rep, (r, o) in enumerate(zip(res, ora)):
        check(r, o, ASYM, n_sites, 0, "%s text=%d rep %d" % (mode, in_text, rep))


# ------------------------------------------------------------------------------------------------ two or more GPUs --

def _n_gpus():
    import torch
    return torch.cuda.device_count()


@pytest.mark.parametrize("mode", ["em", "two_plane"])
def test_group_context_matches_one_gpu(mode):
    if _n_gpus() < 2:
        pytest.skip("needs 2 GPUs")
    n, n_sites, bs = 300, 960, 48
    raw = oracle.synth_raw(61, 0.1, n, n_sites)
    reps = np.stack([boot_counts(20 + k, n_sites // bs) for k in range(3)])
    res = []
    for n_gpus in (1, 2):
        p = nb().Params(n_ind=n, n_sites=n_sites, in_probs=True, indep_geno=mode != "em", evol_model=0, score=ASYM)
        with nb().NgsDistB200(p, n_gpus=n_gpus, shard=nb().SHARD_REPLICATED) as g:
            g.push_sites(raw)
            g.frontend()
            res.append((g.distances(want_num=True, want_cnt=True), g.distances_batch(reps, bs)))
    (one, one_b), (two, two_b) = res
    assert np.array_equal(two["cnt"], one["cnt"])
    assert np.allclose(two["num"], one["num"], rtol=1e-12, atol=0)
    assert np.allclose(two["dist"], one["dist"], rtol=1e-12, atol=0)
    assert np.allclose(two_b, one_b, rtol=1e-12, atol=0)
