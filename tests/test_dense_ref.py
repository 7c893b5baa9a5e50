"""The dense float64 reference (tests/dense_ref.py) against the CPU oracle, on CPU torch.  These tests are what make the
reference trustworthy where tests/test_gpu_full_matrix.py uses it at sizes the oracle cannot reach."""
import numpy as np
import pytest
import torch

import oracle
from dense_ref import DenseRef, boot_counts

MODES = {
    "indep": dict(pairwise_del=False),
    "indep_pdel": dict(pairwise_del=True),
    "call": dict(call_geno=True, pairwise_del=False),
    "call_pdel": dict(call_geno=True, pairwise_del=True),
    "call_thresh": dict(call_geno=True, N_thresh=0.35, call_thresh=0.9, pairwise_del=False),
    "call_thresh_pdel": dict(call_geno=True, N_thresh=0.35, call_thresh=0.9, pairwise_del=True),
}


def reference(raw, mode, avg_nuc_dist, block_size, n_rep, seed, chunk):
    n_sites, n_ind, _ = raw.shape
    kw = MODES[mode]
    counts = boot_counts(seed, n_sites, block_size, n_rep) if n_rep else None
    ref = DenseRef(n_ind, n_sites, score=oracle.score_matrix(avg_nuc_dist), block_size=block_size, counts=counts, **kw)
    t = torch.from_numpy(raw)
    for s0 in range(0, n_sites, chunk):
        ref.add(t[s0:s0 + chunk], s0)
    return ref


def oracle_job(raw, mode, avg_nuc_dist, block_size, n_rep, seed, **kw):
    return oracle.run_job(raw, indep=True, avg_nuc_dist=avg_nuc_dist, n_boot_rep=n_rep, boot_block_size=block_size, seed=seed,
                          **MODES[mode], **kw)


def assert_rel(got, want, tol, what):
    got = np.asarray(got)
    nan = np.isnan(want)
    assert np.array_equal(np.isnan(got), nan), what + ": NaN positions differ"
    err = np.abs(got[~nan] - want[~nan])
    bad = err > tol * np.abs(want[~nan])
    assert not bad.any(), "%s: %d entries off, worst %.3e" % (what, bad.sum(), (err / np.maximum(np.abs(want[~nan]), 1e-300)).max())


def check(ref, ora, mode, **finish_kw):
    exact_num = mode == "call_pdel"
    for r, o in enumerate(ora):
        got = {k: v.numpy() for k, v in ref.finish(r, **finish_kw).items()}
        assert np.array_equal(got["cnt"].astype(np.uint64), o["cnt"]), "cnt rep %d" % r
        assert np.array_equal(got["cnt"], np.round(got["cnt"])), "cnt rep %d not integral" % r
        if exact_num:
            assert np.array_equal(got["num"], o["num"]), "num rep %d not bit-exact" % r
        assert_rel(got["num"], o["num"], 1e-12, "num rep %d" % r)
        assert_rel(got["dist"], o["dist"], 1e-12, "dist rep %d %s" % (r, finish_kw))


@pytest.mark.parametrize("n_ind", [2, 3, 41])
@pytest.mark.parametrize("miss", [0.0, 0.1, 0.3])
@pytest.mark.parametrize("avg_nuc_dist", [False, True])
@pytest.mark.parametrize("mode", sorted(MODES))
def test_modes_models_and_missing_rates(mode, avg_nuc_dist, miss, n_ind):
    """Every mode, score, missing rate and size; replicate 0 and two bootstrap replicates of 7-site blocks over a site
    count 7 does not divide; models 0, 1 and 2, and tot_sites."""
    n_sites, bs, n_rep, seed = 213, 7, 2, 777
    raw = oracle.synth_raw(1000 + n_ind, miss, n_ind, n_sites)
    ref = reference(raw, mode, avg_nuc_dist, bs, n_rep, seed, chunk=64)
    for model in (0, 1, 2):
        check(ref, oracle_job(raw, mode, avg_nuc_dist, bs, n_rep, seed, evol_model=model), mode, evol_model=model)
    check(ref, oracle_job(raw, mode, avg_nuc_dist, bs, n_rep, seed, evol_model=1, tot_sites=500), mode, evol_model=1, tot_sites=500)


@pytest.mark.parametrize("n_sites", [200, 209])
@pytest.mark.parametrize("block_size", [1, 7, 50])
@pytest.mark.parametrize("mode", ["indep_pdel", "call_pdel", "indep"])
def test_bootstrap_block_sizes(mode, block_size, n_sites):
    """Block sizes 1, 7 and 50, with site counts they divide and do not divide (the persistent n_sites % block_size
    truncation), chunks that cut blocks in two, and four replicates."""
    n_ind, n_rep, seed = 23, 4, 4242
    raw = oracle.synth_raw(31, 0.1, n_ind, n_sites)
    ref = reference(raw, mode, False, block_size, n_rep, seed, chunk=37)
    check(ref, oracle_job(raw, mode, False, block_size, n_rep, seed, evol_model=2), mode, evol_model=2)


def test_boot_counts_are_the_oracle_site_maps():
    """The multiplicities are the bincount of rnd_map_data's source blocks, replicate after replicate of one stream."""
    rng = oracle.Taus(99)
    c = boot_counts(99, 1003, 10, 3)
    assert c.shape == (3, 100) and (c.sum(axis=1) == 100).all()
    for r in range(3):
        sm = rng.boot_map(100, 10)
        assert np.array_equal(np.bincount(sm.astype(np.int64) // 10, minlength=100), c[r] * 10)


def test_orientation_follows_the_oracle():
    """An asymmetric score: entry (i, j), i < j, has the lower-index individual take g1."""
    n_ind, n_sites = 9, 150
    raw = oracle.synth_raw(5, 0.1, n_ind, n_sites)
    score = np.array([0.0, 0.3, 1.7, 0.2, 0.0, 0.9, 1.1, 0.4, 0.0])
    ref = DenseRef(n_ind, n_sites, score=score, pairwise_del=True)
    ref.add(torch.from_numpy(raw), 0)
    o = oracle.run_job(raw, indep=True, pairwise_del=True, evol_model=0, score=score)[0]
    got = ref.finish(0, evol_model=0)
    assert_rel(got["num"].numpy(), o["num"], 1e-12, "num")
    iu = np.triu_indices(n_ind, 1)
    flipped = oracle.run_job(raw, indep=True, pairwise_del=True, evol_model=0, score=score.reshape(3, 3).T.ravel())[0]
    assert not np.allclose(got["num"].numpy()[iu], flipped["num"][iu], rtol=1e-9, atol=0)
