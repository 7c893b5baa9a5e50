"""Called-genotype integer path (K2c dist_umma.cu, int8 tensor cores on 2-bit codes) through the C ABI.

Everything is integer until num = acc / S, so against the oracle: cnt bit-exact everywhere; num and model-0 distances
bit-exact with --pairwise_del or without missing data; 1e-9 otherwise (the reference's own sequential FP sum of the
uniform-triple terms is what differs).  The same data forced through the FP64 contraction (ngsd_cfg.reserved bit 1)
must agree too -- the A/B check that both contractions implement the same gen_dist (ngsDist.cpp:325-404).
"""
import numpy as np
import pytest

import oracle
from test_gpu_parity import assert_close, nb

pytestmark = pytest.mark.gpu


def run(raw, genotypes=None, **pk):
    n_sites, n_ind = raw.shape[:2] if genotypes is None else genotypes.shape
    p = nb().Params(n_ind=n_ind, n_sites=n_sites, **pk)
    with nb().NgsDistB200(p) as g:
        if genotypes is None:
            g.push_sites(raw)
        else:
            g.push_genotypes(genotypes)
        return g.run(want_num=True, want_cnt=True)


@pytest.mark.parametrize("pdel", [True, False])
@pytest.mark.parametrize("avg", [False, True])
@pytest.mark.parametrize("miss", [0.0, 0.15])
def test_called_vs_oracle_and_fp64_path(pdel, avg, miss):
    """--call_geno (default thresholds), bootstrap blocks that straddle the 64-site words (block 37), both score matrices."""
    n_ind, n_sites = 203, 3001
    raw = oracle.synth_raw(77, miss, n_ind, n_sites)
    kw = dict(call_geno=True, pairwise_del=pdel, avg_nuc_dist=avg, evol_model=0, n_boot_rep=2, boot_block_size=37, seed=9)
    res = run(raw, in_probs=True, **kw)
    res64 = run(raw, in_probs=True, force_fp64=True, **kw)
    ora = oracle.run_job(raw, indep=True, call_geno=True, pairwise_del=pdel, avg_nuc_dist=avg, evol_model=0, n_boot_rep=2,
                         boot_block_size=37, seed=9)
    assert len(res) == len(ora) == 3
    exact = pdel or miss == 0.0
    for rep, (r, r64, o) in enumerate(zip(res, res64, ora)):
        assert np.array_equal(r["cnt"], o["cnt"]), "cnt rep %d" % rep
        assert np.array_equal(r["cnt"], r64["cnt"])
        if exact:
            assert np.array_equal(r["num"], o["num"]), "num must be bit-exact (rep %d)" % rep
            assert np.array_equal(r["dist"], o["dist"], equal_nan=True), "model-0 distances must be bit-exact (rep %d)" % rep
            assert np.array_equal(r["num"], r64["num"])
        else:
            assert_close(r["num"], o["num"], "num rep %d" % rep)
            assert_close(r["dist"], o["dist"], "dist rep %d" % rep)
            assert_close(r["num"], r64["num"], "int vs fp64 rep %d" % rep)
        assert np.array_equal(r["dist"], r["dist"].T) and (np.diag(r["dist"]) == 0).all()


def test_genotype_input_many_tiles_jc69():
    """Genotype codes {-1,0,1,2} (read_data.cpp:88-95) on 700 individuals (21 tiles), JC69, vs oracle blocks."""
    rng = np.random.RandomState(5)
    n_ind, n_sites = 700, 2500
    geno = rng.randint(-1, 3, size=(n_sites, n_ind)).astype(np.int8)
    P = oracle.frontend_geno(geno)
    for pdel in (False, True):
        r = run(None, genotypes=geno, in_probs=False, indep_geno=True, pairwise_del=pdel, evol_model=2)[0]
        for (r0, c0) in [(0, 0), (64, 600), (636, 636)]:
            o = oracle.distances_block(P, r0, r0 + 64, c0, c0 + 64, indep=True, pairwise_del=pdel, evol_model=2)
            sub = np.triu(np.ones((64, 64), bool), 1) if r0 == c0 else np.ones((64, 64), bool)
            assert np.array_equal(r["cnt"][r0:r0 + 64, c0:c0 + 64][sub], o["cnt"][sub])
            assert_close(r["num"][r0:r0 + 64, c0:c0 + 64][sub], o["num"][sub], "num pdel=%d" % pdel)
            assert_close(r["dist"][r0:r0 + 64, c0:c0 + 64][sub], o["dist"][sub], "dist pdel=%d" % pdel)


@pytest.mark.parametrize("pdel", [True, False])
def test_large_multiplicities_use_weight_layers(pdel):
    """Block multiplicities above one int8 operand byte (127; 42 without --pairwise_del, where the byte carries 3 w) are
    split into layers; linearity in the weights is exact."""
    n_ind, n_sites, bs = 130, 1280, 128
    raw = oracle.synth_raw(3, 0.1, n_ind, n_sites)
    p = nb().Params(n_ind=n_ind, n_sites=n_sites, in_probs=True, call_geno=True, pairwise_del=pdel, evol_model=0,
                    no_block_cache=True)     # the direct weighted contraction is what splits weights into layers
    with nb().NgsDistB200(p) as g:
        g.push_sites(raw)
        nbk = n_sites // bs
        c_big = np.array([300, 0, 1, 127, 128, 42, 43, 0, 85, 254], dtype=np.uint32)
        unit = [np.eye(nbk, dtype=np.uint32)[b] for b in range(nbk)]
        big = g.distances(c_big, bs, want_num=True, want_cnt=True)
        num = np.zeros((n_ind, n_ind))
        cnt = np.zeros((n_ind, n_ind), dtype=np.uint64)
        for b in range(nbk):
            if c_big[b]:
                r = g.distances(unit[b], bs, want_num=True, want_cnt=True)
                num += float(c_big[b]) * np.rint(r["num"] * 18)
                cnt += np.uint64(c_big[b]) * r["cnt"]
    if pdel:
        assert np.array_equal(big["cnt"], cnt)
    else:                                         # without --pairwise_del every pair counts every site of the replicate
        off = ~np.eye(n_ind, dtype=bool)
        assert np.all(big["cnt"][off] == n_sites)
    assert np.array_equal(np.rint(big["num"] * 18), num)        # num is a multiple of 1/18 (1/2 with pairwise_del) far below 2^53


def test_soft_thresholds_fall_back_to_fp64_planes():
    """N_thresh < call_thresh leaves soft triples (gen_func.cpp:908): that data must not take the integer path."""
    n_ind, n_sites = 60, 700
    raw = oracle.synth_raw(21, 0.1, n_ind, n_sites)
    kw = dict(call_geno=True, N_thresh=0.4, call_thresh=0.8, evol_model=0)
    r = run(raw, in_probs=True, **kw)[0]
    o = oracle.run_job(raw, indep=True, **kw)[0]
    assert np.array_equal(r["cnt"], o["cnt"])
    assert_close(r["num"], o["num"])
    # equal thresholds: every triple is called or missing -> integer path, still the reference's answer
    kw = dict(call_geno=True, N_thresh=0.6, call_thresh=0.6, pairwise_del=True, evol_model=0)
    r = run(raw, in_probs=True, **kw)[0]
    o = oracle.run_job(raw, indep=True, **kw)[0]
    assert np.array_equal(r["cnt"], o["cnt"]) and np.array_equal(r["num"], o["num"])


def test_call_decisions_at_the_fast_test_boundaries():
    """The code kernel decides calls on the doubles' high words when the maximum is clear, on an FP64 test when it is
    close, and with the reference's log-space sequence (gen_func.cpp:886-914) at near-ties: triples sitting on every one of
    those boundaries must still come out as the reference calls them."""
    def bump(x, k):              # k units in the high 32-bit word (k * 2^32 ulps)
        return (np.array([x], dtype=np.float64).view(np.uint64) + np.uint64(k << 32)).view(np.float64)[0]
    base = [0.2, 0.3, 0.45, 1e-300, 3e-310, 1e300, 1.0]
    triples = []
    for b in base:
        for k in (0, 1, 2, 3):
            hi = bump(b, k)
            triples += [(hi, b, b * 0.5), (b, hi, b * 0.5), (b * 0.5, b, hi), (hi, b, b), (b, b, hi), (b, hi, hi)]
        triples += [(b, b, b), (b, b, 0.0), (0.0, b, 0.0), (np.nextafter(b, 1e308), b, b), (b, np.nextafter(b, 1e308), 0.0),
                    (b * (1 + 5e-10), b, 0.1 * b), (b, b * (1 + 2e-9), 0.1 * b), (-0.0, b, 0.0)]
    triples += [(0.0, 0.0, 0.0), (5e-324, 0.0, 0.0), (5e-324, 5e-324, 5e-324), (1.7e308, 1.7e308, 1.0), (1.7e308, 1.6e308, 1.7e308)]
    rng = np.random.RandomState(4)
    n_ind, n_sites = 37, 200
    raw = oracle.synth_raw(5, 0.1, n_ind, n_sites)
    for k, t in enumerate(triples):
        raw[rng.randint(n_sites), rng.randint(n_ind)] = t
        raw[k % n_sites, k % n_ind] = t
    P = oracle.frontend(raw, call_geno=True)
    p = nb().Params(n_ind=n_ind, n_sites=n_sites, in_probs=True, call_geno=True, pairwise_del=True)
    with nb().NgsDistB200(p) as g:
        g.push_sites(raw)
        g.frontend()
        Pg, mg = g.posteriors()
    assert np.array_equal(Pg, P)
    assert np.array_equal(mg, 1 - oracle.miss_mask(P))


@pytest.mark.parametrize("n_ind", [203, 128, 5])
def test_packed_genotype_input_is_the_same_input(n_ind):
    """ngsd_push_packed_genotypes (2-bit fields, four individuals per byte; SURVEY §8f N3) against ngsd_push_genotypes of the
    same codes: bit-identical matrices, with the default field coding, the PLINK .bed coding, a padded row stride and
    pushes split at 64-site words."""
    rng = np.random.RandomState(n_ind)
    n_sites = 1000
    geno = rng.randint(-1, 3, size=(n_sites, n_ind)).astype(np.int8)
    kw = dict(in_probs=False, indep_geno=True, pairwise_del=True, evol_model=2)
    ref = run(None, genotypes=geno, **kw)[0]

    def packed_run(packed, cof, split):
        p = nb().Params(n_ind=n_ind, n_sites=n_sites, **kw)
        with nb().NgsDistB200(p) as g:
            if split:
                g.push_packed_genotypes(packed[:640], cof, 0)
                g.push_packed_genotypes(packed[640:], cof, 640)
            else:
                g.push_packed_genotypes(packed, cof)
            return g.run(want_num=True, want_cnt=True)[0]

    bed = nb().pack_genotypes(geno, field_of_code=[1, 0, 2, 3])            # -1 -> 01, 0 -> 00, 1 -> 10, 2 -> 11
    wide = np.concatenate([nb().pack_genotypes(geno), np.full((n_sites, 3), 0xA5, np.uint8)], axis=1)   # row_stride > ceil(n/4)
    for packed, cof, split in [(nb().pack_genotypes(geno), None, False), (bed, nb().PLINK_BED_CODES, True), (wide, None, True)]:
        r = packed_run(packed, cof, split)
        for k in ("dist", "num", "cnt"):
            assert np.array_equal(r[k], ref[k], equal_nan=True), k
    p = nb().Params(n_ind=n_ind, n_sites=n_sites, **kw)
    with nb().NgsDistB200(p) as g:
        with pytest.raises(nb().NgsDistError):
            g.push_packed_genotypes(bed, [0, 3, 1, 2])                      # 3 is not a genotype code
        with pytest.raises(nb().NgsDistError):
            g.push_packed_genotypes(np.zeros((n_sites, (n_ind + 3) // 4 - 1 or 1), np.uint8) if n_ind > 4 else bed, None if n_ind > 4 else [0, -2, 1, 2])
