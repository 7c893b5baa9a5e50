"""Edge tiles of the FP64 contraction (k_dist_dmma): when n_ind is not a multiple of 128, the off-diagonal tiles of the
last row block contract only the 8-column blocks that hold individuals.  Each 8 x 8 block still takes the same DMMA
sequence as in a full tile, so a run on the first n individuals must equal, bit for bit, the [:n, :n] corner of a run on
n' = 128 * ceil(n / 128) individuals (same tile list, same K splits, no edge tiles there).  Also: the executed-DMMA
counter, and the pipelined single-GPU replicate loop against single calls."""
import ctypes

import numpy as np
import pytest

import oracle
from ngsdist_b200 import multi
from test_gpu_parity import nb

pytestmark = pytest.mark.gpu

N_SITES = 3000
SEED = 4242
# n = 256 + r covers every count of real 8-column blocks in the last row block, c8 = ceil(r / 8) = 1 .. 15, at both ends
# of some; r > 120 fills all 16 (no edge tile)
REMS = [1, 8, 9, 16, 17, 24, 25, 32, 40, 48, 56, 64, 72, 80, 88, 96, 104, 112, 113, 120, 121, 127]


def _counts(n_blocks, seed, top):
    rng = np.random.default_rng(seed)
    c = rng.integers(0, 3, n_blocks).astype(np.uint32)
    c[seed % n_blocks] = top
    return c


def _runs(n, pdel, no_cache):
    """Every result of one context, in a fixed order: (label, dict of dist / num / cnt)."""
    raw = oracle.synth_raw(SEED, 0.1, -(-n // 128) * 128, N_SITES)[:, :n, :]
    p = nb().Params(n_ind=n, n_sites=N_SITES, in_probs=True, indep_geno=True, pairwise_del=pdel, evol_model=1,
                    no_block_cache=no_cache)
    out = []
    with nb().NgsDistB200(p) as g:
        g.push_sites(np.ascontiguousarray(raw))
        g.frontend()
        out.append(("replicate 0", g.distances(want_num=True, want_cnt=True)))
        if no_cache:
            bs = 40                                       # whole chunks: uniform-scale splits, unweighted kernel
            out.append(("uniform scale", g.distances(_counts(N_SITES // bs, 1, 5), bs, want_num=True, want_cnt=True)))
            out.append(("per-site weights", g.distances(_counts(N_SITES // 7, 2, 4), 7, want_num=True, want_cnt=True)))
            if pdel:
                for rank in range(3):
                    g.set_tile_shard(rank, 3)
                    out.append(("shard %d/3" % rank, g.distances(want_num=True, want_cnt=True)))
                    out.append(("shard %d/3 per-site" % rank, g.distances(_counts(N_SITES // 7, 3, 3), 7, want_num=True, want_cnt=True)))
                g.set_tile_shard(0, 1)
        else:
            bs = 200
            for k in range(2):                            # the first call builds the block cache, the second reuses it
                r = g.distances(_counts(N_SITES // bs, 4 + k, 3 + k), bs, want_num=True, want_cnt=True)
                assert g.timing().block_cache == 1 + k
                out.append(("block cache %d" % k, r))
    return out


@pytest.mark.parametrize("mode", ["pdel", "pdel_cache", "two_plane"])
@pytest.mark.parametrize("rem", REMS)
def test_edge_tiles_match_padded_twin(rem, mode):
    n = 256 + rem
    pdel, no_cache = mode != "two_plane", mode != "pdel_cache"
    small, big = _runs(n, pdel, no_cache), _runs(-(-n // 128) * 128, pdel, no_cache)
    assert [a for a, _ in small] == [b for b, _ in big]
    shard_sum = {}
    for (label, s), (_, b) in zip(small, big):
        for key in ("dist", "num", "cnt"):
            assert np.array_equal(s[key], b[key][:n, :n], equal_nan=True), (label, key)
        if label.startswith("shard") and not label.endswith("per-site"):
            for key in ("num", "cnt"):
                shard_sum[key] = shard_sum.get(key, 0) + s[key]
    if shard_sum:
        full = small[0][1]
        assert np.array_equal(shard_sum["cnt"], full["cnt"])
        assert np.array_equal(shard_sum["num"], full["num"])


def test_dmma_counter_counts_edge_tiles():
    n, sites = 300, 2000                                  # 3 row blocks: 3 diagonal, (0, 1) full, (0, 2) and (1, 2) edge
    c8 = -(-(n % 128) // 8)
    raw = oracle.synth_raw(7, 0.1, n, sites)
    p = nb().Params(n_ind=n, n_sites=sites, in_probs=True, indep_geno=True, pairwise_del=True, evol_model=1)
    with nb().NgsDistB200(p) as g:
        g.push_sites(raw)
        g.frontend()
        g.distances()
        n_chunks = -(-sites // 8)
        assert g.timing().dist_dmma == n_chunks * 6 * (256 * 1 + 16 * c8 * 2 + 136 * 3)
        g.set_tile_shard(1, 2)                            # ownership by pairs of one row block: (0, 2) alone, then (1, 1) (1, 2)
        g.distances()
        mask = multi.tile_owner_mask(n, 1, 2)
        owned = [(ti, tj) for ti in range(3) for tj in range(ti, 3) if mask[ti * 128, tj * 128 + 1]]
        assert owned
        full = sum(1 for ti, tj in owned if ti != tj and tj != 2)
        edge = sum(1 for ti, tj in owned if ti != tj and tj == 2)
        diag = sum(1 for ti, tj in owned if ti == tj)
        assert g.timing().dist_dmma == n_chunks * 6 * (256 * full + 16 * c8 * edge + 136 * diag)
    n = 250                                               # 122 individuals in the last block fill all 16 column blocks: no edge tile
    p = nb().Params(n_ind=n, n_sites=sites, in_probs=True, indep_geno=True, pairwise_del=True, evol_model=1)
    with nb().NgsDistB200(p) as g:
        g.push_sites(oracle.synth_raw(7, 0.1, n, sites))
        g.frontend()
        g.distances()
        assert g.timing().dist_dmma == n_chunks * 6 * (256 * 1 + 136 * 2)


@pytest.mark.parametrize("bs", [40, 7])
def test_batch_equals_single_calls(bs):
    n, sites, R = 300, 3000, 5
    raw = oracle.synth_raw(11, 0.1, n, sites)
    p = nb().Params(n_ind=n, n_sites=sites, in_probs=True, indep_geno=True, pairwise_del=True, evol_model=1, no_block_cache=True)
    counts = np.stack([_counts(sites // bs, 10 + k, 3 + 2 * k) for k in range(R)])   # a different top multiplicity each
    with nb().NgsDistB200(p) as g:
        g.push_sites(raw)
        g.frontend()
        single = [g.distances(counts[k], bs)["dist"] for k in range(R)]
        dmma = 0
        for k in range(R):
            g.distances(counts[k], bs)
            dmma += g.timing().dist_dmma
        pageable = g.distances_batch(counts, bs)
        assert g.timing().dist_dmma == dmma
        L = nb().lib()
        ptr = L.ngsd_host_alloc(R * n * n * 8)
        try:
            pinned = np.ctypeslib.as_array((ctypes.c_double * (R * n * n)).from_address(ptr)).reshape(R, n, n)
            pinned[:] = np.nan
            g.distances_batch(counts, bs, out=pinned)
            for k in range(R):
                assert np.array_equal(pageable[k], single[k]), k
                assert np.array_equal(pinned[k], single[k]), k
        finally:
            L.ngsd_host_free(ptr)
        again = g.distances(counts[0], bs)["dist"]              # single calls after a batch
        assert np.array_equal(again, single[0])
