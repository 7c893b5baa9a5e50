"""Tile shards on the per pair-site EM path (dist_em.cu).

One GPU: every rank's share computed in turn must tile the full matrix exactly, as the NCCL sum of multi.py assembles it
across GPUs.  Two or more GPUs: a group context against one GPU, and the command line on every golden that takes the EM
path."""
import os
import subprocess

import numpy as np
import pytest

import oracle
from ngsdist_b200 import multi
from test_gpu_parity import nb
from util import GOLDEN, golden_text, manifest, parse_flags

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def em_params(n_ind, n_sites, **kw):
    return nb().Params(n_ind=n_ind, n_sites=n_sites, in_probs=True, indep_geno=False, **kw)


def assemble(g, world, n_ind, call, tile_exact=True):
    """Runs call(g) on every rank of a `world`-way tile shard and sums the results; checks the zeros outside each shard."""
    off = ~np.eye(n_ind, dtype=bool)
    acc = None
    covered = np.zeros((n_ind, n_ind), dtype=int)
    for rank in range(world):
        g.set_tile_shard(rank, world)
        r = call(g)
        own = multi.tile_owner_mask(n_ind, rank, world)
        outside = ~own & off if not tile_exact else ~own
        for k in ("dist", "num", "cnt"):
            assert not r[k][outside].any(), "%s outside the shard of rank %d must be zero" % (k, rank)
        acc = {k: v.copy() for k, v in r.items()} if acc is None else {k: acc[k] + r[k] for k in acc}
        covered += own
    assert (covered[off] == 1).all(), "every off-diagonal entry belongs to exactly one rank"
    return acc


def full_call(block_counts=None, block_size=1):
    return lambda g: g.distances(block_counts, block_size, want_num=True, want_cnt=True)


@pytest.mark.parametrize("model", [0, 2])
@pytest.mark.parametrize("pdel", [False, True])
@pytest.mark.parametrize("world", [2, 3, 5])
def test_em_tile_shards_tile_the_matrix(world, pdel, model):
    n_ind, n_sites = 700, 1200          # 6 row blocks, 21 tiles of 128 (66 of 64)
    raw = oracle.synth_raw(41, 0.1, n_ind, n_sites)
    with nb().NgsDistB200(em_params(n_ind, n_sites, pairwise_del=pdel, evol_model=model)) as g:
        g.push_sites(raw)
        g.frontend()
        full = g.distances(want_num=True, want_cnt=True)
        s = assemble(g, world, n_ind, full_call())
        g.set_tile_shard(0, 1)
        again = g.distances(want_num=True, want_cnt=True)
    assert np.array_equal(s["cnt"], full["cnt"])
    assert np.allclose(s["num"], full["num"], rtol=1e-12, atol=0)   # K splits are planned per shard: summation order differs
    for k in ("dist", "num", "cnt"):
        assert np.array_equal(again[k], full[k]), "the whole matrix again after set_tile_shard(0, 1): " + k


@pytest.mark.parametrize("tot", [0, 5000])
def test_em_tile_shards_fewer_tiles_than_ranks(tot):
    """100 individuals are one 128 x 128 tile: rank 0 owns it, ranks 1 and 2 own nothing (and return zeros)."""
    n_ind, n_sites = 100, 900
    raw = oracle.synth_raw(43, 0.1, n_ind, n_sites)
    with nb().NgsDistB200(em_params(n_ind, n_sites, tot_sites=tot, evol_model=1)) as g:
        g.push_sites(raw)
        g.frontend()
        full = g.distances(want_num=True, want_cnt=True)
        s = assemble(g, 3, n_ind, full_call())
    assert np.array_equal(s["cnt"], full["cnt"])
    assert np.allclose(s["num"], full["num"], rtol=1e-12, atol=0)
    assert np.allclose(s["dist"], full["dist"], rtol=1e-12, atol=0)


def boot_counts(seed, n_blocks, n_rep):
    rng = np.random.default_rng(seed)
    return [np.bincount(rng.integers(0, n_blocks, n_blocks), minlength=n_blocks).astype(np.uint32) for _ in range(n_rep)]


@pytest.mark.parametrize("pdel", [False, True])
def test_em_tile_shards_bootstrap_replicates(pdel):
    """Direct replicates (block cache off) within 1e-12; cached ones bit-identical: splits = blocks on every shard."""
    n_ind, n_sites, bs, world = 700, 1600, 16, 3
    raw = oracle.synth_raw(47, 0.1, n_ind, n_sites)
    reps = boot_counts(5, n_sites // bs, 2)
    for cached in (False, True):
        with nb().NgsDistB200(em_params(n_ind, n_sites, pairwise_del=pdel, evol_model=0, no_block_cache=not cached)) as g:
            g.push_sites(raw)
            g.frontend()
            full = [g.distances(c, bs, want_num=True, want_cnt=True) for c in reps]
            assert g.timing().block_cache == (2 if cached else 0)
            acc = [None, None]
            covered = np.zeros((n_ind, n_ind), dtype=int)
            for rank in range(world):
                g.set_tile_shard(rank, world)
                own = multi.tile_owner_mask(n_ind, rank, world)
                covered += own
                for k, c in enumerate(reps):
                    r = g.distances(c, bs, want_num=True, want_cnt=True)
                    if cached:
                        assert g.timing().block_cache == 1 + k, "the shard builds its cache once, then reuses it"
                    for key in ("dist", "num", "cnt"):
                        assert not r[key][~own].any()
                    acc[k] = r if acc[k] is None else {key: acc[k][key] + r[key] for key in r}
        assert (covered[~np.eye(n_ind, dtype=bool)] == 1).all()
        for f, s in zip(full, acc):
            assert np.array_equal(s["cnt"], f["cnt"])
            if cached:
                assert np.array_equal(s["num"], f["num"]) and np.array_equal(s["dist"], f["dist"])
            else:
                assert np.allclose(s["num"], f["num"], rtol=1e-12, atol=0)


@pytest.mark.parametrize("world", [2, 3])
def test_em_tile_shards_blank_line_nan(world):
    """An empty text line makes every EM sum NaN: the assembled matrices carry the same NaN bits as the whole one."""
    n_ind, n_sites = 300, 640
    raw = oracle.synth_raw(53, 0.1, n_ind, n_sites)
    raw[[17, 400]] = nb().BLANK_SITE
    with nb().NgsDistB200(em_params(n_ind, n_sites, in_text=True, evol_model=0)) as g:
        g.push_sites(raw)
        g.frontend()
        full = g.distances(want_num=True, want_cnt=True)
        s = assemble(g, world, n_ind, full_call(), tile_exact=False)
    off = ~np.eye(n_ind, dtype=bool)
    assert np.isnan(full["dist"][off]).all()
    for k in ("dist", "num"):
        assert np.array_equal(s[k].view(np.uint64), full[k].view(np.uint64)), k
    assert np.array_equal(s["cnt"][off], full["cnt"][off])


# ------------------------------------------------------------------------------------------------ two or more GPUs --

def _n_gpus():
    import torch
    return torch.cuda.device_count()


@pytest.mark.parametrize("pdel", [False, True])
def test_em_group_context_matches_one_gpu(pdel):
    if _n_gpus() < 2:
        pytest.skip("needs 2 GPUs")
    n_ind, n_sites, bs = 700, 1600, 16
    raw = oracle.synth_raw(59, 0.1, n_ind, n_sites)
    reps = np.stack(boot_counts(7, n_sites // bs, 4))
    res = []
    for n_gpus in (1, 2):
        p = em_params(n_ind, n_sites, pairwise_del=pdel, evol_model=0, n_boot_rep=4, boot_block_size=bs)
        with nb().NgsDistB200(p, n_gpus=n_gpus, shard=nb().SHARD_REPLICATED) as g:
            g.push_sites(raw)
            g.frontend()
            m0 = g.distances(want_num=True, want_cnt=True)
            res.append((m0, g.distances_batch(reps, bs)))
    (one, one_b), (two, two_b) = res
    assert np.array_equal(two["cnt"], one["cnt"])
    assert np.allclose(two["num"], one["num"], rtol=1e-12, atol=0)
    assert np.allclose(two["dist"], one["dist"], rtol=1e-12, atol=0)
    assert np.array_equal(two_b, one_b), "cached replicates: the same per-block partials in the same order"


EM_GOLDENS = [(kind, c) for kind in ("binary", "text") for c in manifest()[kind] if not parse_flags(c["flags"])[0]["indep"]]


@pytest.mark.parametrize("kind,case", EM_GOLDENS, ids=lambda x: x if isinstance(x, str) else x["name"])
def test_em_cli_two_gpus_writes_the_reference_file(kind, case, tmp_path):
    if _n_gpus() < 2:
        pytest.skip("needs 2 GPUs")
    out = str(tmp_path / "o.dist")
    cli = os.path.join(ROOT, "ngsdist_b200", "bin", "ngsDist")
    args = [cli, "--geno", os.path.join(GOLDEN, case["input"]), "--n_ind", str(case["n_ind"]), "--n_sites", str(case["n_sites"]), "--out", out,
            "--n_threads", "4", "--verbose", "0", "--n_gpus", "2", "--shard", "auto"] + case["flags"]
    r = subprocess.run(args, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    assert open(out).read() == golden_text(case["name"])
