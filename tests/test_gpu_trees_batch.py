"""ngsd_trees_batch: the NJ and BME trees of a whole batch of matrices in one pass per GPU.  Every tree must be
byte-identical to what ngsd_nj_tree / ngsd_bme_tree give for its matrix alone (the same arithmetic per matrix), whatever
the batch around it, the chunking or the number of GPUs; a non-finite matrix gets status NGSD_ERR_ARG and no tree while
its neighbours are built; the command line's --tree builds its trees through it."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle
from oracle import bme_oracle, nj_oracle
from test_cli import run_cli
from test_gpu_bme import assert_no_near_ties, euclidean, uniform
from test_gpu_nj import additive_tree_matrix
from test_gpu_parity import nb

pytestmark = pytest.mark.gpu

ERR_ARG = -1


def params(n, **kw):
    return nb().Params(n_ind=n, n_sites=64, in_probs=True, indep_geno=True, **kw)


def mixed_sign(n, seed):
    rng = np.random.RandomState(seed)
    D = rng.rand(n, n) - 0.5
    D = (D + D.T) / 2
    np.fill_diagonal(D, 0)
    return D


def mixed_batch(n):
    """Matrices of every kind at once: their trees need different numbers of interchanges (including none)."""
    ms = [euclidean(n, n), uniform(n, n + 1), mixed_sign(n, n + 2), np.ones((n, n)) - np.eye(n), -(np.ones((n, n)) - np.eye(n)),
          euclidean(n, n + 3), uniform(n, n + 4)]
    if n >= 5:
        ms.insert(3, additive_tree_matrix(n, n)[0])
    return np.stack(ms)


def singles(g, mats, method, labels=None):
    one = g.nj_tree if method == "nj" else g.bme_tree
    out = []
    for m in mats:
        r = one(m, labels)
        out.append((r, 0) if method == "nj" else r)
    return out


@pytest.mark.parametrize("method", ["nj", "bme"])
@pytest.mark.parametrize("n", [3, 4, 9, 150, 300])
def test_mixed_batch_equals_single_calls(n, method):
    mats = mixed_batch(n)
    labels = ["T%d" % k for k in range(n)]
    with nb().NgsDistB200(params(n)) as g:
        got = g.trees_batch(mats, method, labels)
        want = singles(g, mats, method, labels)
        assert g.trees_batch(mats[:0], method) == []
    assert got == want
    if method == "bme" and n >= 150:
        assert len({k for _, k in got}) >= 3, "the batch should mix trees that stop after different numbers of rounds"
        assert any(k == 0 for _, k in got)


@pytest.mark.parametrize("method", ["nj", "bme"])
def test_batch_matches_the_cpu_restatement(method):
    n = 150
    mats = np.stack([euclidean(n, 21), uniform(n, 22), mixed_sign(n, 23)])
    labels = ["L%d" % k for k in range(n)]
    with nb().NgsDistB200(params(n)) as g:
        got = g.trees_batch(mats, method, labels)
    for (t, k), D in zip(got, mats):
        if method == "nj":
            want, k_want = nj_oracle.nj(D, labels)[0], 0
        else:
            want, k_want, rounds, _ = bme_oracle.bme(D, labels)
            assert_no_near_ties(rounds)
        gt, gl = nj_oracle.newick_lengths(t)
        wt, wl = nj_oracle.newick_lengths(want)
        assert gt == wt and k == k_want
        assert np.allclose(gl, wl, rtol=0, atol=2e-10)


def replicate_matrices():
    """300 individuals x 5 000 sites: replicate 0 and 20 bootstrap replicates (distances_batch), JC69."""
    n, s = 300, 5000
    p = nb().Params(n_ind=n, n_sites=s, in_probs=True, indep_geno=True, evol_model=2, n_boot_rep=20, boot_block_size=50, seed=7)
    g = nb().NgsDistB200(p)
    g.push_sites(oracle.synth_raw(31, 0.1, n, s))
    return g, np.stack(g.run_batched())


@pytest.mark.parametrize("method", ["nj", "bme"])
def test_bootstrap_replicates_and_their_support(method):
    g, mats = replicate_matrices()
    with g:
        got = g.trees_batch(mats, method)
        want = singles(g, mats, method)
    assert got == want
    assert all(t is not None for t, _ in got)
    trees = [t for t, _ in got]
    assert nb().tree_support(trees[0], trees[1:]) == nb().tree_support(want[0][0], [t for t, _ in want[1:]])


@pytest.mark.parametrize("method", ["nj", "bme"])
def test_a_non_finite_matrix_leaves_its_neighbours_alone(method):
    n = 40
    mats = np.stack([uniform(n, s) for s in range(5)])
    bad = mats.copy()
    bad[2, 3, 7] = bad[2, 7, 3] = np.nan
    bad[4, 0, 1] = bad[4, 1, 0] = np.inf
    with nb().NgsDistB200(params(n)) as g:
        want = g.trees_batch(mats, method)
        got = g.trees_batch(bad, method)
        L = nb().lib()
        offsets, status = np.zeros(6, dtype=np.uint64), np.zeros(5, dtype=np.int32)
        buf = C.create_string_buffer(1 << 20)
        assert L.ngsd_trees_batch(g._h, bad.ctypes.data_as(C.c_void_p), 5, nb().TREE_NJ if method == "nj" else nb().TREE_BME, None, buf,
                                  1 << 20, offsets.ctypes.data_as(C.c_void_p), None, status.ctypes.data_as(C.c_void_p)) == 0
    assert list(status) == [0, 0, ERR_ARG, 0, ERR_ARG]
    assert offsets[3] - offsets[2] == 1                    # the empty string
    assert got[2] == (None, 0) and got[4] == (None, 0)
    assert [got[k] for k in (0, 1, 3)] == [want[k] for k in (0, 1, 3)]


def test_errors_and_the_needed_buffer_size():
    n = 12
    mats = np.stack([uniform(n, s) for s in range(3)])
    L = nb().lib()
    vp = C.c_void_p
    with nb().NgsDistB200(params(n)) as g:
        want = g.trees_batch(mats, "bme")
        need = sum(len(t) + 1 for t, _ in want)
        offsets, nni, status = np.zeros(4, dtype=np.uint64), np.zeros(3, dtype=np.uint64), np.zeros(3, dtype=np.int32)
        args = lambda buf, cap, method=nb().TREE_BME, d=mats.ctypes.data_as(vp), k=3: L.ngsd_trees_batch(
            g._h, d, k, method, None, buf, cap, offsets.ctypes.data_as(vp), nni.ctypes.data_as(vp), status.ctypes.data_as(vp))
        small = C.create_string_buffer(16)
        assert args(small, 16) == ERR_ARG and offsets[3] == need
        assert b"too small" in L.ngsd_last_error(g._h)
        assert args(None, 0) == ERR_ARG and offsets[3] == need
        big = C.create_string_buffer(int(offsets[3]))
        assert args(big, int(offsets[3])) == 0
        assert [big.raw[int(offsets[k]):int(offsets[k + 1]) - 1].decode() for k in range(3)] == [t for t, _ in want]
        assert list(nni) == [k for _, k in want]
        offsets[0] = 99
        assert args(None, 0, k=0, d=None) == 0 and offsets[0] == 0          # n_mat == 0: nothing to do
        assert args(big, 1 << 20, method=7) == ERR_ARG and b"unknown tree method" in L.ngsd_last_error(g._h)
        assert args(big, 1 << 20, d=None) == ERR_ARG and b"NULL" in L.ngsd_last_error(g._h)
        with pytest.raises(ValueError):
            g.trees_batch(mats, "upgma")
    with nb().NgsDistB200(params(2)) as g:
        with pytest.raises(nb().NgsDistError, match="at least 3"):
            g.trees_batch(np.stack([np.ones((2, 2)) - np.eye(2)] * 2), "nj")


def test_chunking_does_not_change_the_trees():
    """Hold most of the free device memory so that only a few matrices fit per chunk."""
    import torch
    n = 1000
    mats = np.stack([euclidean(n, s) for s in range(8)])
    with nb().NgsDistB200(params(n)) as g:
        want_nj = g.trees_batch(mats, "nj")
        want_bme = g.trees_batch(mats, "bme")
        torch.cuda.synchronize()
        free, _ = torch.cuda.mem_get_info()
        per_bme = 2 * n * (n + 1) * 8                     # a BME tree holds about two matrices: about 3 fit beside the library's reserve
        hold = torch.empty(max(0, free - (256 << 20) - 3 * per_bme), dtype=torch.uint8, device="cuda")
        try:
            got_nj = g.trees_batch(mats, "nj")
            got_bme = g.trees_batch(mats, "bme")
        finally:
            del hold
            torch.cuda.empty_cache()
    assert got_nj == want_nj
    assert got_bme == want_bme


def _n_gpus():
    import torch
    return torch.cuda.device_count()


@pytest.mark.parametrize("method", ["nj", "bme"])
def test_group_context_equals_one_gpu(method):
    if _n_gpus() < 2:
        pytest.skip("needs 2 GPUs (%d visible)" % _n_gpus())
    n = 150
    mats = mixed_batch(n)
    with nb().NgsDistB200(params(n)) as g:
        want = g.trees_batch(mats, method)
    with nb().NgsDistB200(params(n), n_gpus=2) as g:
        got = g.trees_batch(mats, method)
        assert g.trees_batch(mats[:1], method) == want[:1]       # one matrix: the second GPU has nothing to do
    assert got == want


def run_tree_cli(tmp_path, geno, n_ind, n_sites, flags, bme):
    out, tree = str(tmp_path / "o.dist"), str(tmp_path / "o.nwk")
    r = run_cli(["--geno", geno, "--n_ind", str(n_ind), "--n_sites", str(n_sites), "--out", out, "--tree", tree, "--verbose", "0"]
                + flags + (["--nni_bme"] if bme else []))
    assert r.returncode == 0, r.stderr[-2000:]
    return open(tree).read().split("\n")[:-1], tree


BOOT_FLAGS = ["--probs", "--indep_geno", "--n_boot_rep", "20", "--boot_block_size", "10", "--seed", "12345", "--evol_model", "0"]


def library_matrices(raw, n_ind, n_sites, **kw):
    p = nb().Params(n_ind=n_ind, n_sites=n_sites, in_probs=True, indep_geno=True, n_boot_rep=20, boot_block_size=10, seed=12345,
                    evol_model=0, **kw)
    g = nb().NgsDistB200(p)
    g.push_sites(raw)
    return g, np.stack([r["dist"] for r in g.run()])


@pytest.mark.parametrize("bme", [False, True])
def test_cli_tree_file_equals_the_library(tmp_path, bme):
    from util import GOLDEN, load_bin
    n_ind, n_sites = 24, 400
    lines, tree = run_tree_cli(tmp_path, os.path.join(GOLDEN, "g24x400.bin"), n_ind, n_sites, BOOT_FLAGS, bme)
    g, mats = library_matrices(load_bin("g24x400.bin", n_ind, n_sites), n_ind, n_sites)
    method = "bme" if bme else "nj"
    with g:
        batch = g.trees_batch(mats, method)
        single = singles(g, mats, method)
    assert batch == single
    assert lines == [t for t, _ in batch]
    assert open(tree + ".support").read() == nb().tree_support(lines[0], lines[1:]) + "\n"


@pytest.mark.parametrize("bme", [False, True])
def test_cli_writes_na_for_a_non_finite_replicate(tmp_path, bme):
    """Individual 5 has data only in the first bootstrap block: under --pairwise_del every replicate that does not draw
    that block has pairs without shared sites, hence no tree; replicate 0 and the others still get theirs."""
    n_ind, n_sites = 12, 200
    raw = oracle.synth_raw(77, 0.0, n_ind, n_sites)
    raw[10:, 5, :] = 1 / 3
    geno = str(tmp_path / "in.bin")
    raw.astype(np.float64).tofile(geno)
    lines, tree = run_tree_cli(tmp_path, geno, n_ind, n_sites, BOOT_FLAGS + ["--pairwise_del"], bme)
    g, mats = library_matrices(raw, n_ind, n_sites, pairwise_del=True)
    with g:
        want = g.trees_batch(mats, "bme" if bme else "nj")
    finite = [bool(np.isfinite(m).all()) for m in mats]
    assert finite[0] and not all(finite) and sum(finite) >= 3
    assert lines == [t if t is not None else "NA" for t, _ in want]
    assert [l != "NA" for l in lines] == finite
    assert open(tree + ".support").read() == nb().tree_support(lines[0], lines[1:]) + "\n"
