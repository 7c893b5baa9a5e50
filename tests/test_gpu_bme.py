"""N4 (SURVEY §8f): balanced minimum-evolution trees refined from the neighbour-joining tree on the device (ngsd_bme_tree,
CLI --tree FILE --nni_bme) against the CPU restatement of the same rules (oracle/bme_oracle.py) and against the
brute-force definitions of the criterion.  FastME, the program the reference's workflow runs, is not a pinned reference."""
import ctypes as C

import numpy as np
import pytest

import oracle
from oracle import bme_oracle, nj_oracle
from test_bme_oracle import generating_lengths
from test_gpu_nj import additive_tree_matrix
from test_gpu_parity import nb

pytestmark = pytest.mark.gpu


def euclidean(n, seed):
    rng = np.random.RandomState(seed)
    X = rng.rand(n, 6)
    D = np.sqrt(((X[:, None, :] - X[None, :, :]) ** 2).sum(axis=2)) + 0.05 * rng.rand(n, n)
    D = (D + D.T) / 2
    np.fill_diagonal(D, 0)
    return D


def uniform(n, seed):
    """Uniform-random symmetric distances: far from any tree, so the NJ tree is far from BME-optimal."""
    rng = np.random.RandomState(seed)
    D = rng.rand(n, n)
    D = (D + D.T) / 2
    np.fill_diagonal(D, 0)
    return D


def assert_no_near_ties(rounds):
    """Precondition: no round is decided by rounding (best against second-best gain, and the final best against the
    threshold), on the scale M of the acceptance rule."""
    for best, second, applied, M in rounds:
        assert best - second > 1e-9 * M if applied else best < -1e-9 * M


def params(n):
    return nb().Params(n_ind=n, n_sites=64, in_probs=True, indep_geno=True)


# (kind, n, seed).  The uniform cases must need at least one interchange from the NJ start; with three leaves there is no
# internal edge, and on four and five leaves NJ already chose the BME tree for every seed tried, so those are exempt.
CASES = [("euclidean", n, n) for n in (3, 4, 5, 9, 150, 300)] + \
        [("uniform", 3, 3), ("uniform", 4, 4), ("uniform", 5, 5), ("uniform", 9, 6), ("uniform", 150, 150), ("uniform", 300, 300)]


@pytest.mark.parametrize("kind,n,seed", CASES)
def test_bme_matches_the_cpu_restatement_and_is_a_local_optimum(kind, n, seed):
    D = (euclidean if kind == "euclidean" else uniform)(n, seed)
    labels = ["L%d" % k for k in range(n)]
    want, want_nni, rounds, L = bme_oracle.bme(D, labels)
    assert_no_near_ties(rounds)
    if kind == "uniform" and n > 5:
        assert want_nni >= 1
    with nb().NgsDistB200(params(n)) as g:
        got, got_nni = g.bme_tree(D, labels)
        nj = g.nj_tree(D, labels)
    gt, gl = nj_oracle.newick_lengths(got)
    wt, wl = nj_oracle.newick_lengths(want)
    assert gt == wt, "different topology"
    assert np.allclose(gl, wl, rtol=0, atol=2e-10)
    assert got_nni == want_nni
    # the NJ tree is unchanged by the shared join loop
    nt, nl = nj_oracle.newick_lengths(nj)
    wnt, wnl = nj_oracle.newick_lengths(nj_oracle.nj(D, labels)[0])
    assert nt == wnt and np.allclose(nl, wnl, rtol=0, atol=2e-10)
    # a local optimum of the criterion, no longer than the NJ tree, with lengths that sum to its length
    L_bme = bme_oracle.pauplin_length(got, D, labels)
    if n > 3:
        assert max(bme_oracle.all_nni_gains(got, D, labels).values()) <= 1e-12 * L_bme
    assert L_bme <= bme_oracle.pauplin_length(nj, D, labels)
    assert abs(sum(gl) - L_bme) <= 1e-9 * L_bme


def test_bme_keeps_the_generating_tree_of_an_additive_matrix():
    n = 40
    D, true_splits = additive_tree_matrix(n, 5)
    gen = generating_lengths(n, 5)
    with nb().NgsDistB200(params(n)) as g:
        t, k = g.bme_tree(D)
    assert k == 0
    assert nj_oracle.splits(t) == true_splits
    got = bme_oracle.edge_lengths(t)
    assert got.keys() == gen.keys()
    assert max(abs(got[s] - gen[s]) for s in gen) <= 1e-10


def test_bme_on_all_equal_distances_makes_no_interchange_and_is_deterministic():
    n = 12
    D = np.ones((n, n)) - np.eye(n)                # every gain is exactly zero: all P are powers of two
    want, want_nni, rounds, _ = bme_oracle.bme(D)
    assert want_nni == 0 and all(r[0] == 0 for r in rounds)
    with nb().NgsDistB200(params(n)) as g:
        a, ka = g.bme_tree(D)
        b, kb = g.bme_tree(D)
    assert a == b and ka == kb == 0
    assert nj_oracle.newick_lengths(a)[0] == nj_oracle.newick_lengths(want)[0]
    assert np.allclose(nj_oracle.newick_lengths(a)[1], nj_oracle.newick_lengths(want)[1], rtol=0, atol=2e-10)


def test_bme_on_the_resident_matrix():
    n = 40
    p = nb().Params(n_ind=n, n_sites=640, in_probs=True, indep_geno=True, evol_model=0)
    with nb().NgsDistB200(p) as g:
        g.push_sites(oracle.synth_raw(8, 0.0, n, 640))
        d = g.run()[0]["dist"]
        t_dev = g.bme_tree()
        assert t_dev == g.bme_tree(d)
    assert nj_oracle.splits(t_dev[0]) == nj_oracle.splits(bme_oracle.bme(d)[0])


def test_bme_refuses_bad_input_and_reports_the_buffer_size_it_needs():
    n = 5
    D = np.ones((n, n)) - np.eye(n)
    D[0, 1] = D[1, 0] = np.nan
    with nb().NgsDistB200(params(n)) as g:
        with pytest.raises(nb().NgsDistError):
            g.bme_tree(D)
        D = uniform(n, 1)
        want, _ = g.bme_tree(D)
        need, k = C.c_uint64(0), C.c_uint64(0)
        buf = C.create_string_buffer(8)
        rc = nb().lib().ngsd_bme_tree(g._h, D.ctypes.data_as(C.c_void_p), None, buf, 8, C.byref(need), C.byref(k))
        assert rc == -1 and need.value == len(want)
        rc = nb().lib().ngsd_bme_tree(g._h, D.ctypes.data_as(C.c_void_p), None, None, 0, C.byref(need), None)
        assert rc == -1 and need.value == len(want)
    with nb().NgsDistB200(params(2)) as g:
        with pytest.raises(nb().NgsDistError):
            g.bme_tree(np.ones((2, 2)) - np.eye(2))


@pytest.mark.parametrize("n,seed", [(12, 2), (60, 3), (150, 4)])
def test_bme_on_mixed_sign_distances_matches_the_cpu_restatement_and_ends(n, seed):
    """Negative entries (a non-default score matrix can give them) make L negative; the acceptance scale is then the
    Pauplin length of |d|, every applied NNI still lowers L, and the device agrees with the oracle."""
    rng = np.random.RandomState(seed)
    D = rng.rand(n, n) - 0.5
    D = (D + D.T) / 2
    np.fill_diagonal(D, 0)
    want, want_nni, rounds, L = bme_oracle.bme(D)
    assert_no_near_ties(rounds)
    assert want_nni >= 1 and L < 0
    with nb().NgsDistB200(params(n)) as g:
        got, got_nni = g.bme_tree(D)
        nj = g.nj_tree(D)
    gt, gl = nj_oracle.newick_lengths(got)
    wt, wl = nj_oracle.newick_lengths(want)
    assert gt == wt and got_nni == want_nni
    assert np.allclose(gl, wl, rtol=0, atol=2e-10)
    M = bme_oracle.pauplin_length(got, np.abs(D))
    assert max(bme_oracle.all_nni_gains(got, D).values()) <= 1e-12 * M
    assert bme_oracle.pauplin_length(got, D) < bme_oracle.pauplin_length(nj, D)


def test_bme_on_all_equal_negative_distances_returns_without_an_interchange():
    n = 12
    D = -(np.ones((n, n)) - np.eye(n))             # every gain is exactly zero and L < 0
    want, want_nni, _, _ = bme_oracle.bme(D)
    assert want_nni == 0
    with nb().NgsDistB200(params(n)) as g:
        got, k = g.bme_tree(D)
    assert k == 0
    assert nj_oracle.newick_lengths(got)[0] == nj_oracle.newick_lengths(want)[0]
    assert np.allclose(nj_oracle.newick_lengths(got)[1], nj_oracle.newick_lengths(want)[1], rtol=0, atol=2e-10)
