"""The three-K-bytes-per-site form of the called-genotype contraction (csrc/dist_umma.cu header) restated on the CPU:
for every pair of codes, every site weight a layer may carry and both score matrices of the reference (parse_args.cpp:25-27,
--avg_nuc_dist), sum_k A[k] B[k] must be S w f(c_i, c_j) exactly, with every operand an int8.  f is the site term of
ngsDist.cpp:351-353 for two called genotypes; a missing genotype is the uniform triple (gen_func.cpp:895-899) or, with
--pairwise_del, a dropped site."""
import itertools

import numpy as np
import pytest

import oracle


def f_table(score, pairwise_del):
    """f[c_i][c_j] for codes 0..2 and 3 = missing (what ngsd_int_lut tabulates, csrc/dist_umma.cu)."""
    s = np.asarray(score, dtype=np.float64).reshape(3, 3)
    p = np.zeros((4, 3))
    p[:3] = np.eye(3)
    p[3] = 0.0 if pairwise_del else 1.0 / 3.0
    return p @ s @ p.T


@pytest.mark.parametrize("avg", [False, True])
@pytest.mark.parametrize("pairwise_del", [False, True])
def test_three_plane_operands_reproduce_the_site_term(avg, pairwise_del):
    score = oracle.score_matrix(avg)
    f = f_table(score, pairwise_del)
    S = 2 if pairwise_del else 18                       # ngsd_int_lut's scale
    m, t = (1, 0) if pairwise_del else (3, 1)
    lut = np.rint(f * S)
    assert np.allclose(lut, f * S, atol=1e-12)
    assert np.all(lut[:3] % m == 0)                     # (S / m) f(k, c) is an integer for k < 3 (else the FP64 path is used)
    wcap = 127 // m                                     # 42 without --pairwise_del: ngsd_int_weight_cap
    for w in (1, 2, wcap):
        for ci, cj in itertools.product(range(4), repeat=2):
            A = np.array([w * (m * (ci == k) + t * (ci == 3)) for k in range(3)])
            B = np.array([lut[k, cj] / m for k in range(3)])
            assert A.max() <= 127 and B.max() <= 127 and A.min() >= 0 and B.min() >= 0
            assert np.all(B == np.rint(B))
            assert int(A @ B) == int(lut[ci, cj]) * w, (ci, cj, w)
