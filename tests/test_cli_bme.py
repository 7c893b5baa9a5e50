"""The command line's --nni_bme: with --tree FILE, one balanced minimum-evolution tree per matrix (ngsd_bme_tree) and
FILE.support built from those trees; without --tree it is refused before any device work."""
import os

import numpy as np
import pytest

import oracle
from oracle import bme_oracle, nj_oracle
from test_cli import MAN, run_cli
from util import GOLDEN, golden_text


def test_cli_nni_bme_needs_tree():
    r = run_cli(["--geno", "x.bin", "--n_ind", "3", "--n_sites", "4", "--out", "o", "--nni_bme", "--verbose", "0"])
    assert r.returncode == 255
    assert "ERROR: [parse_cmd_args]" in r.stderr and "--nni_bme" in r.stderr


@pytest.mark.gpu
def test_cli_nni_bme_writes_one_bme_tree_per_matrix(tmp_path):
    case = [c for c in MAN["binary"] if c["name"] == "c1_indep_boot"][0]
    out, tree = str(tmp_path / "o.dist"), str(tmp_path / "o.nwk")
    r = run_cli(["--geno", os.path.join(GOLDEN, case["input"]), "--n_ind", str(case["n_ind"]), "--n_sites", str(case["n_sites"]), "--out", out,
                 "--tree", tree, "--nni_bme", "--verbose", "0"] + case["flags"])
    assert r.returncode == 0, r.stderr[-2000:]
    assert open(out).read() == golden_text(case["name"])
    trees = open(tree).read().strip().split("\n")
    mats = [m for _, m in oracle.parse_dist(out, case["n_ind"])]
    assert len(trees) == len(mats) == 6
    for t, m in zip(trees, mats):                       # the matrices as written (10 decimals) -> the same tree from the CPU restatement
        want, _, rounds, _ = bme_oracle.bme(m)
        for best, second, applied, M in rounds:         # precondition: no round of these matrices is a rounding tie
            assert best - second > 1e-9 * M if applied else best < -1e-9 * M
        assert nj_oracle.newick_lengths(t)[0] == nj_oracle.newick_lengths(want)[0]
        assert np.allclose(nj_oracle.newick_lengths(t)[1], nj_oracle.newick_lengths(want)[1], atol=1e-8)
    import ngsdist_b200 as nb
    assert open(tree + ".support").read() == nb.tree_support(trees[0], trees[1:], percent=True) + "\n"
