"""Balanced minimum-evolution trees (ngsd_bme_tree) against the neighbour-joining start (ngsd_nj_tree) on one GPU.

  python tools/bench_bme.py [--sizes 500 2000 5000]   per size: ms per tree for nj_tree and bme_tree (host clock around
                                                      calls that end in a device synchronise), interchanges applied, ms
                                                      per BME round, and up to 2 000 individuals Pauplin's length L of
                                                      the NJ and of the BME tree
  python tools/bench_bme.py --compare-lib OLD.so      the same seeded matrices and NJ trees through OLD.so
                                                      (NGSDIST_B200_LIB) and through this build, one process each: the
                                                      matrices must be bit-identical and the NJ Newick strings byte-identical
  python tools/bench_bme.py --dump FILE.npz           (used by --compare-lib) matrices and NJ strings with the library in use

The matrices are ngsd_distances results on synthetic data (ngsd_synth_raw_device, 10 % missing, --indep_geno,
evol_model 2 = JC69), as a user would hand them to a tree program.
"""
import argparse
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

N_SITES = 20000
SEED = 20251018


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                           text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "nvidia-smi not available"
    return q


def matrix(n_ind):
    """JC69 distance matrix of n_ind individuals x N_SITES synthetic sites, and a context that keeps it resident."""
    import torch
    import ngsdist_b200 as nb
    g = nb.NgsDistB200(nb.Params(n_ind=n_ind, n_sites=N_SITES, in_probs=True, indep_geno=True, evol_model=2))
    chunk = 4096
    buf = torch.empty((chunk, n_ind, 3), dtype=torch.float64, device="cuda")
    for s0 in range(0, N_SITES, chunk):
        m = min(chunk, N_SITES - s0)
        g.synth_raw_device(buf.data_ptr(), SEED, 0.1, s0, m)
        g.push_sites_device(buf.data_ptr(), s0, m)
    g.frontend()
    torch.cuda.synchronize()
    d = g.distances()["dist"]
    assert np.isfinite(d).all()
    return g, d


def timed(fn):
    t0 = time.perf_counter()
    r = fn()
    return (time.perf_counter() - t0) * 1e3, r


def bench(sizes, reps):
    from oracle import bme_oracle
    sys.setrecursionlimit(100000)                 # (the oracle's tree walks recurse once per level of a deep tree)
    print("%6s %10s %10s %6s %12s %14s %14s %10s" % ("n_ind", "nj ms", "bme ms", "nni", "ms/round", "L(NJ)", "L(BME)", "L ratio"), flush=True)
    for n in sizes:
        g, d = matrix(n)
        with g:
            g.nj_tree(d)                          # warm-up: module load, first allocations
            g.bme_tree(d)
            nj_ms = min(timed(lambda: g.nj_tree(d))[0] for _ in range(reps))
            bme = [timed(lambda: g.bme_tree(d)) for _ in range(reps)]
            bme_ms = min(t for t, _ in bme)
            newick, n_nni = bme[0][1]
            nj = g.nj_tree(d)
        assert all(r == bme[0][1] for _, r in bme), "bme_tree is not deterministic"
        per_round = (bme_ms - nj_ms) / (n_nni + 1)    # n_nni rounds that applied an interchange and the final one
        if n <= 2000:
            L_nj, L_bme = bme_oracle.pauplin_length(nj, d), bme_oracle.pauplin_length(newick, d)
            ls = "%14.6f %14.6f %10.6f" % (L_nj, L_bme, L_bme / L_nj)
        else:
            ls = "%14s %14s %10s" % ("-", "-", "-")
        print("%6d %10.1f %10.1f %6d %12.3f %s" % (n, nj_ms, bme_ms, n_nni, per_round, ls), flush=True)


def dump(path, sizes):
    out = {}
    for n in sizes:
        g, d = matrix(n)
        with g:
            out["dist_%d" % n] = d
            out["nj_%d" % n] = np.frombuffer(g.nj_tree(d).encode(), dtype=np.uint8)
            out["nj_resident_%d" % n] = np.frombuffer(g.nj_tree().encode(), dtype=np.uint8)
    np.savez(path, **out)


def compare(old, sizes):
    d = tempfile.mkdtemp()
    files = []
    for tag, lib in (("old", os.path.abspath(old)), ("new", os.path.join(ROOT, "ngsdist_b200", "libngsdist_b200.so"))):
        f = os.path.join(d, tag + ".npz")
        env = dict(os.environ, NGSDIST_B200_LIB=lib)
        subprocess.run([sys.executable, os.path.abspath(__file__), "--dump", f, "--sizes"] + [str(n) for n in sizes], env=env, check=True)
        files.append(np.load(f))
    a, b = files
    assert sorted(a.files) == sorted(b.files)
    bad = []
    for k in sorted(a.files):
        same = a[k].dtype == b[k].dtype and a[k].shape == b[k].shape and a[k].tobytes() == b[k].tobytes()
        bad += [] if same else [k]
        print("%-18s %-9d bytes %s" % (k, a[k].nbytes, "identical" if same else "DIFFERS"))
    print("NJ_COMPARE_%s" % ("OK" if not bad else "FAILED"))
    return 0 if not bad else 1


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--sizes", type=int, nargs="+", default=[500, 2000, 5000])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--compare-lib", metavar="OLD.so")
    ap.add_argument("--dump", metavar="FILE.npz")
    a = ap.parse_args()
    if a.dump:
        dump(a.dump, a.sizes)
        return 0
    print(gpu_info(), flush=True)
    rc = compare(a.compare_lib, a.sizes) if a.compare_lib else bench(a.sizes, a.reps) or 0
    print(gpu_info(), flush=True)
    return rc


if __name__ == "__main__":
    sys.exit(main())
