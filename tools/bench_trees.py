"""Trees of a batch of bootstrap matrices (ngsd_trees_batch) against a loop of single calls (ngsd_nj_tree / ngsd_bme_tree).

  python tools/bench_trees.py [--sizes 500 2000 5000] [--batches 1 16 101]
        per size, batch size R and method: ms per tree of one trees_batch call and of a loop of single calls (host clock
        around calls that end in a device synchronise; the better of --reps runs), interchanges applied, and for the
        largest R the split of one batch call into device kernels, device copies and the rest (host layouts, Newick text
        and launch gaps), from a torch.profiler run of its own
  python tools/bench_trees.py --compare-lib OLD.so
        the same seeded matrices through OLD.so (NGSDIST_B200_LIB) and through this build, one process each: the matrices
        must be bit-identical and the ngsd_nj_tree and ngsd_bme_tree strings, on host and resident matrices, byte-identical
  python tools/bench_trees.py --dump FILE.npz      (used by --compare-lib) matrices and strings with the library in use

The matrices are JC69 (evol_model 2) replicate 0 and bootstrap replicates of ngsd_distances_batch on synthetic data
(ngsd_synth_raw_device, 10 % missing, --indep_geno), as the command line hands them to the tree step.
"""
import argparse
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

N_SITES = 20000
BLOCK = 100
SEED = 20251018


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                           text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "nvidia-smi not available"
    return q


def context(n_ind, n_rep):
    """A context over n_ind individuals x N_SITES synthetic sites, its front end done."""
    import torch
    import ngsdist_b200 as nb
    g = nb.NgsDistB200(nb.Params(n_ind=n_ind, n_sites=N_SITES, in_probs=True, indep_geno=True, evol_model=2, n_boot_rep=max(1, n_rep),
                                 boot_block_size=BLOCK, seed=SEED))
    chunk = 4096
    buf = torch.empty((chunk, n_ind, 3), dtype=torch.float64, device="cuda")
    for s0 in range(0, N_SITES, chunk):
        m = min(chunk, N_SITES - s0)
        g.synth_raw_device(buf.data_ptr(), SEED, 0.1, s0, m)
        g.push_sites_device(buf.data_ptr(), s0, m)
    g.frontend()
    torch.cuda.synchronize()
    return g


def replicates(g, n_rep):
    """[n_rep][n][n]: replicate 0 and n_rep - 1 bootstrap replicates (one ngsd_distances_batch)."""
    n = g.p.n_ind
    out = np.empty((n_rep, n, n))
    out[0] = g.distances()["dist"]
    if n_rep > 1:
        rows = [g.next_boot_counts()[0] for _ in range(n_rep - 1)]
        g.distances_batch(np.stack(rows), BLOCK, out=out[1:])
    assert np.isfinite(out).all()
    return out


def timed(fn, reps):
    best, r = None, None
    for _ in range(reps):
        t0 = time.perf_counter()
        r = fn()
        t = (time.perf_counter() - t0) * 1e3
        best = t if best is None else min(best, t)
    return best, r


def breakdown(g, mats, method):
    """Device kernel and copy time of one trees_batch call (torch.profiler), in ms."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        t0 = time.perf_counter()
        g.trees_batch(mats, method)
        wall = (time.perf_counter() - t0) * 1e3
    kern, copy = {}, 0.0
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        us = e.device_time if hasattr(e, "device_time") else e.cuda_time
        if "memcpy" in e.name.lower() or "memset" in e.name.lower():
            copy += us / 1e3
        else:
            kern[e.name] = kern.get(e.name, 0.0) + us / 1e3
    return wall, kern, copy


def bench(sizes, batches, reps):
    print("%6s %5s %6s %12s %12s %8s %10s" % ("n_ind", "R", "method", "batch ms/tr", "single ms/tr", "ratio", "nni/tree"), flush=True)
    for n in sizes:
        R_max = max(batches)
        g = context(n, R_max)
        with g:
            all_mats = replicates(g, R_max)
            g.trees_batch(all_mats[:2], "nj")              # warm-up: module load, first allocations
            g.trees_batch(all_mats[:2], "bme")
            for R in batches:
                mats = np.ascontiguousarray(all_mats[:R])
                for method in ("nj", "bme"):
                    one = g.nj_tree if method == "nj" else g.bme_tree
                    tb, got = timed(lambda: g.trees_batch(mats, method), reps)
                    ts, single = timed(lambda: [one(m) for m in mats], reps if R < 101 or n < 5000 else 1)
                    single = [(s, 0) if method == "nj" else s for s in single]
                    assert got == single, "batched trees differ from single calls"
                    nni = np.mean([k for _, k in got])
                    print("%6d %5d %6s %12.2f %12.2f %8.2f %10.1f" % (n, R, method, tb / R, ts / R, ts / tb, nni), flush=True)
            mats = np.ascontiguousarray(all_mats[:R_max])
            for method in ("nj", "bme"):
                wall, kern, copy = breakdown(g, mats, method)
                dev = sum(kern.values())
                top = ", ".join("%s %.0f" % ((re.findall(r"k_\w+", k) or [k[:20]])[0], v) for k, v in sorted(kern.items(), key=lambda x: -x[1])[:4])
                print("  n %d R %d %s (profiled run): wall %.0f ms = kernels %.0f ms (%s) + copies %.0f ms + host and gaps %.0f ms (%.0f %%)"
                      % (n, R_max, method, wall, dev, top, copy, wall - dev - copy, 100 * (wall - dev - copy) / wall), flush=True)


def dump(path, sizes):
    import ngsdist_b200 as nb
    out = {}
    for n in sizes:
        g = context(n, 2)
        with g:
            d = replicates(g, 2)
            out["dist_%d" % n] = d
            # the resident matrix is the last one ngsd_distances left on the device: replicate 0
            g.distances()
            for tag, fn in (("nj", g.nj_tree), ("bme", lambda *a: g.bme_tree(*a)[0])):
                out["%s_%d" % (tag, n)] = np.frombuffer(fn(d[1]).encode(), dtype=np.uint8)
                out["%s_resident_%d" % (tag, n)] = np.frombuffer(fn().encode(), dtype=np.uint8)
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
        print("%-18s %-11d bytes %s" % (k, a[k].nbytes, "identical" if same else "DIFFERS"))
    print("TREES_COMPARE_%s" % ("OK" if not bad else "FAILED"))
    return 0 if not bad else 1


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--sizes", type=int, nargs="+", default=[500, 2000, 5000])
    ap.add_argument("--batches", type=int, nargs="+", default=[1, 16, 101])
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--compare-lib", metavar="OLD.so")
    ap.add_argument("--dump", metavar="FILE.npz")
    a = ap.parse_args()
    if a.dump:
        dump(a.dump, a.sizes)
        return 0
    print(gpu_info(), flush=True)
    rc = compare(a.compare_lib, a.sizes) if a.compare_lib else bench(a.sizes, a.batches, a.reps) or 0
    print(gpu_info(), flush=True)
    return rc


if __name__ == "__main__":
    sys.exit(main())
