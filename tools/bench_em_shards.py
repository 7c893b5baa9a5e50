"""Per pair-site EM path (default --probs) on tile shards: bit-identity against another build, and scaling over GPUs.

  python tools/bench_em_shards.py compare OLD.so NEW.so   same seeded cases through both libraries (NGSDIST_B200_LIB), one
                                                          process each, unsharded: out, num and cnt must be bit-identical
  python tools/bench_em_shards.py scale [N ...]           group contexts (ngsd_cfg.n_gpus = N, REPLICATED) for N = 1, 2, 4, 8
                                                          as available: matrix 0, block-cache build + replicates, dealt
                                                          replicates, owned 64 x 64 tiles per rank
  python tools/bench_em_shards.py dump FILE.npz           (used by compare) the seeded cases with the library in use
"""
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                           text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "nvidia-smi not available"
    return q


def push_synth(g, seed, n_ind, n_sites, chunk=8192):
    import oracle
    for s0 in range(0, n_sites, chunk):
        n = min(chunk, n_sites - s0)
        g.push_sites(oracle.synth_raw(seed, 0.1, n_ind, n, site0=s0), s0)
    g.frontend()


def boot_counts(seed, n_blocks, n_rep):
    rng = np.random.default_rng(seed)
    return np.stack([np.bincount(rng.integers(0, n_blocks, n_blocks), minlength=n_blocks).astype(np.uint32) for _ in range(n_rep)])


# ---------------------------------------------------------------------------------------------------- bit identity --

def dump(path):
    import ngsdist_b200 as nb
    res = {}
    n_ind, n_sites = 500, 100000                                                  # C2
    for name, kw in (("c2_em", dict(evol_model=2)), ("c2_em_pdel", dict(pairwise_del=True, evol_model=0))):
        with nb.NgsDistB200(nb.Params(n_ind=n_ind, n_sites=n_sites, indep_geno=False, **kw)) as g:
            push_synth(g, 20251018, n_ind, n_sites)
            r = g.distances(want_num=True, want_cnt=True)
        for k, v in r.items():
            res["%s_%s" % (name, k)] = v
    bs = 1000
    reps = boot_counts(3, n_sites // bs, 3)
    with nb.NgsDistB200(nb.Params(n_ind=n_ind, n_sites=n_sites, indep_geno=False, pairwise_del=True, evol_model=0)) as g:
        push_synth(g, 20251019, n_ind, n_sites)
        for k, c in enumerate(reps):                                              # block cache: build, then reuse
            r = g.distances(c, bs, want_num=True, want_cnt=True)
            assert g.timing().block_cache == (1 if k == 0 else 2)
            for key, v in r.items():
                res["boot%d_%s" % (k, key)] = v
    np.savez(path, **res)


def compare(old, new):
    import tempfile
    d = tempfile.mkdtemp()
    files = []
    for tag, lib in (("old", old), ("new", new)):
        f = os.path.join(d, tag + ".npz")
        env = dict(os.environ, NGSDIST_B200_LIB=os.path.abspath(lib))
        subprocess.run([sys.executable, os.path.abspath(__file__), "dump", f], env=env, check=True)
        files.append(np.load(f))
    a, b = files
    assert sorted(a.files) == sorted(b.files)
    bad = [k for k in sorted(a.files) if not np.array_equal(a[k].view(np.uint64), b[k].view(np.uint64))]
    for k in sorted(a.files):
        print("%-22s %s" % (k, "bit-identical" if k not in bad else "DIFFERS"))
    print("EM_COMPARE_%s" % ("OK" if not bad else "FAILED"))
    return 0 if not bad else 1


# --------------------------------------------------------------------------------------------------------- scaling --

def owned_tiles64(n_ind, world):
    """Owned 64 x 64 tiles per rank under ngsd_set_tile_shard's dealing of 128 x 128 tiles (see multi.tile_owner_mask)."""
    from ngsdist_b200 import multi
    tiles, n64 = multi.tile_list(n_ind), (n_ind + 63) // 64
    held, per, t = [0] * world, [0] * world, 0
    while t < len(tiles):
        ln = 2 if t + 1 < len(tiles) and tiles[t + 1][0] == tiles[t][0] else 1
        to = held.index(min(held))
        held[to] += ln
        for ti, tj in tiles[t:t + ln]:
            per[to] += sum(1 for a in (0, 1) for b in (0, 1) if 2 * ti + a <= 2 * tj + b and 2 * tj + b < n64)
        t += ln
    return min(per), max(per)


def timed(fn):
    t0 = time.perf_counter()
    r = fn()
    return time.perf_counter() - t0, r


def scale(ns):
    import ngsdist_b200 as nb
    rows = []
    for n_ind, n_sites, reps_plan in ((500, 100000, ((1000, 20), (1, 20))), (2000, 200000, ((1000, 20),))):
        for N in ns:
            for bs, n_rep in reps_plan:
                p = nb.Params(n_ind=n_ind, n_sites=n_sites, indep_geno=False, evol_model=2, n_boot_rep=n_rep, boot_block_size=bs)
                with nb.NgsDistB200(p, n_gpus=N, shard=nb.SHARD_REPLICATED) as g:
                    push_synth(g, 20251018, n_ind, n_sites)
                    g.distances()                                                 # warm-up: module load, shards, buffers
                    m0 = min(timed(g.distances)[0] for _ in range(3)) if bs == reps_plan[0][0] else float("nan")
                    reps = boot_counts(11, n_sites // bs, n_rep)
                    t_first, _ = timed(lambda: g.distances_batch(reps[:1], bs))   # block 1000: builds the cache
                    t_rest, _ = timed(lambda: g.distances_batch(reps[1:], bs))
                lo, hi = owned_tiles64(n_ind, N)
                rows.append((n_ind, n_sites, N, bs, m0, t_first, t_rest / (n_rep - 1), lo, hi))
                print("n_ind %5d  n_sites %7d  N %d  block %5d  matrix0 %8.1f ms  first replicate %8.1f ms  then %8.2f ms/replicate  "
                      "64-tiles per rank %d..%d" % (n_ind, n_sites, N, bs, m0 * 1e3, t_first * 1e3, t_rest / (n_rep - 1) * 1e3, lo, hi),
                      flush=True)
    return rows


def main():
    if len(sys.argv) < 2 or sys.argv[1] not in ("compare", "scale", "dump"):
        print(__doc__)
        return 2
    if sys.argv[1] == "dump":
        dump(sys.argv[2])
        return 0
    print(gpu_info(), flush=True)
    if sys.argv[1] == "compare":
        return compare(sys.argv[2], sys.argv[3])
    import torch
    avail = torch.cuda.device_count()
    ns = [int(x) for x in sys.argv[2:]] or [n for n in (1, 2, 4, 8) if n <= avail]
    scale(ns)
    print(gpu_info(), flush=True)
    return 0


if __name__ == "__main__":
    sys.exit(main())
