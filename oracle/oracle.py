"""ctypes front for oracle/libngsdist_oracle.so plus a runner for oracle/_ref/ngsDist.

TEST INFRASTRUCTURE ONLY (see package docstring).  Function names follow the reference's
(`read_geno` normalisation, `call_geno`, `gen_dist`, `rnd_map_data`; file:line in ngsdist_oracle.c).
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libngsdist_oracle.so")
REF_BIN = os.path.join(_HERE, "_ref", "ngsDist")

DEFAULT_SCORE = np.array([0, 0.5, 1, 0.5, 0, 0.5, 1, 0.5, 0], dtype=np.float64)  # parse_args.cpp:25-27


def score_matrix(avg_nuc_dist=False):
    s = DEFAULT_SCORE.copy()
    if avg_nuc_dist:
        s[4] = 0.5  # parse_args.cpp:134-137
    return s


def build(force=False):
    """Compile the C restatement (and, when /root/reference is present, oracle/_ref/ngsDist)."""
    if force or not os.path.exists(_LIB_PATH):
        subprocess.check_call(["make", "-s", "-C", _HERE, "oracle"])
    if os.path.isdir("/root/reference") and (force or not os.path.exists(REF_BIN)):
        subprocess.check_call(["make", "-s", "-C", _HERE, "ref"])


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_LIB_PATH)
        u64, i32, dbl, vp = C.c_uint64, C.c_int, C.c_double, C.c_void_p
        L.ngsd_oracle_taus_set.argtypes = [vp, C.c_uint32]
        L.ngsd_oracle_taus_get.argtypes = [vp]
        L.ngsd_oracle_taus_get.restype = C.c_uint32
        L.ngsd_oracle_boot_map.argtypes = [vp, u64, u64, vp]
        L.ngsd_oracle_frontend.argtypes = [vp, u64, u64, i32, i32, i32, dbl, dbl, vp]
        L.ngsd_oracle_frontend.restype = i32
        L.ngsd_oracle_frontend_geno.argtypes = [vp, u64, u64, vp]
        L.ngsd_oracle_frontend_geno.restype = i32
        L.ngsd_oracle_miss_mask.argtypes = [vp, u64, u64, vp]
        L.ngsd_oracle_em2.argtypes = [vp, vp, vp, dbl, i32]
        L.ngsd_oracle_em2.restype = i32
        L.ngsd_oracle_distances.argtypes = [vp, u64, u64, vp, u64, vp, i32, i32, u64, i32, vp, vp, vp, vp]
        L.ngsd_oracle_distances.restype = i32
        L.ngsd_oracle_distances_block.argtypes = [vp, u64, u64, vp, u64, vp, i32, i32, u64, i32, u64, u64, u64, u64, vp, vp, vp]
        L.ngsd_oracle_distances_block.restype = i32
        L.ngsd_oracle_synth_raw.argtypes = [u64, dbl, u64, u64, u64, vp]
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


class Taus:
    """gsl_rng_taus (SURVEY App. B)."""

    def __init__(self, seed):
        self.state = np.zeros(3, dtype=np.uint32)
        lib().ngsd_oracle_taus_set(_p(self.state), int(seed) & 0xFFFFFFFF)

    def get(self):
        return int(lib().ngsd_oracle_taus_get(_p(self.state)))

    def boot_map(self, n_blocks, block_size):
        """rnd_map_data (ngsDist.cpp:416-437): source site for each resampled site."""
        m = np.zeros(n_blocks * block_size, dtype=np.uint64)
        lib().ngsd_oracle_boot_map(_p(self.state), n_blocks, block_size, _p(m))
        return m


def synth_raw(seed, miss_rate, n_ind, n_sites, site0=0):
    """Synthetic raw GLs, binary layout [site][ind][3], normal scale (SURVEY §8(d))."""
    raw = np.empty((n_sites, n_ind, 3), dtype=np.float64)
    lib().ngsd_oracle_synth_raw(seed, float(miss_rate), n_ind, site0, n_sites, _p(raw))
    return raw


def frontend(raw, kind=0, in_log=False, call_geno=False, N_thresh=0.0, call_thresh=0.0):
    """raw [site][ind][3] -> P [ind][site][3] in normal space.  kind 0 binary, 1 text --probs."""
    raw = np.ascontiguousarray(raw, dtype=np.float64)
    n_sites, n_ind, _ = raw.shape
    P = np.empty((n_ind, n_sites, 3), dtype=np.float64)
    rc = lib().ngsd_oracle_frontend(_p(raw), n_ind, n_sites, kind, int(in_log), int(call_geno), N_thresh, call_thresh, _p(P))
    if rc == 1:
        raise ValueError("NaN found! Is the file format correct?")
    if rc == 2:
        raise ValueError("missing data threshold must be smaller than calling genotype threshold!")
    return P


def frontend_geno(codes):
    """codes [site][ind] int in {-1,0,1,2} -> P [ind][site][3]."""
    codes = np.ascontiguousarray(codes, dtype=np.int32)
    n_sites, n_ind = codes.shape
    P = np.empty((n_ind, n_sites, 3), dtype=np.float64)
    rc = lib().ngsd_oracle_frontend_geno(_p(codes), n_ind, n_sites, _p(P))
    if rc:
        raise ValueError("wrong GENO file format. Genotypes must be coded as {-1,0,1,2} !")
    return P


def miss_mask(P):
    n_ind, n_sites, _ = P.shape
    m = np.empty((n_ind, n_sites), dtype=np.uint8)
    lib().ngsd_oracle_miss_mask(_p(P), n_ind, n_sites, _p(m))
    return m


def em2(a, b, tole=0.001, max_iter=50):
    sfs = np.full(9, 1.0 / 9)
    a = np.ascontiguousarray(a, dtype=np.float64)
    b = np.ascontiguousarray(b, dtype=np.float64)
    it = lib().ngsd_oracle_em2(_p(sfs), _p(a), _p(b), tole, max_iter)
    return sfs, it


def distances(P, score=None, indep=True, pairwise_del=False, tot_sites=0, evol_model=1, site_map=None, n_eff=None,
              want_iters=False):
    """gen_dist over all pairs.  Returns dict(dist, num, cnt[, em_iters]) of n_ind x n_ind arrays."""
    P = np.ascontiguousarray(P, dtype=np.float64)
    n_ind, n_sites, _ = P.shape
    score = DEFAULT_SCORE if score is None else np.ascontiguousarray(score, dtype=np.float64).reshape(9)
    if site_map is not None:
        site_map = np.ascontiguousarray(site_map, dtype=np.uint64)
        n_eff = len(site_map) if n_eff is None else n_eff
    elif n_eff is None:
        n_eff = n_sites
    dist = np.zeros((n_ind, n_ind)); num = np.zeros((n_ind, n_ind)); cnt = np.zeros((n_ind, n_ind), dtype=np.uint64)
    iters = np.zeros((n_ind, n_ind), dtype=np.uint64) if want_iters else None
    rc = lib().ngsd_oracle_distances(_p(P), n_ind, n_sites, _p(site_map), n_eff, _p(score), int(indep), int(pairwise_del),
                                     int(tot_sites), int(evol_model), _p(dist), _p(num), _p(cnt), _p(iters))
    if rc:
        raise ValueError("invalid evolutionary model specified!")
    out = dict(dist=dist, num=num, cnt=cnt)
    if want_iters:
        out["em_iters"] = iters
    return out


def distances_block(P, r0, r1, c0, c1, score=None, indep=True, pairwise_del=False, tot_sites=0, evol_model=1,
                    site_map=None, n_eff=None):
    P = np.ascontiguousarray(P, dtype=np.float64)
    n_ind, n_sites, _ = P.shape
    score = DEFAULT_SCORE if score is None else np.ascontiguousarray(score, dtype=np.float64).reshape(9)
    if site_map is not None:
        site_map = np.ascontiguousarray(site_map, dtype=np.uint64)
        n_eff = len(site_map) if n_eff is None else n_eff
    elif n_eff is None:
        n_eff = n_sites
    h, w = r1 - r0, c1 - c0
    dist = np.zeros((h, w)); num = np.zeros((h, w)); cnt = np.zeros((h, w), dtype=np.uint64)
    rc = lib().ngsd_oracle_distances_block(_p(P), n_ind, n_sites, _p(site_map), n_eff, _p(score), int(indep), int(pairwise_del),
                                           int(tot_sites), int(evol_model), r0, r1, c0, c1, _p(dist), _p(num), _p(cnt))
    if rc:
        raise ValueError("invalid evolutionary model specified!")
    return dict(dist=dist, num=num, cnt=cnt)


def run_job(raw, *, in_log=False, call_geno=False, N_thresh=0.0, call_thresh=0.0, avg_nuc_dist=False, indep=True,
            pairwise_del=False, tot_sites=0, evol_model=1, n_boot_rep=0, boot_block_size=1, seed=12345, kind=0, blank_sites=(),
            genotypes=False, score=None):
    """Whole job the way main() runs it (ngsDist.cpp:156-289): returns the list of 1+n_boot_rep result dicts.
    blank_sites: sites that were empty text lines -- read_geno leaves them at the -1e15 fill without normalising
    (read_data.cpp:58-59), so after ngsDist.cpp:165-174 every individual holds (0,0,0) there, or the missing-data triple
    exp(log(1/3)) when call_geno ran on the all-equal fill (gen_func.cpp:895-905).  genotypes: raw is [site][ind] codes.
    score: the 3 x 3 matrix params.score[g1][g2] (9 values, row-major) instead of the one avg_nuc_dist selects."""
    if genotypes:
        P = frontend_geno(raw)
    else:
        P = frontend(raw, kind=kind, in_log=in_log, call_geno=call_geno, N_thresh=N_thresh, call_thresh=call_thresh)
    for s in blank_sites:
        P[:, s, :] = np.exp(np.log(1.0 / 3)) if call_geno else 0.0
    if call_geno or genotypes:
        indep = True  # ngsDist.cpp:55-62
    n_sites = P.shape[1]
    rng = Taus(seed)
    out = []
    kw = dict(score=score_matrix(avg_nuc_dist) if score is None else score, indep=indep, pairwise_del=pairwise_del, tot_sites=tot_sites, evol_model=evol_model)
    for rep in range(n_boot_rep + 1):
        if rep == 0:
            out.append(distances(P, **kw))
        else:
            n_sites -= n_sites % boot_block_size  # ngsDist.cpp:236 (persistent)
            sm = rng.boot_map(n_sites // boot_block_size, boot_block_size)
            out.append(distances(P, site_map=sm, **kw))
    return out


# ---------------------------------------------------------------- reference binary ------------------------------


def have_ref():
    return os.path.exists(REF_BIN) and os.access(REF_BIN, os.X_OK)


def parse_dist(path, n_ind):
    """Parse a .dist file (ngsDist.cpp:282-287): list of (labels, matrix)."""
    mats = []
    with open(path) as fh:
        lines = fh.read().split("\n")
    k = 0
    while k < len(lines):
        if lines[k] == "" and k + 1 < len(lines) and lines[k + 1].strip() == str(n_ind):
            rows, labels = [], []
            for r in range(n_ind):
                f = lines[k + 2 + r].split("\t")
                labels.append(f[0])
                rows.append([float(x) for x in f[1:]])
            mats.append((labels, np.array(rows)))
            k += 2 + n_ind
        else:
            k += 1
    return mats


def run_reference(raw, flags, n_threads=1, workdir=None, keep=False, geno_path=None, n_ind=None, n_sites=None, timeout=3600):
    """Run oracle/_ref/ngsDist on a binary [site][ind][3] input (or on `geno_path`) with `flags` (list of CLI tokens).
    Returns (list of matrices, raw .dist text)."""
    if not have_ref():
        raise RuntimeError("oracle/_ref/ngsDist not built (run `make -C oracle ref` where /root/reference exists)")
    tmp = workdir or tempfile.mkdtemp(prefix="ngsd_ref_")
    if geno_path is None:
        raw = np.ascontiguousarray(raw, dtype=np.float64)
        n_sites, n_ind, _ = raw.shape
        geno_path = os.path.join(tmp, "in.bin")
        raw.tofile(geno_path)
    out = os.path.join(tmp, "out.dist")
    cmd = [REF_BIN, "--geno", geno_path, "--n_ind", str(n_ind), "--n_sites", str(n_sites), "--out", out,
           "--n_threads", str(n_threads), "--verbose", "0"] + list(flags)
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=timeout)
    if r.returncode != 0:
        raise RuntimeError("reference failed (%d): %s" % (r.returncode, r.stderr.decode()[-2000:]))
    with open(out) as fh:
        text = fh.read()
    mats = [m for _, m in parse_dist(out, n_ind)]
    if not keep and workdir is None:
        import shutil
        shutil.rmtree(tmp, ignore_errors=True)
    return mats, text
