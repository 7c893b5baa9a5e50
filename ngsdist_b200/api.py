"""ctypes mirror of include/ngsdist_b200.h.

`Params` carries the fields of the reference's `params` struct (ngsDist.hpp:11-44) that the hot path reads, under
the reference's own names; `NgsDistB200` drives the library the way main() drives gen_dist (ngsDist.cpp:156-289):
front end once, then one matrix for the full data set and one per bootstrap replicate, with the host-side
gsl_rng_taus stream deciding the block multiplicities.
"""
import ctypes as C
import os
import subprocess
from dataclasses import dataclass, field

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.environ.get("NGSDIST_B200_LIB") or os.path.join(_HERE, "libngsdist_b200.so")   # (override: A/B builds of the same ABI)

ABI_SYMBOLS = [
    "ngsd_abi_version", "ngsd_default_cfg", "ngsd_create", "ngsd_destroy", "ngsd_last_error", "ngsd_push_sites",
    "ngsd_push_sites_device", "ngsd_push_genotypes", "ngsd_push_packed_genotypes", "ngsd_frontend", "ngsd_distances", "ngsd_taus_seed", "ngsd_taus_get",
    "ngsd_boot_block_counts", "ngsd_get_posteriors", "ngsd_synth_raw_device", "ngsd_get_timing", "ngsd_stream",
    "ngsd_probe_fp64_tflops", "ngsd_probe_int8_tmacs", "ngsd_probe_umma_tmacs", "ngsd_host_alloc", "ngsd_host_free", "ngsd_set_tile_shard", "ngsd_device_results", "ngsd_finish",
    "ngsd_distances_batch", "ngsd_comm_unique_id", "ngsd_comm_attach", "ngsd_comm_allgather_operands", "ngsd_comm_reduce_sites", "ngsd_comm_reduce_tiles",
    "ngsd_comm_barrier", "ngsd_comm_stats", "ngsd_bind_host_to_device", "ngsd_deferred_stats", "ngsd_push_sites_packed", "ngsd_nj_tree", "ngsd_tree_support",
    "ngsd_bme_tree", "ngsd_trees_batch",
]
ABI_VERSION = 2
COMM_ID_BYTES = 128
SHARD_AUTO, SHARD_REPLICATED, SHARD_SITES = 0, 1, 2
TREE_NJ, TREE_BME = 0, 1


class NgsDistError(RuntimeError):
    """An error the reference would have reported through error(__FUNCTION__, msg) (gen_func.cpp:12-18)."""

    def __init__(self, code, msg):
        super().__init__("[ngsd %d] %s" % (code, msg))
        self.code = code
        self.msg = msg


class _Cfg(C.Structure):
    _fields_ = [("n_ind", C.c_uint64), ("n_sites", C.c_uint64), ("tot_sites", C.c_uint64), ("score", C.c_double * 9),
                ("evol_model", C.c_int32), ("pairwise_del", C.c_int32), ("indep_geno", C.c_int32), ("call_geno", C.c_int32),
                ("N_thresh", C.c_double), ("call_thresh", C.c_double), ("input_is_log", C.c_int32), ("input_kind", C.c_int32),
                ("device", C.c_int32), ("reserved", C.c_int32), ("n_gpus", C.c_int32), ("shard", C.c_int32),
                ("boot_block_size", C.c_uint64)]


class Timing(C.Structure):
    _fields_ = [("frontend_ms", C.c_float), ("count_ms", C.c_float), ("dist_ms", C.c_float), ("epilogue_ms", C.c_float),
                ("total_ms", C.c_float), ("launches", C.c_int32), ("dist_ctas", C.c_int32), ("dist_dmma", C.c_uint64),
                ("active_sites", C.c_uint64), ("dist_imma", C.c_uint64), ("block_cache", C.c_int32), ("pad_", C.c_int32)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


def lib_path():
    return _LIB


def build_library(verbose=False):
    """Compile csrc/*.cu for sm_100a into libngsdist_b200.so (nvcc cross-compiles without a GPU)."""
    cmd = ["make", "-C", os.path.join(_HERE, "csrc"), "-j8"] + ([] if verbose else ["-s"])
    subprocess.check_call(cmd)
    return _LIB


_lib = None


def lib():
    """Load the shared library; never falls back to anything else."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB):
        raise ImportError("libngsdist_b200.so is not built (run `python -c 'import __graft_entry__ as g; g.build()'` or "
                          "`make -C ngsdist_b200/csrc`); ngsdist_b200 has no CPU fallback")
    L = C.CDLL(_LIB)
    vp, u64, i32, dbl = C.c_void_p, C.c_uint64, C.c_int, C.c_double
    L.ngsd_abi_version.restype = i32
    L.ngsd_default_cfg.argtypes = [C.POINTER(_Cfg)]
    L.ngsd_default_cfg.restype = None
    L.ngsd_create.argtypes = [C.POINTER(_Cfg), C.POINTER(vp)]
    L.ngsd_destroy.argtypes = [vp]
    L.ngsd_last_error.argtypes = [vp]
    L.ngsd_last_error.restype = C.c_char_p
    L.ngsd_push_sites.argtypes = [vp, vp, u64, u64]
    L.ngsd_push_sites_device.argtypes = [vp, vp, u64, u64]
    L.ngsd_push_genotypes.argtypes = [vp, vp, u64, u64]
    L.ngsd_push_packed_genotypes.argtypes = [vp, vp, u64, vp, u64, u64]
    L.ngsd_frontend.argtypes = [vp]
    L.ngsd_distances.argtypes = [vp, vp, u64, u64, vp, vp, vp]
    L.ngsd_taus_seed.argtypes = [vp, C.c_uint32]
    L.ngsd_taus_seed.restype = None
    L.ngsd_taus_get.argtypes = [vp]
    L.ngsd_taus_get.restype = C.c_uint32
    L.ngsd_boot_block_counts.argtypes = [vp, u64, vp]
    L.ngsd_boot_block_counts.restype = None
    L.ngsd_get_posteriors.argtypes = [vp, vp, vp]
    L.ngsd_synth_raw_device.argtypes = [vp, vp, u64, dbl, u64, u64]
    L.ngsd_get_timing.argtypes = [vp, C.POINTER(Timing)]
    L.ngsd_stream.argtypes = [vp]
    L.ngsd_stream.restype = vp
    L.ngsd_probe_fp64_tflops.argtypes = [i32, C.POINTER(dbl)]
    L.ngsd_probe_int8_tmacs.argtypes = [i32, C.POINTER(dbl)]
    L.ngsd_probe_umma_tmacs.argtypes = [i32, C.POINTER(dbl)]
    L.ngsd_host_alloc.argtypes = [u64]
    L.ngsd_host_alloc.restype = vp
    L.ngsd_host_free.argtypes = [vp]
    L.ngsd_host_free.restype = None
    L.ngsd_set_tile_shard.argtypes = [vp, C.c_uint32, C.c_uint32]
    L.ngsd_device_results.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp)]
    L.ngsd_finish.argtypes = [vp, vp]
    L.ngsd_distances_batch.argtypes = [vp, vp, u64, u64, u64, vp]
    L.ngsd_comm_unique_id.argtypes = [vp]
    L.ngsd_comm_attach.argtypes = [vp, vp, C.c_uint32, C.c_uint32]
    L.ngsd_comm_allgather_operands.argtypes = [vp, vp]
    L.ngsd_comm_reduce_sites.argtypes = [vp, C.c_uint32, u64, vp]
    L.ngsd_comm_reduce_tiles.argtypes = [vp, C.c_uint32, C.c_int32, vp, vp, vp]
    L.ngsd_comm_barrier.argtypes = [vp]
    L.ngsd_comm_stats.argtypes = [vp, C.POINTER(u64), C.POINTER(C.c_float)]
    L.ngsd_bind_host_to_device.argtypes = [i32]
    L.ngsd_deferred_stats.argtypes = [vp, C.POINTER(u64)]
    L.ngsd_push_sites_packed.argtypes = [vp, vp, i32, dbl, u64, u64]
    L.ngsd_nj_tree.argtypes = [vp, vp, vp, vp, u64, C.POINTER(u64)]
    L.ngsd_tree_support.argtypes = [C.c_char_p, vp, u64, i32, vp, u64, C.POINTER(u64)]
    for name in ("ngsd_create", "ngsd_destroy", "ngsd_push_sites", "ngsd_push_sites_device", "ngsd_push_genotypes", "ngsd_push_packed_genotypes", "ngsd_frontend",
                 "ngsd_distances", "ngsd_get_posteriors", "ngsd_synth_raw_device", "ngsd_get_timing", "ngsd_probe_fp64_tflops", "ngsd_probe_int8_tmacs", "ngsd_probe_umma_tmacs",
                 "ngsd_set_tile_shard", "ngsd_device_results", "ngsd_finish", "ngsd_distances_batch", "ngsd_comm_unique_id", "ngsd_comm_attach",
                 "ngsd_comm_allgather_operands", "ngsd_comm_reduce_sites", "ngsd_comm_reduce_tiles", "ngsd_comm_barrier", "ngsd_comm_stats",
                 "ngsd_bind_host_to_device", "ngsd_deferred_stats", "ngsd_push_sites_packed", "ngsd_nj_tree", "ngsd_tree_support"):
        getattr(L, name).restype = i32
    # (a build from before ngsd_bme_tree or ngsd_trees_batch, named by NGSDIST_B200_LIB for an A/B comparison of the other
    # entry points, lacks them; build() and tests/test_abi_surface.py require them of this package's library)
    if hasattr(L, "ngsd_bme_tree"):
        L.ngsd_bme_tree.argtypes = [vp, vp, vp, vp, u64, C.POINTER(u64), C.POINTER(u64)]
        L.ngsd_bme_tree.restype = i32
    if hasattr(L, "ngsd_trees_batch"):
        L.ngsd_trees_batch.argtypes = [vp, vp, u64, C.c_int32, vp, vp, u64, vp, vp, vp]
        L.ngsd_trees_batch.restype = i32
    _lib = L
    return L


def _ptr(a):
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data_as(C.c_void_p)
    return C.c_void_p(int(a))   # raw address (e.g. torch tensor.data_ptr())


@dataclass
class Params:
    """Subset of the reference `params` (ngsDist.hpp:11-44); defaults follow init_pars (parse_args.cpp:6-37)."""
    n_ind: int = 0
    n_sites: int = 0
    tot_sites: int = 0
    in_probs: bool = True
    in_logscale: bool = False
    call_geno: bool = False
    N_thresh: float = 0.0
    call_thresh: float = 0.0
    pairwise_del: bool = False
    avg_nuc_dist: bool = False
    score: list = field(default_factory=lambda: [0, 0.5, 1, 0.5, 0, 0.5, 1, 0.5, 0])
    evol_model: int = 1
    indep_geno: bool = False
    n_boot_rep: int = 0
    boot_block_size: int = 1
    seed: int = 12345
    in_text: bool = False      # text reader semantics (no -inf clamp) instead of the binary reader's
    keep_planes: bool = False  # ngsd_cfg.reserved bit 0: keep all three operand planes (exact ngsd_get_posteriors)
    force_fp64: bool = False   # ngsd_cfg.reserved bit 1: called genotypes through the FP64 contraction (A/B testing)
    no_block_cache: bool = False  # ngsd_cfg.reserved bit 2: contract every bootstrap replicate directly

    def resolved(self):
        """Apply the parse-time implications and main()'s forcing rules (parse_args.cpp:91-94,123-130; ngsDist.cpp:55-62)."""
        p = Params(**{**self.__dict__, "score": list(self.score)})
        if p.avg_nuc_dist:
            p.score[4] = 0.5
        if p.in_logscale:
            p.in_probs = True
        if p.N_thresh != 0 or p.call_thresh != 0:
            p.call_geno = True
        if p.call_geno and not p.in_probs:
            raise NgsDistError(-1, "can only call genotypes from likelihoods/probabilities!")
        if not p.in_probs or p.call_geno:
            p.indep_geno = True
        return p


def tree_support(main_newick, rep_newicks, percent=True):
    """Bootstrap support of `main_newick` from the replicate trees (host code of the library; no GPU involved):
    the main tree with the number (or RAxML-style integer percentage) of replicates holding each internal edge's
    bipartition as node labels."""
    reps = [r.encode() if isinstance(r, str) else r for r in rep_newicks]
    arr = (C.c_char_p * max(1, len(reps)))(*reps) if reps else None
    main = main_newick.encode() if isinstance(main_newick, str) else main_newick
    need = C.c_uint64(0)
    cap = 2 * len(main) + 64
    for _ in range(2):
        buf = C.create_string_buffer(cap)
        rc = lib().ngsd_tree_support(main, arr, len(reps), 1 if percent else 0, buf, cap, C.byref(need))
        if rc == 0:
            return buf.value.decode()
        if need.value + 1 > cap:
            cap = need.value + 1
            continue
        break
    raise ValueError("ngsd_tree_support: malformed Newick or different leaf sets (rc %d)" % rc)


def taus_block_counts(state, n_blocks):
    counts = np.zeros(n_blocks, dtype=np.uint32)
    lib().ngsd_boot_block_counts(_ptr(state), n_blocks, _ptr(counts))
    return counts


def probe_fp64_tflops(device=0):
    v = C.c_double(0)
    rc = lib().ngsd_probe_fp64_tflops(device, C.byref(v))
    if rc:
        raise NgsDistError(rc, "FP64 probe failed")
    return v.value


def probe_umma_tmacs(device=0):
    v = C.c_double(0)
    rc = lib().ngsd_probe_umma_tmacs(device, C.byref(v))
    if rc:
        raise NgsDistError(rc, "tcgen05 int8 probe failed")
    return v.value


def probe_int8_tmacs(device=0):
    v = C.c_double(0)
    rc = lib().ngsd_probe_int8_tmacs(device, C.byref(v))
    if rc:
        raise NgsDistError(rc, "int8 probe failed")
    return v.value


def comm_unique_id():
    """ncclGetUniqueId through the library (rank 0); hand the bytes to every rank for NgsDistB200.comm_attach."""
    buf = (C.c_uint8 * COMM_ID_BYTES)()
    rc = lib().ngsd_comm_unique_id(buf)
    if rc:
        raise NgsDistError(rc, lib().ngsd_last_error(None).decode())
    return bytes(buf)


def bind_host_to_device(device):
    return lib().ngsd_bind_host_to_device(device)


XFER_F32, XFER_U32, XFER_U20X3 = 1, 2, 3


def pack_u20x3(q):
    """[n][n_ind][3] integers < 2^20 -> [n][n_ind] uint64 (q0 | q1 << 20 | q2 << 40), the NGSD_XFER_U20X3 layout."""
    q = np.asarray(q).astype(np.uint64)
    assert (q < (1 << 20)).all()
    return np.ascontiguousarray(q[..., 0] | (q[..., 1] << np.uint64(20)) | (q[..., 2] << np.uint64(40)))


BLANK_SITE = np.array([0x7FF84E4753444231], dtype=np.uint64).view(np.float64)[0]   # NGSD_BLANK_SITE_BITS: an empty text line
BLANK_SITE_CODE = -128

PLINK_BED_CODES = (0, -1, 1, 2)     # .bed 2-bit fields: 0 = homozygous A1, 1 = missing, 2 = heterozygous, 3 = homozygous A2


def pack_genotypes(geno, field_of_code=None):
    """[site][ind] codes {-1,0,1,2} -> [site][ceil(n_ind / 4)] bytes, individual i in bits 2 (i % 4) of byte i / 4.
    field_of_code maps code c (index c + 1, i.e. [-1, 0, 1, 2]) to its 2-bit field; default: the inverse of {0,1,2,-1}."""
    geno = np.asarray(geno, dtype=np.int8)
    f = np.array([3, 0, 1, 2] if field_of_code is None else field_of_code, dtype=np.uint8)[geno.astype(np.int64) + 1]
    n_sites, n_ind = geno.shape
    pad = (-n_ind) % 4
    if pad:
        f = np.concatenate([f, np.zeros((n_sites, pad), dtype=np.uint8)], axis=1)
    f = f.reshape(n_sites, -1, 4)
    return (f[:, :, 0] | (f[:, :, 1] << 2) | (f[:, :, 2] << 4) | (f[:, :, 3] << 6)).astype(np.uint8)


class NgsDistB200:
    """One context = one GPU = the hot path of one ngsDist run."""

    def __init__(self, params: Params, device=0, n_gpus=1, shard=SHARD_AUTO):
        """n_gpus > 1: one context driving devices device .. device + n_gpus - 1 (ngsd_cfg.n_gpus / shard)."""
        self.p = params.resolved()
        L = lib()
        cfg = _Cfg()
        L.ngsd_default_cfg(C.byref(cfg))
        p = self.p
        cfg.n_ind, cfg.n_sites, cfg.tot_sites = p.n_ind, p.n_sites, p.tot_sites
        for k in range(9):
            cfg.score[k] = float(p.score[k])
        cfg.evol_model = p.evol_model
        cfg.pairwise_del = int(p.pairwise_del)
        cfg.indep_geno = int(p.indep_geno)
        cfg.call_geno = int(p.call_geno)
        cfg.N_thresh, cfg.call_thresh = p.N_thresh, p.call_thresh
        cfg.input_is_log = int(p.in_logscale)
        cfg.input_kind = 2 if not p.in_probs else (1 if p.in_text else 0)
        cfg.device = device
        cfg.reserved = (1 if p.keep_planes else 0) | (2 if p.force_fp64 else 0) | (4 if p.no_block_cache else 0)
        cfg.n_gpus = n_gpus if n_gpus > 1 else 0
        cfg.shard = shard
        cfg.boot_block_size = p.boot_block_size if p.n_boot_rep > 0 else 0
        self.n_gpus = max(1, n_gpus)
        self._h = C.c_void_p()
        rc = L.ngsd_create(C.byref(cfg), C.byref(self._h))
        if rc:
            raise NgsDistError(rc, L.ngsd_last_error(None).decode())
        self._taus = np.zeros(3, dtype=np.uint32)
        L.ngsd_taus_seed(_ptr(self._taus), p.seed & 0xFFFFFFFF)
        self._n_sites_boot = p.n_sites   # the persistently truncated n_sites of ngsDist.cpp:236

    # -- lifetime --
    def close(self):
        if getattr(self, "_h", None):
            lib().ngsd_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc):
        if rc:
            raise NgsDistError(rc, lib().ngsd_last_error(self._h).decode())

    # -- front end --
    def push_sites(self, raw, site0=0):
        """raw: numpy [n][n_ind][3] float64 host array exactly as the reader produced it."""
        raw = np.ascontiguousarray(raw, dtype=np.float64)
        assert raw.shape[1:] == (self.p.n_ind, 3), raw.shape
        self._check(lib().ngsd_push_sites(self._h, _ptr(raw), site0, raw.shape[0]))

    def push_sites_ptr(self, host_ptr, site0, n):
        self._check(lib().ngsd_push_sites(self._h, _ptr(host_ptr), site0, n))

    def push_sites_device(self, dev_ptr, site0, n):
        self._check(lib().ngsd_push_sites_device(self._h, _ptr(dev_ptr), site0, n))

    def push_sites_f32(self, raw32, site0=0):
        """Transport tier NGSD_XFER_F32: [n][n_ind][3] float32."""
        raw32 = np.ascontiguousarray(raw32, dtype=np.float32)
        assert raw32.shape[1:] == (self.p.n_ind, 3)
        self._check(lib().ngsd_push_sites_packed(self._h, _ptr(raw32), XFER_F32, 0.0, site0, raw32.shape[0]))

    def push_sites_fixed(self, q, denom, site0=0):
        """Fixed-point transport: q uint32 [n][n_ind][3] (NGSD_XFER_U32) or uint64 [n][n_ind] holding three 20-bit fields
        (NGSD_XFER_U20X3, see pack_u20x3); value = q / denom."""
        q = np.ascontiguousarray(q)
        if q.dtype == np.uint64:
            assert q.shape[1:] == (self.p.n_ind,)
            fmt = XFER_U20X3
        else:
            q = np.ascontiguousarray(q, dtype=np.uint32)
            assert q.shape[1:] == (self.p.n_ind, 3)
            fmt = XFER_U32
        self._check(lib().ngsd_push_sites_packed(self._h, _ptr(q), fmt, float(denom), site0, q.shape[0]))

    def push_sites_packed_ptr(self, host_ptr, fmt, denom, site0, n):
        self._check(lib().ngsd_push_sites_packed(self._h, _ptr(host_ptr), fmt, float(denom), site0, n))

    def push_genotypes(self, codes, site0=0):
        codes = np.ascontiguousarray(codes, dtype=np.int8)
        assert codes.shape[1] == self.p.n_ind
        self._check(lib().ngsd_push_genotypes(self._h, _ptr(codes), site0, codes.shape[0]))

    def push_packed_genotypes(self, packed, code_of_field=None, site0=0, n=None):
        """2-bit genotypes, four individuals per byte, site-major rows (see ngsd_push_packed_genotypes / pack_genotypes)."""
        packed = np.ascontiguousarray(packed, dtype=np.uint8)
        assert packed.ndim == 2
        cof = None if code_of_field is None else np.ascontiguousarray(code_of_field, dtype=np.int8)
        assert cof is None or cof.shape == (4,)
        self._check(lib().ngsd_push_packed_genotypes(self._h, _ptr(packed), packed.shape[1], _ptr(cof), site0,
                                                     packed.shape[0] if n is None else n))

    def frontend(self):
        self._check(lib().ngsd_frontend(self._h))

    def posteriors(self, want_P=True, want_miss=True):
        n, s = self.p.n_ind, self.p.n_sites
        P = np.empty((n, s, 3), dtype=np.float64) if want_P else None
        m = np.empty((n, s), dtype=np.uint8) if want_miss else None
        self._check(lib().ngsd_get_posteriors(self._h, _ptr(P), _ptr(m)))
        return P, m

    # -- distances --
    def distances(self, block_counts=None, block_size=1, want_num=False, want_cnt=False, out=None):
        n = self.p.n_ind
        if out is None:
            out = np.empty((n, n), dtype=np.float64)
        num = np.empty((n, n), dtype=np.float64) if want_num else None
        cnt = np.empty((n, n), dtype=np.uint64) if want_cnt else None
        if block_counts is not None:
            block_counts = np.ascontiguousarray(block_counts, dtype=np.uint32)
            nb = len(block_counts)
            if nb == 0:                          # --boot_block_size > n_sites: a replicate of zero blocks (not replicate 0)
                block_counts = np.zeros(1, dtype=np.uint32)
        else:
            nb = 0
        self._check(lib().ngsd_distances(self._h, _ptr(block_counts), nb, block_size, _ptr(out), _ptr(num), _ptr(cnt)))
        res = dict(dist=out)
        if want_num:
            res["num"] = num
        if want_cnt:
            res["cnt"] = cnt
        return res

    def distances_raw(self, counts_ptr, n_blocks, block_size, out_ptr):
        """Pointer-level call for bench.py (pinned buffers, no numpy allocation in the timed region)."""
        self._check(lib().ngsd_distances(self._h, _ptr(counts_ptr), n_blocks, block_size, _ptr(out_ptr), None, None))

    def next_boot_counts(self):
        """Advance the host RNG by one replicate (ngsDist.cpp:235-238): returns (block_counts, block_size)."""
        bs = self.p.boot_block_size
        self._n_sites_boot -= self._n_sites_boot % bs
        n_blocks = self._n_sites_boot // bs
        return taus_block_counts(self._taus, n_blocks), bs

    def distances_batch(self, counts, block_size, out=None):
        """counts: [n_rep][n_blocks] uint32 -> [n_rep][n][n] matrices (ngsd_distances_batch).  With a communicator attached
        only rank 0 receives them (the other ranks return None)."""
        counts = np.ascontiguousarray(counts, dtype=np.uint32)
        n_rep, n_blocks = counts.shape
        n = self.p.n_ind
        root = getattr(self, "_comm_rank", 0) == 0
        if out is None and root:
            out = np.empty((n_rep, n, n), dtype=np.float64)
        self._check(lib().ngsd_distances_batch(self._h, _ptr(counts), n_rep, n_blocks, block_size, _ptr(out) if root else None))
        return out if root else None

    def run_batched(self):
        """main()'s replicate loop with the bootstrap replicates in ONE ngsd_distances_batch call: list of matrices."""
        self.frontend()
        res = [self.distances()["dist"]]
        if self.p.n_boot_rep > 0:
            rows = []
            for _ in range(self.p.n_boot_rep):
                c, bs = self.next_boot_counts()
                rows.append(c)
            nb_ = min(len(r) for r in rows)          # the truncation is persistent, so every replicate has the same count
            res += list(self.distances_batch(np.stack([r[:nb_] for r in rows]), self.p.boot_block_size))
        return res

    def run(self, want_num=False, want_cnt=False):
        """The replicate loop of main() (ngsDist.cpp:217-289): list of 1 + n_boot_rep result dicts."""
        self.frontend()
        res = []
        for rep in range(self.p.n_boot_rep + 1):
            if rep == 0:
                res.append(self.distances(want_num=want_num, want_cnt=want_cnt))
            else:
                counts, bs = self.next_boot_counts()
                res.append(self.distances(counts, bs, want_num=want_num, want_cnt=want_cnt))
        return res

    # -- multi-GPU (see multi.py) --
    def set_tile_shard(self, rank, world):
        self._check(lib().ngsd_set_tile_shard(self._h, rank, world))

    def device_results(self):
        """Device addresses of the n_ind x n_ind result buffers (dist f64, num f64, cnt u64) of the last ngsd_distances."""
        o, n, c = C.c_void_p(), C.c_void_p(), C.c_void_p()
        self._check(lib().ngsd_device_results(self._h, C.byref(o), C.byref(n), C.byref(c)))
        return o.value, n.value, c.value

    def partial_sums(self, block_counts=None, block_size=1):
        """Raw sums of this context's sites; results stay on the device (site-sharded runs)."""
        if block_counts is not None:
            block_counts = np.ascontiguousarray(block_counts, dtype=np.uint32)
            nb_ = len(block_counts)
        else:
            nb_ = 0
        self._check(lib().ngsd_distances(self._h, _ptr(block_counts), nb_, block_size, None, None, None))

    def finish(self, out=None):
        n = self.p.n_ind
        if out is None:
            out = np.empty((n, n), dtype=np.float64)
        self._check(lib().ngsd_finish(self._h, _ptr(out)))
        return out

    # -- one process per GPU: NCCL below the C ABI (ngsd_comm_*) --
    def comm_attach(self, comm_id, rank, world):
        """comm_id: the 128 bytes rank 0 got from comm_unique_id(), carried to every rank by the host."""
        buf = (C.c_uint8 * COMM_ID_BYTES).from_buffer_copy(bytes(comm_id))
        self._check(lib().ngsd_comm_attach(self._h, buf, rank, world))
        self._comm_rank, self._comm_world = rank, world

    def comm_allgather_operands(self, site_begin):
        sb = np.ascontiguousarray(site_begin, dtype=np.uint64)
        self._check(lib().ngsd_comm_allgather_operands(self._h, _ptr(sb)))

    def comm_reduce_sites(self, root, n_eff_total, out=None):
        n = self.p.n_ind
        if out is None and self._comm_rank == root:
            out = np.empty((n, n), dtype=np.float64)
        self._check(lib().ngsd_comm_reduce_sites(self._h, root, n_eff_total, _ptr(out) if self._comm_rank == root else None))
        return out if self._comm_rank == root else None

    def comm_reduce_tiles(self, root, want_num_cnt=False, out=None):
        n = self.p.n_ind
        is_root = self._comm_rank == root
        if out is None and is_root:
            out = np.empty((n, n), dtype=np.float64)
        num = np.empty((n, n), dtype=np.float64) if (want_num_cnt and is_root) else None
        cnt = np.empty((n, n), dtype=np.uint64) if (want_num_cnt and is_root) else None
        self._check(lib().ngsd_comm_reduce_tiles(self._h, root, int(want_num_cnt), _ptr(out) if is_root else None, _ptr(num), _ptr(cnt)))
        if not is_root:
            return None
        res = dict(dist=out)
        if want_num_cnt:
            res.update(num=num, cnt=cnt)
        return res

    def comm_barrier(self):
        self._check(lib().ngsd_comm_barrier(self._h))

    def comm_stats(self):
        b, ms = C.c_uint64(0), C.c_float(0)
        self._check(lib().ngsd_comm_stats(self._h, C.byref(b), C.byref(ms)))
        return b.value, ms.value

    # -- measurement --
    def timing(self):
        t = Timing()
        self._check(lib().ngsd_get_timing(self._h, C.byref(t)))
        return t

    def synth_raw_device(self, dev_ptr, seed, miss_rate, site0, n):
        self._check(lib().ngsd_synth_raw_device(self._h, _ptr(dev_ptr), seed, float(miss_rate), site0, n))

    def stream(self):
        return lib().ngsd_stream(self._h)

    def nj_tree(self, dist=None, labels=None):
        """Neighbour-joining tree (Newick) of the last matrix on the device, or of `dist` (n x n host array)."""
        d = None if dist is None else np.ascontiguousarray(dist, dtype=np.float64)
        lab = None
        if labels is not None:
            lab = (C.c_char_p * len(labels))(*[str(x).encode() for x in labels])
        need = C.c_uint64(0)
        cap = 64 * self.p.n_ind + 1024
        for _ in range(2):
            buf = C.create_string_buffer(cap)
            rc = lib().ngsd_nj_tree(self._h, _ptr(d), lab, buf, cap, C.byref(need))
            if rc == 0:
                return buf.value.decode()
            if need.value + 1 > cap:
                cap = need.value + 1
                continue
            self._check(rc)
        self._check(rc)

    def bme_tree(self, dist=None, labels=None):
        """Balanced minimum-evolution tree (Newick, balanced branch lengths) refined by BME interchanges from the
        neighbour-joining tree of the last matrix on the device, or of `dist`; returns (newick, interchanges applied)."""
        d = None if dist is None else np.ascontiguousarray(dist, dtype=np.float64)
        lab = None
        if labels is not None:
            lab = (C.c_char_p * len(labels))(*[str(x).encode() for x in labels])
        need, n_nni = C.c_uint64(0), C.c_uint64(0)
        cap = 64 * self.p.n_ind + 1024
        for _ in range(2):
            buf = C.create_string_buffer(cap)
            rc = lib().ngsd_bme_tree(self._h, _ptr(d), lab, buf, cap, C.byref(need), C.byref(n_nni))
            if rc == 0:
                return buf.value.decode(), n_nni.value
            if need.value + 1 > cap:
                cap = need.value + 1
                continue
            self._check(rc)
        self._check(rc)

    def trees_batch(self, dists, method="nj", labels=None):
        """Trees of a batch of n x n host matrices (ngsd_trees_batch: one pass per GPU for the whole batch), method "nj"
        (nj_tree) or "bme" (bme_tree).  Returns one (newick, interchanges applied) per matrix, in input order; newick is
        None for a matrix with non-finite entries.  Every string equals what nj_tree / bme_tree give for that matrix."""
        n = self.p.n_ind
        d = np.ascontiguousarray(dists, dtype=np.float64)
        if d.size == 0:
            d = d.reshape(0, n, n)
        assert d.ndim == 3 and d.shape[1:] == (n, n), d.shape
        m = {"nj": TREE_NJ, "bme": TREE_BME}.get(method)
        if m is None:
            raise ValueError("method must be 'nj' or 'bme', not %r" % (method,))
        n_mat = d.shape[0]
        lab = None
        if labels is not None:
            lab = (C.c_char_p * len(labels))(*[str(x).encode() for x in labels])
        offsets = np.zeros(n_mat + 1, dtype=np.uint64)
        nni = np.zeros(max(1, n_mat), dtype=np.uint64)
        status = np.zeros(max(1, n_mat), dtype=np.int32)
        cap = n_mat * (64 * n + 1024)
        for _ in range(2):
            buf = C.create_string_buffer(max(1, cap))
            rc = lib().ngsd_trees_batch(self._h, _ptr(d), n_mat, m, lab, buf, cap, _ptr(offsets), _ptr(nni), _ptr(status))
            if rc == 0 or int(offsets[n_mat]) <= cap:
                break
            cap = int(offsets[n_mat])
        self._check(rc)
        raw = buf.raw
        out = []
        for k in range(n_mat):
            s = raw[int(offsets[k]):int(offsets[k + 1]) - 1].decode()
            out.append((s if status[k] == 0 else None, int(nni[k])))
        return out

    def deferred_stats(self):
        """Individual-sites the host's libm decided (knife edges of the reference's comparisons)."""
        n = C.c_uint64(0)
        self._check(lib().ngsd_deferred_stats(self._h, C.byref(n)))
        return n.value
