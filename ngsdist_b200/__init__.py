"""ngsdist_b200: B200-native (sm_100a) implementation of ngsDist's pairwise-distance hot path.

The product is the C-ABI shared library `libngsdist_b200.so` (include/ngsdist_b200.h, sources in csrc/);
this package is a thin ctypes mirror of it for tests and bench.py.  There is no CPU fallback: importing
works without a GPU, but every compute entry point fails loudly when the library or a CUDA device is missing.
"""
from .api import (NgsDistError, Params, NgsDistB200, Timing, lib, lib_path, build_library, taus_block_counts, probe_fp64_tflops, probe_int8_tmacs, probe_umma_tmacs,
                  ABI_SYMBOLS, pack_genotypes, PLINK_BED_CODES, comm_unique_id, bind_host_to_device, SHARD_AUTO, SHARD_REPLICATED,
                  SHARD_SITES, BLANK_SITE, BLANK_SITE_CODE, pack_u20x3, XFER_F32, XFER_U32, XFER_U20X3, tree_support, TREE_NJ, TREE_BME)
from . import api

__all__ = ["tree_support", "NgsDistError", "Params", "NgsDistB200", "Timing", "lib", "lib_path", "build_library", "taus_block_counts",
           "probe_fp64_tflops", "probe_int8_tmacs", "probe_umma_tmacs", "ABI_SYMBOLS", "pack_genotypes", "PLINK_BED_CODES", "comm_unique_id", "bind_host_to_device",
           "SHARD_AUTO", "SHARD_REPLICATED", "SHARD_SITES", "TREE_NJ", "TREE_BME", "api"]
