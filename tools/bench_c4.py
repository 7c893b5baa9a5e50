"""Called-genotype integer path (K2c k_dist_umma) at a C4-like shape; development / profiling helper.
   N_IND, N_SITES, PDEL (0/1), MISS, FORCE_FP64 (1 = reserved bit 1: run the same data through the FP64 contraction)."""
import os, sys, statistics, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import ngsdist_b200 as nb
n_ind, n_sites = int(os.environ.get("N_IND", 5000)), int(os.environ.get("N_SITES", 200000))
pdel = bool(int(os.environ.get("PDEL", 1)))
miss = float(os.environ.get("MISS", 0.05))
p = nb.Params(n_ind=n_ind, n_sites=n_sites, in_probs=True, call_geno=True, pairwise_del=pdel, evol_model=0,
              force_fp64=bool(int(os.environ.get("FORCE_FP64", 0))))
g = nb.NgsDistB200(p)
chunk = 4096
buf = torch.empty((chunk, n_ind, 3), dtype=torch.float64, device="cuda")
t0 = time.perf_counter()
fe = 0.0
for s0 in range(0, n_sites, chunk):
    m = min(chunk, n_sites - s0)
    g.synth_raw_device(buf.data_ptr(), 20251018, miss, s0, m)
    g.push_sites_device(buf.data_ptr(), s0, m)
    fe += g.timing().frontend_ms
g.frontend()
out = torch.empty((n_ind, n_ind), dtype=torch.float64).pin_memory()
ts, tc = [], []
for _ in range(4):
    g.distances_raw(None, 0, 1, out.data_ptr())
    t = g.timing()
    ts.append(t.dist_ms); tc.append(t.count_ms)
ps = n_ind * (n_ind - 1) // 2 * n_sites
t = g.timing()
best = min(ts)
print("called %dx%d pdel=%d: frontend %.1f ms (%.0f GB/s raw), dist %.2f ms (min %.2f), count %.2f ms, total %.2f ms -> %.3e pair-sites/s; IMMA %.1f TMAC/s executed"
      % (n_ind, n_sites, pdel, fe, n_ind * n_sites * 24 / fe * 1e-6, statistics.median(ts), best, statistics.median(tc), t.total_ms,
         ps / (best * 1e-3), t.dist_imma * 4096 / (best * 1e-3) * 1e-12))

# PACKED=1: end to end from HOST memory through ngsd_push_packed_genotypes (2-bit genotypes, 0.25 B per individual-site)
if int(os.environ.get("PACKED", 0)):
    import numpy as np
    g.close()
    stride = (n_ind + 3) // 4
    host = torch.empty((n_sites, stride), dtype=torch.uint8).pin_memory()
    blk = torch.from_numpy(np.random.RandomState(1).randint(0, 256, size=(min(n_sites, 65536), stride), dtype=np.uint8))
    for s0 in range(0, n_sites, blk.shape[0]):
        m = min(blk.shape[0], n_sites - s0)
        host[s0:s0 + m] = torch.roll(blk[:m], s0 // blk.shape[0], dims=1)
    pg = nb.Params(n_ind=n_ind, n_sites=n_sites, in_probs=False, indep_geno=True, pairwise_del=pdel, evol_model=0)
    for it in range(2):
        g2 = nb.NgsDistB200(pg)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        g2.push_packed_genotypes(host.numpy())
        g2.frontend()
        t1 = time.perf_counter()
        g2.distances_raw(None, 0, 1, out.data_ptr())
        t2 = time.perf_counter()
        g2.close()
    print("packed host input %dx%d pdel=%d (25 %% missing): %.1f MB pushed in %.1f ms (%.1f GB/s), distances + D2H %.1f ms, end to end %.1f ms -> %.3e pair-sites/s"
          % (n_ind, n_sites, pdel, host.numel() / 1e6, (t1 - t0) * 1e3, host.numel() / (t1 - t0) * 1e-9, (t2 - t1) * 1e3, (t2 - t0) * 1e3, ps / (t2 - t0)))
