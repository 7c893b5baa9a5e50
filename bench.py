#!/usr/bin/env python
"""bench.py -- pair-site evaluations per second of the ngsDist hot path on B200 (BASELINE.json metric).

Workload = BASELINE.json configs[2] "C3", the shape the north-star target is quoted on: synthetic GLs, 2 000 individuals
x 1 000 000 sites, 10 % missing, `--probs --indep_geno --pairwise_del`, bootstrap with `--boot_block_size 1000 --seed
12345`, every replicate contracted directly with its block-multiplicity weights (the graded diag(w_r) GEMMs, `reserved`
bit 2 -- not the block cache).  One step = one pass of the hot path over the data set:

    front end K1 (raw -> packed operands) -> REPS_PER_STEP bootstrap replicates (K3 counts + K2 weighted FP64 DMMA
    contraction + K4 epilogue each) -> the matrices in host memory on rank 0.

REPS_PER_STEP of the job's 100 replicates are run per step (a bounded sample; the per-replicate cost is constant, so the
job is 100 / REPS_PER_STEP steps plus replicate 0).  The total work per step is FIXED ("strong" scaling): with N ranks
(torchrun, one per GPU) replicate r runs on rank r % N inside ONE ngsd_distances_batch call and the matrices are
gathered on rank 0 by NCCL send/recv issued below the C ABI; the host RNG (gsl_rng_taus) advances identically on every
rank.  pair-sites are counted nominally: pairs x n_eff x replicates.

  value : raw GLs (48 GB) resident in HBM on every rank when the timed region starts; every rank runs the (HBM-bound,
          ~25 ms) front end on all sites itself -- cheaper than moving 96 GB of operands over NVLink.
  e2e   : the same step through the C ABI from HOST buffers: rank g pushes its 1/N of the sites from pinned memory over
          its own PCIe link (ngsd_push_sites), ONE NCCL all-gather of the packed operands (ngsd_comm_allgather_operands)
          makes them resident everywhere, then the same batch; matrices land in rank 0's host memory.
  c4_tiles / c5_sites (N > 1): the two other multi-GPU configs of BASELINE.json -- called genotypes with the output
          triangle tiles dealt to the ranks, and site shards with one NCCL reduce -- each with its collective's bytes and ms.
  --impl reference : the UNMODIFIED reference (oracle/_ref/ngsDist, built from /root/reference with the gsl_rng_taus
          shim) on the host cores, same flags, bounded sample of the C3 data set per step.
  --dump-outputs DIR : after the timed steps, DIR/dist.npy holds the distance matrices of the last timed step (see
          dump_outputs); inputs and bootstrap draws are seeded, so two builds run with the same arguments can be compared.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_IND = 2000
N_SITES = 1_000_000
MISS = 0.10
BLOCK = 1000
BOOT_SEED = 12345
REPS_PER_STEP = 16
SEED = 20251018
METRIC = "pair_site_evals_per_sec"
UNIT = "pair-sites/s"
WORKLOAD = ("C3: synthetic GL 2000 ind x 1M sites, 10% missing, --probs --indep_geno --pairwise_del, bootstrap block 1000 seed 12345, "
            "weighted contraction per replicate")
REF_FLAGS = ["--probs", "--indep_geno", "--pairwise_del", "--boot_block_size", str(BLOCK), "--seed", str(BOOT_SEED)]
DUMP_BYTES = 48 << 20       # --dump-outputs stays under 64 MB
DUMP_SEED = 7


def pairs(n):
    return n * (n - 1) // 2


def dump_outputs(path, mats):
    """Write mats [replicate][n_ind][n_ind] (float64, the matrices a caller of ngsd_distances_batch receives) to
    path/dist.npy: whole when they fit DUMP_BYTES, otherwise as [replicate][k], the same k entries of every matrix,
    drawn once with DUMP_SEED and kept in row-major order (the same entries on every run of the same shape)."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    R, n, _ = mats.shape
    flat = mats.reshape(R, n * n)
    if flat.nbytes > DUMP_BYTES:
        k = DUMP_BYTES // (8 * R)
        idx = np.sort(np.random.default_rng(DUMP_SEED).choice(n * n, size=k, replace=False))
        flat = flat[:, idx]
    np.save(os.path.join(path, "dist.npy"), np.ascontiguousarray(flat, dtype=np.float64))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(",")]
            if len(f) >= 8:
                self.rows.append(f)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        num = lambda x: x.replace(".", "").isdigit()
        sm = [float(r[1]) for r in self.rows if num(r[1])]
        mx = [float(r[2]) for r in self.rows if num(r[2])]
        pw = [float(r[3]) for r in self.rows if num(r[3])]
        busy = [s for s, p in zip(sm, pw) if p > 350.0] or sm          # samples under load
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(r[4 + k] == "Active" for r in self.rows)]
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "power_w_max": max(pw) if pw else None, "samples": len(self.rows)}


# ------------------------------------------------------------------------------------------------ reference arm --

def run_reference_sample(n_ind, n_sites, n_rep, threads, workdir):
    """Hot-path seconds of the unmodified reference on the first n_sites sites of the C3 data set, replicate 0 plus n_rep
    bootstrap replicates: whole-process wall time minus a load-only run of the same file read as 2 individuals (same
    reader work, 1 pair)."""
    import oracle
    path = os.path.join(workdir, "ref_%dx%d.bin" % (n_ind, n_sites))
    if not os.path.exists(path):
        oracle.synth_raw(SEED, MISS, n_ind, n_sites).tofile(path)

    def run(ni, ns, reps):
        out = os.path.join(workdir, "ref.dist")
        cmd = [oracle.REF_BIN, "--geno", path, "--n_ind", str(ni), "--n_sites", str(ns), "--out", out, "--n_threads", str(threads),
               "--verbose", "0", "--n_boot_rep", str(reps)] + REF_FLAGS
        t0 = time.perf_counter()
        subprocess.run(cmd, check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        return time.perf_counter() - t0

    wall = run(n_ind, n_sites, n_rep)
    load = run(2, n_ind * n_sites // 2, 0)
    return max(wall - load, 1e-6), wall, load


def reference_arm(args, rank):
    import oracle
    if rank != 0:
        return
    if not oracle.have_ref():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/ngsDist not built (needs /root/reference at build time)"}))
        return
    threads = os.cpu_count() or 1
    work = tempfile.mkdtemp(prefix="ngsd_bench_ref_")
    # Size the per-step sample so that the whole run stays within a few minutes.  The reference does ~10^8 pair-sites/s on a
    # host at this shape (one heap object per individual-site: DRAM latency bound), a C3 replicate is 2 * 10^12, so a step is a
    # sample: replicate 0 + 1 bootstrap replicate on the first `sites` sites (whole 1000-site blocks) of the first `ni`
    # individuals.  Calibrate on a small case, then take the largest sample that fits the per-step budget.
    hot, _, _ = run_reference_sample(500, BLOCK, 1, threads, work)
    rate = pairs(500) * BLOCK * 2 / hot
    budget_s = 200.0
    per_step = 0.55 * budget_s / (args.steps + args.warmup)
    ni, sites = 250, BLOCK
    for cand in (2000, 1000, 500):
        if pairs(cand) * BLOCK * 2 / rate <= per_step:
            ni = cand
            sites = int(min(10, per_step * rate / (pairs(cand) * BLOCK * 2))) * BLOCK
            break
    for _ in range(args.warmup):
        run_reference_sample(ni, sites, 1, threads, work)
    hots = []
    for _ in range(args.steps):
        hot, wall, load = run_reference_sample(ni, sites, 1, threads, work)
        hots.append(hot)
    total = sum(hots)
    value = pairs(ni) * sites * 2 * args.steps / total
    sample = ("the first %d individuals x the first %d sites of the C3 generator, replicate 0 + 1 bootstrap replicate per step (the full shape "
              "needs 96 GB of heap and weeks on these cores); whole-process wall minus a load-only run of the same file" % (ni, sites))
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total / args.steps * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "impl": "reference",
            "config": {"workload": WORKLOAD, "sample_individuals": ni, "sample_sites": sites, "sample_matrices": 2, "threads": threads,
                       "sampled": "pair-sites/s of the reference does not grow with the shape; the full shape cannot run on the reference at all"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "reference", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------ our arm --

def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--core-only", action="store_true", help="skip the extras (profiling runs)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--n-ind", type=int, default=N_IND)
    ap.add_argument("--n-sites", type=int, default=N_SITES)
    ap.add_argument("--reps", type=int, default=REPS_PER_STEP)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the distance matrices of the last timed step to DIR/dist.npy")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        reference_arm(args, rank)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    import ngsdist_b200 as nb
    from ngsdist_b200 import multi

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    numa_node = nb.bind_host_to_device(local)       # this rank's CPU threads and pinned pages next to its GPU
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    n_ind, n_sites, R = args.n_ind, args.n_sites, args.reps
    W = max(args.warmup, 3)
    full_shape = (n_ind, n_sites) == (N_IND, N_SITES)
    n_blocks = n_sites // BLOCK
    n_eff = n_blocks * BLOCK

    def share_id():
        box = [nb.comm_unique_id() if rank == 0 else None]
        if world > 1:
            dist.broadcast_object_list(box, src=0)
        return box[0]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    p = nb.Params(n_ind=n_ind, n_sites=n_sites, in_probs=True, indep_geno=True, pairwise_del=True, evol_model=1, n_boot_rep=100,
                  boot_block_size=BLOCK, seed=BOOT_SEED, no_block_cache=True)
    g = nb.NgsDistB200(p, device=local)
    if world > 1:
        g.comm_attach(share_id(), rank, world)
    stream = torch.cuda.ExternalStream(g.stream(), device=torch.device("cuda", local))
    # resident input: the raw GLs of all sites, generated on the device chunk by chunk (SURVEY §8(d) generator)
    raw_dev = torch.empty((n_sites, n_ind, 3), dtype=torch.float64, device="cuda")
    GEN = 65536
    for s0 in range(0, n_sites, GEN):
        g.synth_raw_device(raw_dev[s0:].data_ptr(), SEED, MISS, s0, min(GEN, n_sites - s0))
    out_pin = torch.empty((R, n_ind, n_ind), dtype=torch.float64, pin_memory=True) if rank == 0 else None
    out_ptr = out_pin.data_ptr() if rank == 0 else None
    boot = multi.BootStream(n_sites, BLOCK, BOOT_SEED)       # host RNG: identical on every rank

    launches = [0]
    acc = {"dist_ms": 0.0, "count_ms": 0.0, "epi_ms": 0.0, "fe_ms": 0.0, "dmma": 0, "reps": 0, "comm_ms": 0.0, "comm_bytes": 0}

    def draw_counts():
        return np.stack([boot.next_counts() for _ in range(R)])

    def batch(counts):
        g._check(nb.lib().ngsd_distances_batch(g._h, counts.ctypes.data, R, n_blocks, BLOCK, out_ptr))
        t = g.timing()
        acc["dist_ms"] += t.dist_ms; acc["count_ms"] += t.count_ms; acc["epi_ms"] += t.epilogue_ms; acc["dmma"] += t.dist_dmma
        acc["reps"] += len(range(rank, R, world))
        launches[0] += t.launches
        if world > 1:
            b, ms = g.comm_stats()
            acc["comm_ms"] += ms; acc["comm_bytes"] += b

    def step_resident():
        counts = draw_counts()
        g.push_sites_device(raw_dev.data_ptr(), 0, n_sites)
        acc["fe_ms"] += g.timing().frontend_ms
        launches[0] += 1
        batch(counts)

    def timed(fn, steps):
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(stream)
        for _ in range(steps):
            fn()
        e1.record(stream)
        barrier()
        return max_over_ranks(e0.elapsed_time(e1))

    for _ in range(W):
        step_resident()
    launches[0] = 0
    for k in acc:
        acc[k] = 0
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_total = timed(step_resident, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out_pin.numpy())          # before the e2e steps below reuse out_pin
    n_launch = launches[0]
    res = dict(acc)
    tim = g.timing()

    # ---- e2e: host buffers through the C ABI; every rank pushes its own 1/N of the sites ----
    e2e = None
    if not args.no_e2e:
        align = 64
        sb = [n_sites // align * r // world * align for r in range(world)] + [n_sites]
        my0, my1 = sb[rank], sb[rank + 1]
        raw_pin = torch.empty((my1 - my0, n_ind, 3), dtype=torch.float64, pin_memory=True)
        raw_pin.copy_(raw_dev[my0:my1])
        del raw_dev
        torch.cuda.empty_cache()
        h2d = {"ms": 0.0, "bytes": 0}

        def step_e2e():
            counts = draw_counts()
            t0 = time.perf_counter()
            g.push_sites_ptr(raw_pin.data_ptr(), my0, my1 - my0)
            h2d["ms"] += (time.perf_counter() - t0) * 1e3
            h2d["bytes"] += raw_pin.numel() * 8
            if world > 1:
                g.comm_allgather_operands(sb)
            batch(counts)

        step_e2e()
        for k in acc:
            acc[k] = 0
        h2d = {"ms": 0.0, "bytes": 0}
        e2e_steps = max(2, min(args.steps, 3))
        ms_e2e = timed(step_e2e, e2e_steps)
        h2d_gbs = h2d["bytes"] / max(h2d["ms"], 1e-9) * 1e-6
        all_gbs = None
        if world > 1:
            t = torch.tensor([h2d_gbs], device="cuda", dtype=torch.float64)
            lst = [torch.zeros_like(t) for _ in range(world)]
            dist.all_gather(lst, t)
            all_gbs = [round(float(x.item()), 2) for x in lst]
        e2e = {"value": pairs(n_ind) * n_eff * R * e2e_steps / (ms_e2e * 1e-3), "unit": UNIT,
               "h2d_bytes_per_step": n_sites * n_ind * 24, "d2h_bytes_per_step": R * n_ind * n_ind * 8,
               "ms_per_step": ms_e2e / e2e_steps, "steps": e2e_steps,
               "h2d_gbs_per_rank": all_gbs if all_gbs else [round(h2d_gbs, 2)], "h2d_ms_per_step_rank0": h2d["ms"] / e2e_steps,
               "numa_node_rank0": numa_node,
               "path": "pinned host raw (1/N of the sites per rank) -> ngsd_push_sites -> " +
                       ("ngsd_comm_allgather_operands (NCCL) -> " if world > 1 else "") + "ngsd_distances_batch -> host matrices on rank 0"}
        del raw_pin
    else:
        del raw_dev
    peak = nb.probe_fp64_tflops(local) if rank == 0 else None
    g.close()
    torch.cuda.empty_cache()

    extras = {}
    if not args.core_only and full_shape:
        if world == 1:
            extras = single_gpu_extras(nb, torch, np, local, multi)
        else:
            extras = multi_gpu_extras(nb, torch, np, dist, multi, rank, world, local, share_id, barrier, max_over_ranks)

    units_step = pairs(n_ind) * n_eff * R                 # nominal pair-site evaluations per step, whole job
    value = units_step * args.steps / (ms_total * 1e-3)

    if rank == 0:
        traffic = None
        try:
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as fh:
                tr = json.load(fh)["k_dist_dmma_c3_weighted"]
            if full_shape:
                traffic = tr["dram_bytes_read"] + tr["dram_bytes_write"]
        except Exception:
            pass
        # SURVEY §8(d) accounting rule: roofline.achieved = FP64 tensor FLOP/s EXECUTED by the kernel (DMMA.8x8x4 count x 512
        # FLOP, diagonal-tile waste included, zero-weight chunks excluded) against the measured DMMA issue peak; `useful` =
        # nominal pair-sites x 6 FLOP (3 FMA per pair-site, ngsDist.cpp:351-353) over the same kernel time.
        reps_rank0 = max(res["reps"], 1)
        kernel_ms = res["dist_ms"] / reps_rank0
        executed = res["dmma"] * 512.0 / (res["dist_ms"] * 1e-3) * 1e-12
        useful = 6.0 * pairs(n_ind) * n_eff * reps_rank0 / (res["dist_ms"] * 1e-3) * 1e-12
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": W,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": WORKLOAD if full_shape else "synthetic GL %d x %d, C3 flags" % (n_ind, n_sites),
                       "n_ind": n_ind, "n_sites": n_sites, "pairs": pairs(n_ind), "replicates_per_step": R, "job_replicates": 100,
                       "extrapolation": "a step runs %d of the job's 100 bootstrap replicates (constant cost per replicate); job = 100/%d steps + replicate 0" % (R, R),
                       "l2": "inputs_larger_than_l2 (48 GB raw, 2 x 48 GB packed operands)",
                       "sharding": "replicate r on rank r % N inside ngsd_distances_batch; matrices gathered on rank 0 by NCCL send/recv below the C ABI"
                                   if world > 1 else "single GPU",
                       "timed": "front end on all sites (every rank) + %d weighted replicates (counts + contraction + epilogue) + gather + D2H of the matrices" % R},
            "clocks": clocks,
            "gpu_launches": n_launch,
            "step_share_rank0_ms": {"frontend": res["fe_ms"] / args.steps, "contraction": res["dist_ms"] / args.steps,
                                    "mask_count_overlapped": res["count_ms"] / args.steps, "epilogue": res["epi_ms"] / args.steps,
                                    "gather_nccl": res["comm_ms"] / args.steps, "step": ms_total / args.steps},
            "collective": {"kind": "ncclSend/ncclRecv gather of the replicate matrices to rank 0" if world > 1 else None,
                           "bytes_per_step_rank0": res["comm_bytes"] / args.steps, "ms_per_step_rank0": res["comm_ms"] / args.steps},
            "roofline": {"bound": "tensor", "kernel": "k_dist_dmma<weighted, 3 planes> (FP64 DMMA.8x8x4 contraction)", "achieved": executed, "peak": peak,
                         "unit": "TFLOP/s", "frac": executed / peak, "traffic": traffic,
                         "traffic_note": "DRAM bytes read+written by one weighted k_dist_dmma launch at C3 (ncu --set full, profiles/); active operands ~61 GB",
                         "peak_source": "live DMMA.8x8x4 issue-rate probe in this run (MEASURED_PEAKS.json has no FP64 figure; cuBLAS Dgemm measured 35.5)",
                         "executed_flops_per_launch": res["dmma"] * 512.0 / reps_rank0, "kernel_ms": kernel_ms,
                         "useful_tflops_at_6flop_per_pair_site": useful, "useful_frac": useful / peak,
                         "note": "achieved = executed DMMA FLOP/s; chunks whose bootstrap weight is 0 (~37 % per replicate) are skipped, so "
                                 "`useful` (nominal pair-sites x 6 FLOP) exceeds `achieved` and is not a roofline fraction"},
        }
        if e2e is not None:
            line["e2e"] = e2e
        line.update(extras)
        if world == 1 and not args.no_cpu_baseline:
            import oracle
            if oracle.have_ref():
                threads = os.cpu_count() or 1
                work = tempfile.mkdtemp(prefix="ngsd_bench_cpu_")
                sites = BLOCK
                hot, wall, load = run_reference_sample(N_IND, sites, 1, threads, work)
                line["cpu_baseline"] = {"value": pairs(N_IND) * sites * 2 / hot, "unit": UNIT, "cores": threads, "kind": "reference",
                                        "sample": "oracle/_ref/ngsDist --n_threads %d, C3 flags, %d ind x the first %d sites, replicate 0 + 1 bootstrap "
                                                  "replicate: %.1f s wall - %.1f s load-only" % (threads, N_IND, sites, wall, load)}
            else:
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "reference", "sample": "oracle/_ref/ngsDist missing"}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------- extras ----

def single_gpu_extras(nb, torch, np, local, multi):
    """The other contractions of gen_dist on one GPU: C2 through the sum-to-one FP64 contraction and through the per
    pair-site EM (the reference's literal default), the called-genotype int8 path at the C4 geometry, and the bootstrap
    block cache next to the weighted contraction."""
    out = {}
    # ---- C2 (BASELINE configs[1]): 500 x 100 000, --evol_model 2; with --indep_geno (2-plane DMMA) and without (EM) ----
    n, s = 500, 100_000
    raw = torch.empty((s, n, 3), dtype=torch.float64, device="cuda")
    res = {}
    for name, indep in (("indep_geno", True), ("em_default", False)):
        gq = nb.NgsDistB200(nb.Params(n_ind=n, n_sites=s, in_probs=True, indep_geno=indep, evol_model=2), device=local)
        if name == "indep_geno":
            gq.synth_raw_device(raw.data_ptr(), SEED, 0.0, 0, s)
        o = torch.empty((n, n), dtype=torch.float64, pin_memory=True)
        ms, kms, fe = [], [], []
        for it in range(5):
            gq.push_sites_device(raw.data_ptr(), 0, s)
            f = gq.timing().frontend_ms
            gq.distances_raw(None, 0, 1, o.data_ptr())
            t = gq.timing()
            if it >= 2:
                ms.append(f + t.total_ms); kms.append(t.dist_ms); fe.append(f)
        res[name] = {"ms_per_matrix": statistics.median(ms), "kernel_ms": statistics.median(kms), "frontend_ms": statistics.median(fe),
                     "value": pairs(n) * s / (statistics.median(ms) * 1e-3), "unit": UNIT}
        if indep:
            res[name]["frontend_gbs_algorithmic_48B"] = n * s * 48 / (statistics.median(fe) * 1e-3) * 1e-9
        gq.close()
    # ---- transport tiers on C2 (VERDICT r1 item 8): the same matrix end to end from host memory, 24 B vs 8 B per individual-site ----
    try:
        pz = raw / raw.sum(dim=2, keepdim=True)
        q = torch.round(pz * 1e6).to(torch.int64)                         # 6-decimal posteriors (what ANGSD -doGeno 8 prints)
        # the doubles a text reader gets from them: the IEEE quotient (a 0-dim CUDA divisor -- torch turns a division by a
        # Python scalar into a multiplication by its reciprocal, which is not the same double)
        dec = q.to(torch.float64) / torch.tensor(1e6, dtype=torch.float64, device="cuda")
        packed = (q[..., 0] | (q[..., 1] << 20) | (q[..., 2] << 40)).contiguous()
        h_dec = torch.empty(dec.shape, dtype=torch.float64, pin_memory=True); h_dec.copy_(dec)
        h_pk = torch.empty(packed.shape, dtype=torch.int64, pin_memory=True); h_pk.copy_(packed)
        del pz, q, dec, packed
        tiers = {}
        mats = {}
        for name in ("f64", "u20x3"):
            gt = nb.NgsDistB200(nb.Params(n_ind=n, n_sites=s, in_probs=True, indep_geno=True, evol_model=2, in_text=True), device=local)
            o = torch.empty((n, n), dtype=torch.float64, pin_memory=True)
            best = None
            for it in range(5):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                if name == "f64":
                    gt.push_sites_ptr(h_dec.data_ptr(), 0, s)
                else:
                    gt.push_sites_packed_ptr(h_pk.data_ptr(), nb.XFER_U20X3, 1e6, 0, s)
                gt.distances_raw(None, 0, 1, o.data_ptr())
                dt = time.perf_counter() - t0
                if it >= 2:
                    best = dt if best is None else min(best, dt)
            mats[name] = o.clone()
            tiers[name] = {"ms": best * 1e3, "h2d_bytes": n * s * (24 if name == "f64" else 8), "value": pairs(n) * s / best, "unit": UNIT}
            gt.close()
        tiers["bit_identical"] = bool(torch.equal(mats["f64"], mats["u20x3"]))
        res["e2e_transport"] = {"workload": "C2 from pinned host memory, 6-decimal posteriors: doubles vs 3 x 20-bit fixed point (ngsd_push_sites_packed)", **tiers}
        del h_dec, h_pk
    except Exception as ex:
        res["e2e_transport"] = {"error": str(ex)[:200]}
    del raw
    out["c2"] = {"workload": "C2: 500 ind x 100k sites, --probs --evol_model 2: with --indep_geno (2-plane DMMA contraction) and the literal default "
                             "(per pair-site EM, emOptim2.cpp em2, kernel k_dist_em); front end + contraction + epilogue, device time", **res}
    # ---- called genotypes, C4 geometry at 1/50 of the sites ----
    cn, cs = 5000, 100_000
    called = {}
    for pdel in (False, True):
        gc = nb.NgsDistB200(nb.Params(n_ind=cn, n_sites=cs, in_probs=True, call_geno=True, pairwise_del=pdel, evol_model=0), device=local)
        chunk = 4096
        buf = torch.empty((chunk, cn, 3), dtype=torch.float64, device="cuda")
        fe_ms = 0.0
        for s0 in range(0, cs, chunk):
            m = min(chunk, cs - s0)
            gc.synth_raw_device(buf.data_ptr(), SEED, 0.05, s0, m)
            gc.push_sites_device(buf.data_ptr(), s0, m)
            fe_ms += gc.timing().frontend_ms
        del buf
        gc.frontend()
        oc = torch.empty((cn, cn), dtype=torch.float64, pin_memory=True)
        gc.distances_raw(None, 0, 1, oc.data_ptr())
        c_ms = []
        for _ in range(3):
            gc.distances_raw(None, 0, 1, oc.data_ptr())
            tc = gc.timing()
            c_ms.append(tc.dist_ms)
        k_ms = statistics.median(c_ms)
        row = {"kernel_ms": k_ms, "value": pairs(cn) * cs / (k_ms * 1e-3), "unit": UNIT}
        if not pdel:
            peak = nb.probe_umma_tmacs(local)
            exe = tc.dist_imma * 4096.0 / (k_ms * 1e-3) * 1e-12
            row.update({"frontend_ms": fe_ms, "frontend_gbs_raw": cn * cs * 24 / (fe_ms * 1e-3) * 1e-9,
                        "roofline": {"bound": "tensor", "kernel": "k_dist_umma (tcgen05.mma kind::i8, UTCIMMA)", "achieved": exe, "peak": peak,
                                     "unit": "TMAC/s", "frac": exe / peak, "peak_source": "live back-to-back tcgen05.mma 128x128x32 issue-rate probe in this run",
                                     "note": "achieved = executed int8 MACs (3 K bytes per site since round 2, 4 before); the kernel is bound by the shared-memory pipe (DESIGN.md section 3)"}})
        called["pairwise_del" if pdel else "no_pairwise_del"] = row
        gc.close()
        del oc
    out["called_path"] = {"workload": "C4 geometry at 1/50 of the sites: 5000 ind x 100k sites, 5 % missing, --call_geno (integer path, bit-exact)", **called}
    # ---- the bootstrap block cache (effective throughput) next to the weighted contraction of the headline ----
    bn, bsites = 2000, 100_000
    gb = nb.NgsDistB200(nb.Params(n_ind=bn, n_sites=bsites, in_probs=True, indep_geno=True, pairwise_del=True, evol_model=1, n_boot_rep=4,
                                  boot_block_size=BLOCK, seed=BOOT_SEED), device=local)
    buf = torch.empty((8192, bn, 3), dtype=torch.float64, device="cuda")
    for s0 in range(0, bsites, 8192):
        m = min(8192, bsites - s0)
        gb.synth_raw_device(buf.data_ptr(), SEED, MISS, s0, m)
        gb.push_sites_device(buf.data_ptr(), s0, m)
    del buf
    gb.frontend()
    ob = torch.empty((bn, bn), dtype=torch.float64, pin_memory=True)
    ms = []
    for rep in range(4):
        counts, bs_ = gb.next_boot_counts()
        gb.distances_raw(counts.ctypes.data, len(counts), bs_, ob.data_ptr())
        tb = gb.timing()
        ms.append((tb.total_ms, tb.block_cache))
    gb.close()
    steady = [m for m, flag in ms if flag != 1]
    out["bootstrap_block_cache"] = {"workload": "C3 geometry at 1/10 of the sites, per-block partials contracted once, every replicate a weighted split reduction",
                                    "first_call_ms": ms[0][0], "ms_per_replicate": statistics.median(steady),
                                    "value": pairs(bn) * bsites / (statistics.median(steady) * 1e-3), "unit": UNIT,
                                    "note": "effective throughput; the headline and its roofline are the weighted contraction"}
    return out


def multi_gpu_extras(nb, torch, np, dist, multi, rank, world, local, share_id, barrier, max_over_ranks):
    """BASELINE configs[3] and [4] on N ranks, every collective issued by the library (NCCL below the C ABI)."""
    out = {}
    dev = torch.device("cuda", local)

    def span(stream, fn):
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(stream)
        fn()
        e1.record(stream)
        barrier()
        return max_over_ranks(e0.elapsed_time(e1))

    # ---- C4: called genotypes 5 000 x 5 000 000, site-sharded front end -> all-gather of the 2-bit codes -> tiles dealt to the ranks ----
    cn, cs = 5000, 5_000_000
    sb = [cs // 64 * r // world * 64 for r in range(world)] + [cs]
    my0, my1 = sb[rank], sb[rank + 1]
    gc = nb.NgsDistB200(nb.Params(n_ind=cn, n_sites=cs, in_probs=True, call_geno=True, pairwise_del=True, evol_model=0), device=local)
    gc.comm_attach(share_id(), rank, world)
    st = torch.cuda.ExternalStream(gc.stream(), device=dev)
    chunk = 8192
    buf = torch.empty((chunk, cn, 3), dtype=torch.float64, device="cuda")
    fe_ms = 0.0
    for s0 in range(my0, my1, chunk):                     # 600 GB of raw GLs never exist at once: generated per chunk on the device
        m = min(chunk, my1 - s0)
        gc.synth_raw_device(buf.data_ptr(), SEED, 0.05, s0, m)
        gc.push_sites_device(buf.data_ptr(), s0, m)
        fe_ms += gc.timing().frontend_ms
    del buf
    ag_first_ms = span(st, lambda: gc.comm_allgather_operands(sb))      # first exchange on this communicator
    ag_ms = span(st, lambda: gc.comm_allgather_operands(sb))            # steady state (same bytes again)
    ag_bytes = gc.comm_stats()[0]
    gc.set_tile_shard(rank, world)
    oc = torch.empty((cn, cn), dtype=torch.float64, pin_memory=True) if rank == 0 else None
    optr = oc.data_ptr() if rank == 0 else None

    def c4_matrix():
        gc.partial_sums()
        gc._check(nb.lib().ngsd_comm_reduce_tiles(gc._h, 0, 0, optr, None, None))

    c4_matrix()
    ms = [span(st, c4_matrix) for _ in range(3)]
    k_ms = max_over_ranks(gc.timing().dist_ms)
    rb, rms = gc.comm_stats()
    fe_max = max_over_ranks(fe_ms)
    tot = fe_max + ag_ms + statistics.median(ms)
    out["c4_tiles"] = {"workload": "C4: called genotypes 5000 ind x 5M sites, 5 %% missing, --call_geno --pairwise_del (int8 tcgen05 path, bit-exact), "
                                   "site-sharded front end + NCCL all-gather of the 2-bit codes, output-triangle tiles dealt to %d ranks, NCCL assembly on rank 0" % world,
                       "frontend_ms_max_rank": fe_max, "allgather_ms": ag_ms, "allgather_first_call_ms": ag_first_ms, "allgather_bytes_per_rank": ag_bytes,
                       "matrix_ms": statistics.median(ms), "contraction_ms_max_rank": k_ms, "assembly_bytes": rb, "assembly_ms_rank0": rms,
                       "total_ms": tot, "value": pairs(cn) * cs / (tot * 1e-3), "value_matrix_only": pairs(cn) * cs / (statistics.median(ms) * 1e-3), "unit": UNIT}
    gc.close()
    del oc
    torch.cuda.empty_cache()

    # ---- C5 geometry: 20 000 individuals, --avg_nuc_dist --indep_geno, sites sharded, ONE reduce of the packed upper triangle ----
    n5, s5 = 20000, 10_000_000 // 64
    shards = multi.site_shards(s5, 64, world)
    l0, l1 = shards[rank]
    g5 = nb.NgsDistB200(nb.Params(n_ind=n5, n_sites=l1 - l0, in_probs=True, indep_geno=True, avg_nuc_dist=True, evol_model=1), device=local)
    g5.comm_attach(share_id(), rank, world)
    st = torch.cuda.ExternalStream(g5.stream(), device=dev)
    chunk = 2048
    buf = torch.empty((chunk, n5, 3), dtype=torch.float64, device="cuda")
    fe_ms = 0.0
    for s0 in range(l0, l1, chunk):
        m = min(chunk, l1 - s0)
        g5.synth_raw_device(buf.data_ptr(), SEED, 0.0, s0, m)
        g5.push_sites_device(buf.data_ptr(), s0 - l0, m)
        fe_ms += g5.timing().frontend_ms
    del buf
    o5 = torch.empty((n5, n5), dtype=torch.float64, pin_memory=True) if rank == 0 else None
    o5p = o5.data_ptr() if rank == 0 else None
    parts = {"dist": 0.0}

    def c5_matrix():
        g5.partial_sums()
        parts["dist"] = g5.timing().total_ms
        g5._check(nb.lib().ngsd_comm_reduce_sites(g5._h, 0, s5, o5p))

    c5_matrix()
    ms = [span(st, c5_matrix) for _ in range(2)]
    rb, rms = g5.comm_stats()
    k_ms = max_over_ranks(parts["dist"])
    out["c5_sites"] = {"workload": "C5 geometry at 1/64 of the sites: 20000 ind x %d sites, --avg_nuc_dist --indep_geno, sites sharded over %d ranks, "
                                   "ONE ncclReduce of the packed upper triangle of num (cnt is a constant without --pairwise_del), epilogue on the root" % (s5, world),
                       "matrix_ms": statistics.median(ms), "partial_sums_ms_max_rank": k_ms, "frontend_ms_max_rank": max_over_ranks(fe_ms),
                       "reduce_bytes": rb, "reduce_ms_rank0": rms, "full_num_cnt_matrices_bytes": n5 * n5 * 16,
                       "value": pairs(n5) * s5 / (statistics.median(ms) * 1e-3), "unit": UNIT}
    g5.close()
    return out


if __name__ == "__main__":
    main()
