// Multi-GPU layer of libngsdist_b200.so (SURVEY §8e, §2.1 rows C1 / C2): everything a box of B200s needs sits below the
// C ABI, linked against NCCL directly.
//
// The reference has ONE parallel strategy: a task per pair of individuals through a pthread pool in one address space
// (ngsDist.cpp:197-269, gen_dist_slave :408-412).  At box level the path shards three ways instead:
//   replicates : ngsd_distances_batch deals bootstrap replicate r to GPU r % N (the replicate loop ngsDist.cpp:217-289)
//   tiles      : ngsd_distances on REPLICATED data deals the upper-triangle tiles of one matrix to the GPUs
//   sites      : every GPU contracts its own site range; ONE ncclReduce of the packed upper triangle of num (and of cnt
//                only under --pairwise_del), then the non-linear tail of gen_dist (ngsDist.cpp:372-401) on the root.
// Two ways to get there share the code below:
//   * ngsd_cfg.n_gpus > 1  -- one process: the "group" context owns one ordinary context per GPU ("kids") and one host
//                             thread per GPU for the calls that block; NCCL communicators from ncclCommInitAll;
//   * ngsd_comm_attach     -- one process per GPU (torchrun, MPI ...): ncclCommInitRank from a 128-byte id.
#include <nccl.h>
#include <sched.h>
#include <stdlib.h>
#include <sys/syscall.h>
#include <unistd.h>

#include <algorithm>
#include <new>
#include <numeric>
#include <string>
#include <thread>

#include "ngsd_internal.h"

#define NGSD_NCCL(ctx, call)                                                                              \
  do {                                                                                                    \
    ncclResult_t r_ = (call);                                                                             \
    if (r_ != ncclSuccess) {                                                                              \
      ngsd_set_error((ctx), "NCCL error: %s (%s:%d: %s)", ncclGetErrorString(r_), __FILE__, __LINE__, #call); \
      return NGSD_ERR_COMM;                                                                               \
    }                                                                                                     \
  } while (0)

namespace {

// packed upper triangle: pair (i < j) at i (n - 1) - i (i - 1) / 2 + (j - i - 1)
__device__ __forceinline__ uint64_t tri_index(uint64_t i, uint64_t j, uint64_t n) { return i * (n - 1) - i * (i - 1) / 2 + (j - i - 1); }

template <typename T>
__global__ void k_tri_pack(const T *__restrict__ full, uint64_t n, T *__restrict__ tri) {
  const uint64_t idx = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n * n) return;
  const uint64_t i = idx / n, j = idx - i * n;
  if (i < j) tri[tri_index(i, j, n)] = full[idx];
}

template <typename T>
__global__ void k_tri_unpack(const T *__restrict__ tri, uint64_t n, T *__restrict__ full) {
  const uint64_t idx = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n * n) return;
  const uint64_t i = idx / n, j = idx - i * n;
  if (i == j) full[idx] = (T) 0;
  else full[idx] = tri[i < j ? tri_index(i, j, n) : tri_index(j, i, n)];
}

// error / information bits of the front end (ngsd_ctx::d_err) as one int per bit, so that a max-reduce is a bitwise OR
__global__ void k_flags_split(const int *err, int *bits) { if (threadIdx.x < 8) bits[threadIdx.x] = (*err >> threadIdx.x) & 1; }
__global__ void k_flags_merge(int *err, const int *bits) {
  if (threadIdx.x == 0) {
    int v = 0;
    for (int b = 0; b < 8; b++) v |= (bits[b] ? 1 : 0) << b;
    *err |= v;
  }
}

ncclComm_t comm_of(const ngsd_ctx *c) { return (ncclComm_t) c->comm; }

int ensure_events(ngsd_ctx *c) {
  for (auto &e : c->ev_comm)
    if (!e) NGSD_CUDA(c, cudaEventCreate(&e));
  return NGSD_OK;
}

int ensure_tri(ngsd_ctx *c, uint64_t elems) {
  if (c->tri_cap >= elems) return NGSD_OK;
  cudaFree(c->d_tri);
  c->d_tri = nullptr;
  c->tri_cap = 0;
  NGSD_CUDA(c, cudaMalloc((void **) &c->d_tri, std::max<uint64_t>(elems, 1) * sizeof(double)));
  c->tri_cap = elems;
  return NGSD_OK;
}

int ensure_gather(ngsd_ctx *c, uint64_t elems) {
  if (c->gather_cap >= elems) return NGSD_OK;
  cudaFree(c->d_gather);
  c->d_gather = nullptr;
  c->gather_cap = 0;
  NGSD_CUDA(c, cudaMalloc((void **) &c->d_gather, std::max<uint64_t>(elems, 1) * sizeof(double)));
  c->gather_cap = elems;
  return NGSD_OK;
}

void finish_stats(ngsd_ctx *c, uint64_t bytes) {
  float ms = 0.f;
  if (cudaEventElapsedTime(&ms, c->ev_comm[0], c->ev_comm[1]) != cudaSuccess) ms = 0.f;
  c->comm_ms = ms;
  c->comm_bytes = bytes;
}

// ------------------------------------------------------------------------------------------ collectives ----
// Every function takes the local participants: one context per process (ngsd_comm_attach) or all kids of a group; the
// NCCL calls of all local participants go into one ncclGroupStart / ncclGroupEnd.

// Row C1: site shards -> raw sums on `root` -> tail of gen_dist there.
int reduce_sites_impl(ngsd_ctx *err_to, const std::vector<ngsd_ctx *> &cs, uint32_t root, uint64_t n_eff_total, double *out_host,
                      double *num_opt, uint64_t *cnt_opt) {
  const uint64_t n = cs[0]->n_ind, n2 = n * n, tri = n * (n - 1) / 2;
  const bool with_cnt = cs[0]->cfg.pairwise_del != 0;
  const unsigned blocks = (unsigned) ((n2 + 255) / 256);
  for (ngsd_ctx *c : cs) {
    if (!c->comm) { ngsd_set_error(err_to, "no communicator: call ngsd_comm_attach first"); return NGSD_ERR_COMM; }
    if (!c->d_out) { ngsd_set_error(err_to, "no partial sums yet: call ngsd_distances(out = NULL) first"); return NGSD_ERR_STATE; }
    NGSD_CUDA(err_to, cudaSetDevice(c->device));
    int rc = ensure_tri(c, tri);
    if (!rc) rc = ensure_events(c);
    if (rc) { if (c != err_to) ngsd_set_error(err_to, "%s", c->err); return rc; }
    NGSD_CUDA(err_to, cudaEventRecord(c->ev_comm[0], c->stream));
    k_tri_pack<double><<<blocks, 256, 0, c->stream>>>(c->d_num, n, c->d_tri);
    NGSD_CUDA(err_to, cudaGetLastError());
  }
  NGSD_NCCL(err_to, ncclGroupStart());
  for (ngsd_ctx *c : cs) NGSD_NCCL(err_to, ncclReduce(c->d_tri, c->d_tri, tri, ncclDouble, ncclSum, (int) root, comm_of(c), c->stream));
  NGSD_NCCL(err_to, ncclGroupEnd());
  for (ngsd_ctx *c : cs) {
    NGSD_CUDA(err_to, cudaSetDevice(c->device));
    if (c->comm_rank == root) k_tri_unpack<double><<<blocks, 256, 0, c->stream>>>(c->d_tri, n, c->d_num);
    if (with_cnt) k_tri_pack<uint64_t><<<blocks, 256, 0, c->stream>>>(c->d_cntout, n, reinterpret_cast<uint64_t *>(c->d_tri));
    NGSD_CUDA(err_to, cudaGetLastError());
  }
  if (with_cnt) {
    NGSD_NCCL(err_to, ncclGroupStart());
    for (ngsd_ctx *c : cs) NGSD_NCCL(err_to, ncclReduce(c->d_tri, c->d_tri, tri, ncclUint64, ncclSum, (int) root, comm_of(c), c->stream));
    NGSD_NCCL(err_to, ncclGroupEnd());
  }
  for (ngsd_ctx *c : cs) {
    NGSD_CUDA(err_to, cudaSetDevice(c->device));
    if (c->comm_rank == root) {
      if (with_cnt) k_tri_unpack<uint64_t><<<blocks, 256, 0, c->stream>>>(reinterpret_cast<uint64_t *>(c->d_tri), n, c->d_cntout);
      NGSD_CUDA(err_to, ngsd_launch_finish(c, with_cnt ? 0 : std::max<uint64_t>(n_eff_total, 1)));   // the epilogue is non-linear: after the reduction
      if (!with_cnt && n_eff_total == 0) NGSD_CUDA(err_to, cudaMemsetAsync(c->d_cntout, 0, n2 * sizeof(uint64_t), c->stream));
      NGSD_CUDA(err_to, cudaEventRecord(c->ev_comm[1], c->stream));
      if (out_host) NGSD_CUDA(err_to, cudaMemcpyAsync(out_host, c->d_out, n2 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
      if (num_opt) NGSD_CUDA(err_to, cudaMemcpyAsync(num_opt, c->d_num, n2 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
      if (cnt_opt) NGSD_CUDA(err_to, cudaMemcpyAsync(cnt_opt, c->d_cntout, n2 * sizeof(uint64_t), cudaMemcpyDeviceToHost, c->stream));
    } else {
      NGSD_CUDA(err_to, cudaEventRecord(c->ev_comm[1], c->stream));
    }
  }
  for (ngsd_ctx *c : cs) {
    NGSD_CUDA(err_to, cudaSetDevice(c->device));
    NGSD_CUDA(err_to, cudaStreamSynchronize(c->stream));
    finish_stats(c, tri * 8 * (with_cnt ? 2 : 1));
  }
  return NGSD_OK;
}

// Tile shards -> full matrices on `root` (entries a rank does not own are exact zeros: the sum is an assembly).
int reduce_tiles_impl(ngsd_ctx *err_to, const std::vector<ngsd_ctx *> &cs, uint32_t root, bool with_num_cnt, double *out_host, double *num_opt,
                      uint64_t *cnt_opt) {
  const uint64_t n = cs[0]->n_ind, n2 = n * n;
  for (ngsd_ctx *c : cs) {
    if (!c->comm) { ngsd_set_error(err_to, "no communicator: call ngsd_comm_attach first"); return NGSD_ERR_COMM; }
    if (!c->d_out) { ngsd_set_error(err_to, "no results yet: call ngsd_distances(out = NULL) first"); return NGSD_ERR_STATE; }
    NGSD_CUDA(err_to, cudaSetDevice(c->device));
    int rc = ensure_events(c);
    if (rc) return rc;
    NGSD_CUDA(err_to, cudaEventRecord(c->ev_comm[0], c->stream));
  }
  NGSD_NCCL(err_to, ncclGroupStart());
  for (ngsd_ctx *c : cs) {
    NGSD_NCCL(err_to, ncclReduce(c->d_out, c->d_out, n2, ncclDouble, ncclSum, (int) root, comm_of(c), c->stream));
    if (with_num_cnt) {
      NGSD_NCCL(err_to, ncclReduce(c->d_num, c->d_num, n2, ncclDouble, ncclSum, (int) root, comm_of(c), c->stream));
      NGSD_NCCL(err_to, ncclReduce(c->d_cntout, c->d_cntout, n2, ncclUint64, ncclSum, (int) root, comm_of(c), c->stream));
    }
  }
  NGSD_NCCL(err_to, ncclGroupEnd());
  for (ngsd_ctx *c : cs) {
    NGSD_CUDA(err_to, cudaSetDevice(c->device));
    NGSD_CUDA(err_to, cudaEventRecord(c->ev_comm[1], c->stream));
    if (c->comm_rank == root) {
      if (out_host) NGSD_CUDA(err_to, cudaMemcpyAsync(out_host, c->d_out, n2 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
      if (num_opt && with_num_cnt) NGSD_CUDA(err_to, cudaMemcpyAsync(num_opt, c->d_num, n2 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
      if (cnt_opt && with_num_cnt) NGSD_CUDA(err_to, cudaMemcpyAsync(cnt_opt, c->d_cntout, n2 * sizeof(uint64_t), cudaMemcpyDeviceToHost, c->stream));
    }
  }
  for (ngsd_ctx *c : cs) {
    NGSD_CUDA(err_to, cudaSetDevice(c->device));
    NGSD_CUDA(err_to, cudaStreamSynchronize(c->stream));
    finish_stats(c, n2 * 8 * (with_num_cnt ? 3 : 1));
  }
  return NGSD_OK;
}

struct Seg { char *p; uint64_t bytes; };

// the pieces of the resident layouts (DESIGN §2) that hold the sites [s0, s1) of a context created for all sites
void site_range_segments(ngsd_ctx *c, uint64_t s0, uint64_t s1, bool last, std::vector<Seg> &out) {
  out.clear();
  const uint64_t w0 = s0 / 64, w1 = last ? c->NW : s1 / 64;
  const uint64_t c0 = s0 / (uint64_t) c->sc, c1 = last ? c->NC : s1 / (uint64_t) c->sc;
  for (uint64_t rb = 0; rb < c->RB; rb++) {
    if (!c->int_path && c1 > c0) {
      out.push_back({(char *) (c->Apack + (rb * c->NC + c0) * c->tile_doubles), (c1 - c0) * c->tile_doubles * sizeof(double)});
      out.push_back({(char *) (c->Bpack + (rb * c->NC + c0) * c->tile_doubles), (c1 - c0) * c->tile_doubles * sizeof(double)});
    }
    if (rb == 0 && w1 > w0) out.push_back({(char *) (c->d_blank + w0), (w1 - w0) * sizeof(uint64_t)});
    if (w1 > w0) {
      out.push_back({(char *) (c->mask + (rb * c->NW + w0) * 128), (w1 - w0) * 128 * sizeof(uint64_t)});
      if (c->int_path) {
        out.push_back({(char *) (c->codes + (rb * c->NW + w0) * 512), (w1 - w0) * 512 * sizeof(uint32_t)});
        out.push_back({(char *) (c->codes4 + (rb * c->NW + w0) * 1024), (w1 - w0) * 1024 * sizeof(uint32_t)});
      }
    }
  }
  if (c->planes == 2 && !c->int_path && w1 > w0) out.push_back({(char *) (c->Cplane + w0 * c->n_pad * 64), (w1 - w0) * c->n_pad * 64 * sizeof(double)});
}

// Row C2: every rank front-ended only its own site range; all-to-all of the packed pieces (grouped ncclSend / ncclRecv:
// on NVSwitch every pair of GPUs talks at full bandwidth, so this is one hop per byte).
int allgather_impl(ngsd_ctx *err_to, const std::vector<ngsd_ctx *> &cs, const uint64_t *site_begin) {
  const uint32_t world = cs[0]->comm_world;
  const uint64_t align = (cs[0]->planes == 2 && !cs[0]->int_path) ? 192 : 64;
  if (site_begin[0] != 0 || site_begin[world] != cs[0]->n_sites) { ngsd_set_error(err_to, "site ranges must cover [0, n_sites)"); return NGSD_ERR_ARG; }
  for (uint32_t r = 0; r < world; r++) {
    if (site_begin[r + 1] < site_begin[r] || (r + 1 < world && site_begin[r + 1] % align)) {
      ngsd_set_error(err_to, "site range boundaries must be ascending multiples of %llu", (unsigned long long) align);
      return NGSD_ERR_ARG;
    }
  }
  std::vector<Seg> seg;
  // knife-edge triples are settled by the host (and patched into the resident layout) BEFORE the pieces travel
  bool any_deficit = false;
  for (ngsd_ctx *c : cs) {
    if (!c->comm) { ngsd_set_error(err_to, "no communicator: call ngsd_comm_attach first"); return NGSD_ERR_COMM; }
    ngsd_frontend_resolve(c);                 // a failure here shows up again in ngsd_frontend_flags below
    any_deficit |= !c->deficit.empty();
  }
  if (any_deficit && cs.size() == world) {    // one process: every GPU gets every row's deficit list
    std::vector<ngsd_ctx::deficit_entry> all;
    for (ngsd_ctx *c : cs) all.insert(all.end(), c->deficit.begin(), c->deficit.end());
    for (ngsd_ctx *c : cs) { c->deficit = all; c->deficit_dirty = true; }
    any_deficit = false;
  }
  for (ngsd_ctx *c : cs) {
    NGSD_CUDA(err_to, cudaSetDevice(c->device));
    int rc = ensure_events(c);
    if (!rc) rc = ensure_tri(c, 8);
    if (rc) return rc;
    if (any_deficit) {                        // one process per GPU: the lists are host state of other processes -> refuse on every rank
      int f = 0;
      NGSD_CUDA(err_to, cudaMemcpyAsync(&f, c->d_err, sizeof(int), cudaMemcpyDeviceToHost, c->stream));   // stream-ordered: see copy_sync in api.cu
      NGSD_CUDA(err_to, cudaStreamSynchronize(c->stream));
      f |= 16;
      NGSD_CUDA(err_to, cudaMemcpyAsync(c->d_err, &f, sizeof(int), cudaMemcpyHostToDevice, c->stream));
      NGSD_CUDA(err_to, cudaStreamSynchronize(c->stream));
    }
    NGSD_CUDA(err_to, cudaEventRecord(c->ev_comm[0], c->stream));
  }
  std::vector<uint64_t> moved(cs.size(), 0);
  NGSD_NCCL(err_to, ncclGroupStart());
  for (size_t k = 0; k < cs.size(); k++) {
    ngsd_ctx *c = cs[k];
    const uint32_t me = c->comm_rank;
    for (uint32_t p = 0; p < world; p++) {
      if (p == me) continue;
      site_range_segments(c, site_begin[me], site_begin[me + 1], me + 1 == world, seg);
      for (const Seg &s : seg) { NGSD_NCCL(err_to, ncclSend(s.p, s.bytes, ncclChar, (int) p, comm_of(c), c->stream)); moved[k] += s.bytes; }
      site_range_segments(c, site_begin[p], site_begin[p + 1], p + 1 == world, seg);
      for (const Seg &s : seg) { NGSD_NCCL(err_to, ncclRecv(s.p, s.bytes, ncclChar, (int) p, comm_of(c), c->stream)); moved[k] += s.bytes; }
    }
  }
  NGSD_NCCL(err_to, ncclGroupEnd());
  // a front-end error on any rank (NaN, bad genotype code) must stop every rank: OR-reduce the flag words
  for (ngsd_ctx *c : cs) {
    NGSD_CUDA(err_to, cudaSetDevice(c->device));
    k_flags_split<<<1, 32, 0, c->stream>>>(c->d_err, reinterpret_cast<int *>(c->d_tri));
  }
  NGSD_NCCL(err_to, ncclGroupStart());
  for (ngsd_ctx *c : cs) NGSD_NCCL(err_to, ncclAllReduce(c->d_tri, c->d_tri, 8, ncclInt32, ncclMax, comm_of(c), c->stream));
  NGSD_NCCL(err_to, ncclGroupEnd());
  for (ngsd_ctx *c : cs) {
    NGSD_CUDA(err_to, cudaSetDevice(c->device));
    k_flags_merge<<<1, 32, 0, c->stream>>>(c->d_err, reinterpret_cast<const int *>(c->d_tri));
  }
  for (size_t k = 0; k < cs.size(); k++) {
    ngsd_ctx *c = cs[k];
    NGSD_CUDA(err_to, cudaSetDevice(c->device));
    NGSD_CUDA(err_to, cudaEventRecord(c->ev_comm[1], c->stream));
    NGSD_CUDA(err_to, cudaStreamSynchronize(c->stream));
    finish_stats(c, moved[k]);
  }
  for (ngsd_ctx *c : cs) {
    int rc = ngsd_frontend_flags(c);
    if (rc) { if (c != err_to) ngsd_set_error(err_to, "%s", c->err); return rc; }
    ngsd_mark_all_pushed(c);
  }
  return NGSD_OK;
}

int barrier_impl(ngsd_ctx *err_to, const std::vector<ngsd_ctx *> &cs) {
  for (ngsd_ctx *c : cs) {
    if (!c->comm) { ngsd_set_error(err_to, "no communicator"); return NGSD_ERR_COMM; }
    NGSD_CUDA(err_to, cudaSetDevice(c->device));
    int rc = ensure_tri(c, 1);
    if (rc) return rc;
  }
  NGSD_NCCL(err_to, ncclGroupStart());
  for (ngsd_ctx *c : cs) NGSD_NCCL(err_to, ncclAllReduce(c->d_tri, c->d_tri, 1, ncclDouble, ncclSum, comm_of(c), c->stream));
  NGSD_NCCL(err_to, ncclGroupEnd());
  for (ngsd_ctx *c : cs) {
    NGSD_CUDA(err_to, cudaSetDevice(c->device));
    NGSD_CUDA(err_to, cudaStreamSynchronize(c->stream));
  }
  return NGSD_OK;
}

// one host thread per GPU for calls that block on their stream
template <typename F>
int for_each_kid(ngsd_ctx *parent, F fn) {
  const size_t N = parent->kids.size();
  std::vector<int> rc(N, NGSD_OK);
  std::vector<std::thread> th;
  for (size_t g = 1; g < N; g++) th.emplace_back([&, g]() { rc[g] = fn(parent->kids[g], (uint32_t) g); });
  rc[0] = fn(parent->kids[0], 0u);
  for (auto &t : th) t.join();
  for (size_t g = 0; g < N; g++)
    if (rc[g]) { ngsd_set_error(parent, "GPU %d: %s", parent->kids[g]->device, parent->kids[g]->err); return rc[g]; }
  return NGSD_OK;
}

uint64_t gcd64(uint64_t a, uint64_t b) { while (b) { const uint64_t t = a % b; a = b; b = t; } return a; }

void sum_timing(ngsd_timing &acc, const ngsd_timing &t) {
  acc.frontend_ms = std::max(acc.frontend_ms, t.frontend_ms);
  acc.count_ms = std::max(acc.count_ms, t.count_ms);
  acc.dist_ms = std::max(acc.dist_ms, t.dist_ms);
  acc.epilogue_ms = std::max(acc.epilogue_ms, t.epilogue_ms);
  acc.total_ms = std::max(acc.total_ms, t.total_ms);
  acc.launches += t.launches;
  acc.dist_ctas = std::max(acc.dist_ctas, t.dist_ctas);
  acc.dist_dmma += t.dist_dmma;
  acc.dist_imma += t.dist_imma;
  acc.active_sites = std::max(acc.active_sites, t.active_sites);
  acc.block_cache = std::max(acc.block_cache, t.block_cache);
}

}  // namespace

void ngsd_comm_release(ngsd_ctx *ctx) {
  if (ctx->comm && !ctx->parent) ncclCommDestroy(comm_of(ctx));   // a group destroys its kids' communicators itself
  ctx->comm = nullptr;
  cudaFree(ctx->d_tri);
  cudaFree(ctx->d_gather);
  ctx->d_tri = ctx->d_gather = nullptr;
  ctx->tri_cap = ctx->gather_cap = 0;
  for (auto &e : ctx->ev_comm)
    if (e) { cudaEventDestroy(e); e = nullptr; }
}

// ------------------------------------------------------------------------------------------------ group ----

int ngsd_group_create(const ngsd_cfg *cfg, ngsd_ctx **out) {
  const int N = cfg->n_gpus;
  ngsd_ctx *parent = new (std::nothrow) ngsd_ctx();
  if (!parent) { ngsd_set_error(nullptr, "out of host memory"); return NGSD_ERR_ARG; }
  parent->cfg = *cfg;
  parent->device = cfg->device;
  parent->n_ind = cfg->n_ind;
  parent->n_sites = cfg->n_sites;
  ngsd_cfg kc = *cfg;
  kc.n_gpus = 0;
  kc.shard = 0;
  auto fail = [&](int rc) {
    std::string msg = ngsd_last_error(nullptr);
    for (ngsd_ctx *k : parent->kids) { k->parent = nullptr; k->comm = nullptr; ngsd_destroy(k); }
    parent->kids.clear();
    delete parent;
    ngsd_set_error(nullptr, "%s", msg.c_str());
    return rc;
  };
  int mode = cfg->shard;
  ngsd_ctx *first = nullptr;
  if (mode != NGSD_SHARD_SITES) {   // REPLICATED needs every site on every GPU: try it on the first one
    kc.device = cfg->device;
    int rc = ngsd_create(&kc, &first);
    size_t fr = 0, tot = 0;
    if (rc == NGSD_OK) { cudaSetDevice(kc.device); cudaMemGetInfo(&fr, &tot); }
    if (rc == NGSD_OK && (mode == NGSD_SHARD_REPLICATED || fr >= ((size_t) 8 << 30))) {
      mode = NGSD_SHARD_REPLICATED;
    } else if (mode == NGSD_SHARD_REPLICATED) {
      return fail(rc);
    } else {
      if (first) ngsd_destroy(first);
      first = nullptr;
      if (rc != NGSD_OK && rc != NGSD_ERR_CUDA) return fail(rc);   // a configuration error, not memory
      cudaGetLastError();
      mode = NGSD_SHARD_SITES;
    }
  }
  parent->shard_mode = mode;
  uint64_t align = 64;
  if (mode == NGSD_SHARD_REPLICATED) {
    if (first->planes == 2 && !first->int_path) align = 192;
  } else {
    const uint64_t bs = std::max<uint64_t>(1, cfg->boot_block_size);
    align = 64 / gcd64(64, bs) * bs;                            // whole bootstrap blocks and whole 64-site words
  }
  // a data set too small to give every GPU a whole unit of sites runs on fewer of them (one: an ordinary context)
  const int N_use = (int) std::max<uint64_t>(1, std::min<uint64_t>((uint64_t) N, cfg->n_sites / align));
  if (N_use == 1) {
    if (!first) {
      kc.device = cfg->device;
      int rc = ngsd_create(&kc, &first);
      if (rc) return fail(rc);
    }
    delete parent;
    *out = first;
    return NGSD_OK;
  }
  parent->site_begin.assign(N_use + 1, 0);
  for (int g = 1; g < N_use; g++) parent->site_begin[g] = (cfg->n_sites / align * (uint64_t) g / (uint64_t) N_use) * align;
  parent->site_begin[N_use] = cfg->n_sites;
  for (int g = 0; g < N_use; g++) {
    ngsd_ctx *k = nullptr;
    if (g == 0 && first) {
      k = first;
    } else {
      kc.device = cfg->device + g;
      if (mode == NGSD_SHARD_SITES) kc.n_sites = parent->site_begin[g + 1] - parent->site_begin[g];
      int rc = ngsd_create(&kc, &k);
      if (rc) return fail(rc);
    }
    k->parent = parent;
    k->comm_rank = (uint32_t) g;
    k->comm_world = (uint32_t) N_use;
    parent->kids.push_back(k);
  }
  std::vector<ncclComm_t> comms(N_use);
  std::vector<int> devs(N_use);
  for (int g = 0; g < N_use; g++) devs[g] = cfg->device + g;
  ncclResult_t r = ncclCommInitAll(comms.data(), N_use, devs.data());
  if (r != ncclSuccess) {
    ngsd_set_error(nullptr, "NCCL error: %s (ncclCommInitAll over %d devices)", ncclGetErrorString(r), N_use);
    return fail(NGSD_ERR_COMM);
  }
  for (int g = 0; g < N_use; g++) parent->kids[g]->comm = comms[g];
  for (ngsd_ctx *k : parent->kids) {                       // connect every pair now (NCCL sets channels up lazily), see ngsd_comm_attach
    cudaSetDevice(k->device);
    if (ensure_tri(k, 2 * ((uint64_t) 1 << 19) * N_use)) return fail(NGSD_ERR_CUDA);
  }
  const uint64_t kWarm = (uint64_t) 1 << 19;
  bool okc = ncclGroupStart() == ncclSuccess;
  for (ngsd_ctx *k : parent->kids)
    for (int p = 0; p < N_use && okc; p++) {
      if ((uint32_t) p == k->comm_rank) continue;
      okc = okc && ncclSend(k->d_tri + (uint64_t) p * kWarm, kWarm, ncclDouble, p, comm_of(k), k->stream) == ncclSuccess;
      okc = okc && ncclRecv(k->d_tri + (uint64_t) (N_use + p) * kWarm, kWarm, ncclDouble, p, comm_of(k), k->stream) == ncclSuccess;
    }
  okc = (ncclGroupEnd() == ncclSuccess) && okc;
  for (ngsd_ctx *k : parent->kids) { cudaSetDevice(k->device); okc = okc && cudaStreamSynchronize(k->stream) == cudaSuccess; }
  if (!okc) { ngsd_set_error(nullptr, "NCCL error while connecting the GPUs of the group"); return fail(NGSD_ERR_COMM); }
  *out = parent;
  return NGSD_OK;
}

int ngsd_group_destroy(ngsd_ctx *parent) {
  for (ngsd_ctx *k : parent->kids) {
    cudaSetDevice(k->device);
    if (k->stream) cudaStreamSynchronize(k->stream);
    if (k->comm) ncclCommDestroy(comm_of(k));
    k->comm = nullptr;
    k->parent = nullptr;
    ngsd_destroy(k);
  }
  parent->kids.clear();
  delete parent;
  return NGSD_OK;
}

int ngsd_group_push(ngsd_ctx *parent, int what, const void *ptr, uint64_t bytes_per_site, uint64_t row_stride, const int8_t *code_of_field,
                    uint64_t site0, uint64_t n) {
  if (!ptr) { ngsd_set_error(parent, "null input pointer"); return NGSD_ERR_ARG; }
  if (n == 0 || site0 + n > parent->n_sites) { ngsd_set_error(parent, "push beyond n_sites"); return NGSD_ERR_ARG; }
  struct Piece { ngsd_ctx *k; uint64_t g0, n; };
  std::vector<Piece> pieces;
  const size_t N = parent->kids.size();
  for (size_t g = 0; g < N; g++) {
    const uint64_t a = std::max(site0, parent->site_begin[g]), b = std::min(site0 + n, parent->site_begin[g + 1]);
    if (b > a) pieces.push_back({parent->kids[g], a, b - a});
  }
  std::vector<int> rc(pieces.size(), NGSD_OK);
  auto run = [&](size_t q) {
    const Piece &pc = pieces[q];
    const char *src = (const char *) ptr + (pc.g0 - site0) * bytes_per_site;
    const uint64_t local0 = parent->shard_mode == NGSD_SHARD_SITES ? pc.g0 - parent->site_begin[pc.k->comm_rank] : pc.g0;
    switch (what) {
      case 0: rc[q] = ngsd_push_sites(pc.k, (const double *) src, local0, pc.n); break;
      case 1: rc[q] = ngsd_push_genotypes(pc.k, (const int8_t *) src, local0, pc.n); break;
      case 2: rc[q] = ngsd_push_packed_genotypes(pc.k, (const uint8_t *) src, row_stride, code_of_field, local0, pc.n); break;
      case 10 + NGSD_XFER_F32: case 10 + NGSD_XFER_U32: case 10 + NGSD_XFER_U20X3: {   // transport tiers: code_of_field carries &denom
        double denom;
        memcpy(&denom, code_of_field, sizeof(denom));
        rc[q] = ngsd_push_sites_packed(pc.k, src, what - 10, denom, local0, pc.n);
        break;
      }
      default: {
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, src) != cudaSuccess || at.type != cudaMemoryTypeDevice || at.device != pc.k->device) {
          cudaGetLastError();
          ngsd_set_error(pc.k, "device input for sites %llu.. must live on device %d, the GPU that owns them", (unsigned long long) pc.g0, pc.k->device);
          rc[q] = NGSD_ERR_ARG;
        } else {
          rc[q] = ngsd_push_sites_device(pc.k, (const double *) src, local0, pc.n);
        }
      }
    }
  };
  std::vector<std::thread> th;
  for (size_t q = 1; q < pieces.size(); q++) th.emplace_back(run, q);
  run(0);
  for (auto &t : th) t.join();
  for (size_t q = 0; q < pieces.size(); q++)
    if (rc[q]) { ngsd_set_error(parent, "GPU %d: %s", pieces[q].k->device, pieces[q].k->err); return rc[q]; }
  return NGSD_OK;
}

int ngsd_group_frontend(ngsd_ctx *parent) {
  if (parent->shard_mode == NGSD_SHARD_SITES) return for_each_kid(parent, [](ngsd_ctx *k, uint32_t) { return ngsd_frontend(k); });
  // REPLICATED: every kid holds its own range; check that, then all-gather
  for (size_t g = 0; g < parent->kids.size(); g++) {
    ngsd_ctx *k = parent->kids[g];
    const uint64_t w0 = parent->site_begin[g] / 64, w1 = (parent->site_begin[g + 1] + 63) / 64;
    for (uint64_t w = w0; w < w1; w++)
      if (!k->pushed[w]) {
        ngsd_set_error(parent, "front end incomplete: sites %llu.. were never pushed", (unsigned long long) (w * 64));
        return NGSD_ERR_STATE;
      }
  }
  if (parent->kids[0]->frontend_done && parent->kids[0]->words_pushed == parent->kids[0]->NW) return NGSD_OK;   // already gathered
  return allgather_impl(parent, parent->kids, parent->site_begin.data());
}

int ngsd_group_distances(ngsd_ctx *parent, const uint32_t *block_counts, uint64_t n_blocks, uint64_t block_size, double *out, double *num_opt,
                         uint64_t *cnt_opt) {
  const uint32_t N = (uint32_t) parent->kids.size();
  ngsd_ctx *root = parent->kids[0];
  if (!root->frontend_done) {
    int rc = ngsd_group_frontend(parent);
    if (rc) return rc;
  }
  int rc;
  if (parent->shard_mode == NGSD_SHARD_SITES) {
    const bool weighted = block_counts != nullptr;
    if (weighted && (block_size == 0 || n_blocks * block_size > parent->n_sites)) { ngsd_set_error(parent, "invalid bootstrap geometry"); return NGSD_ERR_ARG; }
    if (weighted)
      for (uint32_t g = 1; g < N; g++)
        if (parent->site_begin[g] % block_size) {
          ngsd_set_error(parent, "site shards are not aligned to blocks of %llu sites: set ngsd_cfg.boot_block_size", (unsigned long long) block_size);
          return NGSD_ERR_ARG;
        }
    rc = for_each_kid(parent, [&](ngsd_ctx *k, uint32_t g) {
      if (!weighted) return ngsd_distances(k, nullptr, 0, 1, nullptr, nullptr, nullptr);
      const uint64_t b0 = std::min(n_blocks, parent->site_begin[g] / block_size);
      const uint64_t b1 = g + 1 == N ? n_blocks : std::min(n_blocks, parent->site_begin[g + 1] / block_size);
      return ngsd_distances(k, block_counts + b0, b1 - b0, block_size, nullptr, nullptr, nullptr);
    });
    if (rc) return rc;
    const uint64_t n_eff = weighted ? n_blocks * block_size : parent->n_sites;
    rc = reduce_sites_impl(parent, parent->kids, 0, n_eff, out, num_opt, cnt_opt);
  } else {
    if (!parent->kids_tile_sharded) {
      rc = for_each_kid(parent, [&](ngsd_ctx *k, uint32_t g) { return ngsd_set_tile_shard(k, g, N); });
      if (rc) return rc;
      parent->kids_tile_sharded = true;
    }
    rc = for_each_kid(parent, [&](ngsd_ctx *k, uint32_t) { return ngsd_distances(k, block_counts, n_blocks, block_size, nullptr, nullptr, nullptr); });
    if (rc) return rc;
    rc = reduce_tiles_impl(parent, parent->kids, 0, num_opt || cnt_opt, out, num_opt, cnt_opt);
  }
  if (rc) return rc;
  parent->timing = ngsd_timing();
  for (ngsd_ctx *k : parent->kids) sum_timing(parent->timing, k->timing);
  return NGSD_OK;
}

// One process per GPU: replicate r on rank r % world, matrices gathered on rank 0 (NCCL send / recv).
static int comm_distances_batch(ngsd_ctx *ctx, const uint32_t *block_counts, uint64_t n_rep, uint64_t n_blocks, uint64_t block_size, double *out) {
  const uint32_t world = ctx->comm_world, me = ctx->comm_rank;
  const uint64_t n2 = ctx->n_ind * ctx->n_ind;
  if (me == 0 && !out && n_rep) { ngsd_set_error(ctx, "rank 0 needs an output buffer"); return NGSD_ERR_ARG; }
  NGSD_CUDA(ctx, cudaSetDevice(ctx->device));
  int rc = ensure_events(ctx);
  if (rc) return rc;
  if (me == 0) { rc = ensure_gather(ctx, (uint64_t) (world - 1) * n2); if (rc) return rc; }
  ngsd_timing sum = ngsd_timing();
  uint64_t moved = 0;
  float comm_ms = 0.f;
  for (uint64_t base = 0; base < n_rep; base += world) {
    const uint64_t r = base + me;
    if (r < n_rep) {
      rc = ngsd_distances(ctx, block_counts + r * n_blocks, n_blocks, block_size, me == 0 ? out + r * n2 : nullptr, nullptr, nullptr);
      if (rc) return rc;
      sum.total_ms += ctx->timing.total_ms; sum.dist_ms += ctx->timing.dist_ms; sum.count_ms += ctx->timing.count_ms;
      sum.epilogue_ms += ctx->timing.epilogue_ms; sum.launches += ctx->timing.launches; sum.dist_dmma += ctx->timing.dist_dmma;
      sum.dist_imma += ctx->timing.dist_imma; sum.active_sites += ctx->timing.active_sites; sum.dist_ctas = ctx->timing.dist_ctas;
    }
    NGSD_CUDA(ctx, cudaEventRecord(ctx->ev_comm[0], ctx->stream));
    NGSD_NCCL(ctx, ncclGroupStart());
    if (me == 0) {
      for (uint32_t g = 1; g < world && base + g < n_rep; g++) {
        NGSD_NCCL(ctx, ncclRecv(ctx->d_gather + (uint64_t) (g - 1) * n2, n2, ncclDouble, (int) g, comm_of(ctx), ctx->stream));
        moved += n2 * 8;
      }
    } else if (r < n_rep) {
      NGSD_NCCL(ctx, ncclSend(ctx->d_out, n2, ncclDouble, 0, comm_of(ctx), ctx->stream));
      moved += n2 * 8;
    }
    NGSD_NCCL(ctx, ncclGroupEnd());
    NGSD_CUDA(ctx, cudaEventRecord(ctx->ev_comm[1], ctx->stream));
    if (me == 0)
      for (uint32_t g = 1; g < world && base + g < n_rep; g++)
        NGSD_CUDA(ctx, cudaMemcpyAsync(out + (base + g) * n2, ctx->d_gather + (uint64_t) (g - 1) * n2, n2 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    NGSD_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, ctx->ev_comm[0], ctx->ev_comm[1]);
    comm_ms += ms;
  }
  ctx->timing = sum;
  ctx->comm_bytes = moved;
  ctx->comm_ms = comm_ms;
  return NGSD_OK;
}

int ngsd_group_distances_batch(ngsd_ctx *ctx, const uint32_t *block_counts, uint64_t n_rep, uint64_t n_blocks, uint64_t block_size, double *out) {
  if (ctx->kids.empty()) return comm_distances_batch(ctx, block_counts, n_rep, n_blocks, block_size, out);
  ngsd_ctx *parent = ctx;
  if (!out && n_rep) { ngsd_set_error(parent, "null output"); return NGSD_ERR_ARG; }
  const uint32_t N = (uint32_t) parent->kids.size();
  const uint64_t n2 = parent->n_ind * parent->n_ind;
  if (!parent->kids[0]->frontend_done) {
    int rc = ngsd_group_frontend(parent);
    if (rc) return rc;
  }
  // The per pair-site EM with the bootstrap block cache (blocks of whole site chunks, at least two, cache not turned off
  // by ngsd_cfg.reserved bit 2): every replicate on every GPU, each on its own tiles, so that each GPU builds the cache of
  // its tiles once.  The kids stay tile-sharded from matrix 0 on: ngsd_set_tile_shard would drop the cache.  Otherwise
  // whole replicates are dealt to the GPUs, which at one site per block is the better use of them.
  const ngsd_ctx *k0 = parent->kids[0];
  const bool em_tiles = !parent->cfg.indep_geno && block_size % (uint64_t) k0->sc == 0 && n_blocks >= 2 && !(parent->cfg.reserved & 4);
  if (parent->shard_mode == NGSD_SHARD_SITES || em_tiles) {   // every replicate needs every GPU
    ngsd_timing acc = ngsd_timing();
    for (uint64_t r = 0; r < n_rep; r++) {
      int rc = ngsd_group_distances(parent, block_counts + r * n_blocks, n_blocks, block_size, out + r * n2, nullptr, nullptr);
      if (rc) return rc;
      acc.total_ms += parent->timing.total_ms; acc.dist_ms += parent->timing.dist_ms; acc.launches += parent->timing.launches;
      acc.dist_dmma += parent->timing.dist_dmma; acc.dist_imma += parent->timing.dist_imma;
    }
    parent->timing = acc;
    return NGSD_OK;
  }
  if (parent->kids_tile_sharded) {   // back to whole matrices per GPU
    int rc = for_each_kid(parent, [&](ngsd_ctx *k, uint32_t) { return ngsd_set_tile_shard(k, 0, 1); });
    if (rc) return rc;
    parent->kids_tile_sharded = false;
  }
  std::vector<ngsd_timing> acc(N, ngsd_timing());
  int rc = for_each_kid(parent, [&](ngsd_ctx *k, uint32_t g) {
    for (uint64_t r = g; r < n_rep; r += N) {   // the matrix goes to the host through this GPU's own PCIe link
      int rc1 = ngsd_distances(k, block_counts + r * n_blocks, n_blocks, block_size, out + r * n2, nullptr, nullptr);
      if (rc1) return rc1;
      acc[g].total_ms += k->timing.total_ms; acc[g].dist_ms += k->timing.dist_ms; acc[g].count_ms += k->timing.count_ms;
      acc[g].epilogue_ms += k->timing.epilogue_ms; acc[g].launches += k->timing.launches; acc[g].dist_dmma += k->timing.dist_dmma;
      acc[g].dist_imma += k->timing.dist_imma; acc[g].dist_ctas = k->timing.dist_ctas; acc[g].block_cache = k->timing.block_cache;
    }
    return (int) NGSD_OK;
  });
  if (rc) return rc;
  parent->timing = ngsd_timing();
  for (uint32_t g = 0; g < N; g++) sum_timing(parent->timing, acc[g]);
  return NGSD_OK;
}

int ngsd_group_get_posteriors(ngsd_ctx *parent, double *P_host, uint8_t *miss_host) {
  if (!parent->kids[0]->frontend_done) {
    int rc = ngsd_group_frontend(parent);
    if (rc) return rc;
  }
  if (parent->shard_mode != NGSD_SHARD_SITES) {
    int rc = ngsd_get_posteriors(parent->kids[0], P_host, miss_host);
    if (rc) ngsd_set_error(parent, "%s", parent->kids[0]->err);
    return rc;
  }
  const uint64_t n_ind = parent->n_ind, S = parent->n_sites;
  for (size_t g = 0; g < parent->kids.size(); g++) {
    ngsd_ctx *k = parent->kids[g];
    const uint64_t s0 = parent->site_begin[g], ns = k->n_sites;
    std::vector<double> P(P_host ? n_ind * ns * 3 : 0);
    std::vector<uint8_t> M(miss_host ? n_ind * ns : 0);
    int rc = ngsd_get_posteriors(k, P_host ? P.data() : nullptr, miss_host ? M.data() : nullptr);
    if (rc) { ngsd_set_error(parent, "%s", k->err); return rc; }
    for (uint64_t i = 0; i < n_ind; i++) {
      if (P_host) memcpy(P_host + (i * S + s0) * 3, P.data() + i * ns * 3, ns * 3 * sizeof(double));
      if (miss_host) memcpy(miss_host + i * S + s0, M.data() + i * ns, ns);
    }
  }
  return NGSD_OK;
}

int ngsd_group_get_timing(ngsd_ctx *parent, ngsd_timing *t) {
  if (parent->timing.total_ms < 0 || (parent->timing.launches == 0 && parent->timing.total_ms == 0)) {   // after pushes: the kids' front-end times
    ngsd_timing acc = ngsd_timing();
    for (ngsd_ctx *k : parent->kids) {
      ngsd_timing tk;
      if (ngsd_get_timing(k, &tk) == NGSD_OK) sum_timing(acc, tk);
    }
    *t = acc;
    return NGSD_OK;
  }
  *t = parent->timing;
  return NGSD_OK;
}

// ngsd_trees_batch: GPU g builds the trees of matrices [n_mat g / N, n_mat (g + 1) / N), uploading only those
int ngsd_group_trees(ngsd_ctx *parent, const double *dist_host, uint64_t n_mat, int method, const char *const *labels, std::string *out,
                     uint64_t *n_nni, int32_t *status) {
  const uint64_t N = parent->kids.size(), n2 = parent->kids[0]->n_ind * parent->kids[0]->n_ind;
  return for_each_kid(parent, [&](ngsd_ctx *k, uint32_t g) {
    const uint64_t b = n_mat * g / N, e = n_mat * (g + 1) / N;
    return b == e ? NGSD_OK : ngsd_trees_run(k, dist_host + b * n2, nullptr, e - b, method, labels, out + b, n_nni + b, status + b);
  });
}

// ------------------------------------------------------------------------------------------------ C ABI ----

extern "C" {

int ngsd_comm_unique_id(uint8_t id[NGSD_COMM_ID_BYTES]) {
  static_assert(sizeof(ncclUniqueId) <= NGSD_COMM_ID_BYTES, "ncclUniqueId does not fit NGSD_COMM_ID_BYTES");
  if (!id) return NGSD_ERR_ARG;
  ncclUniqueId u;
  ncclResult_t r = ncclGetUniqueId(&u);
  if (r != ncclSuccess) { ngsd_set_error(nullptr, "NCCL error: %s (ncclGetUniqueId)", ncclGetErrorString(r)); return NGSD_ERR_COMM; }
  memset(id, 0, NGSD_COMM_ID_BYTES);
  memcpy(id, &u, sizeof(u));
  return NGSD_OK;
}

int ngsd_comm_attach(ngsd_ctx *ctx, const uint8_t id[NGSD_COMM_ID_BYTES], uint32_t rank, uint32_t world) {
  if (!ctx || !id) return NGSD_ERR_ARG;
  if (!ctx->kids.empty() || ctx->parent) { ngsd_set_error(ctx, "a multi-GPU context owns its communicator"); return NGSD_ERR_ARG; }
  if (ctx->comm) { ngsd_set_error(ctx, "communicator already attached"); return NGSD_ERR_STATE; }
  if (world == 0 || rank >= world) { ngsd_set_error(ctx, "invalid rank %u of %u", rank, world); return NGSD_ERR_ARG; }
  NGSD_CUDA(ctx, cudaSetDevice(ctx->device));
  ncclUniqueId u;
  memcpy(&u, id, sizeof(u));
  ncclComm_t comm = nullptr;
  NGSD_NCCL(ctx, ncclCommInitRank(&comm, (int) world, u, (int) rank));
  ctx->comm = comm;
  ctx->comm_rank = rank;
  ctx->comm_world = world;
  // NCCL connects lazily: the first collective and the first send / recv between two ranks pay for the channel set-up
  // (seconds on a fresh communicator).  Do both here, so that "attached" means "connected" and no data-path call does.
  // (with messages large enough that NCCL opens all the channels it will ever use between two ranks, and with each kind
  // of collective the data path issues: measured on 8 B200s, a first ncclReduce on a communicator that had only done an
  // all-reduce still cost 0.46 s, a first 2 GB exchange after a 4 MB one 0.9 s)
  const uint64_t kWarm = (uint64_t) 1 << 22;                             // 32 MiB per peer and direction
  double *tmp = nullptr;
  NGSD_CUDA(ctx, cudaMalloc((void **) &tmp, 2 * kWarm * world * sizeof(double)));
  NGSD_CUDA(ctx, cudaMemsetAsync(tmp, 0, 2 * kWarm * world * sizeof(double), ctx->stream));
  ncclResult_t r1 = ncclAllReduce(tmp, tmp, kWarm, ncclDouble, ncclSum, comm, ctx->stream);
  if (r1 == ncclSuccess) r1 = ncclReduce(tmp, tmp, kWarm, ncclDouble, ncclSum, 0, comm, ctx->stream);
  if (r1 == ncclSuccess) r1 = ncclReduce(tmp, tmp, kWarm, ncclUint64, ncclSum, 0, comm, ctx->stream);
  if (r1 == ncclSuccess) r1 = ncclGroupStart();
  for (uint32_t p = 0; p < world && r1 == ncclSuccess; p++) {
    if (p == rank) continue;
    r1 = ncclSend(tmp + (uint64_t) p * kWarm, kWarm, ncclDouble, (int) p, comm, ctx->stream);
    if (r1 == ncclSuccess) r1 = ncclRecv(tmp + (uint64_t) (world + p) * kWarm, kWarm, ncclDouble, (int) p, comm, ctx->stream);
  }
  if (r1 == ncclSuccess) r1 = ncclGroupEnd();
  cudaError_t e1 = cudaStreamSynchronize(ctx->stream);
  cudaFree(tmp);
  if (r1 != ncclSuccess) { ngsd_set_error(ctx, "NCCL error: %s (communicator warm-up)", ncclGetErrorString(r1)); return NGSD_ERR_COMM; }
  NGSD_CUDA(ctx, e1);
  NGSD_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return NGSD_OK;
}

int ngsd_comm_allgather_operands(ngsd_ctx *ctx, const uint64_t *site_begin) {
  if (!ctx || !site_begin) return NGSD_ERR_ARG;
  if (!ctx->kids.empty()) return ngsd_group_frontend(ctx);
  return allgather_impl(ctx, std::vector<ngsd_ctx *>{ctx}, site_begin);
}

int ngsd_comm_reduce_sites(ngsd_ctx *ctx, uint32_t root, uint64_t n_eff_total, double *out_host) {
  if (!ctx) return NGSD_ERR_ARG;
  if (!ctx->kids.empty()) { ngsd_set_error(ctx, "a multi-GPU context reduces inside ngsd_distances"); return NGSD_ERR_ARG; }
  if (root >= ctx->comm_world) { ngsd_set_error(ctx, "invalid root"); return NGSD_ERR_ARG; }
  return reduce_sites_impl(ctx, std::vector<ngsd_ctx *>{ctx}, root, n_eff_total, out_host, nullptr, nullptr);
}

int ngsd_comm_reduce_tiles(ngsd_ctx *ctx, uint32_t root, int32_t with_num_cnt, double *out_host, double *num_host, uint64_t *cnt_host) {
  if (!ctx) return NGSD_ERR_ARG;
  if (!ctx->kids.empty()) { ngsd_set_error(ctx, "a multi-GPU context assembles inside ngsd_distances"); return NGSD_ERR_ARG; }
  if (root >= ctx->comm_world) { ngsd_set_error(ctx, "invalid root"); return NGSD_ERR_ARG; }
  return reduce_tiles_impl(ctx, std::vector<ngsd_ctx *>{ctx}, root, with_num_cnt != 0, out_host, num_host, cnt_host);
}

int ngsd_comm_barrier(ngsd_ctx *ctx) {
  if (!ctx) return NGSD_ERR_ARG;
  if (!ctx->kids.empty()) return barrier_impl(ctx, ctx->kids);
  return barrier_impl(ctx, std::vector<ngsd_ctx *>{ctx});
}

int ngsd_comm_stats(const ngsd_ctx *ctx, uint64_t *bytes, float *ms) {
  if (!ctx) return NGSD_ERR_ARG;
  const ngsd_ctx *c = ctx->kids.empty() ? ctx : ctx->kids[0];
  if (bytes) *bytes = c->comm_bytes;
  if (ms) *ms = c->comm_ms;
  return NGSD_OK;
}

// sysfs: /sys/bus/pci/devices/<domain:bus:dev.fn>/{numa_node,local_cpulist}
int ngsd_bind_host_to_device(int device) {
  char bus[32] = {0};
  if (cudaDeviceGetPCIBusId(bus, sizeof(bus), device) != cudaSuccess) { cudaGetLastError(); return -1; }
  for (char *p = bus; *p; p++) *p = (char) tolower(*p);
  char path[128];
  snprintf(path, sizeof(path), "/sys/bus/pci/devices/%s/numa_node", bus);
  int node = -1;
  if (FILE *f = fopen(path, "r")) { if (fscanf(f, "%d", &node) != 1) node = -1; fclose(f); }
  snprintf(path, sizeof(path), "/sys/bus/pci/devices/%s/local_cpulist", bus);
  if (FILE *f = fopen(path, "r")) {
    char list[4096] = {0};
    if (fgets(list, sizeof(list), f)) {
      cpu_set_t set;
      CPU_ZERO(&set);
      int any = 0;
      for (char *tok = strtok(list, ",\n"); tok; tok = strtok(nullptr, ",\n")) {
        int a = 0, b = 0;
        const int k = sscanf(tok, "%d-%d", &a, &b);
        if (k == 1) b = a;
        if (k >= 1)
          for (int cpu = a; cpu <= b && cpu < CPU_SETSIZE; cpu++) { CPU_SET(cpu, &set); any = 1; }
      }
      if (any) sched_setaffinity(0, sizeof(set), &set);
    }
    fclose(f);
  }
  if (node >= 0 && node < 64) {   // MPOL_PREFERRED: pages this thread touches from now on come from the GPU's node
    unsigned long mask = 1ul << node;
    syscall(SYS_set_mempolicy, 1 /* MPOL_PREFERRED */, &mask, 65ul);
  }
  return node;
}

}  // extern "C"
