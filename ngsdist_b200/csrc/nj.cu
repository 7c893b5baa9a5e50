// N4 (SURVEY §8f, ranked last): neighbour-joining trees from the distance matrices while they are still on the device.
//
// The reference stops at the `.dist` file; its README (README.md:83-98) hands the 1 + n_boot_rep matrices to FastME for
// one tree per matrix and to RAxML for the bootstrap support.  The tree step is O(n^3) per matrix on data the device
// already holds, so it is offered here as an additive entry point.  There is NO reference implementation to pin against
// (FastME is an external program): this follows the published algorithm -- Saitou & Nei 1987 in the Studier & Keppler
// 1988 formulation --
//     Q(i,j) = (m - 2) d(i,j) - r_i - r_j,  r_i = sum_k d(i,k)            pick the active pair with the smallest Q
//     limb_i = d(i,j) / 2 + (r_i - r_j) / (2 (m - 2)),  limb_j = d(i,j) - limb_i
//     d(u,k) = (d(i,k) + d(j,k) - d(i,j)) / 2                              the new node u takes slot i, slot j retires
// until three nodes are left, which are joined in a trifurcation -- and is checked against a CPU restatement of the same
// rules (oracle/nj_oracle.py; ties: smallest i, then smallest j; the exact tie between complementary pairs when four nodes
// are left is settled by looking only at the pairs of the smallest active index).
//
// Per join two launches and no host round trip: k_nj_rowmin (one block per row: the row's best partner) and k_nj_join
// (one block: best row, limb lengths, the O(n) update of row / column u and of the row sums, the join record).  The host
// replays the n - 3 join records into Newick once at the end.  Sum over joins of the active m^2 entries = n^3 / 3 reads:
// 21 GB at n = 2 000 (4 ms of HBM time; launch-bound at ~8 us per join), 21 TB at n = 20 000.
//
// Batches (ngsd_trees_batch; ngsd_nj_tree and ngsd_bme_tree are batches of one): every kernel takes its matrix from
// blockIdx.y and each matrix has its own working copy, row sums, active flags, node count, row minima, join records and
// `bad` flag, so one loop of n - 3 steps builds the trees of a whole chunk of matrices with the launches of one tree.
// The arithmetic, block sizes and tie rules of every matrix are those of a single tree, so every tree is byte-identical
// to the one the matrix gives alone.  A chunk is as many matrices as fit in the free device memory at call time.
#include <math.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <unordered_map>
#include <vector>

#include "ngsd_internal.h"

namespace {

__global__ void __launch_bounds__(256) k_nj_rowsum(const double *__restrict__ W, uint64_t ws, uint64_t n, double *__restrict__ r_all,
                                                   int *__restrict__ bad) {
  __shared__ double red[256];
  const uint64_t i = blockIdx.x;
  const double *__restrict__ D = W + blockIdx.y * ws;
  double *__restrict__ r = r_all + blockIdx.y * n;
  double s = 0;
  int nf = 0;
  for (uint64_t k = threadIdx.x; k < n; k += 256) {
    const double v = D[i * n + k];
    if (k != i) { s += v; nf |= !isfinite(v); }
  }
  red[threadIdx.x] = s;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int) threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) r[i] = red[0];
  if (nf) atomicOr(bad + blockIdx.y, 1);
}

// (Q, j) of the best partner j > i of row i; rows that are retired or have no partner report +inf
__global__ void __launch_bounds__(256, 6) k_nj_rowmin(const double *__restrict__ W, uint64_t ws, const double *__restrict__ r_all,
                                                   const uint8_t *__restrict__ active_all, uint64_t n, const uint32_t *__restrict__ m_all,
                                                   double *__restrict__ rowq_all, uint32_t *__restrict__ rowj_all) {
  __shared__ double sq[256];
  __shared__ uint32_t sj[256];
  const uint64_t i = blockIdx.x;
  const double *__restrict__ D = W + blockIdx.y * ws;
  const double *__restrict__ r = r_all + blockIdx.y * n;
  const uint8_t *__restrict__ active = active_all + blockIdx.y * n;
  if (!active[i]) {                                            // a retired row: no partner, and no block reduction to wait for
    if (threadIdx.x == 0) { rowq_all[blockIdx.y * n + i] = INFINITY; rowj_all[blockIdx.y * n + i] = 0xFFFFFFFFu; }
    return;
  }
  const uint32_t m = m_all[blockIdx.y];
  const double mm2 = (double) (m - 2);
  double best = INFINITY;
  uint32_t bj = 0xFFFFFFFFu;
  // With four nodes left Q(i,j) equals Q of the complementary pair exactly (both choices give the same unrooted tree, but
  // rounding would pick the Newick rooting at random): each of the three pairings is represented once, by the pair that
  // holds the smallest active index -- only that row takes part.
  bool skip_row = false;
  if (m == 4) {
    int f = 0;
    for (uint64_t k = threadIdx.x; k < i; k += 256) f |= active[k];
    skip_row = __syncthreads_or(f) != 0;
  }
  if (!skip_row) {
    const double ri = r[i];
    for (uint64_t j = i + 1 + threadIdx.x; j < n; j += 256) {
      if (!active[j]) continue;
      const double q = mm2 * D[i * n + j] - ri - r[j];
      if (q < best) { best = q; bj = (uint32_t) j; }          // ascending j per thread: the first minimum wins
    }
  }
  sq[threadIdx.x] = best;
  sj[threadIdx.x] = bj;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int) threadIdx.x < o) {
      const double q2 = sq[threadIdx.x + o];
      const uint32_t j2 = sj[threadIdx.x + o];
      if (q2 < sq[threadIdx.x] || (q2 == sq[threadIdx.x] && j2 < sj[threadIdx.x])) { sq[threadIdx.x] = q2; sj[threadIdx.x] = j2; }
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) { rowq_all[blockIdx.y * n + i] = sq[0]; rowj_all[blockIdx.y * n + i] = sj[0]; }
}

// one block per matrix (blockIdx.x)
__global__ void __launch_bounds__(1024) k_nj_join(double *__restrict__ W, uint64_t ws, double *__restrict__ r_all, uint8_t *__restrict__ active_all,
                                                  uint64_t n, uint32_t *__restrict__ m_all, const double *__restrict__ rowq_all,
                                                  const uint32_t *__restrict__ rowj_all, NjJoin *__restrict__ joins_all, uint32_t step) {
  __shared__ double sq[1024];
  __shared__ uint32_t si[1024];
  __shared__ double sred[1024];
  __shared__ uint32_t pick[2];
  double *__restrict__ D = W + blockIdx.x * ws;
  double *__restrict__ r = r_all + blockIdx.x * n;
  uint8_t *__restrict__ active = active_all + blockIdx.x * n;
  const double *__restrict__ rowq = rowq_all + blockIdx.x * n;
  const uint32_t *__restrict__ rowj = rowj_all + blockIdx.x * n;
  double best = INFINITY;
  uint32_t bi = 0xFFFFFFFFu;
  for (uint64_t i = threadIdx.x; i < n; i += 1024) {
    const double q = rowq[i];
    if (q < best) { best = q; bi = (uint32_t) i; }
  }
  sq[threadIdx.x] = best;
  si[threadIdx.x] = bi;
  __syncthreads();
  for (int o = 512; o > 0; o >>= 1) {
    if ((int) threadIdx.x < o) {
      const double q2 = sq[threadIdx.x + o];
      const uint32_t i2 = si[threadIdx.x + o];
      if (q2 < sq[threadIdx.x] || (q2 == sq[threadIdx.x] && i2 < si[threadIdx.x])) { sq[threadIdx.x] = q2; si[threadIdx.x] = i2; }
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) { pick[0] = si[0]; pick[1] = si[0] == 0xFFFFFFFFu ? 0xFFFFFFFFu : rowj[si[0]]; }
  __syncthreads();
  const uint64_t i = pick[0], j = pick[1];
  if (i == 0xFFFFFFFFu || j == 0xFFFFFFFFu) return;           // (non-finite input: reported by the caller)
  const uint32_t m = m_all[blockIdx.x];
  const double dij = D[i * n + j], ri = r[i], rj = r[j];
  double ru = 0;
  for (uint64_t k = threadIdx.x; k < n; k += 1024) {
    if (!active[k] || k == i || k == j) continue;
    const double dik = D[i * n + k], djk = D[j * n + k];
    const double duk = (dik + djk - dij) / 2;
    r[k] += duk - dik - djk;
    D[i * n + k] = duk;
    D[k * n + i] = duk;
    ru += duk;
  }
  sred[threadIdx.x] = ru;
  __syncthreads();
  for (int o = 512; o > 0; o >>= 1) {
    if ((int) threadIdx.x < o) sred[threadIdx.x] += sred[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const double li = dij / 2 + (ri - rj) / (2 * (double) (m - 2));
    joins_all[blockIdx.x * (n - 2) + step] = {(uint32_t) i, (uint32_t) j, li, dij - li};
    r[i] = sred[0];
    active[j] = 0;
    m_all[blockIdx.x] = m - 1;
  }
}

// one warp per matrix: the three slots left (in increasing order) and their distances
__global__ void __launch_bounds__(32) k_nj_last(const double *__restrict__ W, uint64_t ws, const uint8_t *__restrict__ active_all, uint64_t n,
                                                NjLast *__restrict__ last) {
  const double *__restrict__ D = W + blockIdx.x * ws;
  const uint8_t *__restrict__ active = active_all + blockIdx.x * n;
  uint32_t a = 0, b = 0, c = 0, found = 0;
  for (uint64_t base = 0; base < n && found < 3; base += 32) {
    const uint64_t k = base + threadIdx.x;
    uint32_t bits = __ballot_sync(0xFFFFFFFFu, k < n && active[k]);
    for (; bits && found < 3; bits &= bits - 1, found++) {
      const uint32_t x = (uint32_t) base + __ffs(bits) - 1;
      if (found == 0) a = x; else if (found == 1) b = x; else c = x;
    }
  }
  if (threadIdx.x == 0) last[blockIdx.x] = {{a, b, c}, 0, {D[a * n + b], D[a * n + c], D[b * n + c]}};
}

struct NjBuffers {
  double *r = nullptr, *rowq = nullptr;
  uint32_t *rowj = nullptr, *m = nullptr;
  uint8_t *active = nullptr;
  NjJoin *joins = nullptr;
  NjLast *last = nullptr;
  int *bad = nullptr;
  ~NjBuffers() { cudaFree(r); cudaFree(rowq); cudaFree(rowj); cudaFree(m); cudaFree(active); cudaFree(joins); cudaFree(last); cudaFree(bad); }
};

// device bytes of one matrix besides its working copy (NjBuffers)
uint64_t nj_bytes(uint64_t n) { return n * (2 * sizeof(double) + sizeof(uint32_t) + 1) + (n - 2) * sizeof(NjJoin) + sizeof(NjLast) + 8; }

// the join loop over `count` working copies (device, stride ws), each overwritten: one launch per kernel and step serves them all
int nj_chunk(ngsd_ctx *ctx, double *W, uint64_t ws, uint32_t count, NjBatch *out) {
  const uint64_t n = ctx->n_ind;
  cudaStream_t st = ctx->stream;
  NjBuffers b;
  NGSD_CUDA(ctx, cudaMalloc((void **) &b.r, count * n * sizeof(double)));
  NGSD_CUDA(ctx, cudaMalloc((void **) &b.rowq, count * n * sizeof(double)));
  NGSD_CUDA(ctx, cudaMalloc((void **) &b.rowj, count * n * sizeof(uint32_t)));
  NGSD_CUDA(ctx, cudaMalloc((void **) &b.m, count * sizeof(uint32_t)));
  NGSD_CUDA(ctx, cudaMalloc((void **) &b.active, count * n));
  NGSD_CUDA(ctx, cudaMalloc((void **) &b.joins, count * (n - 2) * sizeof(NjJoin)));
  NGSD_CUDA(ctx, cudaMalloc((void **) &b.last, count * sizeof(NjLast)));
  NGSD_CUDA(ctx, cudaMalloc((void **) &b.bad, count * sizeof(int)));
  const std::vector<uint32_t> m0(count, (uint32_t) n);
  NGSD_CUDA(ctx, cudaMemcpyAsync(b.m, m0.data(), count * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
  NGSD_CUDA(ctx, cudaMemsetAsync(b.active, 1, count * n, st));
  NGSD_CUDA(ctx, cudaMemsetAsync(b.bad, 0, count * sizeof(int), st));
  k_nj_rowsum<<<dim3((unsigned) n, count), 256, 0, st>>>(W, ws, n, b.r, b.bad);
  for (uint32_t step = 0; step + 3 < n + 0u; step++) {          // n - 3 joins: three nodes are left
    k_nj_rowmin<<<dim3((unsigned) n, count), 256, 0, st>>>(W, ws, b.r, b.active, n, b.m, b.rowq, b.rowj);
    k_nj_join<<<count, 1024, 0, st>>>(W, ws, b.r, b.active, n, b.m, b.rowq, b.rowj, b.joins, step);
  }
  k_nj_last<<<count, 32, 0, st>>>(W, ws, b.active, n, b.last);
  NGSD_CUDA(ctx, cudaGetLastError());
  out->n = (uint32_t) n;
  out->count = count;
  out->joins.resize(count * (n - 2));
  out->last.resize(count);
  out->bad.resize(count);
  NGSD_CUDA(ctx, cudaMemcpyAsync(out->joins.data(), b.joins, count * (n - 2) * sizeof(NjJoin), cudaMemcpyDeviceToHost, st));
  NGSD_CUDA(ctx, cudaMemcpyAsync(out->last.data(), b.last, count * sizeof(NjLast), cudaMemcpyDeviceToHost, st));
  NGSD_CUDA(ctx, cudaMemcpyAsync(out->bad.data(), b.bad, count * sizeof(int), cudaMemcpyDeviceToHost, st));
  NGSD_CUDA(ctx, cudaStreamSynchronize(st));
  return NGSD_OK;
}

void append_len(std::string &s, double v) {
  char b[64];
  snprintf(b, sizeof(b), ":%.10f", v);
  s += b;
}

// replay the joins of matrix k: the subtree living in every slot, as Newick text
std::string nj_newick(const NjBatch &nj, uint32_t k, const char *const *labels) {
  const uint32_t n = nj.n;
  std::vector<std::string> sub(n);
  for (uint64_t i = 0; i < n; i++) sub[i] = labels && labels[i] ? std::string(labels[i]) : "Ind_" + std::to_string(i);
  for (const NjJoin *jn = nj.joins.data() + (uint64_t) k * (n - 2), *e = jn + (n - 3); jn != e; jn++) {
    std::string s = "(" + sub[jn->i];
    append_len(s, jn->li);
    s += "," + sub[jn->j];
    append_len(s, jn->lj);
    s += ")";
    sub[jn->i].swap(s);
    sub[jn->j].clear();
  }
  const NjLast &l = nj.last[k];
  const double *d3 = l.d3;                                      // d(a,b), d(a,c), d(b,c)
  const double la = (d3[0] + d3[1] - d3[2]) / 2, lb = (d3[0] + d3[2] - d3[1]) / 2, lc = (d3[1] + d3[2] - d3[0]) / 2;
  std::string out = "(" + sub[l.rem[0]];
  append_len(out, la);
  out += "," + sub[l.rem[1]];
  append_len(out, lb);
  out += "," + sub[l.rem[2]];
  append_len(out, lc);
  out += ");";
  return out;
}

// one tree through the batch driver: ngsd_nj_tree and ngsd_bme_tree
int one_tree(ngsd_ctx *ctx, const double *dist_host, int method, const char *const *labels, char *newick, uint64_t newick_cap,
             uint64_t *newick_len, uint64_t *n_nni) {
  if (!ctx || !newick_len) return NGSD_ERR_ARG;
  if (!ctx->kids.empty()) ctx = ctx->kids[0];
  if (ctx->n_ind < 3) { ngsd_set_error(ctx, "a tree needs at least 3 individuals"); return NGSD_ERR_ARG; }
  if (!dist_host && !ctx->d_out) { ngsd_set_error(ctx, "no distance matrix yet: call ngsd_distances first or pass one"); return NGSD_ERR_STATE; }
  std::string out;
  uint64_t k = 0;
  int32_t status = NGSD_OK;
  if (int rc = ngsd_trees_run(ctx, dist_host, dist_host ? nullptr : ctx->d_out, 1, method, labels, &out, &k, &status)) return rc;
  if (status) { ngsd_set_error(ctx, "the distance matrix holds non-finite values (pairs without shared sites?): no tree"); return status; }
  if (n_nni) *n_nni = k;
  *newick_len = out.size();
  if (!newick || newick_cap < out.size() + 1) { ngsd_set_error(ctx, "newick buffer too small: %llu bytes needed", (unsigned long long) out.size() + 1); return NGSD_ERR_ARG; }
  memcpy(newick, out.c_str(), out.size() + 1);
  return NGSD_OK;
}

}  // namespace

int ngsd_trees_run(ngsd_ctx *ctx, const double *dist_host, const double *dist_dev, uint64_t n_mat, int method, const char *const *labels,
                   std::string *out, uint64_t *n_nni, int32_t *status) {
  const uint64_t n = ctx->n_ind, n2 = n * n;
  const bool bme = method == NGSD_TREE_BME;
  NGSD_CUDA(ctx, cudaSetDevice(ctx->device));
  // BME reuses NJ's working copy for its n (n + 1) prefix sums, and keeps the input matrix (a host matrix is uploaded once)
  const uint64_t ws = bme ? n * (n + 1) : n2;
  const bool upload_d = bme && dist_host;
  const uint64_t per = ws * sizeof(double) + (upload_d ? n2 * sizeof(double) : 0) + nj_bytes(n) + (bme ? ngsd_bme_bytes(n) : 0);
  size_t free_b = 0, total_b = 0;
  NGSD_CUDA(ctx, cudaMemGetInfo(&free_b, &total_b));
  const uint64_t reserve = 256ull << 20;                       // allocation granularity and whatever else the device needs meanwhile
  const uint64_t fit = free_b > reserve ? (free_b - reserve) / per : 0;
  const uint32_t C = (uint32_t) std::max<uint64_t>(1, std::min<uint64_t>({fit, n_mat, 65535}));   // (65535: gridDim.y)
  struct Chunk {
    double *W = nullptr, *D = nullptr;
    ~Chunk() { cudaFree(W); cudaFree(D); }
  } c;
  NGSD_CUDA(ctx, cudaMalloc((void **) &c.W, C * ws * sizeof(double)));
  if (upload_d) NGSD_CUDA(ctx, cudaMalloc((void **) &c.D, C * n2 * sizeof(double)));
  cudaStream_t st = ctx->stream;
  for (uint64_t c0 = 0; c0 < n_mat; c0 += C) {
    const uint32_t cnt = (uint32_t) std::min<uint64_t>(C, n_mat - c0);
    const double *src = dist_host ? dist_host + c0 * n2 : dist_dev;   // (a device matrix comes alone)
    if (upload_d) NGSD_CUDA(ctx, cudaMemcpyAsync(c.D, src, cnt * n2 * sizeof(double), cudaMemcpyHostToDevice, st));
    if (dist_host && !bme) {
      NGSD_CUDA(ctx, cudaMemcpyAsync(c.W, src, cnt * n2 * sizeof(double), cudaMemcpyHostToDevice, st));
    } else {
      const double *D = upload_d ? c.D : dist_dev;
      for (uint32_t k = 0; k < cnt; k++)
        NGSD_CUDA(ctx, cudaMemcpyAsync(c.W + k * ws, D + k * n2, n2 * sizeof(double), cudaMemcpyDeviceToDevice, st));
    }
    NjBatch nj;
    if (int rc = nj_chunk(ctx, c.W, ws, cnt, &nj)) return rc;
    for (uint32_t k = 0; k < cnt; k++) {
      status[c0 + k] = nj.bad[k] ? NGSD_ERR_ARG : NGSD_OK;
      n_nni[c0 + k] = 0;
      out[c0 + k].clear();
    }
    if (bme) {
      if (int rc = ngsd_bme_chunk(ctx, upload_d ? c.D : dist_dev, n2, c.W, ws, nj, labels, out + c0, n_nni + c0)) return rc;
    } else {
      ngsd_parallel_for(cnt, [&](uint64_t k) { if (!nj.bad[k]) out[c0 + k] = nj_newick(nj, (uint32_t) k, labels); });
    }
  }
  return NGSD_OK;
}

extern "C" int ngsd_trees_batch(ngsd_ctx *ctx, const double *dist_host, uint64_t n_mat, int32_t method, const char *const *labels, char *newicks,
                                uint64_t cap, uint64_t *offsets, uint64_t *n_nni, int32_t *status) {
  if (!ctx) return NGSD_ERR_ARG;
  if (n_mat == 0) {
    if (offsets) offsets[0] = 0;
    return NGSD_OK;
  }
  if (!dist_host) { ngsd_set_error(ctx, "no distance matrices: dist_host is NULL"); return NGSD_ERR_ARG; }
  if (!offsets || !status) { ngsd_set_error(ctx, "offsets and status are required"); return NGSD_ERR_ARG; }
  if (method != NGSD_TREE_NJ && method != NGSD_TREE_BME) { ngsd_set_error(ctx, "unknown tree method %d (NGSD_TREE_NJ or NGSD_TREE_BME)", (int) method); return NGSD_ERR_ARG; }
  const uint64_t n = (ctx->kids.empty() ? ctx : ctx->kids[0])->n_ind;
  if (n < 3) { ngsd_set_error(ctx, "a tree needs at least 3 individuals"); return NGSD_ERR_ARG; }
  std::vector<std::string> out(n_mat);
  std::vector<uint64_t> nni(n_mat, 0);
  const int rc = ctx->kids.empty() ? ngsd_trees_run(ctx, dist_host, nullptr, n_mat, method, labels, out.data(), nni.data(), status)
                                   : ngsd_group_trees(ctx, dist_host, n_mat, method, labels, out.data(), nni.data(), status);
  if (rc) return rc;
  uint64_t pos = 0;
  for (uint64_t k = 0; k < n_mat; k++) {
    offsets[k] = pos;
    pos += out[k].size() + 1;
  }
  offsets[n_mat] = pos;
  if (n_nni) memcpy(n_nni, nni.data(), n_mat * sizeof(uint64_t));
  if (!newicks || cap < pos) { ngsd_set_error(ctx, "newick buffer too small: %llu bytes needed", (unsigned long long) pos); return NGSD_ERR_ARG; }
  for (uint64_t k = 0; k < n_mat; k++) memcpy(newicks + offsets[k], out[k].c_str(), out[k].size() + 1);
  return NGSD_OK;
}

extern "C" int ngsd_nj_tree(ngsd_ctx *ctx, const double *dist_host, const char *const *labels, char *newick, uint64_t newick_cap,
                            uint64_t *newick_len) {
  return one_tree(ctx, dist_host, NGSD_TREE_NJ, labels, newick, newick_cap, newick_len, nullptr);
}

extern "C" int ngsd_bme_tree(ngsd_ctx *ctx, const double *dist_host, const char *const *labels, char *newick, uint64_t newick_cap,
                             uint64_t *newick_len, uint64_t *n_nni) {
  return one_tree(ctx, dist_host, NGSD_TREE_BME, labels, newick, newick_cap, newick_len, n_nni);
}

// ---------------------------------------------------------------------------------------------------------------------
// Bootstrap support: the last step of the reference's workflow (README.md:83-98 runs `raxmlHPC -f b -t main -z boots`).
// Host code only (no context, no device): Newick in, Newick with support labels on the internal nodes out.
// A bipartition is identified by the XOR of per-leaf 128-bit keys over one side (XOR with the key of all leaves gives the
// other side; the smaller of the two is the canonical one), so a tree is hashed in one pass and a replicate costs O(n).
namespace {

struct TsNode {
  int parent = -1;
  std::vector<int> kids;
  std::string label, length;                      // length: the text after ':' as it was written
  int leaf = -1;                                  // index of the leaf's label in the main tree's leaf order
  uint64_t h0 = 0, h1 = 0;                        // XOR of the leaf keys below
  uint32_t n_below = 0;
};

struct TsTree {
  std::vector<TsNode> nodes;                      // nodes[0] = root
  uint32_t n_leaves = 0;
};

inline uint64_t ts_mix(uint64_t z) {
  z += 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

// Newick subset: nested parentheses, unquoted or 'single-quoted' labels, optional ":length", optional labels on internal
// nodes (ignored), terminated by ';'.  Returns false on malformed input.
bool ts_parse(const char *s, TsTree *t) {
  t->nodes.clear();
  t->nodes.emplace_back();
  t->n_leaves = 0;
  int cur = 0;
  const char *p = s;
  auto skip_ws = [&]() { while (*p == ' ' || *p == '\t' || *p == '\n' || *p == '\r') p++; };
  auto read_label = [&](std::string *out) {
    skip_ws();
    out->clear();
    if (*p == '\'') {
      p++;
      while (*p && !(*p == '\'' && p[1] != '\'')) { if (*p == '\'') p++; out->push_back(*p++); }
      if (*p != '\'') return false;
      p++;
    } else {
      while (*p && !strchr("():,; \t\n\r", *p)) out->push_back(*p++);
    }
    return true;
  };
  auto read_length = [&](std::string *out) {
    skip_ws();
    out->clear();
    if (*p != ':') return;
    p++;
    skip_ws();
    while (*p && !strchr("(),; \t\n\r", *p)) out->push_back(*p++);
  };
  skip_ws();
  if (*p != '(') return false;
  int depth = 0;
  bool expect_node = true;                        // after '(' or ',': a subtree or a leaf must follow
  while (*p) {
    skip_ws();
    if (*p == '(') {
      if (!expect_node) return false;
      if (depth > 0) {                            // (the first '(' opens the root, node 0)
        TsNode n;
        n.parent = cur;
        t->nodes.push_back(n);
        const int id = (int) t->nodes.size() - 1;
        t->nodes[cur].kids.push_back(id);
        cur = id;
      }
      depth++;
      p++;
      expect_node = true;
    } else if (*p == ',') {
      if (expect_node || depth == 0) return false;
      p++;
      expect_node = true;
    } else if (*p == ')') {
      if (expect_node || depth == 0) return false;
      p++;
      depth--;
      std::string lab, len;
      if (!read_label(&lab)) return false;
      read_length(&len);
      t->nodes[cur].length = len;                 // (a label on an internal node is dropped: support goes there)
      if (depth == 0) {
        skip_ws();
        if (*p != ';') return false;
        break;
      }
      cur = t->nodes[cur].parent;
      expect_node = false;
    } else {
      if (!expect_node || depth == 0) return false;
      TsNode n;
      n.parent = cur;
      if (!read_label(&n.label) || n.label.empty()) return false;
      read_length(&n.length);
      n.leaf = 0;
      t->nodes.push_back(n);
      t->nodes[cur].kids.push_back((int) t->nodes.size() - 1);
      t->n_leaves++;
      expect_node = false;
    }
  }
  return depth == 0 && *p == ';' && t->n_leaves >= 2;
}

// leaf indices from `index` (label -> position), subtree hashes bottom-up.  false: unknown or repeated label
bool ts_hash(TsTree *t, const std::unordered_map<std::string, int> &index) {
  std::vector<uint8_t> seen(index.size(), 0);
  for (int v = (int) t->nodes.size() - 1; v >= 0; v--) {          // children always have larger ids than their parent
    TsNode &n = t->nodes[v];
    if (n.kids.empty()) {
      auto it = index.find(n.label);
      if (it == index.end() || seen[it->second]) return false;
      seen[it->second] = 1;
      n.leaf = it->second;
      n.h0 = ts_mix(2 * (uint64_t) n.leaf + 1);
      n.h1 = ts_mix(ts_mix(2 * (uint64_t) n.leaf + 2));
      n.n_below = 1;
    }
    if (n.parent >= 0) {
      TsNode &q = t->nodes[n.parent];
      q.h0 ^= n.h0;
      q.h1 ^= n.h1;
      q.n_below += n.n_below;
    }
  }
  return t->n_leaves == index.size();
}

struct TsKey {
  uint64_t a, b;
  bool operator==(const TsKey &o) const { return a == o.a && b == o.b; }
};
struct TsKeyHash {
  size_t operator()(const TsKey &k) const { return (size_t) (k.a ^ (k.b * 0x9E3779B97F4A7C15ull)); }
};

// canonical keys of the non-trivial bipartitions of a hashed tree, each once; node -> key index in `of_node` (or -1)
void ts_splits(const TsTree &t, std::vector<TsKey> *keys, std::vector<int> *of_node) {
  const TsNode &root = t.nodes[0];
  const uint64_t all0 = root.h0, all1 = root.h1;
  keys->clear();
  if (of_node) of_node->assign(t.nodes.size(), -1);
  std::unordered_map<TsKey, int, TsKeyHash> once;
  for (size_t v = 1; v < t.nodes.size(); v++) {
    const TsNode &n = t.nodes[v];
    if (n.kids.empty() || n.n_below < 2 || n.n_below + 2 > t.n_leaves) continue;   // trivial: a leaf or all but one leaf
    // canonical side: the smaller of the two keys (the side below, and everything else)
    const TsKey k1{n.h0, n.h1}, k2{n.h0 ^ all0, n.h1 ^ all1};
    const TsKey k = (k1.a < k2.a || (k1.a == k2.a && k1.b <= k2.b)) ? k1 : k2;
    auto it = once.find(k);
    int id;
    if (it == once.end()) {
      id = (int) keys->size();
      keys->push_back(k);
      once.emplace(k, id);
    } else {
      id = it->second;
    }
    if (of_node) (*of_node)[v] = id;
  }
}

void ts_write(const TsTree &t, int v, const std::vector<std::string> &support, std::string *out) {
  const TsNode &n = t.nodes[v];
  if (n.kids.empty()) {
    *out += n.label;
  } else {
    out->push_back('(');
    for (size_t k = 0; k < n.kids.size(); k++) {
      if (k) out->push_back(',');
      ts_write(t, n.kids[k], support, out);
    }
    out->push_back(')');
    *out += support[v];
  }
  if (!n.length.empty()) {
    out->push_back(':');
    *out += n.length;
  }
}

}  // namespace

extern "C" int ngsd_tree_support(const char *main_newick, const char *const *rep_newicks, uint64_t n_reps, int percent, char *out,
                                 uint64_t out_cap, uint64_t *out_len) {
  if (!main_newick || (n_reps && !rep_newicks) || !out_len) return NGSD_ERR_ARG;
  TsTree mt;
  if (!ts_parse(main_newick, &mt)) return NGSD_ERR_ARG;
  std::unordered_map<std::string, int> index;
  for (const TsNode &n : mt.nodes)
    if (n.kids.empty() && n.parent >= 0) {
      if (!index.emplace(n.label, (int) index.size()).second) return NGSD_ERR_ARG;     // repeated label
    }
  if (!ts_hash(&mt, index)) return NGSD_ERR_ARG;
  std::vector<TsKey> mkeys;
  std::vector<int> of_node;
  ts_splits(mt, &mkeys, &of_node);
  std::unordered_map<TsKey, uint64_t, TsKeyHash> count;
  for (const TsKey &k : mkeys) count.emplace(k, 0);
  uint64_t used = 0;
  TsTree rt;
  std::vector<TsKey> rkeys;
  for (uint64_t r = 0; r < n_reps; r++) {
    if (!rep_newicks[r]) return NGSD_ERR_ARG;
    if (!strcmp(rep_newicks[r], "NA")) continue;                   // a replicate without a tree (non-finite matrix) is skipped
    if (!ts_parse(rep_newicks[r], &rt) || !ts_hash(&rt, index)) return NGSD_ERR_ARG;
    ts_splits(rt, &rkeys, nullptr);
    for (const TsKey &k : rkeys) {
      auto it = count.find(k);
      if (it != count.end()) it->second++;
    }
    used++;
  }
  std::vector<std::string> support(mt.nodes.size());
  for (size_t v = 1; v < mt.nodes.size(); v++) {
    if (of_node[v] < 0) continue;
    const uint64_t c = count[mkeys[of_node[v]]];
    char buf[32];
    if (percent) snprintf(buf, sizeof buf, "%d", used ? (int) (0.5 + 100.0 * (double) c / (double) used) : 0);
    else snprintf(buf, sizeof buf, "%lu", (unsigned long) c);
    support[v] = buf;
  }
  std::string s;
  ts_write(mt, 0, support, &s);
  s.push_back(';');
  *out_len = s.size();
  if (!out || s.size() + 1 > out_cap) return NGSD_ERR_ARG;
  memcpy(out, s.c_str(), s.size() + 1);
  return NGSD_OK;
}
