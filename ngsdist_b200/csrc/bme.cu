// N4 (SURVEY §8f): balanced minimum-evolution refinement of the neighbour-joining tree, on the device.
//
// The reference's workflow (README.md:83-98) hands every matrix to FastME, whose criterion is balanced minimum evolution
// (BME; Desper & Gascuel 2002): the length of a tree is Pauplin's  L(T) = sum_{i<j} 2^(1 - tau_ij) d_ij,  tau_ij the number
// of edges between leaves i and j.  ngsd_bme_tree starts from the NJ tree (the join loop of nj.cu), applies the best BME
// nearest-neighbour interchange while its gain exceeds 1e-12 M, M = sum_{i<j} 2^(1 - tau_ij) |d_ij| (M = L when no distance is
// negative), and writes the tree with balanced branch lengths.  Every applied NNI lowers L, so no tree comes back and the
// loop ends for every finite matrix, whatever the signs of its entries; with M as the scale a matrix of all-equal negative
// distances (every gain exactly 0) stops at once instead of taking zero-gain moves.
//
// Rules (restated by oracle/bme_oracle.py; DESIGN §3 N4).  The tree is rooted at individual 0; internal node ids are the NJ
// join order (join t makes node n + t, the final trifurcation centre is 2n - 3) and an NNI renames nothing.  With
// P_ij = 2^-tau_ij d_ij and S_XY = sum_{i in X, j in Y} P_ij, every internal edge (u, v), v an internal child of u, has
//   A = everything not below u,  B = v's sibling,  C, D = v's children (C holds the smaller individual index)
//   gain(B<->C) = S_AB + S_CD - 2 (S_AC + S_BD)      gain(B<->D) = S_AB + S_CD - 2 (S_AD + S_BC)      (= L(T) - L(T'))
//   length(u, v) = 2 (S_AC + S_AD + S_BC + S_BD) - 2 (S_AB + S_CD)
// and the pendant edge of leaf i, whose neighbour's other two subtrees are X and Y, has length 2 (S_iX + S_iY - S_XY).
// One NNI per round, the largest gain (ties: smallest (v, variant), B<->C is variant 0).
//
// One round: the host lays the tree out in DFS order (children by smallest individual index) -- then B, C, D are one
// position range each and A at most two -- and uploads the O(n) layout; k_bme_rows writes, for every position p, the
// prefix sums R_p[q] = sum_{k<q} P_pk (tau from a running minimum of the LCA depths of neighbouring positions), and
// k_bme_gains evaluates every edge from O(|B| + |C| + |D|) differences of R and picks the best NNI with a deterministic
// last-block reduction.  One upload, two kernels and a 24-byte copy per round; k_bme_lengths gives the 2n - 3 lengths at
// the end.  A block sum S_XY = sum_{p in X} (R_p[hi] - R_p[lo]) is off by about eps times the absolute row totals of X, so
// every gain is good to about eps M, far inside the 1e-12 M acceptance threshold.
#include <math.h>
#include <string.h>

#include <array>
#include <string>
#include <vector>

#include "ngsd_internal.h"

namespace {

constexpr int kThreads = 256;
constexpr int kEdgeWords = 9;   // lo_u, hi_u, lo_B, hi_B, lo_C, hi_C, lo_D, hi_D, v
constexpr int kLeafWords = 7;   // p_i, lo_X, hi_X, and Y as two ranges

struct BmeBest { double gain, M; uint32_t key, pad; };   // best gain, sum of |P| over ordered pairs, 2 v + variant

// inclusive scan over the 256 threads of the block in thread order; `sh` holds 8 values and is free again on return
template <class T, class Op>
__device__ __forceinline__ T block_scan(T x, T *sh, Op op) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int o = 1; o < 32; o <<= 1) {
    const T y = __shfl_up_sync(0xFFFFFFFFu, x, o);
    if (lane >= o) x = op(y, x);
  }
  if (lane == 31) sh[w] = x;
  __syncthreads();
  T pre = sh[0];
  for (int k = 1; k < w; k++) pre = op(pre, sh[k]);
  if (w > 0) x = op(pre, x);
  __syncthreads();
  return x;
}

struct MinOp { __device__ uint32_t operator()(uint32_t a, uint32_t b) const { return a < b ? a : b; } };
struct AddOp { __device__ double operator()(double a, double b) const { return a + b; } };

// Row p of the DFS layout: R[p][0] = 0 and R[p][q + 1] = sum_{k <= q} P(perm[p], perm[k]), P = 2^-tau d, P_pp = 0, and
// Rabs[p] = sum_q |P(perm[p], perm[q])|.  The depth of the LCA of positions p < q is min(h[p .. q - 1]): a forward running minimum for q > p, a backward one for q < p.
// Slot blockIdx.y is tree act[slot]: its layout is slots[slot], its matrix, prefix rows and Rabs those of the tree.
__global__ void __launch_bounds__(kThreads) k_bme_rows(const double *__restrict__ D, uint64_t dstride, uint32_t n, const uint32_t *__restrict__ act,
                                                       const uint32_t *__restrict__ slots, uint64_t lay_words, double *__restrict__ R,
                                                       uint64_t rstride, double *__restrict__ Rabs_all) {
  __shared__ uint32_t shu[8];
  __shared__ double shd[8];
  __shared__ uint32_t carry_u;
  __shared__ double carry_d;
  const uint32_t t = act[blockIdx.y];
  const uint32_t *__restrict__ perm = slots + blockIdx.y * lay_words, *__restrict__ dep = perm + n, *__restrict__ h = perm + 2 * n;
  double *__restrict__ Rabs = Rabs_all + (uint64_t) t * n;
  const uint32_t p = blockIdx.x;
  const double *__restrict__ Drow = D + t * dstride + (uint64_t) perm[p] * n;
  double *__restrict__ Rrow = R + t * rstride + (uint64_t) p * (n + 1);
  const int dp = (int) dep[p];
  double a = 0;
  if (threadIdx.x == 0) { carry_u = 0xFFFFFFFFu; Rrow[0] = 0; Rrow[p + 1] = 0; }
  __syncthreads();
  for (uint32_t base = p + 1; base < n; base += kThreads) {
    const uint32_t q = base + threadIdx.x;
    uint32_t m = block_scan(q < n ? h[q - 1] : 0xFFFFFFFFu, shu, MinOp());
    m = min(m, carry_u);
    if (q < n) {
      const double x = ldexp(Drow[perm[q]], -(dp + (int) dep[q] - 2 * (int) m));
      Rrow[q + 1] = x;
      a += fabs(x);
    }
    __syncthreads();
    if (threadIdx.x == kThreads - 1) carry_u = m;
    __syncthreads();
  }
  if (threadIdx.x == 0) carry_u = 0xFFFFFFFFu;
  __syncthreads();
  for (uint32_t base = 0; base < p; base += kThreads) {
    const int64_t q = (int64_t) p - 1 - base - threadIdx.x;
    uint32_t m = block_scan(q >= 0 ? h[q] : 0xFFFFFFFFu, shu, MinOp());
    m = min(m, carry_u);
    if (q >= 0) {
      const double x = ldexp(Drow[perm[q]], -(dp + (int) dep[q] - 2 * (int) m));
      Rrow[q + 1] = x;
      a += fabs(x);
    }
    __syncthreads();
    if (threadIdx.x == kThreads - 1) carry_u = m;
    __syncthreads();
  }
  a = block_scan(a, shd, AddOp());
  if (threadIdx.x == kThreads - 1) Rabs[p] = a;
  if (threadIdx.x == 0) carry_d = 0;
  __syncthreads();
  for (uint32_t base = 0; base < n; base += kThreads) {
    const uint32_t q = base + threadIdx.x;
    double s = block_scan(q < n ? Rrow[q + 1] : 0.0, shd, AddOp());
    s += carry_d;
    __syncthreads();
    if (q < n) Rrow[q + 1] = s;
    if (threadIdx.x == kThreads - 1) carry_d = s;
    __syncthreads();
  }
}

// sum over the block of six doubles; the result is valid in thread 0
__device__ __forceinline__ void block_sum6(double s[6]) {
  __shared__ double sh[8][6];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int k = 0; k < 6; k++)
    for (int o = 16; o > 0; o >>= 1) s[k] += __shfl_down_sync(0xFFFFFFFFu, s[k], o);
  if (lane == 0)
    for (int k = 0; k < 6; k++) sh[w][k] = s[k];
  __syncthreads();
  if (threadIdx.x == 0)
    for (int k = 0; k < 6; k++) {
      double t = sh[0][k];
      for (int j = 1; j < kThreads / 32; j++) t += sh[j][k];
      s[k] = t;
    }
}

// S_AB, S_CD, S_AC, S_BD, S_AD, S_BC of one internal edge (valid in thread 0); the rows are B, C and D, the columns the
// other ranges (A = [0, lo_u) and [hi_u, n))
__device__ __forceinline__ void edge_sums(const double *__restrict__ R, uint32_t n, const uint32_t *__restrict__ e, double s[6]) {
  const uint32_t lo_u = e[0], hi_u = e[1], lo_B = e[2], hi_B = e[3], lo_C = e[4], hi_C = e[5], lo_D = e[6], hi_D = e[7];
  for (int k = 0; k < 6; k++) s[k] = 0;
  for (uint32_t p = lo_B + threadIdx.x; p < hi_B; p += kThreads) {
    const double *Rr = R + (uint64_t) p * (n + 1);
    s[0] += Rr[lo_u] + (Rr[n] - Rr[hi_u]);
    s[3] += Rr[hi_D] - Rr[lo_D];
    s[5] += Rr[hi_C] - Rr[lo_C];
  }
  for (uint32_t p = lo_C + threadIdx.x; p < hi_C; p += kThreads) {
    const double *Rr = R + (uint64_t) p * (n + 1);
    s[1] += Rr[hi_D] - Rr[lo_D];
    s[2] += Rr[lo_u] + (Rr[n] - Rr[hi_u]);
  }
  for (uint32_t p = lo_D + threadIdx.x; p < hi_D; p += kThreads) {
    const double *Rr = R + (uint64_t) p * (n + 1);
    s[4] += Rr[lo_u] + (Rr[n] - Rr[hi_u]);
  }
  block_sum6(s);
}

__device__ __forceinline__ bool better(double g, uint32_t k, double g2, uint32_t k2) { return g > g2 || (g == g2 && k < k2); }

// One CTA per internal edge of slot blockIdx.y (tree act[slot]): its two gains, the better of them; the last CTA of the
// slot to finish reduces the tree's edges (and M) into best[slot]
__global__ void __launch_bounds__(kThreads) k_bme_gains(const double *__restrict__ R_all, uint64_t rstride, const double *__restrict__ Rabs_all,
                                                        uint32_t n, const uint32_t *__restrict__ act, const uint32_t *__restrict__ slots,
                                                        uint64_t lay_words, double *__restrict__ part_g_all, uint32_t *__restrict__ part_k_all,
                                                        uint32_t *__restrict__ ticket_all, BmeBest *__restrict__ best_all) {
  __shared__ bool last;
  __shared__ double sg[kThreads], sM[kThreads];
  __shared__ uint32_t sk[kThreads];
  const uint32_t t = act[blockIdx.y];
  const uint32_t *e = slots + blockIdx.y * lay_words + 3 * n + (uint64_t) blockIdx.x * kEdgeWords;
  double s[6];
  edge_sums(R_all + t * rstride, n, e, s);
  double *__restrict__ part_g = part_g_all + (uint64_t) t * n;
  uint32_t *__restrict__ part_k = part_k_all + (uint64_t) t * n, *__restrict__ ticket = ticket_all + t;
  if (threadIdx.x == 0) {
    const uint32_t v = e[8];
    const double g0 = s[0] + s[1] - 2 * (s[2] + s[3]), g1 = s[0] + s[1] - 2 * (s[4] + s[5]);
    const bool one = g1 > g0;
    part_g[blockIdx.x] = one ? g1 : g0;
    part_k[blockIdx.x] = 2 * v + (one ? 1 : 0);
    __threadfence();
    last = atomicAdd(ticket, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!last) return;
  __threadfence();
  double g = -INFINITY, M = 0;
  uint32_t k = 0xFFFFFFFFu;
  for (uint32_t b = threadIdx.x; b < gridDim.x; b += kThreads) {
    const double g2 = __ldcg(part_g + b);
    const uint32_t k2 = __ldcg(part_k + b);
    if (better(g2, k2, g, k)) { g = g2; k = k2; }
  }
  for (uint32_t p = threadIdx.x; p < n; p += kThreads) M += __ldcg(Rabs_all + (uint64_t) t * n + p);
  sg[threadIdx.x] = g; sk[threadIdx.x] = k; sM[threadIdx.x] = M;
  __syncthreads();
  for (int o = kThreads / 2; o > 0; o >>= 1) {
    if ((int) threadIdx.x < o) {
      if (better(sg[threadIdx.x + o], sk[threadIdx.x + o], sg[threadIdx.x], sk[threadIdx.x])) {
        sg[threadIdx.x] = sg[threadIdx.x + o];
        sk[threadIdx.x] = sk[threadIdx.x + o];
      }
      sM[threadIdx.x] += sM[threadIdx.x + o];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    best_all[blockIdx.y] = {sg[0], sM[0], sk[0], 0};
    *ticket = 0;
  }
}

// The 2n - 3 balanced lengths of slot blockIdx.y (tree act[slot]): CTA b < n_int is internal edge b, the others the pendant
// edges in `leaves` order
__global__ void __launch_bounds__(kThreads) k_bme_lengths(const double *__restrict__ R_all, uint64_t rstride, uint32_t n, uint32_t n_int,
                                                          const uint32_t *__restrict__ act, const uint32_t *__restrict__ slots, uint64_t lay_words,
                                                          double *__restrict__ len_all) {
  const double *__restrict__ R = R_all + act[blockIdx.y] * rstride;
  const uint32_t *__restrict__ edges = slots + blockIdx.y * lay_words + 3 * n, *__restrict__ leaves = edges + (uint64_t) n_int * kEdgeWords;
  double *__restrict__ len = len_all + blockIdx.y * 2 * (uint64_t) n;
  double s[6];
  if (blockIdx.x < n_int) {
    edge_sums(R, n, edges + (uint64_t) blockIdx.x * kEdgeWords, s);
    if (threadIdx.x == 0) len[blockIdx.x] = 2 * (s[2] + s[3] + s[4] + s[5]) - 2 * (s[0] + s[1]);
    return;
  }
  const uint32_t *f = leaves + (uint64_t) (blockIdx.x - n_int) * kLeafWords;
  const uint32_t pi = f[0], lo_X = f[1], hi_X = f[2], a0 = f[3], b0 = f[4], a1 = f[5], b1 = f[6];
  for (int k = 0; k < 6; k++) s[k] = 0;
  if (threadIdx.x == 0) {
    const double *Rr = R + (uint64_t) pi * (n + 1);
    s[0] = (Rr[hi_X] - Rr[lo_X]) + ((Rr[b0] - Rr[a0]) + (Rr[b1] - Rr[a1]));
  }
  for (uint32_t p = lo_X + threadIdx.x; p < hi_X; p += kThreads) {
    const double *Rr = R + (uint64_t) p * (n + 1);
    s[1] += (Rr[b0] - Rr[a0]) + (Rr[b1] - Rr[a1]);
  }
  block_sum6(s);
  if (threadIdx.x == 0) len[blockIdx.x] = 2 * (s[0] - s[1]);
}

// The tree rooted at individual 0: kid[w] of internal node w, ordered by smallest individual index after layout()
struct BmeTree {
  uint32_t n = 0, u0 = 0;                   // u0: the neighbour of individual 0
  std::vector<uint32_t> parent;
  std::vector<std::array<uint32_t, 2>> kid;
  std::vector<uint32_t> lo, hi, dep, minleaf, order;

  bool leaf(uint32_t w) const { return w < n; }

  // NJ joins -> adjacency -> rooted at individual 0
  void build(uint32_t n_, const NjJoin *joins, const uint32_t rem[3]) {
    n = n_;
    const uint32_t N = 2 * n - 2;
    std::vector<std::vector<uint32_t>> adj(N);
    std::vector<uint32_t> slot(n);
    for (uint32_t k = 0; k < n; k++) slot[k] = k;
    auto link = [&](uint32_t a, uint32_t b) { adj[a].push_back(b); adj[b].push_back(a); };
    for (uint32_t t = 0; t + 3 < n; t++) {
      link(n + t, slot[joins[t].i]);
      link(n + t, slot[joins[t].j]);
      slot[joins[t].i] = n + t;
    }
    for (int a = 0; a < 3; a++) link(2 * n - 3, slot[rem[a]]);
    parent.assign(N, 0xFFFFFFFFu);
    kid.assign(N, {0, 0});
    u0 = adj[0][0];
    std::vector<uint32_t> st{u0};
    parent[u0] = 0;
    while (!st.empty()) {
      const uint32_t w = st.back();
      st.pop_back();
      int c = 0;
      for (uint32_t x : adj[w])
        if (x != parent[w]) { parent[x] = w; kid[w][c++] = x; if (!leaf(x)) st.push_back(x); }
    }
  }

  // DFS positions (individual 0 first, children by smallest individual index), depths, and the per-round arrays:
  // perm[pos], dep of the leaf at pos, h[k] = depth of the LCA of positions k and k + 1
  void layout(uint32_t *perm, uint32_t *pdep, uint32_t *h) {
    const uint32_t N = 2 * n - 2;
    order.clear();
    std::vector<uint32_t> st{u0};
    while (!st.empty()) {                     // preorder, any child order
      const uint32_t w = st.back();
      st.pop_back();
      order.push_back(w);
      if (!leaf(w)) { st.push_back(kid[w][0]); st.push_back(kid[w][1]); }
    }
    minleaf.assign(N, 0);
    for (size_t k = order.size(); k-- > 0;) {
      const uint32_t w = order[k];
      if (leaf(w)) { minleaf[w] = w; continue; }
      if (minleaf[kid[w][1]] < minleaf[kid[w][0]]) std::swap(kid[w][0], kid[w][1]);
      minleaf[w] = minleaf[kid[w][0]];
    }
    lo.assign(N, 0); hi.assign(N, 0); dep.assign(N, 0);
    order.clear();
    dep[u0] = 1;
    st.assign(1, u0);
    uint32_t pos = 1;
    perm[0] = 0; pdep[0] = 0; h[0] = 0;
    lo[0] = 0; hi[0] = 1;
    while (!st.empty()) {                     // preorder, kid[0] first
      const uint32_t w = st.back();
      st.pop_back();
      order.push_back(w);
      if (leaf(w)) { lo[w] = pos; hi[w] = pos + 1; perm[pos] = w; pdep[pos] = dep[w]; pos++; continue; }
      dep[kid[w][0]] = dep[kid[w][1]] = dep[w] + 1;
      st.push_back(kid[w][1]);
      st.push_back(kid[w][0]);
    }
    for (size_t k = order.size(); k-- > 0;) {
      const uint32_t w = order[k];
      if (leaf(w)) continue;
      lo[w] = lo[kid[w][0]];
      hi[w] = hi[kid[w][1]];
      h[hi[kid[w][0]] - 1] = dep[w];
    }
  }

  // candidate sites: every internal node v but u0, in increasing id
  void edges(uint32_t *e) const {
    for (uint32_t v = n; v < 2 * n - 2; v++) {
      if (v == u0) continue;
      const uint32_t u = parent[v], B = kid[u][0] == v ? kid[u][1] : kid[u][0], C = kid[v][0], D = kid[v][1];
      const uint32_t w[kEdgeWords] = {lo[u], hi[u], lo[B], hi[B], lo[C], hi[C], lo[D], hi[D], v};
      memcpy(e, w, sizeof w);
      e += kEdgeWords;
    }
  }

  // pendant edges of leaves 0..n-1: X one subtree at the leaf's neighbour, Y the rest of it (at most two ranges)
  void leaves(uint32_t *f) const {
    for (uint32_t i = 0; i < n; i++, f += kLeafWords) {
      if (i == 0) {
        const uint32_t a = kid[u0][0], b = kid[u0][1];
        const uint32_t w[kLeafWords] = {0, lo[a], hi[a], lo[b], hi[b], 0, 0};
        memcpy(f, w, sizeof w);
        continue;
      }
      const uint32_t u = parent[i], X = kid[u][0] == i ? kid[u][1] : kid[u][0];
      const uint32_t w[kLeafWords] = {lo[i], lo[X], hi[X], 0, lo[u], hi[u], n};
      memcpy(f, w, sizeof w);
    }
  }

  void nni(uint32_t key) {
    const uint32_t v = key >> 1, u = parent[v];
    const int bi = kid[u][0] == v ? 1 : 0, ci = (int) (key & 1);
    const uint32_t B = kid[u][bi], C = kid[v][ci];
    kid[u][bi] = C; parent[C] = u;
    kid[v][ci] = B; parent[B] = v;
  }
};

void append_len(std::string &s, double v) {
  char b[64];
  snprintf(b, sizeof(b), ":%.10f", v);
  s += b;
}

// the Newick string of a refined tree from its 2n - 3 lengths (internal edges in increasing v skipping u0, then the leaves)
std::string bme_newick(const BmeTree &t, const double *len, const char *const *labels) {
  const uint32_t n = t.n, n_int = n - 3;
  // length of the edge above every node (individual 0: its pendant edge)
  std::vector<double> above(2 * n - 2, 0.0);
  for (uint32_t v = n, e = 0; v < 2 * n - 2; v++)
    if (v != t.u0) above[v] = len[e++];
  for (uint32_t i = 0; i < n; i++) above[i] = len[n_int + i];
  auto label = [&](uint32_t k) { return labels && labels[k] ? std::string(labels[k]) : "Ind_" + std::to_string(k); };
  std::string out = "(" + label(0);
  append_len(out, above[0]);
  std::vector<std::pair<uint32_t, int>> stack;
  for (int c = 0; c < 2; c++) {
    out += ",";
    stack.assign(1, {t.kid[t.u0][c], 0});
    while (!stack.empty()) {
      const auto [w, s] = stack.back();
      stack.pop_back();
      if (t.leaf(w)) { out += label(w); append_len(out, above[w]); continue; }
      if (s == 0) { out += "("; stack.push_back({w, 1}); stack.push_back({t.kid[w][0], 0}); }
      else if (s == 1) { out += ","; stack.push_back({w, 2}); stack.push_back({t.kid[w][1], 0}); }
      else { out += ")"; append_len(out, above[w]); }
    }
  }
  out += ");";
  return out;
}

// per tree of a chunk: Rabs, part_g, len (2n) in doubles, part_k, the ticket and BmeBest; the device copy of the layouts
// (act, then one slot per tree) lives in `lay`, its pinned host twin in `hlay`
struct BmeBuffers {
  double *Rabs = nullptr, *part_g = nullptr, *len = nullptr;
  uint32_t *part_k = nullptr, *ticket = nullptr, *lay = nullptr, *hlay = nullptr;
  BmeBest *best = nullptr;
  ~BmeBuffers() { cudaFree(Rabs); cudaFree(part_g); cudaFree(len); cudaFree(part_k); cudaFree(ticket); cudaFree(lay); cudaFree(best); cudaFreeHost(hlay); }
};

uint64_t lay_words_of(uint64_t n) { return 3 * n + (n - 3) * kEdgeWords + n * kLeafWords; }   // perm, dep, h, the edges, the leaves

}  // namespace

uint64_t ngsd_bme_bytes(uint64_t n) {
  return n * (4 * sizeof(double) + sizeof(uint32_t)) + sizeof(uint32_t) + sizeof(BmeBest) + (1 + lay_words_of(n)) * sizeof(uint32_t);
}

// One round: the host applies each active tree's NNI and lays the tree out (one host thread per tree); one upload of all
// layouts; k_bme_rows and k_bme_gains over every active tree; one copy of a BmeBest per active tree.  A tree whose best
// gain is not above 1e-12 M leaves the active set with its R rows as its final layout left them; one k_bme_lengths pass
// over all trees ends the chunk.
int ngsd_bme_chunk(ngsd_ctx *ctx, const double *D, uint64_t dstride, double *R, uint64_t rstride, const NjBatch &nj, const char *const *labels,
                   std::string *out, uint64_t *n_nni) {
  const uint32_t n = nj.n, C = nj.count, n_int = n - 3;
  const uint64_t edge_end = 3 * (uint64_t) n + (uint64_t) n_int * kEdgeWords, lay_words = lay_words_of(n);
  cudaStream_t st = ctx->stream;
  BmeBuffers b;
  NGSD_CUDA(ctx, cudaMalloc((void **) &b.Rabs, (uint64_t) C * n * sizeof(double)));
  NGSD_CUDA(ctx, cudaMalloc((void **) &b.part_g, (uint64_t) C * n * sizeof(double)));
  NGSD_CUDA(ctx, cudaMalloc((void **) &b.len, (uint64_t) C * 2 * n * sizeof(double)));
  NGSD_CUDA(ctx, cudaMalloc((void **) &b.part_k, (uint64_t) C * n * sizeof(uint32_t)));
  NGSD_CUDA(ctx, cudaMalloc((void **) &b.ticket, C * sizeof(uint32_t)));
  NGSD_CUDA(ctx, cudaMalloc((void **) &b.lay, (C + C * lay_words) * sizeof(uint32_t)));
  NGSD_CUDA(ctx, cudaMalloc((void **) &b.best, C * sizeof(BmeBest)));
  NGSD_CUDA(ctx, cudaMallocHost((void **) &b.hlay, (C + C * lay_words) * sizeof(uint32_t)));
  NGSD_CUDA(ctx, cudaMemsetAsync(b.ticket, 0, C * sizeof(uint32_t), st));
  uint32_t *hact = b.hlay, *hslots = b.hlay + C;
  const uint32_t *dact = b.lay, *dslots = b.lay + C;
  std::vector<BmeTree> t(C);
  std::vector<uint32_t> act;                        // the trees still improving, in slot order
  for (uint32_t k = 0; k < C; k++) {
    if (nj.bad[k]) continue;
    t[k].build(n, nj.joins.data() + (uint64_t) k * (n - 2), nj.last[k].rem);
    act.push_back(k);
  }
  const std::vector<uint32_t> good = act;
  std::vector<BmeBest> hbest(C);
  while (!act.empty()) {
    const uint32_t A = (uint32_t) act.size();
    memcpy(hact, act.data(), A * sizeof(uint32_t));
    ngsd_parallel_for(A, [&](uint64_t s) {
      uint32_t *L = hslots + s * lay_words;
      t[act[s]].layout(L, L + n, L + 2 * n);
      t[act[s]].edges(L + 3 * n);
    });
    NGSD_CUDA(ctx, cudaMemcpyAsync(b.lay, b.hlay, (C + (A - 1) * lay_words + edge_end) * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    k_bme_rows<<<dim3(n, A), kThreads, 0, st>>>(D, dstride, n, dact, dslots, lay_words, R, rstride, b.Rabs);
    if (n_int == 0) {                               // three leaves: no internal edge, nothing to interchange
      NGSD_CUDA(ctx, cudaStreamSynchronize(st));
      break;
    }
    k_bme_gains<<<dim3(n_int, A), kThreads, 0, st>>>(R, rstride, b.Rabs, n, dact, dslots, lay_words, b.part_g, b.part_k, b.ticket, b.best);
    NGSD_CUDA(ctx, cudaGetLastError());
    NGSD_CUDA(ctx, cudaMemcpyAsync(hbest.data(), b.best, A * sizeof(BmeBest), cudaMemcpyDeviceToHost, st));
    NGSD_CUDA(ctx, cudaStreamSynchronize(st));
    uint32_t keep = 0;
    for (uint32_t s = 0; s < A; s++) {
      if (!(hbest[s].gain > 1e-12 * hbest[s].M)) continue;
      t[act[s]].nni(hbest[s].key);
      n_nni[act[s]]++;
      act[keep++] = act[s];
    }
    act.resize(keep);
  }
  const uint32_t G = (uint32_t) good.size();
  if (G == 0) return NGSD_OK;
  memcpy(hact, good.data(), G * sizeof(uint32_t));
  ngsd_parallel_for(G, [&](uint64_t s) {
    uint32_t *L = hslots + s * lay_words;
    t[good[s]].edges(L + 3 * n);
    t[good[s]].leaves(L + edge_end);
  });
  NGSD_CUDA(ctx, cudaMemcpyAsync(b.lay, b.hlay, (C + G * lay_words) * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
  k_bme_lengths<<<dim3(n_int + n, G), kThreads, 0, st>>>(R, rstride, n, n_int, dact, dslots, lay_words, b.len);
  NGSD_CUDA(ctx, cudaGetLastError());
  std::vector<double> len((uint64_t) G * 2 * n);
  NGSD_CUDA(ctx, cudaMemcpyAsync(len.data(), b.len, len.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
  NGSD_CUDA(ctx, cudaStreamSynchronize(st));
  ngsd_parallel_for(G, [&](uint64_t s) { out[good[s]] = bme_newick(t[good[s]], len.data() + s * 2 * n, labels); });
  return NGSD_OK;
}
