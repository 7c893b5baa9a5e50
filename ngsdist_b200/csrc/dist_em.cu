// K2b dist_em: the default --probs path of gen_dist, i.e. WITHOUT indep_geno (ngsDist.cpp:340-353): for every
// pair-site the 9-cell joint genotype table is re-estimated by em2() (emOptim2.cpp:112-135; emStep2 :91-109,
// lik2 :77-89, normalize :69-75) from ONE site of data, tol 0.001, <= 50 iterations, and the distance term is
// sum(score o sfs_T).  That is not bilinear in (p_i, p_j), so it cannot be a GEMM (SURVEY D2); it runs on the FP64
// CUDA cores.
//
// Closed form (SURVEY App. C, validated there on 6e6 pair-sites and here against the oracle): with a uniform start,
// after t EM steps sfs_t = (a^t / S_a(t)) (x) (b^t / S_b(t)) with element-wise powers and S_x(t) = sum_g x_g^t, and the
// reference's log-likelihood after step t is log(S(t+1) / S(t)), S = S_a * S_b, S(0) = 9.  It stops at the first
// T in 1..49 with |log r_T - log r_{T-1}| < 0.001  <=>  rho_a(T) * rho_b(T) < e^0.001, where
//     rho_x(t) = S_x(t+1) * S_x(t-1) / S_x(t)^2   (>= 1 by log-convexity of power sums),
// else at T = 50.  Everything that depends on ONE individual is therefore separable from the pair:
//     rho_x(t), t = 1..49          the stopping sequence
//     ahat_x(t) = x^t / S_x(t)      the individual's factor of sfs_t
// and the pair-site term is  ahat_i(T)^T . score . ahat_j(T)  with T = first t whose rho product is below e^0.001.
//
// Kernel structure (k_dist_em3): one CTA owns a 64 x 64 tile of pairs and a range of 8-site chunks.  Per TWO sites it
// alternates
//   build : 2 sites x 128 individual-sites x EM steps 1..26 -> shared-memory tables (rho and ahat for rows and columns),
//           one thread per (site, individual, half of the steps); each individual-site also records t* (the last step
//           at which rho still rises), the search interval [lo, hi] of the stop and its state at step 27;
//   pairs : every thread finds T for its 8 pairs per site by bisection on the rho tables -- valid because rho_i * rho_j
//           is non-increasing beyond max(t*_i, t*_j) (the steps up to it are scanned linearly, which is rare: t* = 0
//           for > 96 % of Dirichlet individual-sites) -- and adds the pair term of the ahat factors at T (8 FMA).
//           A pair that has not stopped by step 26 continues by direct iteration from the saved state at step 27.
// A warp works on ONE row and 32 columns at a time, so row-table reads are broadcasts / few distinct addresses and
// column-table reads ([t][column] layout) are conflict-free whatever t each lane is at.  ~50 FP64 instructions per
// pair-site instead of ~200 for the direct iteration, and no data-dependent trip counts in the common case.
// Powers are taken of x / max(x) so nothing underflows; rho and ahat are scale invariant.
#include <algorithm>

#include "ngsd_internal.h"

namespace {

constexpr int kEdge = NGSD_EM_EDGE;             // pairs tile: 64 rows x 64 columns
constexpr int kIter = 50;                       // maxIter of em2 (ngsDist.cpp:349)
constexpr int kThreads = 512;                   // 16 warps: the kernel is bound by FP64 / shared-memory latency
constexpr double kExpTol = 1.0010005001667084;  // e^0.001 (tole of ngsDist.cpp:349)
constexpr double kRise = 1e-13;                 // a rho step counts as "rising" above rounding noise only
constexpr int kWin = 26;                        // EM steps held in the tables
constexpr int kWLd = 27;                        // row-table stride (odd: conflict-free build stores)

struct EmArgs {
  const double *Apack;          // packed posterior planes (A operand of dist_dmma, 3-plane layout)
  const double *weights;        // [NC*8] per-site bootstrap weights or nullptr
  const uint32_t *chunk_ids;    // active chunk list or nullptr (identity)
  const uint32_t *tiles;        // [n_tiles][2] (ti, tj) of the owned 64 x 64 tiles
  double *partials;             // [n_splits][n_tiles][64][64]
  uint64_t NC, n_sites;
  uint32_t n_chunks, n_splits, n_tiles;
  double K[9];                  // score folded with a2 = 1 - a0 - a1, b2 = 1 - b0 - b1 (see pair_term)
};

// 1 / s: MUFU.RCP64H seed (>= 20 bits) + two Newton steps (error ~1 ulp); s is a normal number in [1/3, 3] here.
__device__ __forceinline__ double fast_rcp(double s) {
  double x;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(x) : "d"(s));
  double e = fma(-s, x, 1.0);
  x = fma(x, e, x);
  e = fma(-s, x, 1.0);
  return fma(x, e, x);
}

struct Pow3 { double v0, v1, v2; };
__device__ __forceinline__ Pow3 mul3(const Pow3 &a, const Pow3 &b) { return {a.v0 * b.v0, a.v1 * b.v1, a.v2 * b.v2}; }
__device__ __forceinline__ double sum3(const Pow3 &a) { return (a.v0 + a.v1) + a.v2; }

// sum_{g1,g2} score[g1][g2] a_g1 b_g2 with a2 = 1 - a0 - a1 and b2 = 1 - b0 - b1 (both triples sum to one):
//   K0 + b0 K3 + b1 K4 + a0 (K1 + b0 K5 + b1 K6) + a1 (K2 + b0 K7 + b1 K8)          8 FMA
__device__ __forceinline__ double pair_term(const double (&K)[9], double a0, double a1, double b0, double b1) {
  const double r0 = fma(b1, K[6], fma(b0, K[5], K[1]));
  const double r1 = fma(b1, K[8], fma(b0, K[7], K[2]));
  const double r2 = fma(b1, K[4], fma(b0, K[3], K[0]));
  return fma(a0, r0, fma(a1, r1, r2));
}

// ---------------------------------------------------------------------------------------------------------------------
// k_dist_em3 (round 2): the closed form above with three changes that follow from measurements of the round-1 kernel
// k_dist_em (50-step tables, one site per build / pairs round; since removed).
//  * ncu + arithmetic: the build was FP64-pipe bound (128 individual-sites x 50 steps per 4096 pairs), the pair phase
//    shared-memory bound (12 LDS.64 per pair in the bisection + 4 for the factors).  On the bench data 99.9 % of the pairs
//    stop within 26 EM steps (mean 7.8) -- but nearly every 64 x 64 tile has one pair that does not, so windowing the
//    tables per tile does not help (tried: k_dist_em2, 164 ms against 115 ms).  Instead:
//  * tables hold steps 1..26 only (half the build); a pair without a stop by then (0.08 %) continues by DIRECT iteration
//    from the two individuals' saved state at step 27 (x, x^27, S(26), S(27)) -- the same recurrences, so the same T;
//  * every individual-site also records  lo = first t with rho < e^0.001  and  hi = 1 + last t with rho >= e^0.0005.
//    rho >= 1 always (log-convexity of power sums), hence a pair can only stop at t >= max(lo_i, lo_j) and has stopped
//    by max(hi_i, hi_j): the bisection runs on that interval -- typically 1-3 steps wide instead of 26 -- and rounds in
//    which no lane of the warp can move are skipped.  (Margins of 1e-9 on both thresholds keep rounding out of it: the
//    interval always holds the first t whose rho product, of the same values, is below e^0.001.)
//  * with 26-step tables two sites fit in shared memory at once: one barrier pair per TWO sites and twice the
//    independent work per phase.
constexpr int kW_RhoRow = 0;                                 // [64][27]     rho of row r at step t:    [r * 27 + t]        t = 1..26
constexpr int kW_RhoCol = kW_RhoRow + kEdge * kWLd;          // [27][64]     rho of column c at step t: [t * 64 + c]
constexpr int kW_FacRow = kW_RhoCol + (kWin + 1) * kEdge;    // [2][64][27]  ahat_g of row r:           [(g * 64 + r) * 27 + t - 1]
constexpr int kW_FacCol = kW_FacRow + 2 * kEdge * kWLd;      // [26][2][64]  ahat_g of column c:        [((t - 1) * 2 + g) * 64 + c]
constexpr int kW_Tail = kW_FacCol + kWin * 2 * kEdge;        // [128][8]     x0 x1 x2, x^27 (3), S(26), S(27) per individual
constexpr int kW_Doubles = kW_Tail + 128 * 8;                // 11200 doubles = 87.5 KiB per site
constexpr int k3_Raw = 2 * kW_Doubles;                       // staged chunk (also absorbs the masked over-reads of the bisection)
constexpr int k3_Wgt = k3_Raw + 2 * 6 * 256;
constexpr int k3_Doubles = k3_Wgt + 8;
constexpr size_t kSmem3Bytes = (size_t) k3_Doubles * 8 + 2 * 4 * 128 * sizeof(int);   // per site: tstar, lo, hi, valid [128] each
constexpr double kTolLo = kExpTol * (1.0 + 1e-9);            // a single rho below this is necessary for a stop
constexpr double kSqrtTolHi = 1.0005001250208359 * (1.0 - 1e-9);   // e^0.0005: both rho below this is sufficient

struct TailState { Pow3 x, p; double Sp, Sc; };

// EM steps of one half (qtr: t = 1..13 or 14..26) of one individual-site.  SIDE 0 = row of the tile (tables indexed
// [individual][t]), 1 = column ([t][individual]).  Stores rho(t) and the factors ahat(t) of these steps and returns t*
// (the last step at which rho rises); also gives lo / hi of this thread's steps (first t with rho < kTolLo, 1 + last t
// with rho >= kSqrtTolHi) and, from the second half, the state at t = 27.  A rolled two-step loop keeps the kernel
// inside the instruction cache without register moves.
template <int SIDE>
__device__ __forceinline__ int build_steps26(const Pow3 &x, int qtr, double *rho_t, double *fac, int *lo_out, int *hi_out, TailState *tail) {
  constexpr int RS = SIDE == 0 ? 1 : kEdge;
  constexpr int FS = SIDE == 0 ? 1 : 2 * kEdge;
  constexpr int FG = SIDE == 0 ? kEdge * kWLd : kEdge;
  Pow3 p;
  double Sp, Sc, rp;
  int t;
  if (qtr == 0) {
    p = x; Sp = 3.0; Sc = sum3(x); rp = INFINITY; t = 1;
  } else {                                                              // x^12 by square-and-multiply, then two more steps
    const Pow3 x2 = mul3(x, x), x4 = mul3(x2, x2), x8 = mul3(x4, x4);
    const Pow3 b = mul3(x8, x4);
    t = 14;
    const double Sm2 = sum3(b);
    const Pow3 pm1 = mul3(b, x);
    Sp = sum3(pm1);
    p = mul3(pm1, x);
    Sc = sum3(p);
    const double ip = fast_rcp(Sp);
    rp = ((Sc * Sm2) * ip) * ip;                                        // rho(13)
  }
  int tstar = 0, lo = 99, hi = 0;
  rho_t += t * RS;
  fac += (t - 1) * FS;
  auto step = [&](const Pow3 &pc, double Spv, double Scv, double rpv, Pow3 &pn, double &Snv, double &rhov, int tt, int off) {
    pn = mul3(pc, x);
    Snv = sum3(pn);
    const double inv = fast_rcp(Scv);
    rhov = ((Snv * Spv) * inv) * inv;
    if (rhov - rpv > kRise) tstar = tt;
    if (rhov < kTolLo) lo = min(lo, tt);
    if (!(rhov < kSqrtTolHi)) hi = tt + 1;
    rho_t[off * RS] = rhov;
    fac[off * FS] = pc.v0 * inv;
    fac[off * FS + FG] = pc.v1 * inv;
  };
  {                                                                     // 13 steps: one, then six pairs (ping-pong, no register moves)
    Pow3 n; double Sn, rho;
    step(p, Sp, Sc, rp, n, Sn, rho, t, 0);
    p = n; Sp = Sc; Sc = Sn; rp = rho;
    t++; rho_t += RS; fac += FS;
  }
#pragma unroll 1
  for (int k = 6; k > 0; k--) {
    Pow3 n; double Sn, rho;
    step(p, Sp, Sc, rp, n, Sn, rho, t, 0);
    step(n, Sc, Sn, rho, p, Sp, rp, t + 1, 1);                          // now p = x^(t+2), Sp(out) = S(t+2), rp = rho(t+1)
    const double S1 = Sn;
    Sc = Sp; Sp = S1;
    t += 2; rho_t += 2 * RS; fac += 2 * FS;
  }
  if (tail) { tail->x = x; tail->p = p; tail->Sp = Sp; tail->Sc = Sc; }   // state at t = 27: p = x^27, Sp = S(26), Sc = S(27)
  *lo_out = lo;
  *hi_out = hi;
  return tstar;
}

// 4 pairs of one thread for one site: rows r0 and r0 + 16, columns lane and lane + 32.
template <bool WEIGHTED>
__device__ __forceinline__ void pair_group26(const double *tb, const int *meta, const int (&tcol)[2], const int (&locol)[2], const int (&hicol)[2],
                                             const bool (&vcol)[2], bool diag, int r0, int lane, double w, const double (&K)[9], double *acc) {
  constexpr int L = kWin;
  const double *rho_row = tb + kW_RhoRow, *rho_col = tb + kW_RhoCol, *fac_row = tb + kW_FacRow, *fac_col = tb + kW_FacCol;
  const int *ts = meta, *lo = meta + 128, *hi = meta + 256, *valid = meta + 384;
  int pos[4], cap[4], tfix[4];
  bool ok[4];
  int wide = 0;                                         // widest search interval of this thread's pairs
#pragma unroll
  for (int e = 0; e < 4; e++) {
    const int h = e & 1, r = r0 + 16 * (e >> 1), cc = h * 32 + lane;
    ok[e] = (!diag || cc > r) && vcol[h] && valid[r] != 0;
    const int tm = min(max(ts[r], tcol[h]), L), lop = max(lo[r], locol[h]);
    cap[e] = ok[e] ? min(max(hi[r], hicol[h]), L + 1) : 0;              // the pair has stopped by cap (L + 1: not known to)
    pos[e] = ok[e] ? min(max(tm + 1, lop), L + 1) : 0;                   // ... and not before pos, once the prefix is scanned
    tfix[e] = 0;
    if (ok[e] && tm >= lop) {                           // rare: scan the non-monotone prefix
      for (int t = max(lop, 1); t <= tm; t++)
        if (rho_row[r * kWLd + t] * rho_col[t * kEdge + cc] < kExpTol) { tfix[e] = t; pos[e] = cap[e] = 0; break; }
    }
    wide = max(wide, cap[e] - pos[e]);
  }
  // first t in [pos, cap] whose rho product is below e^0.001 -- cap itself needs no test (every t < pos is known to be
  // above).  Rounds wider than the widest interval in the warp cannot move anybody and are skipped (warp-uniform); the
  // state is one int per pair, addresses are formed at the loads.
  wide = __reduce_max_sync(0xFFFFFFFFu, wide);
#pragma unroll
  for (int s = 16; s >= 1; s >>= 1) {
    if (s > wide) continue;
#pragma unroll
    for (int e = 0; e < 4; e++) {
      const int h = e & 1, r = r0 + 16 * (e >> 1), cc = h * 32 + lane;
      const int qn = pos[e] + s;                                        // probe t = qn - 1
      const double prod = rho_row[r * kWLd + qn - 1] * rho_col[(qn - 1) * kEdge + cc];
      if (qn <= cap[e] && !(prod < kExpTol)) pos[e] = qn;
    }
  }
  unsigned tailmask = 0;
#pragma unroll
  for (int e = 0; e < 4; e++) {
    const int h = e & 1, r = r0 + 16 * (e >> 1), cc = h * 32 + lane;
    const int l = tfix[e] ? tfix[e] : pos[e];
    const bool undecided = ok[e] && l > L;
    const int T1 = ((!ok[e] || undecided) ? 1 : l) - 1;
    const double a0 = fac_row[r * kWLd + T1], a1 = fac_row[(kEdge + r) * kWLd + T1];
    const double b0 = fac_col[(T1 * 2) * kEdge + cc], b1 = fac_col[(T1 * 2 + 1) * kEdge + cc];
    double d = pair_term(K, a0, a1, b0, b1);
    if (WEIGHTED) d *= w;
    if (ok[e] && !undecided) acc[e] += d;
    if (undecided) tailmask |= 1u << e;
  }
  if (tailmask) {                                        // rare (0.08 % of pairs): continue from step 27 with the individuals' saved state
    const double *tail = tb + kW_Tail;
    for (int e = 0; e < 4; e++) {
      if (!((tailmask >> e) & 1u)) continue;
      const int h = e & 1, r = r0 + 16 * (e >> 1), cc = h * 32 + lane;
      const double *sa = tail + r * 8, *sb = tail + (64 + cc) * 8;
      Pow3 xa = {sa[0], sa[1], sa[2]}, pa = {sa[3], sa[4], sa[5]}, xb = {sb[0], sb[1], sb[2]}, pb = {sb[3], sb[4], sb[5]};
      double Spa = sa[6], Sca = sa[7], Spb = sb[6], Scb = sb[7];
      double a0 = 0, a1 = 0, b0 = 0, b1 = 0;
      for (int t = kWin + 1;; t++) {                     // state at t: p = x^t, Sc = S(t), Sp = S(t - 1)
        const double ia = fast_rcp(Sca), ib = fast_rcp(Scb);
        bool stop = t == kIter;
        Pow3 na = pa, nb = pb;
        double Sna = 0, Snb = 0;
        if (!stop) {
          na = mul3(pa, xa); Sna = sum3(na);
          nb = mul3(pb, xb); Snb = sum3(nb);
          const double ra = ((Sna * Spa) * ia) * ia, rb = ((Snb * Spb) * ib) * ib;
          stop = ra * rb < kExpTol;
        }
        if (stop) { a0 = pa.v0 * ia; a1 = pa.v1 * ia; b0 = pb.v0 * ib; b1 = pb.v1 * ib; break; }
        pa = na; Spa = Sca; Sca = Sna;
        pb = nb; Spb = Scb; Scb = Snb;
      }
      double d = pair_term(K, a0, a1, b0, b1);
      if (WEIGHTED) d *= w;
      acc[e] += d;
    }
  }
}

// grid = n_splits * n_tiles (split-major) over the owned tile list; block 512
template <bool WEIGHTED>
__global__ void __launch_bounds__(kThreads, 1) k_dist_em3(EmArgs a) {
  extern __shared__ __align__(16) double sm[];
  double *raw = sm + k3_Raw, *wgt = sm + k3_Wgt;
  int *metab = reinterpret_cast<int *>(sm + k3_Doubles);                 // [2 sites][tstar, lo, hi, valid][128]

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t q = blockIdx.x / a.n_tiles, slot = blockIdx.x - q * a.n_tiles;
  const uint32_t ti = a.tiles[2 * slot], tj = a.tiles[2 * slot + 1];
  const bool diag = ti == tj;
  const uint32_t c0 = (uint32_t) (((uint64_t) q * a.n_chunks) / a.n_splits);
  const uint32_t c1 = (uint32_t) (((uint64_t) (q + 1) * a.n_chunks) / a.n_splits);

  // build role: 512 threads = 2 sites x 2 halves of the 26 steps x 2 sides x 64 individuals; the row / column warps of a
  // (site, half) are rotated over the four SM sub-partitions
  const int b_site = warp >> 3, b_half = (warp >> 2) & 1, b_role = ((warp & 3) + b_half) & 3, b_side = b_role >> 1, b_k = (b_role & 1) * 32 + lane;
  double K[9];
#pragma unroll
  for (int k = 0; k < 9; k++) K[k] = a.K[k];
  double acc[8];
#pragma unroll
  for (int k = 0; k < 8; k++) acc[k] = 0.0;

  for (uint32_t c = c0; c < c1; c++) {
    const uint64_t chunk = a.chunk_ids ? a.chunk_ids[c] : (uint64_t) c;
    __syncthreads();                                          // everyone is done with the previous chunk's staging
#pragma unroll
    for (int h = 0; h < 6; h++) {
      const int seg = h * 2 + (tid >> 8);
      const uint64_t gi0 = (uint64_t) (seg < 6 ? ti : tj) * kEdge;
      const double *src = a.Apack + ((gi0 >> 7) * a.NC + chunk) * (NGSD_K4_3 * NGSD_K4_DOUBLES) + (seg % 6) * 512 + ((gi0 & 127) >> 3) * 32;
      raw[seg * 256 + (tid & 255)] = src[tid & 255];
    }
    if (WEIGHTED && tid < NGSD_SC) wgt[tid] = a.weights[chunk * NGSD_SC + tid];
    __syncthreads();

    for (int s8 = 0; s8 < NGSD_SC; s8 += 2) {                 // two sites per build / pairs round
      // ================= build =================
      bool live[2];
      double wv[2];
#pragma unroll
      for (int k = 0; k < 2; k++) {
        wv[k] = WEIGHTED ? wgt[s8 + k] : 1.0;
        live[k] = chunk * NGSD_SC + s8 + k < a.n_sites && !(WEIGHTED && wv[k] == 0.0);   // CTA-uniform
      }
      if (!live[0] && !live[1]) continue;
      {
        int *meta = metab + b_site * 512;
        if (b_half == 0) { meta[b_side * 64 + b_k] = 0; meta[128 + b_side * 64 + b_k] = 99; meta[256 + b_side * 64 + b_k] = 0; }
      }
      __syncthreads();
      if (live[b_site]) {
        const int s = s8 + b_site;
        double *tb = sm + b_site * kW_Doubles;
        int *meta = metab + b_site * 512;
        const double *rw = raw + (b_side * 6 + (s >> 2)) * 256 + b_k * 4 + (s & 3);
        Pow3 x = {rw[0], rw[2 * 256], rw[4 * 256]};
        const double m = fmax(x.v0, fmax(x.v1, x.v2));
        const bool okx = m > 0;                                            // all-zero = padded or pairwise-deleted
        if (okx) {
          const double im = fast_rcp(m);
          x.v0 *= im; x.v1 *= im; x.v2 *= im;
          int tstar, lo, hi;
          TailState tl;
          if (b_side == 0) tstar = build_steps26<0>(x, b_half, tb + kW_RhoRow + b_k * kWLd, tb + kW_FacRow + b_k * kWLd, &lo, &hi, b_half ? &tl : nullptr);
          else tstar = build_steps26<1>(x, b_half, tb + kW_RhoCol + b_k, tb + kW_FacCol + b_k, &lo, &hi, b_half ? &tl : nullptr);
          const int ind = b_side * 64 + b_k;
          if (tstar) atomicMax(&meta[ind], tstar);
          if (lo < 99) atomicMin(&meta[128 + ind], lo);
          if (hi) atomicMax(&meta[256 + ind], hi);
          if (b_half) {
            double *td = tb + kW_Tail + ind * 8;
            td[0] = tl.x.v0; td[1] = tl.x.v1; td[2] = tl.x.v2; td[3] = tl.p.v0; td[4] = tl.p.v1; td[5] = tl.p.v2; td[6] = tl.Sp; td[7] = tl.Sc;
          }
        }
        if (b_half == 0) meta[384 + b_side * 64 + b_k] = okx ? 1 : 0;
      }
      __syncthreads();

      // ================= pairs: rows warp + 16 k (k = 0..3), columns lane + 32 h =================
#pragma unroll
      for (int k = 0; k < 2; k++) {
        if (!live[k]) continue;
        const double *tb = sm + k * kW_Doubles;
        const int *meta = metab + k * 512;
        int tcol[2], locol[2], hicol[2];
        bool vcol[2];
#pragma unroll
        for (int h = 0; h < 2; h++) {
          const int cidx = 64 + h * 32 + lane;
          tcol[h] = meta[cidx]; locol[h] = meta[128 + cidx]; hicol[h] = meta[256 + cidx]; vcol[h] = meta[384 + cidx] != 0;
        }
        pair_group26<WEIGHTED>(tb, meta, tcol, locol, hicol, vcol, diag, warp, lane, wv[k], K, acc);
        pair_group26<WEIGHTED>(tb, meta, tcol, locol, hicol, vcol, diag, warp + 32, lane, wv[k], K, acc + 4);
      }
      __syncthreads();
    }
  }

  double *dst = a.partials + ((uint64_t) q * a.n_tiles + slot) * (kEdge * kEdge);
#pragma unroll
  for (int k = 0; k < 4; k++)
#pragma unroll
    for (int h = 0; h < 2; h++) {
      const int r = warp + 16 * (k & 1) + 32 * (k >> 1), cc = h * 32 + lane;
      dst[r * kEdge + cc] = (!diag || r < cc) ? acc[(k >> 1) * 4 + (k & 1) * 2 + h] : 0.0;
    }
}

struct EmEpiArgs {
  const double *partials;     // [n_splits][n_tiles64][64][64]
  const uint32_t *slot;       // [n64][n64] position of the 64 x 64 tile (ti, tj) in the owned list (0xFFFFFFFF: not owned)
  uint32_t n64, n_tiles64;
  const double *split_w;      // [n_splits] weight of each split (bootstrap block cache) or nullptr
  const uint32_t *cnt;        // [n_pad][n_pad] or nullptr
  const uint32_t *cnt_cache;  // per-block counts [n_splits][n_tiles128][4][64][64] (bootstrap block cache) or nullptr
  const uint32_t *tile_index; // [RB][RB] position of the 128 x 128 tile (ti, tj) in K3's tile list
  uint32_t n_tiles128, RB;
  double *out, *num;
  uint64_t *cntout;
  uint64_t n_ind, n_pad, const_cnt, tot_sites;
  uint32_t n_splits;
  int evol_model;
};

// tail of gen_dist (ngsDist.cpp:372-401) for the EM path; fixed-order reduction over the K splits.  Pairs of tiles a
// tile shard does not own are left as ngsd_clear_outputs set them (0).
__global__ void __launch_bounds__(256) k_epilogue_em(EmEpiArgs a) {
  const uint64_t j = (uint64_t) blockIdx.x * 16 + (threadIdx.x & 15), i = (uint64_t) blockIdx.y * 16 + (threadIdx.x >> 4);
  if (i >= a.n_ind || j >= a.n_ind) return;
  if (i == j) {
    a.out[i * a.n_ind + i] = 0.0;
    if (a.num) a.num[i * a.n_ind + i] = 0.0;
    if (a.cntout) a.cntout[i * a.n_ind + i] = 0;
    return;
  }
  if (i > j) return;
  const uint32_t s = a.slot[(i / kEdge) * a.n64 + j / kEdge];
  if (s == 0xFFFFFFFFu) return;
  const double *src = a.partials + (uint64_t) s * (kEdge * kEdge) + (i % kEdge) * kEdge + j % kEdge;
  const uint64_t stride = (uint64_t) a.n_tiles64 * (kEdge * kEdge);
  double num = 0;
  if (a.split_w) {
    for (uint32_t q = 0; q < a.n_splits; q++) {
      const double w = a.split_w[q];
      if (w != 0.0) num += w * src[(uint64_t) q * stride];
    }
  } else {
    for (uint32_t q = 0; q < a.n_splits; q++) num += src[(uint64_t) q * stride];
  }
  uint64_t cnt = a.cnt ? (uint64_t) a.cnt[i * a.n_pad + j] : a.const_cnt;
  if (a.cnt_cache) {          // sum_b c[b] * cnt_b(i,j) from the 128 x 128 tile list of K3 (row-major upper triangle in bands)
    const uint32_t t = a.tile_index[(i >> 7) * a.RB + (j >> 7)];
    const int rr = (int) (i & 127), cc = (int) (j & 127);
    const uint32_t *pc = a.cnt_cache + ((uint64_t) t * 4 + (rr >> 6) * 2 + (cc >> 6)) * 4096 + (rr & 63) * 64 + (cc & 63);
    const uint64_t cstride = (uint64_t) a.n_tiles128 * 4 * 4096;
    cnt = 0;
    for (uint32_t q = 0; q < a.n_splits; q++) {
      const double w = a.split_w[q];
      if (w != 0.0) cnt += (uint64_t) w * (uint64_t) pc[(uint64_t) q * cstride];
    }
  }
  if (a.num) a.num[i * a.n_ind + j] = a.num[j * a.n_ind + i] = num;
  if (a.cntout) a.cntout[i * a.n_ind + j] = a.cntout[j * a.n_ind + i] = cnt;
  if (a.tot_sites > 0) cnt = a.tot_sites;
  double d = num / (double) cnt;
  if (a.evol_model == 1) d = -log(1 - d);
  else if (a.evol_model == 2) d = -log(1 - (d * 4 / 3)) * 3 / 4;
  a.out[i * a.n_ind + j] = a.out[j * a.n_ind + i] = d;
}

uint64_t em_n64(const ngsd_ctx *ctx) { return (ctx->n_ind + kEdge - 1) / kEdge; }

}  // namespace

uint64_t ngsd_em_split_doubles(const ngsd_ctx *ctx) { return (uint64_t) ctx->em_n_tiles * (kEdge * kEdge); }

// planned from the tiles this context owns, so that a tile shard still fills the SMs
uint32_t ngsd_em_splits(const ngsd_ctx *ctx, uint32_t n_chunks) {
  const uint64_t tiles = std::max<uint32_t>(ctx->em_n_tiles, 1);
  uint64_t want = ((uint64_t) 8 * ctx->n_sm + tiles - 1) / tiles;             // ~8 units per SM: short tail, 1 CTA per SM
  const uint64_t maxs = std::max<uint64_t>(1, n_chunks / 2);
  const uint64_t cap_mem = std::max<uint64_t>(1, ((uint64_t) 2 << 30) / (tiles * kEdge * kEdge * 8));
  want = std::max<uint64_t>(1, std::min(std::min(want, maxs), cap_mem));
  return (uint32_t) std::min<uint64_t>(want, 65535);
}

cudaError_t ngsd_launch_dist_em(ngsd_ctx *ctx, uint32_t n_chunks, uint32_t n_splits, bool weighted) {
  static bool attr_set[64] = {};
  if (!attr_set[ctx->device & 63]) {
    const void *fns[2] = {(const void *) k_dist_em3<false>, (const void *) k_dist_em3<true>};
    for (const void *f : fns) {
      cudaError_t e = cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) kSmem3Bytes);
      if (e != cudaSuccess) return e;
    }
    attr_set[ctx->device & 63] = true;
  }
  EmArgs a;
  a.Apack = ctx->Apack;
  a.weights = weighted ? ctx->d_weights : nullptr;
  a.chunk_ids = weighted ? ctx->d_chunk_ids : nullptr;
  a.tiles = ctx->d_em_tiles;
  a.partials = ctx->cur_partials;
  a.NC = ctx->NC;
  a.n_sites = ctx->n_sites;
  a.n_chunks = n_chunks;
  a.n_splits = n_splits;
  a.n_tiles = ctx->em_n_tiles;
  const double *D = ctx->cfg.score;   // D[g1 * 3 + g2], g1 = genotype of the row individual (i1 < i2, ngsDist.cpp:351-353)
  a.K[0] = D[8];
  a.K[1] = D[2] - D[8];
  a.K[2] = D[5] - D[8];
  a.K[3] = D[6] - D[8];
  a.K[4] = D[7] - D[8];
  a.K[5] = D[0] - D[2] - D[6] + D[8];
  a.K[6] = D[1] - D[2] - D[7] + D[8];
  a.K[7] = D[3] - D[5] - D[6] + D[8];
  a.K[8] = D[4] - D[5] - D[7] + D[8];
  const uint64_t grid = (uint64_t) n_splits * a.n_tiles;
  if (grid == 0 || grid > 0x7fffffffull) return cudaErrorInvalidConfiguration;
  if (weighted)
    k_dist_em3<true><<<(unsigned) grid, kThreads, kSmem3Bytes, ctx->stream>>>(a);
  else
    k_dist_em3<false><<<(unsigned) grid, kThreads, kSmem3Bytes, ctx->stream>>>(a);
  return cudaGetLastError();
}

cudaError_t ngsd_launch_epilogue_em(ngsd_ctx *ctx, uint32_t n_splits, uint64_t const_cnt, bool use_cnt) {
  EmEpiArgs a;
  a.partials = ctx->cur_partials;
  a.slot = ctx->d_em_slot;
  a.n64 = (uint32_t) em_n64(ctx);
  a.n_tiles64 = ctx->em_n_tiles;
  a.split_w = ctx->cur_split_w;
  a.cnt = (use_cnt && !ctx->cur_cnt_cache) ? ctx->d_cnt : nullptr;
  a.cnt_cache = use_cnt ? ctx->cur_cnt_cache : nullptr;
  a.tile_index = ctx->d_tile_index;
  a.n_tiles128 = ctx->n_tiles;
  a.RB = (uint32_t) ctx->RB;
  a.out = ctx->d_out;
  a.num = ctx->d_num;
  a.cntout = ctx->d_cntout;
  a.n_ind = ctx->n_ind;
  a.n_pad = ctx->n_pad;
  a.const_cnt = const_cnt;
  a.tot_sites = ctx->cfg.tot_sites;
  a.n_splits = n_splits;
  a.evol_model = ctx->cfg.evol_model;
  if (ctx->shard_world > 1) {
    cudaError_t e = ngsd_clear_outputs(ctx);
    if (e != cudaSuccess) return e;
  }
  const uint32_t n16 = (uint32_t) ((ctx->n_ind + 15) / 16);
  k_epilogue_em<<<dim3(n16, n16), 256, 0, ctx->stream>>>(a);
  return cudaGetLastError();
}
