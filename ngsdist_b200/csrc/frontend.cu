// K1 front end: raw genotype likelihoods -> packed FP64 operand planes + presence bit masks.
//
// Replaces, per individual-site (SURVEY §8a H2-H4, Appendix A):
//   shared/read_data.cpp:37-45 (binary) / :83-99 (text)  log-scale conversion + post_prob normalisation + NaN check
//   shared/gen_func.cpp:123-151,920-932                 conv_space, logsum, post_prob
//   ngsDist.cpp:165-174 + gen_func.cpp:73-98,886-914     call_geno (log space) and exp() back to normal space
//   shared/gen_func.cpp:862-868                         miss_data predicate (EPSILON = 1e-5)
// and writes what gen_dist (ngsDist.cpp:325-404) will contract: A = p, B = score.p in DMMA fragment order.
//
// HBM-bound by design: 24 B read + 48 B written per individual-site (32 B in pdel two-plane mode); one thread owns 4
// consecutive sites of one individual so that every global store is a full 32-byte sector and a warp stores 1 KiB
// contiguous per plane.
#include <algorithm>

#include "ngsd_internal.h"

namespace {

constexpr double kNegInfClamp = -1e15;               // "INF" of shared/gen_func.hpp:15
constexpr double kEps = 1e-5;                        // EPSILON, shared/gen_func.hpp:16
constexpr double kThird = 0x1.5555555555555p-2;      // exp(log(1/3)) as glibc evaluates it (SURVEY §8a H3)
constexpr uint64_t kTile3 = NGSD_K4_3 * NGSD_K4_DOUBLES;     // doubles per operand tile: three planes / planes == 2
constexpr uint64_t kTilePd2 = NGSD_K4_PD2 * NGSD_K4_DOUBLES; // pdel two-plane mode

// One 32-byte sector per instruction (sm_100 has 256-bit global stores: STG.E.ENL2.256); p must be 32-byte aligned.
__device__ __forceinline__ void st256(double *p, double a, double b, double c, double d) {
  asm volatile("st.global.v4.f64 [%0], {%1,%2,%3,%4};" ::"l"(p), "d"(a), "d"(b), "d"(c), "d"(d) : "memory");
}

struct FrontCfg {
  int kind;          // ngsd_input_kind
  int in_log;
  int call_geno;
  int pairwise_del;
  int planes;        // 3, or 2 (sum-to-one reduction, see ngsd_internal.h)
  int pdel2;         // pdel two-plane mode (planes == 3 chunks, 2 planes; ngsd_internal.h)
  double pl[2], pr[2], pV[4];   // its shifts l, r and V (row-major)
  int int_path;      // called genotypes: write 2-bit codes for dist_umma.cu instead of FP64 planes
  double N_thresh, call_thresh;
  double score[9];
  ngsd_deferred *defer;      // knife-edge triples handed to the host's libm (api.cu resolve_deferred)
  unsigned *defer_n;
  unsigned defer_cap;
  uint64_t *blank;           // [NW] bit = site came from an empty text line (read_data.cpp:58-59)
};

constexpr double kKnife = 1e-11;                     // half-width of the band around a comparison threshold that goes to the host

// An empty text line leaves the reference's geno at its -1e15 fill for every individual and skips post_prob
// (read_data.cpp:58-59): the host marks such a site with this NaN payload (doubles) or code -128 (genotypes).
__device__ __forceinline__ bool is_blank(double x0) { return (unsigned long long) __double_as_longlong(x0) == NGSD_BLANK_SITE_BITS; }

__device__ __forceinline__ void defer_triple(const FrontCfg &c, uint64_t site, uint64_t ind, double x0, double x1, double x2, int *err) {
  const unsigned k = atomicAdd(c.defer_n, 1u);
  if (k < c.defer_cap) {
    ngsd_deferred d;
    d.site = site; d.ind = (uint32_t) ind; d.flags = 0; d.x[0] = x0; d.x[1] = x1; d.x[2] = x2;
    c.defer[k] = d;
  } else {
    atomicOr(err, 8);        // list full: this triple keeps the device's own evaluation
  }
}

// |p0-p1| or |p1-p2| within kKnife of EPSILON while the other does not already decide miss_data (gen_func.cpp:862-868)
__device__ __forceinline__ bool miss_knife(const double p[3]) {
  const double d01 = fabs(p[0] - p[1]), d12 = fabs(p[1] - p[2]);
  return (fabs(d01 - kEps) < kKnife && d12 < kEps + kKnife) || (fabs(d12 - kEps) < kKnife && d01 < kEps + kKnife);
}

// Normal-space posterior triple of one individual-site, following the reference step by step.
// Returns false when a NaN was produced on the binary path (fatal in the reference).  *knife is set when one of the
// reference's comparisons (first strict maximum, exact tie, N_thresh, call_thresh, EPSILON) is within kKnife of flipping:
// the device's log / exp are within 1 ulp of glibc's, not identical, so those triples are re-evaluated on the host.
__device__ __forceinline__ bool posterior(const FrontCfg &c, double x0, double x1, double x2, double p[3], bool *knife) {
  double L[3] = {x0, x1, x2};
  *knife = false;
  const bool blank = is_blank(x0);
  if (blank) {
    L[0] = L[1] = L[2] = kNegInfClamp;      // the untouched fill; post_prob never ran
  } else if (!c.in_log) {
#pragma unroll
    for (int g = 0; g < 3; g++) {
      L[g] = log(L[g]);
      if (c.kind == NGSD_INPUT_BINARY_GL && L[g] == -INFINITY) L[g] = kNegInfClamp;   // conv_space, gen_func.cpp:127-128
    }
  }
  // logsum + post_prob (gen_func.cpp:135-151, 920-932)
  double M = L[0];
  M = (L[1] >= M ? L[1] : M);
  M = (L[2] >= M ? L[2] : M);
  double norm;
  if (blank) {
    norm = 0;
  } else if (M == -INFINITY) {
    norm = -INFINITY;
  } else {
    double sum = 0;
    sum += exp(L[0] - M);
    sum += exp(L[1] - M);
    sum += exp(L[2] - M);
    norm = log(sum) + M;
  }
#pragma unroll
  for (int g = 0; g < 3; g++) L[g] -= norm;
  bool ok = true;
  if (c.kind == NGSD_INPUT_BINARY_GL && (isnan(L[0]) || isnan(L[1]) || isnan(L[2]))) ok = false;   // read_data.cpp:42-45
  if (c.call_geno) {
    // array_max_pos / array_min_pos: first strict extremum (gen_func.cpp:73-98)
    int max_pos = 0, min_pos = 0;
    double mx = -INFINITY, mn = INFINITY;
#pragma unroll
    for (int g = 0; g < 3; g++) {
      if (L[g] > mx) { max_pos = g; mx = L[g]; }
      if (L[g] < mn) { min_pos = g; mn = L[g]; }
    }
    double max_pp = exp(L[max_pos]);
    if (L[min_pos] == L[max_pos]) max_pp = -1;                      // gen_func.cpp:895-897 (miss_data == 0)
    else {
      // runner-up within kKnife of the maximum (array_max_pos / the exact-tie test could go the other way), or max_pp
      // within kKnife of a threshold it is compared with
      const double second = max_pos == 0 ? fmax(L[1], L[2]) : max_pos == 1 ? fmax(L[0], L[2]) : fmax(L[0], L[1]);
      if (mx - second < kKnife || fabs(max_pp - c.N_thresh) < kKnife || fabs(max_pp - c.call_thresh) < kKnife) *knife = true;
    }
    bool to_missing = max_pp < c.N_thresh;                          // :903-905
    bool to_call = max_pp >= c.call_thresh;                         // :908-913
    if (to_call) {
#pragma unroll
      for (int g = 0; g < 3; g++) p[g] = (g == max_pos) ? 1.0 : 0.0;   // exp(-1e15) = 0, exp(log(1)) = 1
      return ok;
    }
    if (to_missing) {
      p[0] = p[1] = p[2] = kThird;                                  // exp(log(1/3))
      return ok;
    }
  }
#pragma unroll
  for (int g = 0; g < 3; g++) p[g] = exp(L[g]);                     // ngsDist.cpp:172-173
  if (!blank && miss_knife(p)) *knife = true;
  return ok;
}

// Fast path for the un-called front end (no call_geno): the same posterior without the round trip through log space.
//   normal-scale input : p_g = x_g / (x_0 + x_1 + x_2)                       [= exp(log x_g - logsum(log x))]
//   log-scale input    : e_g = exp(L_g - max L), p_g = e_g / (e_0 + e_1 + e_2)  [= exp(L_g - logsum(L))]
// Algebraically identical to post_prob + exp (gen_func.cpp:920-932, ngsDist.cpp:172-173); it differs from the
// reference's own rounding by <= ~|log p| * 2^-52 relative (the reference loses that much in "log(sum) + M"), far
// inside the 1e-9 budget on distances.  Reference corner cases are reproduced explicitly:
//   x_g == 0 -> p_g = 0 (exp(-1e15 - norm) underflows to 0);  all three 0 on the binary path -> exp(-1.125) each
//   (SURVEY App. E-11);  negative / NaN input -> NaN -> fatal on the binary path.
__device__ __forceinline__ bool posterior_fast(const FrontCfg &c, double x0, double x1, double x2, double p[3], bool *knife) {
  double e0 = x0, e1 = x1, e2 = x2;
  *knife = false;
  if (is_blank(x0)) {                           // exp(-1e15) three times (ngsDist.cpp:172-173 on the untouched fill)
    p[0] = p[1] = p[2] = 0.0;
    return true;
  }
  if (c.in_log) {
    double M = x0;
    M = (x1 >= M ? x1 : M);
    M = (x2 >= M ? x2 : M);
    if (M == -INFINITY) {                       // logsum returns -inf -> L - (-inf) = NaN (gen_func.cpp:144-145)
      p[0] = p[1] = p[2] = NAN;
      return c.kind != NGSD_INPUT_BINARY_GL;
    }
    e0 = (x0 == M) ? 1.0 : exp(x0 - M);
    e1 = (x1 == M) ? 1.0 : exp(x1 - M);
    e2 = (x2 == M) ? 1.0 : exp(x2 - M);
  } else {
    if (x0 < 0 || x1 < 0 || x2 < 0) e0 = NAN;   // log(negative) = NaN in the reference
    if (c.kind == NGSD_INPUT_BINARY_GL && x0 == 0 && x1 == 0 && x2 == 0) {
      p[0] = p[1] = p[2] = 0.32465246735834974;  // exp(-1.125): -1e15 - (-1e15 + log 3) after rounding
      *knife = c.planes == 2;                    // does not sum to one: the host records its deficit for the 2-plane contraction
      return true;
    }
  }
  const double sum = (e0 + e1) + e2;
  p[0] = e0 / sum;      // true divisions: x / x must give exactly 1 (hard calls stay hard)
  p[1] = e1 / sum;
  p[2] = e2 / sum;
  bool ok = true;
  if (c.kind == NGSD_INPUT_BINARY_GL && (isnan(p[0]) || isnan(p[1]) || isnan(p[2]))) ok = false;
  *knife = miss_knife(p);                       // x / sum and exp(log x - logsum) agree to ~1e-15: far inside the band
  return ok;
}

// Fast path of call_geno when N_thresh == call_thresh (every triple ends up called or missing; the integer path).
// call_geno (gen_func.cpp:886-914) only needs, in log space: the first strict maximum, the exact-tie test L[min] == L[max]
// and max_pp = exp(L[max]) against the thresholds.  log and "- norm" are monotone, so away from near-ties the order of
// the normalised logs is the order of the raw values, and max_pp = x_max / sum(x) to ~1e-13.  Returns false -- the
// caller then runs the reference's exact log-space sequence -- whenever rounding could make a difference: non-positive
// or non-finite input, two values (or max_pp and a threshold) within 1e-9 of each other.  code: 0..2 called, 3 missing.
__device__ __forceinline__ bool called_code_fast(const FrontCfg &c, double x0, double x1, double x2, unsigned &code) {
  const double kTie = 1e-9;
  unsigned mp = 0;
  double mx = x0, mn;
  if (x1 > mx) { mx = x1; mp = 1; }
  if (x2 > mx) { mx = x2; mp = 2; }
  mn = fmin(x0, fmin(x1, x2));
  double max_pp;
  if (!c.in_log) {
    const double sum = (x0 + x1) + x2;
    if (!(mn >= 0.0) || !(mx > 0.0) || !(sum < INFINITY)) return false;   // negatives, all zero, NaN, inf: reference corner cases
    // (a zero next to a positive maximum is harmless: log(0) = -1e15 / -inf stays the strict minimum after normalisation)
    if (mn == mx) {                                                  // all equal: max_pp = -1, max_pos = 0 (gen_func.cpp:895-897)
      if (-1.0 >= c.call_thresh) { code = 0u; return true; }
      if (-1.0 < c.N_thresh) { code = 3u; return true; }
      return false;
    }
    const double tol = kTie * mx;
    // a runner-up (or the minimum, for the all-equal test) within tol of the maximum could collapse onto it in log space
    const double second = mp == 0 ? fmax(x1, x2) : mp == 1 ? fmax(x0, x2) : fmax(x0, x1);
    if (mx - second <= tol) return false;
    max_pp = (c.N_thresh == 0.0 && c.call_thresh == 0.0) ? 1.0 : mx / sum;   // default thresholds: only the sign matters
  } else {
    if (!(mn > -INFINITY) || !(mx < INFINITY)) return false;
    if (mn == mx) {
      if (-1.0 >= c.call_thresh) { code = 0u; return true; }
      if (-1.0 < c.N_thresh) { code = 3u; return true; }
      return false;
    }
    const double tol = kTie * (1.0 + fabs(mx) + fabs(mn));
    const double second = mp == 0 ? fmax(x1, x2) : mp == 1 ? fmax(x0, x2) : fmax(x0, x1);
    if (mx - second <= tol) return false;
    if (c.N_thresh == 0.0 && c.call_thresh == 0.0) {
      max_pp = 1.0;                                                  // any positive value: only the sign matters
    } else {
      max_pp = 1.0 / ((exp(x0 - mx) + exp(x1 - mx)) + exp(x2 - mx));
    }
  }
  if (fabs(max_pp - c.N_thresh) <= kTie || fabs(max_pp - c.call_thresh) <= kTie) {
    if (!(c.N_thresh == 0.0 && c.call_thresh == 0.0)) return false;  // knife edge at a user threshold (SURVEY App. E-7)
  }
  if (max_pp >= c.call_thresh) { code = mp; return true; }           // gen_func.cpp:908-913
  if (max_pp < c.N_thresh) { code = 3u; return true; }               // gen_func.cpp:903-905
  return false;
}

// 4 codes of 2 bits -> the 4 selector nibbles of a byte permute (PRMT), i.e. the form k_dist_umma consumes them in:
// storing the codes spread once (codes4, 4 bits per site) saves its expander warps the same shuffle for every tile.
__device__ __forceinline__ unsigned spread8(unsigned b) {
  const unsigned s = (b | (b << 4)) & 0x0F0Fu;
  return (s | (s << 2)) & 0x3333u;
}

// Genotype-code input (read_data.cpp:88-95,98 followed by ngsDist.cpp:172-173): exact one-hot / uniform triples.
__device__ __forceinline__ bool posterior_from_code(int g, double p[3]) {
  if (g > 2) { p[0] = p[1] = p[2] = 0; return false; }
  if (g < 0) { p[0] = p[1] = p[2] = kThird; return true; }
  p[0] = (g == 0) ? 1.0 : 0.0; p[1] = (g == 1) ? 1.0 : 0.0; p[2] = (g == 2) ? 1.0 : 0.0;
  return true;
}

__device__ __forceinline__ bool miss_data(const double p[3]) {      // gen_func.cpp:862-868
  return fabs(p[0] - p[1]) < kEps && fabs(p[1] - p[2]) < kEps;
}

// Pdel two-plane operands of one individual-site: A = m (p0 + l0, p1 + l1), B = m V (p0 + r0, p1 + r1).  A present
// triple with a non-finite component poisons both coordinates (the form drops p2, and with it a NaN in p2 alone): its
// row and column turn NaN, as in the three-plane contraction.
__device__ __forceinline__ void pdel2_operands(const FrontCfg &c, const double p[3], bool present, double a[2], double b[2]) {
  if (!present) { a[0] = a[1] = b[0] = b[1] = 0.0; return; }
  double q0 = p[0] + c.pl[0], q1 = p[1] + c.pl[1], t0 = p[0] + c.pr[0], t1 = p[1] + c.pr[1];
  if (!(isfinite(p[0]) && isfinite(p[1]) && isfinite(p[2]))) q0 = q1 = t0 = t1 = NAN;
  a[0] = q0;
  a[1] = q1;
  b[0] = c.pV[0] * t0 + c.pV[1] * t1;
  b[1] = c.pV[2] * t0 + c.pV[3] * t1;
}

// grid (n_pad/32, ceil(n/64)); block (32 individuals, 16 site groups of 4) = one 64-site mask word per individual.
// EXACT = the reference's log-space sequence (needed by call_geno's comparisons); otherwise the fast path above.
template <bool EXACT>
__global__ void __launch_bounds__(512, EXACT ? 1 : 2) k_frontend(FrontCfg c, const double *__restrict__ raw, const int8_t *__restrict__ codes,
                                                      uint64_t n_ind, uint64_t site0, uint64_t n, uint64_t NC, uint64_t NW,
                                                      double *__restrict__ Apack, double *__restrict__ Bpack,
                                                      double *__restrict__ Cplane, uint64_t ldc,
                                                      uint64_t *__restrict__ mask, int *__restrict__ err) {
  __shared__ unsigned nib[16][32];
  const int tx = threadIdx.x, ty = threadIdx.y;
  const uint64_t i = (uint64_t) blockIdx.x * 32 + tx;
  const uint64_t word = site0 / 64 + blockIdx.y;
  const uint64_t s_local0 = (uint64_t) blockIdx.y * 64 + ty * 4;   // first of this thread's 4 sites, relative to site0

  double A[4][3];
  int code[4] = {-1, -1, -1, -1};
  // all loads first (12 independent 8-byte loads per thread; a warp reads 768 contiguous bytes per site)
#pragma unroll
  for (int q = 0; q < 4; q++) {
    const uint64_t sl = s_local0 + q;
    A[q][0] = A[q][1] = A[q][2] = 0;
    if (i < n_ind && sl < n) {
      if (codes) {
        code[q] = (int) codes[sl * n_ind + i];
      } else {
        const double *x = raw + (sl * n_ind + i) * 3;
        A[q][0] = x[0]; A[q][1] = x[1]; A[q][2] = x[2];
      }
    }
  }
  unsigned bits = 0;
  int bad = 0;
#pragma unroll
  for (int q = 0; q < 4; q++) {
    const uint64_t sl = s_local0 + q;
    bool present = false;
    if (i < n_ind && sl < n) {
      bool ok;
      double p[3];
      if (codes) {
        if (code[q] == NGSD_BLANK_SITE_CODE) {                     // empty text line: (0,0,0) after exp (read_data.cpp:58-59)
          p[0] = p[1] = p[2] = 0.0;
          ok = true;
          if (i == 0) { atomicOr((unsigned long long *) &c.blank[(site0 + sl) >> 6], 1ull << ((site0 + sl) & 63)); bad |= 4; }
        } else {
          ok = posterior_from_code(code[q], p);
        }
        if (!ok) bad |= 2;
      } else {
        bool knife;
        ok = EXACT ? posterior(c, A[q][0], A[q][1], A[q][2], p, &knife) : posterior_fast(c, A[q][0], A[q][1], A[q][2], p, &knife);
        if (!ok) bad |= 1;
        if (knife) defer_triple(c, site0 + sl, i, A[q][0], A[q][1], A[q][2], err);
        if (i == 0 && !c.call_geno && is_blank(A[q][0])) { atomicOr((unsigned long long *) &c.blank[(site0 + sl) >> 6], 1ull << ((site0 + sl) & 63)); bad |= 4; }
      }
      present = !miss_data(p);
      if (c.pairwise_del && !present) p[0] = p[1] = p[2] = 0;       // the skip of ngsDist.cpp:335-338, folded into the operands
      A[q][0] = p[0]; A[q][1] = p[1]; A[q][2] = p[2];
    }
    bits |= (present ? 1u : 0u) << q;
  }
  if (bad) atomicOr(err, bad);

  // packed stores: 32 bytes per plane per operand; B = score . p evaluated in the reference's g2 order (ngsDist.cpp:351-353)
  const uint64_t rb = i >> 7, r = i & 127;
  const uint64_t sgrp = site0 / 4 + (uint64_t) blockIdx.y * 16 + ty;     // global 4-site group
  if (c.pdel2) {
    // pdel two-plane: chunk of 8 sites, k4-group = g*2 + h, g = 0..1 (no C plane, no deficit list: a triple that does not
    // sum to one -- all-zero, blank -- is missing under --pairwise_del)
    const uint64_t chunk = sgrp >> 1, h = sgrp & 1;
    const uint64_t base = (rb * NC + chunk) * kTilePd2 + (r >> 3) * 32 + (r & 7) * 4;
    double Av[4][2], Bw[4][2];
#pragma unroll
    for (int q = 0; q < 4; q++) pdel2_operands(c, A[q], (bits >> q) & 1u, Av[q], Bw[q]);
#pragma unroll
    for (int g = 0; g < 2; g++) {
      const uint64_t o = base + (uint64_t) (g * 2 + h) * NGSD_K4_DOUBLES;
      st256(Apack + o, Av[0][g], Av[1][g], Av[2][g], Av[3][g]);
      st256(Bpack + o, Bw[0][g], Bw[1][g], Bw[2][g], Bw[3][g]);
    }
  } else {
    double Bv[3][4];
#pragma unroll
    for (int g = 0; g < 3; g++)
#pragma unroll
      for (int q = 0; q < 4; q++) {
        double b = c.score[3 * g + 0] * A[q][0];
        b += c.score[3 * g + 1] * A[q][1];
        b += c.score[3 * g + 2] * A[q][2];
        Bv[g][q] = b;
      }
    if (c.planes == 3) {
      const uint64_t chunk = sgrp >> 1, h = sgrp & 1;
      const uint64_t base = (rb * NC + chunk) * kTile3 + (r >> 3) * 32 + (r & 7) * 4;
#pragma unroll
      for (int g = 0; g < 3; g++) {
        const uint64_t o = base + (uint64_t) (g * 2 + h) * (16 * 32);
        st256(Apack + o, A[0][g], A[1][g], A[2][g], A[3][g]);
        st256(Bpack + o, Bv[g][0], Bv[g][1], Bv[g][2], Bv[g][3]);
      }
    } else {
      // two planes: A = (p0, p1), B = (B0 - B2, B1 - B2), C = B2; chunk of 12 sites, k4-group = g*3 + h
      const uint64_t chunk = sgrp / 3, h = sgrp % 3;
      const uint64_t base = (rb * NC + chunk) * kTile3 + (r >> 3) * 32 + (r & 7) * 4;
#pragma unroll
      for (int g = 0; g < 2; g++) {
        const uint64_t o = base + (uint64_t) (g * 3 + h) * (16 * 32);
        st256(Apack + o, A[0][g], A[1][g], A[2][g], A[3][g]);
        st256(Bpack + o, Bv[g][0] - Bv[2][0], Bv[g][1] - Bv[2][1], Bv[g][2] - Bv[2][2], Bv[g][3] - Bv[2][3]);
      }
      st256(Cplane + (word * ldc + i) * 64 + ty * 4, Bv[2][0], Bv[2][1], Bv[2][2], Bv[2][3]);   // [word][n_pad][64]: a site range is contiguous (all-gather)
    }
  }

  nib[ty][tx] = bits;
  __syncthreads();
  if (ty == 0) {
    uint64_t w = 0;
#pragma unroll
    for (int k = 0; k < 16; k++) w |= (uint64_t) nib[k][tx] << (4 * k);
    mask[(rb * NW + word) * 128 + r] = w;
  }
}

// The exact log-space sequence of the reference for one triple, out of line: the integer-path kernel below only needs
// it for the rare triples its fast test cannot decide, and inlining it would cost that kernel its occupancy.
// (scalars by value and the result in one word: passing the parameter struct by reference would spill it to local
// memory in every thread of the caller.)  Returns the code, + 4 when a NaN was found on the binary path.
__device__ __noinline__ unsigned called_code_exact(int kind, int in_log, double N_thresh, double call_thresh, double x0, double x1, double x2) {
  FrontCfg c;
  c.kind = kind; c.in_log = in_log; c.call_geno = 1; c.pairwise_del = 0; c.planes = 3; c.pdel2 = 0; c.int_path = 1;
  c.N_thresh = N_thresh; c.call_thresh = call_thresh;
  double p[3];
  bool knife;
  c.defer = nullptr; c.defer_n = nullptr; c.defer_cap = 0; c.blank = nullptr;
  const bool ok = posterior(c, x0, x1, x2, p, &knife);
  const unsigned code = (p[0] == 1.0) ? 0u : (p[1] == 1.0) ? 1u : (p[2] == 1.0) ? 2u : 3u;   // one-hot or the uniform "missing" triple
  return code | (ok ? 0u : 4u);
}

// Front end of the integer path (called genotypes / genotype input; dist_umma.cu): same thread mapping as k_frontend,
// but the only outputs are 2 bits per individual-site (codes [RB][NW][4][128], 16 sites per word, 3 = missing or
// padding) and the presence mask.  HBM-bound: 24 B (or 1 B of genotype code) read per individual-site, 0.4 B written.
__global__ void __launch_bounds__(512, 2) k_frontend_codes(FrontCfg c, const double *__restrict__ raw, const int8_t *__restrict__ codes,
                                                            uint64_t n_ind, uint64_t site0, uint64_t n, uint64_t NW,
                                                            uint32_t *__restrict__ codes_out, uint32_t *__restrict__ codes4_out,
                                                            uint64_t *__restrict__ mask, int *__restrict__ err) {
  __shared__ unsigned cod[16][32];
  const int tx = threadIdx.x, ty = threadIdx.y;
  const uint64_t i = (uint64_t) blockIdx.x * 32 + tx;
  const uint64_t word = site0 / 64 + blockIdx.y;
  const uint64_t s_local0 = (uint64_t) blockIdx.y * 64 + ty * 4;
  double A[4][3];
  int gc[4] = {-1, -1, -1, -1};
#pragma unroll
  for (int q = 0; q < 4; q++) {
    const uint64_t sl = s_local0 + q;
    A[q][0] = A[q][1] = A[q][2] = 0;
    if (i < n_ind && sl < n) {
      if (codes) {
        gc[q] = (int) codes[sl * n_ind + i];
      } else {
        const double *x = raw + (sl * n_ind + i) * 3;
        A[q][0] = x[0]; A[q][1] = x[1]; A[q][2] = x[2];
      }
    }
  }
  unsigned cbits = 0xFF;                  // 2 bits per site; 3 = missing / padding
  unsigned need_fp = 0;                   // sites the integer test below could not decide
  unsigned need_exact = 0;                // sites the FP64 fast test could not decide (near-ties, corner cases): rare
  int bad = 0;
  // Level 1 (normal-scale input, default thresholds: every triple ends up called or missing).  Non-negative finite
  // doubles order like their bit patterns, so the first strict maximum is decided on the high words alone whenever the
  // maximum's high word is >= 2 above the runner-up's (relative gap >= 2^-20, far outside the 1e-9 near-tie band of
  // called_code_fast); an all-equal positive normal triple is missing data (max_pp = -1 < N_thresh = 0,
  // gen_func.cpp:895-905).  Anything else -- negatives, NaN, inf, zeros, denormals, close calls -- goes to level 2.
  const bool level1 = !codes && !c.in_log && c.N_thresh == 0.0 && c.call_thresh == 0.0;
#pragma unroll
  for (int q = 0; q < 4; q++) {
    const uint64_t sl = s_local0 + q;
    if (i < n_ind && sl < n) {
      unsigned cg = 3u;
      if (codes) {
        cg = gc[q] < 0 ? 3u : (unsigned) gc[q];                      // read_data.cpp:88-95: -1 = missing
        if (gc[q] > 2) { bad |= 2; cg = 3u; }
      } else if (level1) {
        const unsigned h0 = (unsigned) __double2hiint(A[q][0]), h1 = (unsigned) __double2hiint(A[q][1]),
                       h2 = (unsigned) __double2hiint(A[q][2]);
        const unsigned m01 = max(h0, h1), mx = max(m01, h2), second = max(min(h0, h1), min(m01, h2));
        const unsigned lo_diff = ((unsigned) __double2loint(A[q][0]) ^ (unsigned) __double2loint(A[q][1])) |
                                 ((unsigned) __double2loint(A[q][1]) ^ (unsigned) __double2loint(A[q][2])) | (h0 ^ h1) | (h1 ^ h2);
        if (mx < 0x7FF00000u && mx - second >= 2u) {
          cg = h2 == mx ? 2u : (h1 == mx ? 1u : 0u);
        } else if (lo_diff == 0u && h0 - 0x00100000u < 0x7FE00000u) {
          cg = 3u;
        } else {
          need_fp |= 1u << q;
        }
      } else {
        need_fp |= 1u << q;
      }
      cbits = (cbits & ~(3u << (2 * q))) | (cg << (2 * q));
    }
  }
  if (need_fp) {                          // level 2: the FP64 test with the reference's tie / threshold semantics
#pragma unroll
    for (int q = 0; q < 4; q++) {
      if (!((need_fp >> q) & 1u)) continue;
      unsigned cg;
      if (!called_code_fast(c, A[q][0], A[q][1], A[q][2], cg)) {
        need_exact |= 1u << q;
        cg = 3u;
      }
      cbits = (cbits & ~(3u << (2 * q))) | (cg << (2 * q));
    }
  }
  if (need_exact) {                       // the reference's exact log-space sequence, values re-read (keeps the hot loop lean);
    for (int q = 0; q < 4; q++) {         // the host's libm has the last word on these triples (resolve_deferred)
      if (!((need_exact >> q) & 1u)) continue;
      const double *x = raw + ((s_local0 + q) * n_ind + i) * 3;
      if (is_blank(x[0])) continue;       // empty text line under call_geno: max_pp = -1 -> missing (code 3 is already set)
      defer_triple(c, site0 + s_local0 + q, i, x[0], x[1], x[2], err);
      unsigned cg = called_code_exact(c.kind, c.in_log, c.N_thresh, c.call_thresh, x[0], x[1], x[2]);
      if (cg & 4u) bad |= 1;
      cbits = (cbits & ~(3u << (2 * q))) | ((cg & 3u) << (2 * q));
    }
  }
  if (bad) atomicOr(err, bad);
  // presence nibble of this thread's 4 sites (miss_data of gen_func.cpp:862-868: exactly the code-3 entries)
  unsigned pres = ~(cbits & (cbits >> 1)) & 0x55u;
  pres = (pres | (pres >> 1)) & 0x33u;
  pres = (pres | (pres >> 2)) & 0x0Fu;
  cod[ty][tx] = cbits | (pres << 8);
  __syncthreads();
  const uint64_t rb = i >> 7, r = i & 127;
  if (ty < 4) {                           // word ty of this individual: sites 16 ty .. 16 ty + 15 of the 64-site word
    const unsigned w = (cod[4 * ty][tx] & 0xFFu) | ((cod[4 * ty + 1][tx] & 0xFFu) << 8) | ((cod[4 * ty + 2][tx] & 0xFFu) << 16) |
                       (cod[4 * ty + 3][tx] << 24);
    codes_out[((rb * NW + word) * 4 + ty) * 128 + r] = w;
  } else if (ty == 4) {                   // presence mask word: 16 nibbles
    unsigned mlo = 0, mhi = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) {
      mlo |= ((cod[k][tx] >> 8) & 0xFu) << (4 * k);
      mhi |= ((cod[k + 8][tx] >> 8) & 0xFu) << (4 * k);
    }
    mask[(rb * NW + word) * 128 + r] = ((uint64_t) mhi << 32) | mlo;
  } else if (ty >= 8) {                   // codes4 word ty - 8: sites 8 k .. 8 k + 7 as selector nibbles
    const int k = ty - 8;
    codes4_out[((rb * NW + word) * 8 + k) * 128 + r] = spread8(cod[2 * k][tx] & 0xFFu) | (spread8(cod[2 * k + 1][tx] & 0xFFu) << 16);
  }
}

// Genotype-code input on the integer path (read_data.cpp:88-95: codes {-1,0,1,2}, anything above 2 is an error): the same
// block shape and output as k_frontend_codes without any of its floating-point state, so that it is a ~20-register
// kernel that can share an SM with a persistent contraction CTA (a packed push overlapping another context's contraction).
__global__ void __launch_bounds__(512, 4) k_codes_from_int8(const int8_t *__restrict__ codes, uint64_t n_ind, uint64_t site0, uint64_t n, uint64_t NW,
                                                            uint32_t *__restrict__ codes_out, uint32_t *__restrict__ codes4_out,
                                                            uint64_t *__restrict__ mask, int *__restrict__ err, uint64_t *__restrict__ blank) {
  __shared__ unsigned cod[16][32];
  const int tx = threadIdx.x, ty = threadIdx.y;
  const uint64_t i = (uint64_t) blockIdx.x * 32 + tx;
  const uint64_t word = site0 / 64 + blockIdx.y;
  const uint64_t s_local0 = (uint64_t) blockIdx.y * 64 + ty * 4;
  unsigned cbits = 0xFF;                  // 2 bits per site; 3 = missing / padding
  int bad = 0;
#pragma unroll
  for (int q = 0; q < 4; q++) {
    const uint64_t sl = s_local0 + q;
    if (i < n_ind && sl < n) {
      const int g = (int) codes[sl * n_ind + i];
      unsigned cg = g < 0 ? 3u : (unsigned) g;                       // -1 = missing
      if (g > 2) { bad = 2; cg = 3u; }
      if (g == NGSD_BLANK_SITE_CODE && i == 0) {                     // empty text line: the site gets weight 0 in the contraction
        atomicOr((unsigned long long *) &blank[(site0 + sl) >> 6], 1ull << ((site0 + sl) & 63));
        bad |= 4;
      }
      cbits = (cbits & ~(3u << (2 * q))) | (cg << (2 * q));
    }
  }
  if (bad) atomicOr(err, bad);
  unsigned pres = ~(cbits & (cbits >> 1)) & 0x55u;                   // presence nibble of this thread's 4 sites
  pres = (pres | (pres >> 1)) & 0x33u;
  pres = (pres | (pres >> 2)) & 0x0Fu;
  cod[ty][tx] = cbits | (pres << 8);
  __syncthreads();
  const uint64_t rb = i >> 7, r = i & 127;
  if (ty < 4) {
    const unsigned w = (cod[4 * ty][tx] & 0xFFu) | ((cod[4 * ty + 1][tx] & 0xFFu) << 8) | ((cod[4 * ty + 2][tx] & 0xFFu) << 16) |
                       (cod[4 * ty + 3][tx] << 24);
    codes_out[((rb * NW + word) * 4 + ty) * 128 + r] = w;
  } else if (ty == 4) {
    unsigned mlo = 0, mhi = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) {
      mlo |= ((cod[k][tx] >> 8) & 0xFu) << (4 * k);
      mhi |= ((cod[k + 8][tx] >> 8) & 0xFu) << (4 * k);
    }
    mask[(rb * NW + word) * 128 + r] = ((uint64_t) mhi << 32) | mlo;
  } else if (ty >= 8) {
    const int k = ty - 8;
    codes4_out[((rb * NW + word) * 8 + k) * 128 + r] = spread8(cod[2 * k][tx] & 0xFFu) | (spread8(cod[2 * k + 1][tx] & 0xFFu) << 16);
  }
}

// Inspection: packed A planes + mask -> [ind][site][3] / [ind][site]
__global__ void k_unpack(const double *__restrict__ Apack, const uint32_t *__restrict__ codes, const uint64_t *__restrict__ mask,
                         uint64_t n_ind, uint64_t n_sites, uint64_t NC, uint64_t NW, int planes, int pdel2, double l0, double l1,
                         double *__restrict__ P, uint8_t *__restrict__ miss) {
  const uint64_t idx = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n_ind * n_sites) return;
  const uint64_t i = idx / n_sites, s = idx % n_sites;
  const uint64_t rb = i >> 7, r = i & 127, sgrp = s >> 2, q = s & 3;
  const bool present = (mask[(rb * NW + (s >> 6)) * 128 + r] >> (s & 63)) & 1;
  if (P) {
    if (codes) {
      const unsigned code = (codes[((rb * NW + (s >> 6)) * 4 + ((s >> 4) & 3)) * 128 + r] >> (2 * (s & 15))) & 3u;
      for (unsigned g = 0; g < 3; g++) P[idx * 3 + g] = code == 3u ? kThird : (code == g ? 1.0 : 0.0);
    } else if (pdel2) {     // A = m (p0 + l0, p1 + l1): missing individual-sites read as zero, as in the three planes
      const uint64_t chunk = sgrp >> 1, h = sgrp & 1;
      const uint64_t base = (rb * NC + chunk) * kTilePd2 + (r >> 3) * 32 + (r & 7) * 4 + q;
      const double p0 = present ? Apack[base + h * 512] - l0 : 0.0, p1 = present ? Apack[base + (2 + h) * 512] - l1 : 0.0;
      P[idx * 3 + 0] = p0; P[idx * 3 + 1] = p1; P[idx * 3 + 2] = present ? 1.0 - p0 - p1 : 0.0;
    } else if (planes == 3) {
      const uint64_t chunk = sgrp >> 1, h = sgrp & 1;
      const uint64_t base = (rb * NC + chunk) * kTile3 + (r >> 3) * 32 + (r & 7) * 4 + q;
      for (int g = 0; g < 3; g++) P[idx * 3 + g] = Apack[base + (uint64_t) (g * 2 + h) * 512];
    } else {
      const uint64_t chunk = sgrp / 3, h = sgrp % 3;
      const uint64_t base = (rb * NC + chunk) * kTile3 + (r >> 3) * 32 + (r & 7) * 4 + q;
      const double p0 = Apack[base + (uint64_t) (0 * 3 + h) * 512], p1 = Apack[base + (uint64_t) (1 * 3 + h) * 512];
      P[idx * 3 + 0] = p0; P[idx * 3 + 1] = p1; P[idx * 3 + 2] = 1.0 - p0 - p1;   // the identity the 2-plane mode relies on
    }
  }
  if (miss) miss[idx] = !present;
}

// ngsd_push_packed_genotypes: 2-bit fields, four individuals per byte -> the int8 codes of read_data.cpp:88-95 that
// k_frontend / k_frontend_codes take (byte f of code_of_field = the code of field value f)
__global__ void k_unpack_2bit(const uint8_t *__restrict__ packed, uint64_t row_stride, uint32_t code_of_field, uint64_t n_ind, uint64_t n,
                              int8_t *__restrict__ codes) {
  const uint64_t idx = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n * n_ind) return;
  const uint64_t s = idx / n_ind, i = idx - s * n_ind;
  const unsigned f = (packed[s * row_stride + (i >> 2)] >> (2 * (i & 3))) & 3u;
  codes[idx] = (int8_t) (code_of_field >> (8 * f));
}

__device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}

// SURVEY §8(d) synthetic generator (transcendental-free; bit-identical to oracle/ngsdist_oracle.c:ngsd_oracle_synth_raw)
__global__ void k_synth(double *__restrict__ raw, uint64_t seed, uint64_t thr, int use_miss, uint64_t n_ind, uint64_t site0, uint64_t n) {
  const uint64_t k = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n * n_ind) return;
  const uint64_t idx = site0 * n_ind + k;
  double *x = raw + k * 3;
  if (use_miss && splitmix64((seed + 1) ^ idx) < thr) {
    x[0] = x[1] = x[2] = 1.0 / 3.0;
    return;
  }
#pragma unroll
  for (uint64_t g = 0; g < 3; g++) {
    const uint64_t hsh = splitmix64(seed ^ splitmix64(idx * 4 + g));
    const double u = ((double) (hsh >> 11) + 0.5) * 0x1p-53;
    const double u2 = u * u, u4 = u2 * u2;
    x[g] = u4 * u4;
  }
}

}  // namespace

static void set_pdel2(FrontCfg &c, const ngsd_ctx *ctx) {
  c.pdel2 = ctx->pdel2 ? 1 : 0;
  for (int k = 0; k < 2; k++) { c.pl[k] = ctx->pd_l[k]; c.pr[k] = ctx->pd_r[k]; }
  for (int k = 0; k < 4; k++) c.pV[k] = ctx->pd_V[k];
}

cudaError_t ngsd_launch_frontend(ngsd_ctx *ctx, const ngsd_frontend_args &a) {
  FrontCfg c;
  c.kind = ctx->cfg.input_kind;
  c.in_log = ctx->cfg.input_is_log;
  c.call_geno = ctx->cfg.call_geno;
  c.pairwise_del = ctx->cfg.pairwise_del;
  c.planes = ctx->planes;
  set_pdel2(c, ctx);
  c.int_path = ctx->int_path ? 1 : 0;
  c.N_thresh = ctx->cfg.N_thresh;
  c.call_thresh = ctx->cfg.call_thresh;
  for (int k = 0; k < 9; k++) c.score[k] = ctx->cfg.score[k];
  c.defer = ctx->d_defer;
  c.defer_n = ctx->d_defer_n;
  c.defer_cap = ctx->defer_cap;
  c.blank = ctx->d_blank;
  // grid.y is limited to 65535 blocks of 64 sites: a push of any size goes out as several launches
  const uint64_t max_sites = (uint64_t) 65535 * 64;
  for (uint64_t off = 0; off < a.n; off += max_sites) {
    const uint64_t n = std::min(max_sites, a.n - off), site0 = a.site0 + off;
    const double *raw = a.raw ? a.raw + off * ctx->n_ind * 3 : nullptr;
    const int8_t *codes = a.codes ? a.codes + off * ctx->n_ind : nullptr;
    dim3 grid((unsigned) (ctx->n_pad / 32), (unsigned) ((n + 63) / 64)), block(32, 16);
    if (ctx->int_path && codes)
      k_codes_from_int8<<<grid, block, 0, ctx->stream>>>(codes, ctx->n_ind, site0, n, ctx->NW, ctx->codes, ctx->codes4, ctx->mask, ctx->d_err, ctx->d_blank);
    else if (ctx->int_path)
      k_frontend_codes<<<grid, block, 0, ctx->stream>>>(c, raw, codes, ctx->n_ind, site0, n, ctx->NW, ctx->codes, ctx->codes4, ctx->mask, ctx->d_err);
    else if (c.call_geno)
      k_frontend<true><<<grid, block, 0, ctx->stream>>>(c, raw, codes, ctx->n_ind, site0, n, ctx->NC, ctx->NW, ctx->Apack, ctx->Bpack,
                                                        ctx->Cplane, ctx->ldc, ctx->mask, ctx->d_err);
    else
      k_frontend<false><<<grid, block, 0, ctx->stream>>>(c, raw, codes, ctx->n_ind, site0, n, ctx->NC, ctx->NW, ctx->Apack, ctx->Bpack,
                                                         ctx->Cplane, ctx->ldc, ctx->mask, ctx->d_err);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
  }
  return cudaSuccess;
}

namespace {

// Knife-edge triples after the host decided them with its own libm (api.cu resolve_deferred): one thread per entry
// rewrites the triple's slots in the resident layout -- operand planes (or 2-bit code) and the presence bit.
// d.x = the normal-space posterior as gen_dist reads it; d.flags bit 0 = miss_data() is true, bits 8..9 = the code.
__global__ void k_patch(FrontCfg c, const ngsd_deferred *__restrict__ list, unsigned n, uint64_t n_pad, uint64_t NC, uint64_t NW,
                        double *__restrict__ Apack, double *__restrict__ Bpack, double *__restrict__ Cplane, uint32_t *__restrict__ codes,
                        uint32_t *__restrict__ codes4, uint64_t *__restrict__ mask) {
  const unsigned k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const ngsd_deferred d = list[k];
  const uint64_t i = d.ind, s = d.site, rb = i >> 7, r = i & 127;
  const bool present = !(d.flags & 1u);
  unsigned long long *mw = (unsigned long long *) &mask[(rb * NW + (s >> 6)) * 128 + r];
  if (present) atomicOr(mw, 1ull << (s & 63)); else atomicAnd(mw, ~(1ull << (s & 63)));
  if (c.int_path) {
    unsigned *cw = &codes[((rb * NW + (s >> 6)) * 4 + ((s >> 4) & 3)) * 128 + r];
    const unsigned sh = 2 * (unsigned) (s & 15);
    atomicAnd(cw, ~(3u << sh));
    atomicOr(cw, ((d.flags >> 8) & 3u) << sh);
    unsigned *cw4 = &codes4[((rb * NW + (s >> 6)) * 8 + ((s >> 3) & 7)) * 128 + r];
    const unsigned sh4 = 4 * (unsigned) (s & 7);
    atomicAnd(cw4, ~(15u << sh4));
    atomicOr(cw4, ((d.flags >> 8) & 3u) << sh4);
    return;
  }
  double p[3] = {d.x[0], d.x[1], d.x[2]};
  if (c.pairwise_del && !present) p[0] = p[1] = p[2] = 0;
  const uint64_t sgrp = s >> 2, q = s & 3;
  if (c.pdel2) {
    double a[2], b[2];
    pdel2_operands(c, p, present, a, b);
    const uint64_t base = (rb * NC + (sgrp >> 1)) * kTilePd2 + (r >> 3) * 32 + (r & 7) * 4 + q;
    for (int g = 0; g < 2; g++) {
      const uint64_t o = base + (uint64_t) (g * 2 + (sgrp & 1)) * 512;
      Apack[o] = a[g];
      Bpack[o] = b[g];
    }
    return;
  }
  double B[3];
#pragma unroll
  for (int g = 0; g < 3; g++) {
    double b = c.score[3 * g + 0] * p[0];
    b += c.score[3 * g + 1] * p[1];
    b += c.score[3 * g + 2] * p[2];
    B[g] = b;
  }
  if (c.planes == 3) {
    const uint64_t base = (rb * NC + (sgrp >> 1)) * kTile3 + (r >> 3) * 32 + (r & 7) * 4 + q;
    for (int g = 0; g < 3; g++) {
      const uint64_t o = base + (uint64_t) (g * 2 + (sgrp & 1)) * 512;
      Apack[o] = p[g];
      Bpack[o] = B[g];
    }
  } else {
    const uint64_t base = (rb * NC + sgrp / 3) * kTile3 + (r >> 3) * 32 + (r & 7) * 4 + q;
    for (int g = 0; g < 2; g++) {
      const uint64_t o = base + (uint64_t) (g * 3 + sgrp % 3) * 512;
      Apack[o] = p[g];
      Bpack[o] = B[g] - B[2];
    }
    Cplane[((s >> 6) * n_pad + i) * 64 + (s & 63)] = B[2];
  }
}

}  // namespace

cudaError_t ngsd_launch_patch(ngsd_ctx *ctx, const ngsd_deferred *list_dev, unsigned n) {
  if (n == 0) return cudaSuccess;
  FrontCfg c;
  memset(&c, 0, sizeof(c));
  c.pairwise_del = ctx->cfg.pairwise_del;
  c.planes = ctx->planes;
  set_pdel2(c, ctx);
  c.int_path = ctx->int_path ? 1 : 0;
  for (int k = 0; k < 9; k++) c.score[k] = ctx->cfg.score[k];
  k_patch<<<(n + 127) / 128, 128, 0, ctx->stream>>>(c, list_dev, n, ctx->n_pad, ctx->NC, ctx->NW, ctx->Apack, ctx->Bpack, ctx->Cplane, ctx->codes,
                                                    ctx->codes4, ctx->mask);
  return cudaGetLastError();
}

namespace {
// transport tiers (ngsd_push_sites_packed): narrow host values -> the doubles the front end reads
__global__ void k_widen(const void *__restrict__ src, int format, double denom, uint64_t n_triples, double *__restrict__ raw) {
  const uint64_t k = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_triples) return;
  double x0, x1, x2;
  if (format == NGSD_XFER_F32) {
    const float *f = reinterpret_cast<const float *>(src) + k * 3;
    x0 = (double) f[0]; x1 = (double) f[1]; x2 = (double) f[2];
  } else if (format == NGSD_XFER_U32) {
    const uint32_t *q = reinterpret_cast<const uint32_t *>(src) + k * 3;
    x0 = (double) q[0] / denom; x1 = (double) q[1] / denom; x2 = (double) q[2] / denom;
  } else {
    const uint64_t q = reinterpret_cast<const uint64_t *>(src)[k];
    x0 = (double) (q & 0xFFFFFu) / denom; x1 = (double) ((q >> 20) & 0xFFFFFu) / denom; x2 = (double) ((q >> 40) & 0xFFFFFu) / denom;
  }
  raw[k * 3 + 0] = x0; raw[k * 3 + 1] = x1; raw[k * 3 + 2] = x2;
}
}  // namespace

cudaError_t ngsd_launch_widen(ngsd_ctx *ctx, const void *src_dev, int format, double denom, uint64_t n, double *raw_dev) {
  const uint64_t tot = n * ctx->n_ind;
  k_widen<<<(unsigned) ((tot + 255) / 256), 256, 0, ctx->stream>>>(src_dev, format, denom, tot, raw_dev);
  return cudaGetLastError();
}

cudaError_t ngsd_launch_unpack_2bit(ngsd_ctx *ctx, const uint8_t *packed_dev, uint64_t row_stride, uint32_t code_of_field, uint64_t n,
                                    int8_t *codes_dev) {
  const uint64_t tot = n * ctx->n_ind;
  k_unpack_2bit<<<(unsigned) ((tot + 255) / 256), 256, 0, ctx->stream>>>(packed_dev, row_stride, code_of_field, ctx->n_ind, n, codes_dev);
  return cudaGetLastError();
}

cudaError_t ngsd_launch_unpack(ngsd_ctx *ctx, double *P_dev, uint8_t *miss_dev) {
  const uint64_t tot = ctx->n_ind * ctx->n_sites;
  k_unpack<<<(unsigned) ((tot + 255) / 256), 256, 0, ctx->stream>>>(ctx->Apack, ctx->codes, ctx->mask, ctx->n_ind, ctx->n_sites, ctx->NC,
                                                                    ctx->NW, ctx->planes, ctx->pdel2 ? 1 : 0, ctx->pd_l[0], ctx->pd_l[1],
                                                                    P_dev, miss_dev);
  return cudaGetLastError();
}

cudaError_t ngsd_launch_synth(ngsd_ctx *ctx, double *raw_dev, uint64_t seed, double miss_rate, uint64_t site0, uint64_t n) {
  long double t = (long double) miss_rate * 18446744073709551616.0L;
  uint64_t thr = t >= 18446744073709551615.0L ? UINT64_MAX : (uint64_t) t;
  const uint64_t tot = n * ctx->n_ind;
  k_synth<<<(unsigned) ((tot + 255) / 256), 256, 0, ctx->stream>>>(raw_dev, seed, thr, miss_rate > 0 ? 1 : 0, ctx->n_ind, site0, n);
  return cudaGetLastError();
}
