// C ABI of libngsdist_b200.so (include/ngsdist_b200.h): context management, the chunked front-end pushes, the
// host-side bootstrap bookkeeping (RNG + block multiplicities, ngsDist.cpp:235-238,416-437) and the orchestration of
// K3 -> K2 -> K4 for one distance matrix.  No CPU implementation of the hot path exists in this library.
#include <math.h>
#include <stdarg.h>
#include <stdlib.h>

#include <algorithm>
#include <new>

#include "ngsd_internal.h"

static char g_create_err[512] = "";

void ngsd_set_error(ngsd_ctx *ctx, const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(ctx ? ctx->err : g_create_err, 512, fmt, ap);
  va_end(ap);
}

namespace {

template <typename T>
cudaError_t dev_alloc(T **p, uint64_t count) {
  return cudaMalloc((void **) p, std::max<uint64_t>(count, 1) * sizeof(T));
}

// grow-on-demand pinned scratch (ctx->h_pin or ctx->h_pin2)
int ensure_pinned(ngsd_ctx *ctx, void **pin, uint64_t *pin_bytes, uint64_t bytes) {
  if (*pin_bytes >= bytes) return NGSD_OK;
  if (*pin) cudaFreeHost(*pin);
  *pin = nullptr;
  *pin_bytes = 0;
  NGSD_CUDA(ctx, cudaHostAlloc(pin, bytes, cudaHostAllocDefault));
  *pin_bytes = bytes;
  return NGSD_OK;
}

// Upper-triangle tile list (ti <= tj) in bands of `band` tile-rows/columns so that consecutive tiles (= the CTAs
// resident together) share row blocks through L2.
std::vector<ngsd_tile> make_tiles(uint32_t RB) {
  std::vector<ngsd_tile> t;
  const uint32_t band = 12;
  for (uint32_t bi = 0; bi < RB; bi += band)
    for (uint32_t bj = bi; bj < RB; bj += band)
      for (uint32_t ti = bi; ti < std::min(bi + band, RB); ti++)
        for (uint32_t tj = std::max(bj, ti); tj < std::min(bj + band, RB); tj++) t.push_back({(uint16_t) ti, (uint16_t) tj});
  return t;
}

// K-split boundaries (in positions of the active chunk list) for the dynamically scheduled (split, tile) units of
// k_dist_dmma.  Two unit sizes: ~8 "main" units per CTA cover the first 84 % of the chunks, then units a quarter of
// that size fill the tail so that the CTAs finish within one small unit of each other.  `cost_tiles` is the tile
// count in full-tile equivalents (a diagonal tile costs 136/256; edge tiles count as full ones, so the splits do not
// depend on how k_dist_dmma contracts them).  The partial workspace (128 KiB per unit) is
// capped at 6 GiB.
std::vector<uint32_t> plan_splits(uint32_t n_chunks, uint32_t n_tiles, double cost_tiles, int grid) {
  std::vector<uint32_t> b;
  b.push_back(0);
  if (n_chunks == 0) { b.push_back(0); return b; }
  const uint64_t max_splits = std::max<uint64_t>(1, ((uint64_t) 6 << 30) / ((uint64_t) n_tiles * NGSD_TILE_ELEMS * 8));
  if (n_chunks < 64 || max_splits < 4) {
    const uint32_t s = (uint32_t) std::min<uint64_t>(max_splits, std::max<uint32_t>(1, n_chunks / 16));
    for (uint32_t k = 1; k <= s; k++) b.push_back((uint32_t) ((uint64_t) k * n_chunks / s));
    return b;
  }
  const double upc = 8.0, ratio = 4.0, frac = 0.84;   // main units per CTA, main / tail unit size, main fraction
  const uint32_t Lm = (uint32_t) (frac * n_chunks);
  uint64_t Sm = (uint64_t) llround(upc * grid / cost_tiles);
  Sm = std::max<uint64_t>(1, std::min<uint64_t>(Sm, Lm / 16));
  Sm = std::min<uint64_t>(Sm, std::max<uint64_t>(1, max_splits * 2 / 3));
  const uint32_t cm = (uint32_t) ((Lm + Sm - 1) / Sm);
  const uint32_t ct = std::max<uint32_t>(8, (uint32_t) (cm / ratio));
  uint64_t St = std::max<uint64_t>(1, (n_chunks - Lm + ct - 1) / ct);
  St = std::min<uint64_t>(St, std::max<uint64_t>(1, max_splits - Sm));
  for (uint64_t k = 1; k <= Sm; k++) b.push_back((uint32_t) (k * Lm / Sm));
  for (uint64_t k = 1; k <= St; k++) b.push_back(Lm + (uint32_t) (k * (n_chunks - Lm) / St));
  return b;
}

void tick(ngsd_ctx *ctx, int k) { cudaEventRecord(ctx->ev[k], ctx->stream); }

// Small host <-> device copies of bookkeeping arrays.  NOT cudaMemcpy: that runs on the legacy default stream, which the
// context's non-blocking streams do not wait for, and a host-to-device copy from pageable memory may return while its
// DMA is still in flight -- a kernel launched next on ctx->stream could read the old contents (seen: k_patch reading the
// deferred list before the host's answers had landed).  Stream-ordered copy + synchronise instead.
cudaError_t copy_sync(ngsd_ctx *ctx, void *dst, const void *src, size_t bytes, cudaMemcpyKind kind) {
  if (bytes == 0) return cudaSuccess;
  cudaError_t e = cudaMemcpyAsync(dst, src, bytes, kind, ctx->stream);
  if (e != cudaSuccess) return e;
  return cudaStreamSynchronize(ctx->stream);
}

// development aid: NGSD_SYNC=1 synchronises after every launch of ngsd_distances and names the one that failed
cudaError_t dbg_sync(ngsd_ctx *ctx, const char *what) {
  static const bool on = getenv("NGSD_SYNC") != nullptr;
  if (!on) return cudaSuccess;
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) fprintf(stderr, "NGSD_SYNC: %s failed: %s\n", what, cudaGetErrorString(e));
  (void) ctx;
  return e;
}

// Copy the matrices of the last ngsd_distances to the caller's buffers (each may be null) and wait for them.
int copy_out(ngsd_ctx *ctx, double *out, double *num_opt, uint64_t *cnt_opt) {
  const uint64_t n2 = ctx->n_ind * ctx->n_ind;
  if (out) NGSD_CUDA(ctx, cudaMemcpyAsync(out, ctx->d_out, n2 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  if (num_opt) NGSD_CUDA(ctx, cudaMemcpyAsync(num_opt, ctx->d_num, n2 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  if (cnt_opt) NGSD_CUDA(ctx, cudaMemcpyAsync(cnt_opt, ctx->d_cntout, n2 * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
  NGSD_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return NGSD_OK;
}

// Host-to-device copy of a small host list, queued on ctx->stream from the pinned scratch h_lists: from pageable memory
// the call could wait for the work queued before it, and the replicate loop enqueues the next matrix while the device
// still runs the last one.  The scratch is rewritten once ctx->ev_pin has passed (distances_enqueue resets it); growing
// it first drains the stream, so no queued copy reads a freed buffer.
int upload_list(ngsd_ctx *ctx, void *dst, const void *src, uint64_t bytes) {
  if (bytes == 0) return NGSD_OK;
  uint64_t at = (ctx->h_lists_used + 15) & ~(uint64_t) 15;
  if (at + bytes > ctx->h_lists_bytes) {
    NGSD_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    int rc = ensure_pinned(ctx, &ctx->h_lists, &ctx->h_lists_bytes, std::max<uint64_t>(2 * ctx->h_lists_bytes, bytes + 4096));
    if (rc) return rc;
    at = 0;
  }
  char *h = (char *) ctx->h_lists + at;
  memcpy(h, src, bytes);
  NGSD_CUDA(ctx, cudaMemcpyAsync(dst, h, bytes, cudaMemcpyHostToDevice, ctx->stream));
  ctx->h_lists_used = at + bytes;
  return NGSD_OK;
}

cudaError_t upload_tile_index(ngsd_ctx *ctx, const std::vector<ngsd_tile> &tiles) {
  std::vector<uint32_t> idx(ctx->RB * ctx->RB, 0xFFFFFFFFu);
  for (size_t t = 0; t < tiles.size(); t++) idx[(uint64_t) tiles[t].ti * ctx->RB + tiles[t].tj] = (uint32_t) t;
  if (!ctx->d_tile_index) {
    cudaError_t e = cudaMalloc((void **) &ctx->d_tile_index, idx.size() * sizeof(uint32_t));
    if (e != cudaSuccess) return e;
  }
  cudaError_t e = copy_sync(ctx, ctx->d_tile_index, idx.data(), idx.size() * sizeof(uint32_t), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) return e;
  // tiles of one row block share their A operand: dist_umma.cu contracts them two at a time (one 128 x 256 MMA)
  std::vector<uint32_t> pairs;
  for (size_t t = 0; t < tiles.size();) {
    if (t + 1 < tiles.size() && tiles[t + 1].ti == tiles[t].ti) {
      pairs.push_back((uint32_t) t); pairs.push_back((uint32_t) t + 1);
      t += 2;
    } else {
      pairs.push_back((uint32_t) t); pairs.push_back(0xFFFFFFFFu);
      t += 1;
    }
  }
  ctx->n_pairs = (uint32_t) (pairs.size() / 2);
  if (!ctx->d_pairs) {
    e = cudaMalloc((void **) &ctx->d_pairs, (ctx->RB * (ctx->RB + 1) + 2) * sizeof(uint32_t));
    if (e != cudaSuccess) return e;
  }
  if (pairs.empty()) return cudaSuccess;
  return copy_sync(ctx, ctx->d_pairs, pairs.data(), pairs.size() * sizeof(uint32_t), cudaMemcpyHostToDevice);
}

// The 64 x 64 tiles of the per pair-site EM path (dist_em.cu) that lie in the owned 128 x 128 tiles: 64-tile (ti, tj)
// belongs to 128-tile (ti / 2, tj / 2).  Listed in upper-triangle order (row by row) whether sharded or not, so that a
// shard's CTAs keep the relative order of the whole matrix's; the slot index maps a 64-tile to its position in the list.
cudaError_t upload_em_tiles(ngsd_ctx *ctx, const std::vector<ngsd_tile> &owned) {
  const uint64_t n64 = (ctx->n_ind + NGSD_EM_EDGE - 1) / NGSD_EM_EDGE;
  std::vector<uint8_t> own(ctx->RB * ctx->RB, 0);
  for (const ngsd_tile &t : owned) own[(uint64_t) t.ti * ctx->RB + t.tj] = 1;
  std::vector<uint32_t> list, slot(n64 * n64, 0xFFFFFFFFu);
  for (uint64_t ti = 0; ti < n64; ti++)
    for (uint64_t tj = ti; tj < n64; tj++)
      if (own[(ti / 2) * ctx->RB + tj / 2]) {
        slot[ti * n64 + tj] = (uint32_t) (list.size() / 2);
        list.push_back((uint32_t) ti);
        list.push_back((uint32_t) tj);
      }
  cudaError_t e = cudaSuccess;
  if (!ctx->d_em_tiles) {
    e = cudaMalloc((void **) &ctx->d_em_tiles, (n64 * (n64 + 1) + 2) * sizeof(uint32_t));
    if (e == cudaSuccess) e = cudaMalloc((void **) &ctx->d_em_slot, slot.size() * sizeof(uint32_t));
    if (e != cudaSuccess) return e;
  }
  ctx->em_n_tiles = (uint32_t) (list.size() / 2);
  if (!list.empty()) e = copy_sync(ctx, ctx->d_em_tiles, list.data(), list.size() * sizeof(uint32_t), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) return e;
  return copy_sync(ctx, ctx->d_em_slot, slot.data(), slot.size() * sizeof(uint32_t), cudaMemcpyHostToDevice);
}

}  // namespace

extern "C" {

int ngsd_abi_version(void) { return NGSD_ABI_VERSION; }

void ngsd_default_cfg(ngsd_cfg *cfg) {
  memset(cfg, 0, sizeof(*cfg));
  const double s[9] = {0, 0.5, 1, 0.5, 0, 0.5, 1, 0.5, 0};   // parse_args.cpp:25-27
  memcpy(cfg->score, s, sizeof(s));
  cfg->evol_model = 1;                                       // parse_args.cpp:28
  cfg->input_kind = NGSD_INPUT_BINARY_GL;
}

const char *ngsd_last_error(const ngsd_ctx *ctx) { return ctx ? ctx->err : g_create_err; }

// Coefficients of the pdel two-plane form (ngsd_internal.h) for score S (S[g1][g2] = score[3*g1 + g2], g1 the row
// individual's genotype), in double with Cramer's rule so that dyadic scores give exact coefficients:
//   V = Z^T S Z,  r = V^-1 Z^T S c,  l = V^-T Z^T S^T c,  kappa = c^T S c - l^T V r     (c = (0,0,1)).
// Taken only when every coefficient is finite, max(|l|, |r|) <= 4 and |kappa| <= 4 max|S|: that keeps the per-site
// terms within a small multiple of the three-plane ones and rejects singular V (--avg_nuc_dist: S has rank 1 on the
// zero-sum plane), near-singular and non-finite scores, which keep the three planes.
static bool pdel2_coefficients(const double *score, double l[2], double r[2], double V[4], double *kappa) {
  auto S = [&](int a, int b) { return score[3 * a + b]; };
  // S Z: columns S e_g - S e_2 (g = 0, 1); then Z^T (S Z): rows e_g - e_2
  double SZ[3][2];
  for (int a = 0; a < 3; a++)
    for (int g = 0; g < 2; g++) SZ[a][g] = S(a, g) - S(a, 2);
  for (int f = 0; f < 2; f++)
    for (int g = 0; g < 2; g++) V[f * 2 + g] = SZ[f][g] - SZ[2][g];
  const double bR[2] = {S(0, 2) - S(2, 2), S(1, 2) - S(2, 2)};   // Z^T S c
  const double bL[2] = {S(2, 0) - S(2, 2), S(2, 1) - S(2, 2)};   // Z^T S^T c
  const double det = V[0] * V[3] - V[1] * V[2];
  r[0] = (V[3] * bR[0] - V[1] * bR[1]) / det;
  r[1] = (V[0] * bR[1] - V[2] * bR[0]) / det;
  l[0] = (V[3] * bL[0] - V[2] * bL[1]) / det;
  l[1] = (V[0] * bL[1] - V[1] * bL[0]) / det;
  *kappa = S(2, 2) - (l[0] * (V[0] * r[0] + V[1] * r[1]) + l[1] * (V[2] * r[0] + V[3] * r[1]));
  double smax = 0;
  for (int k = 0; k < 9; k++) smax = std::max(smax, fabs(score[k]));
  const double vals[9] = {l[0], l[1], r[0], r[1], V[0], V[1], V[2], V[3], *kappa};
  for (double v : vals)
    if (!std::isfinite(v)) return false;
  const double shift = std::max(std::max(fabs(l[0]), fabs(l[1])), std::max(fabs(r[0]), fabs(r[1])));
  return shift <= 4.0 && fabs(*kappa) <= 4.0 * smax;
}

int ngsd_create(const ngsd_cfg *cfg, ngsd_ctx **out) {
  if (!cfg || !out) { ngsd_set_error(nullptr, "null argument"); return NGSD_ERR_ARG; }
  *out = nullptr;
  if (cfg->n_ind == 0) { ngsd_set_error(nullptr, "number of individuals (--n_ind) missing!"); return NGSD_ERR_ARG; }
  if (cfg->n_sites == 0) { ngsd_set_error(nullptr, "number of sites (--n_sites) missing!"); return NGSD_ERR_ARG; }
  if (cfg->n_ind > 65535u * NGSD_TILE) { ngsd_set_error(nullptr, "n_ind too large for the tile index type"); return NGSD_ERR_ARG; }
  if (cfg->tot_sites > 0 && cfg->pairwise_del) {
    ngsd_set_error(nullptr, "cannot specify total number of sites (--tot_sites) with pairwise deletion (--pairwise_del)!");
    return NGSD_ERR_ARG;
  }
  if (cfg->evol_model < 0 || cfg->evol_model > 6) { ngsd_set_error(nullptr, "invalid evolutionary model specified!"); return NGSD_ERR_MODEL; }
  if (cfg->evol_model > 2) {
    static const char *names[] = {"K80", "F81", "HKY85", "TN93"};
    ngsd_set_error(nullptr, "%s model not yet supported", names[cfg->evol_model - 3]);
    return NGSD_ERR_MODEL;
  }
  if (cfg->call_geno && cfg->N_thresh > cfg->call_thresh) {
    ngsd_set_error(nullptr, "missing data threshold must be smaller than calling genotype threshold!");
    return NGSD_ERR_THRESH;
  }
  if (cfg->input_kind < 0 || cfg->input_kind > 2 || (cfg->reserved & ~7)) { ngsd_set_error(nullptr, "invalid input_kind / flags"); return NGSD_ERR_ARG; }
  // internal index types: 64-site word and chunk ids are uint32, per-split shared-site counts are uint32
  if (cfg->n_sites > ((uint64_t) 1 << 32) - 64) { ngsd_set_error(nullptr, "n_sites too large for one context (limit 2^32 - 64 sites per GPU): shard the sites (ngsd_cfg.n_gpus with NGSD_SHARD_SITES)"); return NGSD_ERR_ARG; }
  if (cfg->n_gpus < 0 || cfg->n_gpus > 64 || cfg->shard < 0 || cfg->shard > 2) { ngsd_set_error(nullptr, "invalid n_gpus / shard"); return NGSD_ERR_ARG; }
  if ((cfg->input_kind == NGSD_INPUT_GENOTYPES || cfg->call_geno) && !cfg->indep_geno) {
    ngsd_set_error(nullptr, "indep_geno must be set for genotype input / call_geno (ngsDist.cpp:55-62)");
    return NGSD_ERR_ARG;
  }

  int ndev = 0;
  cudaError_t ce = cudaGetDeviceCount(&ndev);
  if (ce != cudaSuccess || ndev == 0) {
    ngsd_set_error(nullptr, "no CUDA device available (%s); this library has no CPU fallback", cudaGetErrorString(ce));
    return NGSD_ERR_CUDA;
  }
  if (cfg->device < 0 || cfg->device >= ndev) { ngsd_set_error(nullptr, "invalid device ordinal %d", cfg->device); return NGSD_ERR_ARG; }
  if (cfg->n_gpus > 1) {
    if (cfg->device + cfg->n_gpus > ndev) { ngsd_set_error(nullptr, "n_gpus %d from device %d: only %d devices visible", cfg->n_gpus, cfg->device, ndev); return NGSD_ERR_ARG; }
    return ngsd_group_create(cfg, out);
  }

  ngsd_ctx *ctx = new (std::nothrow) ngsd_ctx();
  if (!ctx) { ngsd_set_error(nullptr, "out of host memory"); return NGSD_ERR_ARG; }
  ctx->cfg = *cfg;
  ctx->device = cfg->device;
#define CREATE_CUDA(call)                                                                      \
  do {                                                                                         \
    cudaError_t e_ = (call);                                                                   \
    if (e_ != cudaSuccess) {                                                                   \
      ngsd_set_error(nullptr, "CUDA error: %s (%s)", cudaGetErrorString(e_), #call);           \
      ngsd_destroy(ctx);                                                                       \
      return NGSD_ERR_CUDA;                                                                    \
    }                                                                                          \
  } while (0)
  CREATE_CUDA(cudaSetDevice(ctx->device));
  cudaDeviceProp prop;
  CREATE_CUDA(cudaGetDeviceProperties(&prop, ctx->device));
  if (prop.major != 10) {
    ngsd_set_error(nullptr, "device %d is sm_%d%d; this library is built for sm_100a (B200) only", ctx->device, prop.major, prop.minor);
    ngsd_destroy(ctx);
    return NGSD_ERR_CUDA;
  }
  ctx->n_sm = prop.multiProcessorCount;
  CREATE_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
  CREATE_CUDA(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
  CREATE_CUDA(cudaStreamCreateWithFlags(&ctx->aux_stream, cudaStreamNonBlocking));
  CREATE_CUDA(cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
  CREATE_CUDA(cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming));
  for (auto &set : ctx->ev_sets)
    for (auto &e : set) CREATE_CUDA(cudaEventCreate(&e));
  CREATE_CUDA(cudaEventCreateWithFlags(&ctx->ev_pin, cudaEventDisableTiming));
  for (int b = 0; b < 2; b++) {
    CREATE_CUDA(cudaEventCreateWithFlags(&ctx->ev_copied[b], cudaEventDisableTiming));
    CREATE_CUDA(cudaEventCreateWithFlags(&ctx->stage_free[b], cudaEventDisableTiming));
    CREATE_CUDA(cudaEventCreateWithFlags(&ctx->stage_ready[b], cudaEventDisableTiming));
  }
  ctx->n_ind = cfg->n_ind;
  ctx->n_sites = cfg->n_sites;
  ctx->n_pad = (cfg->n_ind + NGSD_TILE - 1) / NGSD_TILE * NGSD_TILE;
  ctx->RB = ctx->n_pad / NGSD_TILE;
  ctx->NW = (cfg->n_sites + 63) / 64;
  // sum-to-one reduction (2 operand planes) whenever no individual-site is masked out of the contraction
  ctx->planes = (cfg->indep_geno && !cfg->pairwise_del && !(cfg->reserved & 1)) ? 2 : 3;
  ctx->sc = ctx->planes == 3 ? NGSD_SC : NGSD_SC2;
  ctx->NC = ctx->planes == 3 ? ctx->NW * 8 : (ctx->NW * 16 + 2) / 3;
  ctx->pushed.assign(ctx->NW, 0);
  // Called genotypes (every triple one-hot or "missing"): exact integer contraction on the int8 tensor cores, 2 bits per
  // individual-site in HBM instead of FP64 planes (dist_umma.cu).  --call_geno leaves soft triples between the two
  // thresholds (gen_func.cpp:908), so it qualifies only when they coincide (the default 0 / 0).
  const bool hard_calls = cfg->input_kind == NGSD_INPUT_GENOTYPES || (cfg->call_geno && cfg->N_thresh == cfg->call_thresh);
  ctx->int_path = hard_calls && cfg->indep_geno && !(cfg->reserved & 2) &&
                  ngsd_int_lut(cfg->score, cfg->pairwise_del != 0, ctx->int_lut, &ctx->int_scale, &ctx->int_max_byte);
  if (ctx->int_path) {
    ctx->planes = 3;
    ctx->sc = NGSD_SC;
    ctx->NC = ctx->NW * 8;
    CREATE_CUDA(dev_alloc(&ctx->codes, ctx->RB * ctx->NW * 512));
    CREATE_CUDA(dev_alloc(&ctx->codes4, ctx->RB * ctx->NW * 1024));
  }
  // --pairwise_del on the FP64 path: two planes with the mask term folded into the shared-site count (ngsd_internal.h),
  // for contractions of at least NGSD_PDEL2_MIN_PAIR_SITES pair-sites per matrix
  const double pair_sites = (double) cfg->n_ind * (double) (cfg->n_ind - 1) / 2 * (double) cfg->n_sites;
  ctx->pdel2 = cfg->indep_geno && cfg->pairwise_del && !ctx->int_path && !(cfg->reserved & 1) && pair_sites >= (double) NGSD_PDEL2_MIN_PAIR_SITES &&
               pdel2_coefficients(cfg->score, ctx->pd_l, ctx->pd_r, ctx->pd_V, &ctx->pd_kappa);
  if (ctx->pdel2) {
    ctx->k4 = NGSD_K4_PD2;
    ctx->tile_doubles = (uint64_t) NGSD_K4_PD2 * NGSD_K4_DOUBLES;
  }
  const uint64_t plane = ctx->int_path ? 0 : ctx->RB * ctx->NC * ctx->tile_doubles;
  CREATE_CUDA(dev_alloc(&ctx->Apack, plane));
  CREATE_CUDA(dev_alloc(&ctx->Bpack, plane));
  CREATE_CUDA(dev_alloc(&ctx->mask, ctx->RB * ctx->NW * 128));
  // Padding must read as zero: in two-plane mode the last 12-site chunk can hold a k4-group beyond the last 64-site word
  // (NW * 16 groups are written, NC * 3 are contracted), and cudaMalloc hands back whatever an earlier context left there.
  if (plane) {
    CREATE_CUDA(cudaMemsetAsync(ctx->Apack, 0, plane * sizeof(double), ctx->stream));
    CREATE_CUDA(cudaMemsetAsync(ctx->Bpack, 0, plane * sizeof(double), ctx->stream));
  }
  CREATE_CUDA(cudaMemsetAsync(ctx->mask, 0, ctx->RB * ctx->NW * 128 * sizeof(uint64_t), ctx->stream));
  if (ctx->planes == 2) {
    ctx->ldc = ctx->n_pad;   // Cplane is [NW][n_pad][64]: the sites of a 64-site word are contiguous per individual
    CREATE_CUDA(dev_alloc(&ctx->Cplane, ctx->NW * ctx->n_pad * 64));
    CREATE_CUDA(dev_alloc(&ctx->d_cvec, ctx->n_pad));
  }
  CREATE_CUDA(dev_alloc(&ctx->d_err, 1));
  ctx->defer_cap = 1u << 18;
  CREATE_CUDA(dev_alloc(&ctx->d_defer, ctx->defer_cap));
  CREATE_CUDA(dev_alloc(&ctx->d_defer_n, 1));
  CREATE_CUDA(cudaMemsetAsync(ctx->d_defer_n, 0, sizeof(unsigned), ctx->stream));
  CREATE_CUDA(dev_alloc(&ctx->d_blank, ctx->NW));
  CREATE_CUDA(cudaMemsetAsync(ctx->d_blank, 0, ctx->NW * sizeof(uint64_t), ctx->stream));
  CREATE_CUDA(dev_alloc(&ctx->d_sched, 1));
  CREATE_CUDA(cudaMemsetAsync(ctx->d_err, 0, sizeof(int), ctx->stream));
  std::vector<ngsd_tile> tiles = make_tiles((uint32_t) ctx->RB);
  ctx->n_tiles = (uint32_t) tiles.size();
  ctx->n_diag_tiles = (uint32_t) ctx->RB;
  ctx->n_edge_tiles = ngsd_edge_c8(ctx->n_ind) ? (uint32_t) ctx->RB - 1 : 0;
  CREATE_CUDA(dev_alloc(&ctx->d_tiles, tiles.size()));
  CREATE_CUDA(copy_sync(ctx, ctx->d_tiles, tiles.data(), tiles.size() * sizeof(ngsd_tile), cudaMemcpyHostToDevice));
  CREATE_CUDA(upload_tile_index(ctx, tiles));
  if (!cfg->indep_geno) CREATE_CUDA(upload_em_tiles(ctx, tiles));
#undef CREATE_CUDA
  *out = ctx;
  return NGSD_OK;
}

int ngsd_destroy(ngsd_ctx *ctx) {
  if (!ctx) return NGSD_OK;
  if (!ctx->kids.empty()) return ngsd_group_destroy(ctx);
  cudaSetDevice(ctx->device);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  ngsd_comm_release(ctx);
  if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
  if (ctx->aux_stream) cudaStreamSynchronize(ctx->aux_stream);
  cudaFree(ctx->Apack); cudaFree(ctx->Bpack); cudaFree(ctx->mask); cudaFree(ctx->d_err); cudaFree(ctx->Cplane); cudaFree(ctx->d_cvec);
  cudaFree(ctx->stage_dev[0]); cudaFree(ctx->stage_dev[1]);
  cudaFree(ctx->d_tiles); cudaFree(ctx->d_partials); cudaFree(ctx->d_weights); cudaFree(ctx->d_chunk_ids);
  cudaFree(ctx->d_ent_word); cudaFree(ctx->d_ent_mask); cudaFree(ctx->d_cnt); cudaFree(ctx->d_split_begin); cudaFree(ctx->d_split_scale); cudaFree(ctx->d_sched);
  cudaFree(ctx->d_out); cudaFree(ctx->d_out_alt); cudaFree(ctx->d_num); cudaFree(ctx->d_cntout);
  cudaFree(ctx->d_cache); cudaFree(ctx->d_cnt_cache); cudaFree(ctx->d_ent_begin); cudaFree(ctx->d_tile_index); cudaFree(ctx->d_pairs);
  cudaFree(ctx->d_em_tiles); cudaFree(ctx->d_em_slot);
  cudaFree(ctx->codes); cudaFree(ctx->codes4); cudaFree(ctx->d_wsite); cudaFree(ctx->d_word_layer); cudaFree(ctx->d_word_ids);
  cudaFree(ctx->d_defer); cudaFree(ctx->d_defer_n); cudaFree(ctx->d_blank);
  cudaFree(ctx->d_def_rowptr); cudaFree(ctx->d_def_rowind); cudaFree(ctx->d_def_site); cudaFree(ctx->d_def_delta); cudaFree(ctx->d_fix);
  if (ctx->h_pin) cudaFreeHost(ctx->h_pin);
  if (ctx->h_pin2) cudaFreeHost(ctx->h_pin2);
  if (ctx->h_lists) cudaFreeHost(ctx->h_lists);
  cudaFree(ctx->d_cs_begin); cudaFree(ctx->d_cnt_part);
  for (auto &set : ctx->ev_sets)
    for (auto &e : set) if (e) cudaEventDestroy(e);
  if (ctx->ev_pin) cudaEventDestroy(ctx->ev_pin);
  for (int b = 0; b < 2; b++) {
    if (ctx->ev_copied[b]) cudaEventDestroy(ctx->ev_copied[b]);
    if (ctx->stage_free[b]) cudaEventDestroy(ctx->stage_free[b]);
    if (ctx->stage_ready[b]) cudaEventDestroy(ctx->stage_ready[b]);
  }
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  if (ctx->aux_stream) cudaStreamDestroy(ctx->aux_stream);
  if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
  if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
  delete ctx;
  return NGSD_OK;
}

// ---------------------------------------------------------------------------------------------- front end ----

static int check_push(ngsd_ctx *ctx, uint64_t site0, uint64_t n) {
  if (!ctx) return NGSD_ERR_ARG;
  if (n == 0) { ngsd_set_error(ctx, "empty push"); return NGSD_ERR_ARG; }
  if (site0 % 64 != 0) { ngsd_set_error(ctx, "site0 must be a multiple of 64"); return NGSD_ERR_ARG; }
  if (site0 + n > ctx->n_sites) { ngsd_set_error(ctx, "push beyond n_sites"); return NGSD_ERR_ARG; }
  if ((n % 64 != 0) && site0 + n != ctx->n_sites) { ngsd_set_error(ctx, "only the last push may hold a partial 64-site word"); return NGSD_ERR_ARG; }
  return NGSD_OK;
}

static void mark_pushed(ngsd_ctx *ctx, uint64_t site0, uint64_t n) {
  if (!ctx->deficit.empty()) {   // sites pushed again: what the earlier push recorded for them is void
    auto &v = ctx->deficit;
    v.erase(std::remove_if(v.begin(), v.end(), [&](const ngsd_ctx::deficit_entry &e) { return e.site >= site0 && e.site < site0 + n; }), v.end());
    ctx->deficit_dirty = true;
    if (v.empty()) ctx->def_rows = 0;
  }
  for (uint64_t w = site0 / 64; w < (site0 + n + 63) / 64; w++)
    if (!ctx->pushed[w]) { ctx->pushed[w] = 1; ctx->words_pushed++; }
  ctx->frontend_done = false;
  ctx->cache_valid = false;
}

int ngsd_push_sites_device(ngsd_ctx *ctx, const double *raw_dev, uint64_t site0, uint64_t n) {
  if (ctx && !ctx->kids.empty()) return ngsd_group_push(ctx, 3, raw_dev, ctx->n_ind * 3 * sizeof(double), 0, nullptr, site0, n);
  int rc = check_push(ctx, site0, n);
  if (rc) return rc;
  if (ctx->cfg.input_kind == NGSD_INPUT_GENOTYPES) { ngsd_set_error(ctx, "context expects genotype codes"); return NGSD_ERR_ARG; }
  NGSD_CUDA(ctx, cudaSetDevice(ctx->device));
  ctx->timing = ngsd_timing();
  tick(ctx, 0);
  ngsd_frontend_args a{raw_dev, nullptr, site0, n};
  NGSD_CUDA(ctx, ngsd_launch_frontend(ctx, a));
  tick(ctx, 1);
  ctx->timing.launches = 1;
  ctx->timing.total_ms = -1.f;   // resolved lazily in ngsd_get_timing
  mark_pushed(ctx, site0, n);
  return NGSD_OK;
}

static int ensure_staging(ngsd_ctx *ctx, uint64_t bytes_per_site) {
  if (ctx->stage_dev[0]) return NGSD_OK;
  uint64_t sites = ((uint64_t) 64 << 20) / bytes_per_site / 64 * 64;
  sites = std::max<uint64_t>(sites, 64);
  sites = std::min<uint64_t>(sites, (ctx->n_sites + 63) / 64 * 64);
  ctx->stage_sites = sites;
  for (int b = 0; b < 2; b++) {
    NGSD_CUDA(ctx, cudaMalloc((void **) &ctx->stage_dev[b], sites * bytes_per_site));
    NGSD_CUDA(ctx, cudaEventRecord(ctx->stage_free[b], ctx->stream));
  }
  return NGSD_OK;
}

int ngsd_push_sites(ngsd_ctx *ctx, const double *raw_host, uint64_t site0, uint64_t n) {
  if (ctx && !ctx->kids.empty()) return ngsd_group_push(ctx, 0, raw_host, ctx->n_ind * 3 * sizeof(double), 0, nullptr, site0, n);
  int rc = check_push(ctx, site0, n);
  if (rc) return rc;
  if (!raw_host) { ngsd_set_error(ctx, "null raw pointer"); return NGSD_ERR_ARG; }
  if (ctx->cfg.input_kind == NGSD_INPUT_GENOTYPES) { ngsd_set_error(ctx, "context expects genotype codes"); return NGSD_ERR_ARG; }
  NGSD_CUDA(ctx, cudaSetDevice(ctx->device));
  const uint64_t bps = ctx->n_ind * 3 * sizeof(double);
  rc = ensure_staging(ctx, bps);
  if (rc) return rc;
  ctx->stage_bps = bps;
  ctx->timing = ngsd_timing();
  tick(ctx, 0);
  int launches = 0;
  for (uint64_t off = 0; off < n; off += ctx->stage_sites) {
    const uint64_t m = std::min(ctx->stage_sites, n - off);
    const int b = ctx->stage_next;
    ctx->stage_next ^= 1;
    NGSD_CUDA(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->stage_free[b], 0));
    NGSD_CUDA(ctx, cudaMemcpyAsync(ctx->stage_dev[b], raw_host + off * ctx->n_ind * 3, m * bps, cudaMemcpyHostToDevice, ctx->copy_stream));
    NGSD_CUDA(ctx, cudaEventRecord(ctx->stage_ready[b], ctx->copy_stream));
    NGSD_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->stage_ready[b], 0));
    ngsd_frontend_args a{ctx->stage_dev[b], nullptr, site0 + off, m};
    NGSD_CUDA(ctx, ngsd_launch_frontend(ctx, a));
    NGSD_CUDA(ctx, cudaEventRecord(ctx->stage_free[b], ctx->stream));
    launches++;
  }
  tick(ctx, 1);
  ctx->timing.launches = launches;
  ctx->timing.total_ms = -1.f;
  NGSD_CUDA(ctx, cudaStreamSynchronize(ctx->stream));   // the caller may now reuse raw_host
  mark_pushed(ctx, site0, n);
  return NGSD_OK;
}

int ngsd_push_sites_packed(ngsd_ctx *ctx, const void *host, int32_t format, double denom, uint64_t site0, uint64_t n) {
  if (ctx && !ctx->kids.empty()) {
    const uint64_t b = format == NGSD_XFER_U20X3 ? ctx->n_ind * 8 : ctx->n_ind * 12;
    return ngsd_group_push(ctx, 10 + format, host, b, 0, reinterpret_cast<const int8_t *>(&denom), site0, n);
  }
  int rc = check_push(ctx, site0, n);
  if (rc) return rc;
  if (!host) { ngsd_set_error(ctx, "null input pointer"); return NGSD_ERR_ARG; }
  if (ctx->cfg.input_kind == NGSD_INPUT_GENOTYPES) { ngsd_set_error(ctx, "context expects genotype codes"); return NGSD_ERR_ARG; }
  if (format < NGSD_XFER_F32 || format > NGSD_XFER_U20X3) { ngsd_set_error(ctx, "unknown transport format %d", format); return NGSD_ERR_ARG; }
  if (format != NGSD_XFER_F32 && (!(denom > 0) || ctx->cfg.input_is_log)) {
    ngsd_set_error(ctx, "fixed-point transport needs denom > 0 and normal-scale input");
    return NGSD_ERR_ARG;
  }
  NGSD_CUDA(ctx, cudaSetDevice(ctx->device));
  // one staging slot = the chunk's narrow values followed by the doubles they widen to
  const uint64_t in_bps = format == NGSD_XFER_U20X3 ? ctx->n_ind * 8 : ctx->n_ind * 12, raw_bps = ctx->n_ind * 24, bps = in_bps + raw_bps;
  if (ctx->stage_dev[0] && ctx->stage_bps != bps) {
    NGSD_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (int b = 0; b < 2; b++) { cudaFree(ctx->stage_dev[b]); ctx->stage_dev[b] = nullptr; }
  }
  rc = ensure_staging(ctx, bps);
  if (rc) return rc;
  ctx->stage_bps = bps;
  ctx->timing = ngsd_timing();
  tick(ctx, 0);
  int launches = 0;
  for (uint64_t off = 0; off < n; off += ctx->stage_sites) {
    const uint64_t m = std::min(ctx->stage_sites, n - off);
    const int b = ctx->stage_next;
    ctx->stage_next ^= 1;
    double *d_raw = ctx->stage_dev[b];                                               // 32-byte aligned: first
    char *d_in = reinterpret_cast<char *>(ctx->stage_dev[b]) + ctx->stage_sites * raw_bps;
    NGSD_CUDA(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->stage_free[b], 0));
    NGSD_CUDA(ctx, cudaMemcpyAsync(d_in, reinterpret_cast<const char *>(host) + off * in_bps, m * in_bps, cudaMemcpyHostToDevice, ctx->copy_stream));
    NGSD_CUDA(ctx, cudaEventRecord(ctx->stage_ready[b], ctx->copy_stream));
    NGSD_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->stage_ready[b], 0));
    NGSD_CUDA(ctx, ngsd_launch_widen(ctx, d_in, format, denom, m, d_raw));
    ngsd_frontend_args a{d_raw, nullptr, site0 + off, m};
    NGSD_CUDA(ctx, ngsd_launch_frontend(ctx, a));
    NGSD_CUDA(ctx, cudaEventRecord(ctx->stage_free[b], ctx->stream));
    launches += 2;
  }
  tick(ctx, 1);
  ctx->timing.launches = launches;
  ctx->timing.total_ms = -1.f;
  NGSD_CUDA(ctx, cudaStreamSynchronize(ctx->stream));   // the caller may now reuse `host`
  mark_pushed(ctx, site0, n);
  return NGSD_OK;
}

int ngsd_push_genotypes(ngsd_ctx *ctx, const int8_t *codes_host, uint64_t site0, uint64_t n) {
  if (ctx && !ctx->kids.empty()) return ngsd_group_push(ctx, 1, codes_host, ctx->n_ind, 0, nullptr, site0, n);
  int rc = check_push(ctx, site0, n);
  if (rc) return rc;
  if (!codes_host) { ngsd_set_error(ctx, "null codes pointer"); return NGSD_ERR_ARG; }
  if (ctx->cfg.input_kind != NGSD_INPUT_GENOTYPES) { ngsd_set_error(ctx, "context expects genotype likelihoods"); return NGSD_ERR_ARG; }
  NGSD_CUDA(ctx, cudaSetDevice(ctx->device));
  // same double-buffered device staging as ngsd_push_sites: the copy of chunk k + 1 overlaps the front end of chunk k
  const uint64_t bps = ctx->n_ind;
  if (ctx->stage_dev[0] && ctx->stage_bps != bps) {
    NGSD_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (int b = 0; b < 2; b++) { cudaFree(ctx->stage_dev[b]); ctx->stage_dev[b] = nullptr; }
  }
  rc = ensure_staging(ctx, bps);
  if (rc) return rc;
  ctx->stage_bps = bps;
  ctx->timing = ngsd_timing();
  tick(ctx, 0);
  int launches = 0;
  for (uint64_t off = 0; off < n; off += ctx->stage_sites) {
    const uint64_t m = std::min(ctx->stage_sites, n - off);
    const int b = ctx->stage_next;
    ctx->stage_next ^= 1;
    int8_t *d = reinterpret_cast<int8_t *>(ctx->stage_dev[b]);
    NGSD_CUDA(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->stage_free[b], 0));
    NGSD_CUDA(ctx, cudaMemcpyAsync(d, codes_host + off * ctx->n_ind, m * bps, cudaMemcpyHostToDevice, ctx->copy_stream));
    NGSD_CUDA(ctx, cudaEventRecord(ctx->stage_ready[b], ctx->copy_stream));
    NGSD_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->stage_ready[b], 0));
    ngsd_frontend_args a{nullptr, d, site0 + off, m};
    NGSD_CUDA(ctx, ngsd_launch_frontend(ctx, a));
    NGSD_CUDA(ctx, cudaEventRecord(ctx->stage_free[b], ctx->stream));
    launches++;
  }
  tick(ctx, 1);
  ctx->timing.launches = launches;
  ctx->timing.total_ms = -1.f;
  NGSD_CUDA(ctx, cudaStreamSynchronize(ctx->stream));   // the caller may now reuse codes_host
  mark_pushed(ctx, site0, n);
  return NGSD_OK;
}

int ngsd_push_packed_genotypes(ngsd_ctx *ctx, const uint8_t *packed_host, uint64_t row_stride, const int8_t *code_of_field, uint64_t site0,
                               uint64_t n) {
  if (ctx && !ctx->kids.empty()) return ngsd_group_push(ctx, 2, packed_host, row_stride, row_stride, code_of_field, site0, n);
  int rc = check_push(ctx, site0, n);
  if (rc) return rc;
  if (!packed_host) { ngsd_set_error(ctx, "null packed pointer"); return NGSD_ERR_ARG; }
  if (ctx->cfg.input_kind != NGSD_INPUT_GENOTYPES) { ngsd_set_error(ctx, "context expects genotype likelihoods"); return NGSD_ERR_ARG; }
  if (row_stride < (ctx->n_ind + 3) / 4) { ngsd_set_error(ctx, "row_stride is smaller than ceil(n_ind / 4)"); return NGSD_ERR_ARG; }
  static const int8_t identity[4] = {0, 1, 2, -1};
  const int8_t *map = code_of_field ? code_of_field : identity;
  uint32_t map32 = 0;
  for (int f = 0; f < 4; f++) {
    if (map[f] < -1 || map[f] > 2) { ngsd_set_error(ctx, "code_of_field entries must be in {-1,0,1,2}"); return NGSD_ERR_ARG; }
    map32 |= (uint32_t) (uint8_t) map[f] << (8 * f);
  }
  NGSD_CUDA(ctx, cudaSetDevice(ctx->device));
  // one staging slot = the chunk's packed rows followed by its unpacked int8 codes
  const uint64_t bps = row_stride + ctx->n_ind;
  if (ctx->stage_dev[0] && ctx->stage_bps != bps) {          // a different row_stride than the last push: re-size
    NGSD_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (int b = 0; b < 2; b++) { cudaFree(ctx->stage_dev[b]); ctx->stage_dev[b] = nullptr; }
  }
  rc = ensure_staging(ctx, bps);
  if (rc) return rc;
  ctx->stage_bps = bps;
  ctx->timing = ngsd_timing();
  tick(ctx, 0);
  int launches = 0;
  for (uint64_t off = 0; off < n; off += ctx->stage_sites) {
    const uint64_t m = std::min(ctx->stage_sites, n - off);
    const int b = ctx->stage_next;
    ctx->stage_next ^= 1;
    uint8_t *d_packed = reinterpret_cast<uint8_t *>(ctx->stage_dev[b]);
    int8_t *d_codes = reinterpret_cast<int8_t *>(d_packed + ctx->stage_sites * row_stride);
    NGSD_CUDA(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->stage_free[b], 0));
    NGSD_CUDA(ctx, cudaMemcpyAsync(d_packed, packed_host + off * row_stride, m * row_stride, cudaMemcpyHostToDevice, ctx->copy_stream));
    NGSD_CUDA(ctx, cudaEventRecord(ctx->stage_ready[b], ctx->copy_stream));
    NGSD_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->stage_ready[b], 0));
    NGSD_CUDA(ctx, ngsd_launch_unpack_2bit(ctx, d_packed, row_stride, map32, m, d_codes));
    ngsd_frontend_args a{nullptr, d_codes, site0 + off, m};
    NGSD_CUDA(ctx, ngsd_launch_frontend(ctx, a));
    NGSD_CUDA(ctx, cudaEventRecord(ctx->stage_free[b], ctx->stream));
    launches += 2;
  }
  tick(ctx, 1);
  ctx->timing.launches = launches;
  ctx->timing.total_ms = -1.f;
  NGSD_CUDA(ctx, cudaStreamSynchronize(ctx->stream));   // the caller may now reuse packed_host
  mark_pushed(ctx, site0, n);
  return NGSD_OK;
}

void ngsd_mark_all_pushed(ngsd_ctx *ctx) {
  std::fill(ctx->pushed.begin(), ctx->pushed.end(), (uint8_t) 1);
  ctx->words_pushed = ctx->NW;
  ctx->frontend_done = true;
  ctx->cache_valid = false;
}

int ngsd_frontend(ngsd_ctx *ctx) {
  if (!ctx) return NGSD_ERR_ARG;
  if (!ctx->kids.empty()) return ngsd_group_frontend(ctx);
  if (ctx->words_pushed != ctx->NW) {
    ngsd_set_error(ctx, "front end incomplete: %llu of %llu 64-site words pushed", (unsigned long long) ctx->words_pushed, (unsigned long long) ctx->NW);
    return NGSD_ERR_STATE;
  }
  int rc = ngsd_frontend_flags(ctx);
  if (rc) return rc;
  ctx->frontend_done = true;
  return NGSD_OK;
}

// One triple through the reader-side normalisation and the front-end loop of main() exactly as the reference runs them
// on the host, with the host's libm: read_data.cpp:37-45 / :83-99 (log, -inf clamp on the binary path, post_prob),
// gen_func.cpp:135-151 (logsum), :73-98,886-914 (call_geno on log-scale values), ngsDist.cpp:172-173 (exp).
static bool host_posterior(const ngsd_cfg &c, const double x[3], double p[3]) {
  double L[3] = {x[0], x[1], x[2]};
  const bool binary = c.input_kind == NGSD_INPUT_BINARY_GL;
  if (!c.input_is_log)
    for (int g = 0; g < 3; g++) {
      L[g] = log(L[g]);
      if (binary && L[g] == -INFINITY) L[g] = -1e15;
    }
  double M = L[0];
  for (int g = 1; g < 3; g++) M = std::max(L[g], M);
  double norm;
  if (M == -INFINITY) {
    norm = -INFINITY;
  } else {
    double sum = 0;
    for (int g = 0; g < 3; g++) sum += exp(L[g] - M);
    norm = log(sum) + M;
  }
  for (int g = 0; g < 3; g++) L[g] -= norm;
  const bool ok = !(binary && (std::isnan(L[0]) || std::isnan(L[1]) || std::isnan(L[2])));
  if (c.call_geno) {
    int max_pos = 0, min_pos = 0;
    double mx = -INFINITY, mn = INFINITY;
    for (int g = 0; g < 3; g++) {
      if (L[g] > mx) { max_pos = g; mx = L[g]; }
      if (L[g] < mn) { min_pos = g; mn = L[g]; }
    }
    double max_pp = exp(L[max_pos]);
    if (L[min_pos] == L[max_pos]) max_pp = -1;
    if (max_pp < c.N_thresh)
      for (int g = 0; g < 3; g++) L[g] = log((double) 1 / 3);
    if (max_pp >= c.call_thresh) {
      for (int g = 0; g < 3; g++) L[g] = -1e15;
      L[max_pos] = log(1);
    }
  }
  for (int g = 0; g < 3; g++) p[g] = exp(L[g]);
  return ok;
}

// Knife-edge triples (ngsd_deferred): decided here with the host's libm, written back by k_patch.
extern "C" int ngsd_frontend_resolve(ngsd_ctx *ctx) {
  NGSD_CUDA(ctx, cudaSetDevice(ctx->device));
  unsigned n = 0;
  NGSD_CUDA(ctx, cudaMemcpyAsync(&n, ctx->d_defer_n, sizeof(unsigned), cudaMemcpyDeviceToHost, ctx->stream));
  NGSD_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (n == 0) return NGSD_OK;
  n = std::min(n, ctx->defer_cap);
  std::vector<ngsd_deferred> list(n);
  NGSD_CUDA(ctx, copy_sync(ctx, list.data(), ctx->d_defer, (size_t) n * sizeof(ngsd_deferred), cudaMemcpyDeviceToHost));
  bool nan_found = false;
  for (ngsd_deferred &d : list) {
    double p[3];
    if (!host_posterior(ctx->cfg, d.x, p)) nan_found = true;
    const bool miss = fabs(p[0] - p[1]) < 1e-5 && fabs(p[1] - p[2]) < 1e-5;          // gen_func.cpp:862-868
    const unsigned code = p[0] == 1.0 ? 0u : p[1] == 1.0 ? 1u : p[2] == 1.0 ? 2u : 3u;   // one-hot, or the uniform "missing" triple
    d.flags = (miss ? 1u : 0u) | (code << 8);
    d.x[0] = p[0]; d.x[1] = p[1]; d.x[2] = p[2];
    if (ctx->planes == 2 && !ctx->int_path) {
      const double delta = ((p[0] + p[1]) + p[2]) - 1.0;
      if (fabs(delta) > 1e-9) { ctx->deficit.push_back({d.ind, d.site, delta}); ctx->deficit_dirty = true; }
    }
  }
  NGSD_CUDA(ctx, copy_sync(ctx, ctx->d_defer, list.data(), (size_t) n * sizeof(ngsd_deferred), cudaMemcpyHostToDevice));
  NGSD_CUDA(ctx, ngsd_launch_patch(ctx, ctx->d_defer, n));
  NGSD_CUDA(ctx, cudaMemsetAsync(ctx->d_defer_n, 0, sizeof(unsigned), ctx->stream));
  if (nan_found) ctx->deferred_nan = true;
  NGSD_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  ctx->deferred_total += n;
  return NGSD_OK;
}

// The deferred error flags of the pushes so far (NaN on the binary path, genotype codes above 2).
int ngsd_frontend_flags(ngsd_ctx *ctx) {
  int rc0 = ngsd_frontend_resolve(ctx);
  if (rc0) return rc0;
  NGSD_CUDA(ctx, cudaSetDevice(ctx->device));
  int flags = 0;
  NGSD_CUDA(ctx, cudaMemcpyAsync(&flags, ctx->d_err, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  NGSD_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (ctx->deferred_nan) flags |= 1;
  if (flags & 1) { ngsd_set_error(ctx, "NaN found! Is the file format correct?"); return NGSD_ERR_NAN; }
  if (flags & 2) { ngsd_set_error(ctx, "wrong GENO file format. Genotypes must be coded as {-1,0,1,2} !"); return NGSD_ERR_GENO; }
  if (flags & 16) {
    ngsd_set_error(ctx, "all-zero likelihood triples with a site-sharded front end over several processes: create the contexts with ngsd_cfg.reserved bit 0 (three operand planes)");
    return NGSD_ERR_ARG;
  }
  ctx->any_blank = (flags & 4) != 0;
  if (ctx->any_blank) {        // sites that were empty text lines: the integer path gives them weight 0 (distances_int)
    ctx->h_blank.resize(ctx->NW);
    NGSD_CUDA(ctx, copy_sync(ctx, ctx->h_blank.data(), ctx->d_blank, ctx->NW * sizeof(uint64_t), cudaMemcpyDeviceToHost));
  }
  return NGSD_OK;
}

int ngsd_get_posteriors(ngsd_ctx *ctx, double *P_host, uint8_t *miss_host) {
  if (!ctx) return NGSD_ERR_ARG;
  if (!ctx->kids.empty()) return ngsd_group_get_posteriors(ctx, P_host, miss_host);
  NGSD_CUDA(ctx, cudaSetDevice(ctx->device));
  const uint64_t tot = ctx->n_ind * ctx->n_sites;
  double *dP = nullptr;
  uint8_t *dM = nullptr;
  if (P_host) NGSD_CUDA(ctx, cudaMalloc((void **) &dP, tot * 3 * sizeof(double)));
  if (miss_host) NGSD_CUDA(ctx, cudaMalloc((void **) &dM, tot));
  cudaError_t e = ngsd_launch_unpack(ctx, dP, dM);
  if (e == cudaSuccess && P_host) e = cudaMemcpyAsync(P_host, dP, tot * 3 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess && miss_host) e = cudaMemcpyAsync(miss_host, dM, tot, cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  cudaFree(dP);
  cudaFree(dM);
  NGSD_CUDA(ctx, e);
  return NGSD_OK;
}

// ---------------------------------------------------------------------------------------------- distances ----

static int ensure_dist_buffers(ngsd_ctx *ctx, uint64_t slots);
static int ensure_entries(ngsd_ctx *ctx, uint64_t n);

// Row triples that do not sum to one (2-plane mode, see ngsd_ctx::deficit): CSR by individual, last push of a site wins.
static int upload_deficit(ngsd_ctx *ctx) {
  if (!ctx->deficit_dirty && ctx->d_fix) return NGSD_OK;
  auto &v = ctx->deficit;
  std::stable_sort(v.begin(), v.end(), [](const ngsd_ctx::deficit_entry &a, const ngsd_ctx::deficit_entry &b) {
    return a.ind != b.ind ? a.ind < b.ind : a.site < b.site;
  });
  std::vector<ngsd_ctx::deficit_entry> u;
  for (size_t k = 0; k < v.size(); k++) {
    if (!u.empty() && u.back().ind == v[k].ind && u.back().site == v[k].site) u.back() = v[k];
    else u.push_back(v[k]);
  }
  v.swap(u);
  std::vector<uint32_t> rowptr, rowind;
  std::vector<uint64_t> site(v.size());
  std::vector<double> delta(v.size());
  for (size_t k = 0; k < v.size(); k++) {
    if (rowind.empty() || rowind.back() != v[k].ind) { rowind.push_back(v[k].ind); rowptr.push_back((uint32_t) k); }
    site[k] = v[k].site;
    delta[k] = v[k].delta;
  }
  rowptr.push_back((uint32_t) v.size());
  if (v.size() > ctx->def_cap) {
    cudaFree(ctx->d_def_rowptr); cudaFree(ctx->d_def_rowind); cudaFree(ctx->d_def_site); cudaFree(ctx->d_def_delta);
    ctx->d_def_rowptr = ctx->d_def_rowind = nullptr; ctx->d_def_site = nullptr; ctx->d_def_delta = nullptr;
    ctx->def_cap = 0;
    const uint64_t cap = v.size() * 2 + 16;
    NGSD_CUDA(ctx, dev_alloc(&ctx->d_def_rowptr, cap + 1));
    NGSD_CUDA(ctx, dev_alloc(&ctx->d_def_rowind, cap));
    NGSD_CUDA(ctx, dev_alloc(&ctx->d_def_site, cap));
    NGSD_CUDA(ctx, dev_alloc(&ctx->d_def_delta, cap));
    ctx->def_cap = cap;
  }
  if (!ctx->d_fix) NGSD_CUDA(ctx, dev_alloc(&ctx->d_fix, ctx->n_ind * ctx->n_ind));
  NGSD_CUDA(ctx, copy_sync(ctx, ctx->d_def_rowptr, rowptr.data(), rowptr.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
  NGSD_CUDA(ctx, copy_sync(ctx, ctx->d_def_rowind, rowind.data(), rowind.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
  NGSD_CUDA(ctx, copy_sync(ctx, ctx->d_def_site, site.data(), site.size() * sizeof(uint64_t), cudaMemcpyHostToDevice));
  NGSD_CUDA(ctx, copy_sync(ctx, ctx->d_def_delta, delta.data(), delta.size() * sizeof(double), cudaMemcpyHostToDevice));
  ctx->def_rows = (uint32_t) rowind.size();
  ctx->deficit_dirty = false;
  return NGSD_OK;
}

// The input of k_dist_umma (K2c, dist_umma.cu), for the integer path's sums and for the tensor-core count pass of the
// FP64 path:
//  * per-site weight bytes in layers of at most `cap` each: the bootstrap multiplicities (ngsDist.cpp:416-437), 1 for
//    replicate 0 (block_counts == nullptr), 0 beyond the sites in use and, with zero_blanks, at sites that were empty
//    text lines;
//  * the list of 64-site words to contract as (word id, layer | bit 31 when all 64 weights of the word are 1): every
//    word with a non-zero weight or, with cache_words > 0, the first cache_words words in order (the K splits of the
//    bootstrap block cache are the words of one block each).
// Both are staged in the pinned scratch *pin, the device buffers d_wsite, d_word_ids and d_word_layer grow on demand and
// the copies are queued on ctx->stream.  *n_words = length of the list.
static int build_word_list(ngsd_ctx *ctx, const uint32_t *block_counts, uint64_t n_blocks, uint64_t block_size, uint32_t maxw,
                           uint32_t cap, bool zero_blanks, uint64_t cache_words, void **pin, uint64_t *pin_bytes, uint64_t *n_words) {
  const uint64_t NW = ctx->NW, nsp = NW * 64;
  const uint32_t layers = (maxw + cap - 1) / cap;
  const uint64_t bytes_w = (uint64_t) layers * nsp, n_list = (uint64_t) layers * NW, bytes_w64 = (bytes_w + 63) / 64 * 64;
  int rc = ensure_pinned(ctx, pin, pin_bytes, bytes_w64 + 2 * n_list * sizeof(uint32_t) + 64);
  if (rc) return rc;
  uint8_t *h_w = (uint8_t *) *pin;
  uint32_t *h_ids = (uint32_t *) (h_w + bytes_w64), *h_layer = h_ids + n_list;
  memset(h_w, 0, bytes_w);
  if (!block_counts) {
    memset(h_w, 1, ctx->n_sites);
  } else {
    for (uint64_t b = 0; b < n_blocks; b++) {
      uint32_t left = block_counts[b];
      for (uint32_t l = 0; l < layers && left; l++) {
        const uint32_t w = std::min(left, cap);
        memset(h_w + (uint64_t) l * nsp + b * block_size, (int) w, block_size);
        left -= w;
      }
    }
  }
  if (zero_blanks)
    for (uint64_t w = 0; w < NW; w++)
      for (uint64_t m = ctx->h_blank[w]; m; m &= m - 1)
        for (uint32_t l = 0; l < layers; l++) h_w[(uint64_t) l * nsp + w * 64 + (uint64_t) __builtin_ctzll(m)] = 0;
  const uint64_t scan = cache_words ? cache_words : NW;
  uint64_t n = 0;
  for (uint32_t l = 0; l < layers; l++)
    for (uint64_t w = 0; w < scan; w++) {
      const uint64_t *p8 = (const uint64_t *) (h_w + (uint64_t) l * nsp + w * 64);
      if (cache_words || (p8[0] | p8[1] | p8[2] | p8[3] | p8[4] | p8[5] | p8[6] | p8[7])) {
        const uint64_t one = 0x0101010101010101ull;
        const bool unit = p8[0] == one && p8[1] == one && p8[2] == one && p8[3] == one && p8[4] == one && p8[5] == one && p8[6] == one && p8[7] == one;
        h_ids[n] = (uint32_t) w;
        h_layer[n] = l | (unit ? 0x80000000u : 0u);             // bit 31: the kernel may skip the weight bytes of this word
        n++;
      }
    }
  if (bytes_w > ctx->wsite_cap) {
    cudaFree(ctx->d_wsite);
    ctx->d_wsite = nullptr;
    ctx->wsite_cap = 0;
    NGSD_CUDA(ctx, dev_alloc(&ctx->d_wsite, bytes_w));
    ctx->wsite_cap = bytes_w;
  }
  if (n_list > ctx->word_cap) {
    cudaFree(ctx->d_word_ids);
    cudaFree(ctx->d_word_layer);
    ctx->d_word_ids = ctx->d_word_layer = nullptr;
    ctx->word_cap = 0;
    NGSD_CUDA(ctx, dev_alloc(&ctx->d_word_ids, n_list));
    NGSD_CUDA(ctx, dev_alloc(&ctx->d_word_layer, n_list));
    ctx->word_cap = n_list;
  }
  if (n) {
    NGSD_CUDA(ctx, cudaMemcpyAsync(ctx->d_wsite, h_w, bytes_w, cudaMemcpyHostToDevice, ctx->stream));
    NGSD_CUDA(ctx, cudaMemcpyAsync(ctx->d_word_ids, h_ids, n * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    NGSD_CUDA(ctx, cudaMemcpyAsync(ctx->d_word_layer, h_layer, n * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
  }
  *n_words = n;
  return NGSD_OK;
}

// Cut K splits (boundaries in the word list) so that none holds more than max_words words: the int32 accumulators of
// k_dist_umma must not overflow.
static void cap_splits(std::vector<uint32_t> &splits, uint32_t max_words) {
  std::vector<uint32_t> cut(1, 0);
  for (size_t k = 1; k < splits.size(); k++) {
    while (splits[k] - cut.back() > max_words) cut.push_back(cut.back() + max_words);
    if (splits[k] > cut.back()) cut.push_back(splits[k]);
  }
  if (cut.size() < 2) cut.push_back(0);
  splits.swap(cut);
}

// One matrix on the called-genotype integer path (K2c dist_umma.cu): same contract as ngsd_distances.
static int distances_int(ngsd_ctx *ctx, const uint32_t *block_counts, uint64_t n_blocks, uint64_t block_size, double *out,
                         double *num_opt, uint64_t *cnt_opt) {
  const bool weighted = block_counts != nullptr;
  const uint64_t n_eff = weighted ? n_blocks * block_size : ctx->n_sites;
  uint32_t maxw = 1;
  uint64_t active_sites = n_eff;
  if (weighted) {
    active_sites = 0;
    for (uint64_t b = 0; b < n_blocks; b++) {
      maxw = std::max(maxw, block_counts[b]);
      active_sites += block_counts[b] ? block_size : 0;
    }
  }
  const bool do_count = ctx->cfg.pairwise_del != 0;
  // ---- bootstrap block cache (see ngsd_distances): per-block int32 partials, blocks = whole 64-site words ----
  const uint64_t unit_ints = do_count ? 2 * NGSD_TILE_ELEMS : NGSD_TILE_ELEMS;
  bool use_cache = false, build_cache = false;
  if (weighted && !(ctx->cfg.reserved & 4) && block_size % 64 == 0 && n_blocks >= 2 &&
      ctx->n_tiles > 0 && n_blocks < 0x7fffffffull / ctx->n_tiles &&
      (uint64_t) std::max(ctx->int_max_byte, 1) * block_size < 2147483647ull) {
    const uint64_t need = (n_blocks * (uint64_t) ctx->n_tiles * unit_ints + 1) / 2;   // in doubles
    if (ctx->cache_valid && ctx->cache_blocks == n_blocks && ctx->cache_bs == block_size) {
      use_cache = true;
    } else {
      size_t fr = 0, tot = 0;
      NGSD_CUDA(ctx, cudaMemGetInfo(&fr, &tot));
      if (need * sizeof(double) + ((uint64_t) 3 << 30) <= (uint64_t) fr + ctx->cache_doubles * sizeof(double)) {
        if (need > ctx->cache_doubles) {
          cudaFree(ctx->d_cache);
          ctx->d_cache = nullptr;
          ctx->cache_doubles = 0;
          ctx->cache_valid = false;
          NGSD_CUDA(ctx, dev_alloc(&ctx->d_cache, need));
          ctx->cache_doubles = need;
        }
        use_cache = build_cache = true;
      }
    }
  }
  if (use_cache) maxw = 1;                                     // the contraction (if any) runs unweighted, K splits = blocks
  const uint32_t wcap = ngsd_int_weight_cap(ctx);              // site weights are int8 operand bytes: <= 127 (42) per layer
  // Sites that were empty text lines hold (0,0,0) in the reference (read_data.cpp:58-59): nothing to add for any pair,
  // but still counted without --pairwise_del.  A 2-bit code cannot say that, a site weight of 0 can.
  const bool blanks = ctx->any_blank && !ctx->cfg.pairwise_del;
  uint64_t n_words = use_cache ? n_blocks * (block_size / 64) : 0;
  const bool contract = !use_cache || build_cache;            // (otherwise the cached partials of this geometry are resident)
  if (contract) {
    int rc = build_word_list(ctx, use_cache ? nullptr : block_counts, n_blocks, block_size, maxw, wcap, blanks, n_words, &ctx->h_pin,
                             &ctx->h_pin_bytes, &n_words);
    if (rc) return rc;
  }

  if (ctx->n_tiles == 0 || n_words == 0) {   // a tile shard that owns nothing (or no active site): all-zero sums
    int rc = ensure_dist_buffers(ctx, 1);
    if (rc) return rc;
    const uint64_t n2 = ctx->n_ind * ctx->n_ind;
    NGSD_CUDA(ctx, cudaMemsetAsync(ctx->d_out, 0, n2 * sizeof(double), ctx->stream));
    NGSD_CUDA(ctx, cudaMemsetAsync(ctx->d_num, 0, n2 * sizeof(double), ctx->stream));
    NGSD_CUDA(ctx, cudaMemsetAsync(ctx->d_cntout, 0, n2 * sizeof(uint64_t), ctx->stream));
    if (ctx->n_tiles == 0) {
      ctx->timing = ngsd_timing();
      return copy_out(ctx, out, num_opt, cnt_opt);
    }
  }

  // K splits of the word list; an int32 accumulator must hold max_byte * weight * sites of one split
  std::vector<uint32_t> splits;
  std::vector<double> scales;
  if (use_cache) {
    splits.resize(n_blocks + 1);
    for (uint64_t b = 0; b <= n_blocks; b++) splits[b] = (uint32_t) (b * (block_size / 64));
    scales.resize(n_blocks);
    for (uint64_t b = 0; b < n_blocks; b++) scales[b] = (double) block_counts[b];
  } else {
    splits = plan_splits((uint32_t) n_words, ctx->n_tiles, (double) ctx->n_tiles, ctx->n_sm);
    const uint64_t per_word = (uint64_t) std::max(ctx->int_max_byte, 1) * std::min<uint32_t>(maxw, wcap) * 64;
    cap_splits(splits, (uint32_t) std::max<uint64_t>(1, 2147483647ull / per_word));
  }
  const uint32_t n_splits = (uint32_t) splits.size() - 1;
  const uint64_t n_units = (uint64_t) n_splits * ctx->n_tiles;
  const int grid = (int) std::min<uint64_t>(ctx->n_sm, std::max<uint64_t>(n_units, 1));
  int rc = ensure_dist_buffers(ctx, use_cache ? 1 : (do_count ? n_units + 1 : n_units / 2 + 1));   // int32 partials: sum tile (+ count tile) per unit
  if (rc) return rc;
  if (splits.size() > ctx->split_cap) {
    cudaFree(ctx->d_split_begin);
    ctx->d_split_begin = nullptr;
    ctx->split_cap = 0;
    NGSD_CUDA(ctx, dev_alloc(&ctx->d_split_begin, splits.size() + 64));
    cudaFree(ctx->d_split_scale);
    ctx->d_split_scale = nullptr;
    NGSD_CUDA(ctx, dev_alloc(&ctx->d_split_scale, splits.size() + 64));
    ctx->split_cap = (uint32_t) splits.size() + 64;
  }

  ctx->cur_partials = use_cache ? ctx->d_cache : ctx->d_partials;      // (after every (re)allocation above)
  ctx->cur_split_w = use_cache ? ctx->d_split_scale : nullptr;
  ctx->timing = ngsd_timing();
  NGSD_CUDA(ctx, cudaMemcpyAsync(ctx->d_split_begin, splits.data(), splits.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
  if (use_cache) NGSD_CUDA(ctx, cudaMemcpyAsync(ctx->d_split_scale, scales.data(), scales.size() * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  const bool run_kernel = n_words && contract;
  int launches = 0;
  tick(ctx, 2);
  tick(ctx, 3);
  if (run_kernel) {
    const uint32_t pstride = do_count ? 2 * NGSD_TILE_ELEMS : NGSD_TILE_ELEMS;
    NGSD_CUDA(ctx, ngsd_launch_dist_umma(ctx, (uint32_t) n_units, grid, pstride, false));
    // with --pairwise_del a second pass over the same units: the shared-site counts, as the second tile of each slot
    if (do_count) NGSD_CUDA(ctx, ngsd_launch_dist_umma(ctx, (uint32_t) n_units, grid, pstride, true));
    launches += do_count ? 2 : 1;
  }
  tick(ctx, 4);
  tick(ctx, 8);
  if (n_words) {
    NGSD_CUDA(ctx, ngsd_launch_epilogue_int(ctx, n_splits, n_eff, do_count));
    launches += 2;
  }
  tick(ctx, 5);
  rc = copy_out(ctx, out, num_opt, cnt_opt);
  if (rc) return rc;
  float ms;
  ctx->timing.count_ms = 0;                                  // part of dist_ms: the count GEMM runs inside K2c
  cudaEventElapsedTime(&ms, ctx->ev[3], ctx->ev[4]); ctx->timing.dist_ms = ms;
  cudaEventElapsedTime(&ms, ctx->ev[8], ctx->ev[5]); ctx->timing.epilogue_ms = ms;
  cudaEventElapsedTime(&ms, ctx->ev[2], ctx->ev[5]); ctx->timing.total_ms = ms;
  ctx->timing.launches = launches;
  ctx->timing.dist_ctas = grid;
  // IMMA-equivalents (4096 MAC each): 6 k-steps of 32 K bytes per word in the three-byte form (+2 for the count pass),
  // 128 per k-step and tile
  ctx->timing.dist_imma = run_kernel ? (uint64_t) n_words * (6 + (do_count ? 2 : 0)) * ctx->n_tiles * 128ull : 0;
  ctx->timing.active_sites = active_sites;
  ctx->timing.block_cache = use_cache ? (build_cache ? 1 : 2) : 0;
  if (use_cache) {
    ctx->cache_valid = true;
    ctx->cache_blocks = n_blocks;
    ctx->cache_bs = block_size;
  }
  ctx->cur_partials = ctx->d_partials;
  ctx->cur_split_w = nullptr;
  return NGSD_OK;
}

static int ensure_dist_buffers(ngsd_ctx *ctx, uint64_t slots) {
  const uint64_t n2 = ctx->n_ind * ctx->n_ind;
  if (!ctx->d_out) {
    NGSD_CUDA(ctx, dev_alloc(&ctx->d_out, n2));
    NGSD_CUDA(ctx, dev_alloc(&ctx->d_num, n2));
    NGSD_CUDA(ctx, dev_alloc(&ctx->d_cntout, n2));
    if (!ctx->int_path) {
      NGSD_CUDA(ctx, dev_alloc(&ctx->d_weights, ctx->NC * NGSD_SC_MAX));
      NGSD_CUDA(ctx, dev_alloc(&ctx->d_chunk_ids, ctx->NC));
    }
    if (ctx->cfg.pairwise_del && !ctx->int_path) NGSD_CUDA(ctx, dev_alloc(&ctx->d_cnt, ctx->n_pad * ctx->n_pad));
  }
  if (slots > ctx->partial_slots) {
    cudaFree(ctx->d_partials);
    ctx->d_partials = nullptr;
    ctx->partial_slots = 0;
    NGSD_CUDA(ctx, dev_alloc(&ctx->d_partials, slots * NGSD_TILE_ELEMS));
    ctx->partial_slots = slots;
  }
  return NGSD_OK;
}

static int ensure_entries(ngsd_ctx *ctx, uint64_t n) {
  if (n <= ctx->ent_cap) return NGSD_OK;
  cudaFree(ctx->d_ent_word);
  cudaFree(ctx->d_ent_mask);
  ctx->d_ent_word = nullptr;
  ctx->d_ent_mask = nullptr;
  ctx->ent_cap = 0;
  const uint64_t cap = n + n / 4 + 64;
  NGSD_CUDA(ctx, dev_alloc(&ctx->d_ent_word, cap));
  NGSD_CUDA(ctx, dev_alloc(&ctx->d_ent_mask, cap));
  ctx->ent_cap = cap;
  return NGSD_OK;
}

// --pairwise_del counts of the FP64 path as an int8 GEMM on the tensor cores (north_star (3): "integer mask GEMM"):
// the word list of the per-site weights (build_word_list, layers of <= 127), K splits for load balance, then
// k_dist_umma<true> + k_cnt_reduce into ctx->d_cnt.  Queued on ctx->stream.
static int count_on_tensor_cores(ngsd_ctx *ctx, const uint32_t *block_counts, uint64_t n_blocks, uint64_t block_size, uint32_t maxw, int *launches) {
  uint64_t n_words = 0;
  int rc = build_word_list(ctx, block_counts, n_blocks, block_size, maxw, 127, false, 0, &ctx->h_pin2, &ctx->h_pin2_bytes, &n_words);
  if (rc) return rc;
  if (n_words == 0) {
    NGSD_CUDA(ctx, cudaMemsetAsync(ctx->d_cnt, 0, ctx->n_pad * ctx->n_pad * sizeof(uint32_t), ctx->stream));
    return NGSD_OK;
  }
  std::vector<uint32_t> splits = plan_splits((uint32_t) n_words, ctx->n_tiles, (double) ctx->n_tiles, ctx->n_sm);
  cap_splits(splits, 2147483647u / (127u * 64u));   // an int32 accumulator holds 127 * 64 per word
  const uint32_t n_splits = (uint32_t) splits.size() - 1;
  if (splits.size() > ctx->cs_cap) {
    cudaFree(ctx->d_cs_begin);
    ctx->d_cs_begin = nullptr;
    ctx->cs_cap = 0;
    NGSD_CUDA(ctx, dev_alloc(&ctx->d_cs_begin, splits.size() + 64));
    ctx->cs_cap = (uint32_t) splits.size() + 64;
  }
  const uint64_t part = (uint64_t) n_splits * ctx->n_tiles * NGSD_TILE_ELEMS;
  if (part > ctx->cnt_part_ints) {
    cudaFree(ctx->d_cnt_part);
    ctx->d_cnt_part = nullptr;
    ctx->cnt_part_ints = 0;
    NGSD_CUDA(ctx, dev_alloc(&ctx->d_cnt_part, part));
    ctx->cnt_part_ints = part;
  }
  rc = upload_list(ctx, ctx->d_cs_begin, splits.data(), splits.size() * sizeof(uint32_t));
  if (rc) return rc;
  if (ctx->shard_world > 1) NGSD_CUDA(ctx, cudaMemsetAsync(ctx->d_cnt, 0, ctx->n_pad * ctx->n_pad * sizeof(uint32_t), ctx->stream));
  ngsd_count_umma_args ca{ctx->d_cs_begin, n_splits, ctx->d_cnt_part, ctx->d_wsite, ctx->d_word_ids, ctx->d_word_layer};
  NGSD_CUDA(ctx, ngsd_launch_count_umma(ctx, ca));
  *launches += 2;
  return NGSD_OK;
}

// One distance matrix of one GPU in three steps: distances_enqueue does the host bookkeeping (weights, chunk list, weight
// classes, count-pass word list, K splits) and queues the uploads and kernels; the caller copies ctx->d_out to the host;
// distances_collect reads the device times.  The paths that end early (degenerate replicates, the integer path) copy
// their matrix themselves and report job->copied.
struct dist_job {
  bool copied = false;        // the matrix is already in the caller's buffers and job->timing is complete
  bool count_timed = false;   // ev[6..7] bracket a count pass
  cudaEvent_t *ev = nullptr;  // the event set the matrix was timed with
  ngsd_timing timing = {};
};

static int distances_enqueue(ngsd_ctx *ctx, const uint32_t *block_counts, uint64_t n_blocks, uint64_t block_size, double *out,
                             double *num_opt, uint64_t *cnt_opt, dist_job *job) {
  *job = dist_job();
  job->ev = ctx->ev;
  NGSD_CUDA(ctx, cudaSetDevice(ctx->device));
  if (!ctx->frontend_done) {
    int rc = ngsd_frontend(ctx);
    if (rc) return rc;
  }
  // the pinned scratch may still feed the uploads of the matrix enqueued before this one
  NGSD_CUDA(ctx, cudaEventSynchronize(ctx->ev_pin));
  ctx->h_lists_used = 0;
  const bool em_path = !ctx->cfg.indep_geno;   // default --probs: per pair-site em2 (ngsDist.cpp:348-349)
  const bool weighted = block_counts != nullptr;
  uint64_t n_eff = ctx->n_sites;
  if (weighted) {
    if (block_size == 0 || n_blocks * block_size > ctx->n_sites) {
      ngsd_set_error(ctx, "invalid bootstrap geometry: %llu blocks of %llu sites", (unsigned long long) n_blocks, (unsigned long long) block_size);
      return NGSD_ERR_ARG;
    }
    n_eff = n_blocks * block_size;
    if (n_blocks == 0) {
      // --boot_block_size > n_sites: the reference truncates n_sites to 0 (ngsDist.cpp:236) and still writes a matrix --
      // every pair has dist = 0 over cnt = 0 sites, i.e. 0/0 (or 0/tot_sites) through ngsDist.cpp:372-401.  The same
      // degenerate replicate is what a site shard without any block contributes: all-zero sums.
      int rc0 = ensure_dist_buffers(ctx, 1);
      if (rc0) return rc0;
      const uint64_t n2z = ctx->n_ind * ctx->n_ind;
      NGSD_CUDA(ctx, cudaMemsetAsync(ctx->d_num, 0, n2z * sizeof(double), ctx->stream));
      NGSD_CUDA(ctx, cudaMemsetAsync(ctx->d_cntout, 0, n2z * sizeof(uint64_t), ctx->stream));
      NGSD_CUDA(ctx, ngsd_launch_finish(ctx));
      if (em_path) NGSD_CUDA(ctx, ngsd_clear_unowned(ctx));
      rc0 = copy_out(ctx, out, num_opt, cnt_opt);
      if (rc0) return rc0;
      ctx->timing = ngsd_timing();
      ctx->timing.launches = 1;
      job->copied = true;
      return NGSD_OK;
    }
  }
  if (ctx->int_path) {
    job->copied = true;
    return distances_int(ctx, block_counts, n_blocks, block_size, out, num_opt, cnt_opt);
  }
  if (em_path && ctx->any_blank && !ctx->cfg.pairwise_del) {
    // An empty text line is (0,0,0) for every individual (read_data.cpp:58-59); em2 on it divides 0 by 0
    // (emOptim2.cpp:69-75 normalize), so every pair's sum turns NaN as soon as one such site is in the replicate.
    bool hit = false;
    for (uint64_t w = 0; w < ctx->NW && !hit; w++)
      for (uint64_t m = ctx->h_blank[w]; m && !hit; m &= m - 1) {
        const uint64_t s_ = w * 64 + (uint64_t) __builtin_ctzll(m);
        hit = weighted ? (s_ < n_eff && block_counts[s_ / block_size] > 0) : true;
      }
    if (hit) {
      int rc0 = ensure_dist_buffers(ctx, 1);
      if (rc0) return rc0;
      const uint64_t n2z = ctx->n_ind * ctx->n_ind;
      NGSD_CUDA(ctx, cudaMemsetAsync(ctx->d_num, 0xFF, n2z * sizeof(double), ctx->stream));   // all-ones = the negative quiet NaN x86 gives 0/0
      NGSD_CUDA(ctx, ngsd_launch_finish(ctx, n_eff));
      NGSD_CUDA(ctx, ngsd_clear_unowned(ctx));
      rc0 = copy_out(ctx, out, num_opt, cnt_opt);
      if (rc0) return rc0;
      ctx->timing = ngsd_timing();
      ctx->timing.launches = 1;
      job->copied = true;
      return NGSD_OK;
    }
  }
  const uint64_t SC = (uint64_t) ctx->sc;
  const uint64_t NCu = (ctx->n_sites + SC - 1) / SC;   // chunks that hold data

  // ---- host-side bootstrap bookkeeping: per-site weights, active chunk list, K3 entries of the block cache ----
  uint64_t n_chunks = NCu, n_entries = 0, active_sites = n_eff;
  bool uniform_scale = false;
  std::vector<uint32_t> class_end;      // (uniform_scale) end position of each weight class in the sorted chunk list
  std::vector<double> class_weight;
  uint32_t maxw = 1;
  if (weighted)
    for (uint64_t b = 0; b < n_blocks; b++) maxw = std::max(maxw, block_counts[b]);
  const uint64_t ent_max = ctx->cfg.pairwise_del ? ctx->NW + 2 * n_blocks + 2 : 0;   // a block touches <= block_size / 64 + 2 words
  const uint64_t bytes_w = ctx->NC * SC * sizeof(double), bytes_c = ctx->NC * sizeof(uint32_t);
  const uint64_t bytes_e = ent_max * (sizeof(uint32_t) + sizeof(uint64_t));
  int rc = ensure_pinned(ctx, &ctx->h_pin, &ctx->h_pin_bytes, bytes_w + bytes_c + bytes_e + 64);
  if (rc) return rc;
  double *h_w = (double *) ctx->h_pin;
  uint64_t *h_em = (uint64_t *) ((char *) ctx->h_pin + bytes_w);
  uint32_t *h_c = (uint32_t *) ((char *) h_em + ent_max * sizeof(uint64_t));
  uint32_t *h_ew = h_c + ctx->NC;
  // ---- bootstrap block cache -------------------------------------------------------------------------------------
  // Resampling is by whole blocks (ngsDist.cpp:416-437), so num_r(i,j) = sum_b c_r[b] * G_b(i,j) with G_b the sum over
  // the sites of source block b: compute the per-block partials ONCE (K splits = blocks) and every replicate is a
  // weighted split reduction in the epilogue -- ~100x less work per replicate at C3 (SURVEY §7 design option (a)).
  // It needs blocks that are whole site chunks and room for n_blocks partials; otherwise (and with ngsd_cfg.reserved
  // bit 2, which benchmarks of the per-replicate weighted contraction set) the replicate is contracted directly.
  const uint64_t em_split_doubles = em_path ? ngsd_em_split_doubles(ctx) : 0;
  bool use_cache = false, build_cache = false;
  if (weighted && !(ctx->cfg.reserved & 4) && block_size % SC == 0 && n_blocks >= 2 &&
      n_blocks < 0x7fffffffull / std::max<uint32_t>(ctx->n_tiles, 1)) {
    const uint64_t need = em_path ? n_blocks * em_split_doubles : n_blocks * (uint64_t) ctx->n_tiles * NGSD_TILE_ELEMS;
    // with --pairwise_del the per-block shared-site counts are cached next to the sums (one K3 split per block)
    const uint64_t need_cnt = (ctx->cfg.pairwise_del && n_blocks <= 65535) ? n_blocks * (uint64_t) ctx->n_tiles * NGSD_TILE_ELEMS : 0;
    if (ctx->cache_valid && ctx->cache_blocks == n_blocks && ctx->cache_bs == block_size) {
      use_cache = true;
    } else {
      size_t fr = 0, tot = 0;
      NGSD_CUDA(ctx, cudaMemGetInfo(&fr, &tot));
      const uint64_t avail = (uint64_t) fr + ctx->cache_doubles * sizeof(double) + ctx->cnt_cache_elems * sizeof(uint32_t);
      if (need * sizeof(double) + need_cnt * sizeof(uint32_t) + ((uint64_t) 3 << 30) <= avail) {
        if (need_cnt > ctx->cnt_cache_elems) {
          cudaFree(ctx->d_cnt_cache);
          ctx->d_cnt_cache = nullptr;
          ctx->cnt_cache_elems = 0;
          NGSD_CUDA(ctx, dev_alloc(&ctx->d_cnt_cache, need_cnt));
          ctx->cnt_cache_elems = need_cnt;
        }
        if (need > ctx->cache_doubles) {
          cudaFree(ctx->d_cache);
          ctx->d_cache = nullptr;
          ctx->cache_doubles = 0;
          ctx->cache_valid = false;
          NGSD_CUDA(ctx, dev_alloc(&ctx->d_cache, need));
          ctx->cache_doubles = need;
        }
        use_cache = build_cache = true;
      }
    }
  }

  const bool need_site_weights = weighted && (!use_cache || ctx->planes == 2);   // cached replicates only need them for the c-vector
  if (weighted && !need_site_weights) {
    active_sites = 0;
    for (uint64_t b = 0; b < n_blocks; b++) active_sites += block_counts[b] ? block_size : 0;
  }
  if (need_site_weights) {
    active_sites = 0;
    memset(h_w, 0, bytes_w);
    for (uint64_t b = 0; b < n_blocks; b++) {
      if (!block_counts[b]) continue;
      const double w = (double) block_counts[b];
      for (uint64_t s = b * block_size; s < (b + 1) * block_size; s++) h_w[s] = w;
      active_sites += block_size;
    }
    n_chunks = 0;
    for (uint64_t c = 0; c < NCu && !use_cache; c++) {
      bool any = false;
      for (uint64_t k = 0; k < SC; k++) any |= h_w[c * SC + k] != 0.0;
      if (any) h_c[n_chunks++] = (uint32_t) c;
    }
    // Blocks that are whole chunks (block_size % 8 == 0): every chunk has ONE weight.  Order the chunk list by weight
    // class (stable), let every K split lie inside one class and carry the weight as a per-split scale: the inner loop
    // of k_dist_dmma then needs no per-site multiplies at all (DMMA and DMUL share one pipe).
    uniform_scale = (block_size % SC == 0) && !em_path;
    if (uniform_scale && !use_cache) {
      std::vector<uint32_t> sorted;
      sorted.reserve(n_chunks);
      class_end.clear();
      class_weight.clear();
      for (uint32_t v = 1; v <= maxw; v++) {
        const size_t before = sorted.size();
        for (uint64_t k = 0; k < n_chunks; k++)
          if (h_w[(uint64_t) h_c[k] * SC] == (double) v) sorted.push_back(h_c[k]);
        if (sorted.size() > before) { class_end.push_back((uint32_t) sorted.size()); class_weight.push_back((double) v); }
      }
      memcpy(h_c, sorted.data(), n_chunks * sizeof(uint32_t));
    }
  }
  if (ctx->n_tiles == 0) {   // a tile shard that owns nothing: all-zero contribution
    int rc0 = ensure_dist_buffers(ctx, 1);
    if (rc0) return rc0;
    const uint64_t n2z = ctx->n_ind * ctx->n_ind;
    NGSD_CUDA(ctx, cudaMemsetAsync(ctx->d_out, 0, n2z * sizeof(double), ctx->stream));
    NGSD_CUDA(ctx, cudaMemsetAsync(ctx->d_num, 0, n2z * sizeof(double), ctx->stream));
    NGSD_CUDA(ctx, cudaMemsetAsync(ctx->d_cntout, 0, n2z * sizeof(uint64_t), ctx->stream));
    ctx->timing = ngsd_timing();
    job->copied = true;
    return copy_out(ctx, out, num_opt, cnt_opt);
  }
  // The shared-site counts of --pairwise_del come from one of two sources: the per-block counts of the block cache
  // (K3 builds them next to the per-block sums, one split per source block; the cache build above sized d_cnt_cache
  // for this geometry), or the int8 count pass on the tensor cores.
  const bool cnt_from_cache = use_cache && ctx->cfg.pairwise_del && n_blocks <= 65535 && ctx->d_cnt_cache != nullptr;
  const bool cnt_on_tc = ctx->cfg.pairwise_del && !cnt_from_cache;
  const bool run_k3 = cnt_from_cache && build_cache;
  std::vector<uint32_t> ent_begin;
  if (run_k3) {   // K3 entries: the sites of every block as (word, mask) pairs
    ent_begin.resize(n_blocks + 1);
    for (uint64_t b = 0; b < n_blocks; b++) {
      ent_begin[b] = (uint32_t) n_entries;
      uint64_t s0 = b * block_size, s1 = s0 + block_size;
      while (s0 < s1) {   // the block's bits, word by word
        const uint64_t w = s0 >> 6, lo = s0 & 63, hi = std::min<uint64_t>(64, lo + (s1 - s0));
        h_ew[n_entries] = (uint32_t) w;
        h_em[n_entries] = (hi == 64 ? ~0ull : ((1ull << hi) - 1)) & ~((1ull << lo) - 1);
        n_entries++;
        s0 += hi - lo;
      }
    }
    ent_begin[n_blocks] = (uint32_t) n_entries;
    if (n_blocks + 1 > ctx->ent_begin_cap) {
      cudaFree(ctx->d_ent_begin);
      ctx->d_ent_begin = nullptr;
      ctx->ent_begin_cap = 0;
      NGSD_CUDA(ctx, dev_alloc(&ctx->d_ent_begin, n_blocks + 1));
      ctx->ent_begin_cap = n_blocks + 1;
    }
  }

  ngsd_dist_plan plan;
  uint32_t em_splits = 0;
  plan.weighted = weighted;
  plan.n_chunks = (uint32_t) n_chunks;
  plan.grid = ctx->n_sm;
  const double cost_tiles = (double) (ctx->n_tiles - ctx->n_diag_tiles) + ctx->n_diag_tiles * (136.0 / 256.0);
  std::vector<uint32_t> splits;
  std::vector<double> scales;
  plan.uniform_scale = uniform_scale;
  if (use_cache) {            // K splits = source blocks, unweighted, identity chunk list
    const uint32_t per = (uint32_t) (block_size / SC);
    splits.resize(n_blocks + 1);
    for (uint64_t b = 0; b <= n_blocks; b++) splits[b] = (uint32_t) (b * per);
    scales.resize(n_blocks);
    for (uint64_t b = 0; b < n_blocks; b++) scales[b] = (double) block_counts[b];
    plan.weighted = false;
    plan.uniform_scale = false;
    plan.n_chunks = (uint32_t) (n_blocks * per);
  } else {
    splits = plan_splits(plan.n_chunks, ctx->n_tiles, cost_tiles, plan.grid);
  }
  if (uniform_scale && !use_cache) {   // cut the splits at the class boundaries and record each split's weight
    std::vector<uint32_t> cut;
    size_t k = 0;
    cut.push_back(0);
    for (size_t q = 1; q < splits.size(); q++) {
      while (k < class_end.size() && class_end[k] < splits[q]) {
        if (class_end[k] > cut.back()) cut.push_back(class_end[k]);
        k++;
      }
      if (splits[q] > cut.back()) cut.push_back(splits[q]);
    }
    splits.swap(cut);
    k = 0;
    for (size_t q = 0; q + 1 < splits.size(); q++) {
      while (k < class_end.size() && class_end[k] <= splits[q]) k++;
      scales.push_back(k < class_weight.size() ? class_weight[k] : 1.0);
    }
  }
  plan.n_splits = (uint32_t) splits.size() - 1;
  plan.n_units = plan.n_splits * ctx->n_tiles;
  plan.grid = (int) std::min<uint64_t>(plan.grid, plan.n_units);
  if (em_path) {
    em_splits = use_cache ? (uint32_t) n_blocks : ngsd_em_splits(ctx, plan.n_chunks);
    plan.n_units = (uint32_t) (((uint64_t) em_splits * em_split_doubles + NGSD_TILE_ELEMS - 1) / NGSD_TILE_ELEMS);   // workspace slots
  }
  if (splits.size() > ctx->split_cap) {
    cudaFree(ctx->d_split_begin);
    ctx->d_split_begin = nullptr;
    ctx->split_cap = 0;
    NGSD_CUDA(ctx, dev_alloc(&ctx->d_split_begin, splits.size() + 64));
    cudaFree(ctx->d_split_scale);
    ctx->d_split_scale = nullptr;
    NGSD_CUDA(ctx, dev_alloc(&ctx->d_split_scale, splits.size() + 64));
    ctx->split_cap = (uint32_t) splits.size() + 64;
  }
  rc = ensure_dist_buffers(ctx, use_cache ? 1 : plan.n_units);
  if (rc) return rc;
  if (ctx->cfg.pairwise_del) {
    rc = ensure_entries(ctx, n_entries);
    if (rc) return rc;
  }
  ctx->cur_partials = use_cache ? ctx->d_cache : ctx->d_partials;
  ctx->cur_split_w = use_cache ? ctx->d_split_scale : nullptr;
  ctx->cur_cnt_cache = cnt_from_cache ? ctx->d_cnt_cache : nullptr;

  ctx->timing = ngsd_timing();
  rc = upload_list(ctx, ctx->d_split_begin, splits.data(), splits.size() * sizeof(uint32_t));
  if (rc) return rc;
  if (uniform_scale || use_cache) {
    rc = upload_list(ctx, ctx->d_split_scale, scales.data(), scales.size() * sizeof(double));
    if (rc) return rc;
  }
  if (weighted) {
    if (need_site_weights && (!uniform_scale || ctx->planes == 2))   // per-site weights: scaled B fragments and/or the weighted c-vector
      NGSD_CUDA(ctx, cudaMemcpyAsync(ctx->d_weights, h_w, bytes_w, cudaMemcpyHostToDevice, ctx->stream));
    if (!use_cache) NGSD_CUDA(ctx, cudaMemcpyAsync(ctx->d_chunk_ids, h_c, n_chunks * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
  }
  if (n_entries) {
    NGSD_CUDA(ctx, cudaMemcpyAsync(ctx->d_ent_word, h_ew, n_entries * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    NGSD_CUDA(ctx, cudaMemcpyAsync(ctx->d_ent_mask, h_em, n_entries * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream));
  }
  if (run_k3) {
    rc = upload_list(ctx, ctx->d_ent_begin, ent_begin.data(), ent_begin.size() * sizeof(uint32_t));
    if (rc) return rc;
  }
  int launches = 0;
  const bool do_count = ctx->cfg.pairwise_del != 0;
  tick(ctx, 2);
  if (cnt_on_tc) {   // counts on the int8 tensor cores, ahead of the contraction on the same stream
    NGSD_CUDA(ctx, cudaEventRecord(ctx->ev[6], ctx->stream));
    int rcc = count_on_tensor_cores(ctx, block_counts, n_blocks, block_size, maxw, &launches);
    if (rcc) return rcc;
    NGSD_CUDA(ctx, cudaEventRecord(ctx->ev[7], ctx->stream));
  }
  NGSD_CUDA(ctx, cudaEventRecord(ctx->ev_pin, ctx->stream));   // every upload from pinned scratch is queued above
  if (run_k3) NGSD_CUDA(ctx, cudaEventRecord(ctx->ev_fork, ctx->stream));   // K3 entry lists are on the device
  tick(ctx, 3);
  // K2 / K2b first, so that its persistent CTAs own every SM; K3 (building the block cache's counts) is then launched on
  // the auxiliary stream and its (small) CTAs co-reside with them: integer AND+POPC in the shadow of the FP64 contraction.
  if (use_cache && !build_cache) {
    // the per-block partials of this geometry are resident: nothing to contract
  } else if (em_path) {
    NGSD_CUDA(ctx, ngsd_launch_dist_em(ctx, plan.n_chunks, em_splits, plan.weighted));
    launches++;
  } else if (plan.n_chunks > 0) {
    NGSD_CUDA(ctx, ngsd_launch_dist_dmma(ctx, plan));
    launches++;
  } else {
    NGSD_CUDA(ctx, cudaMemsetAsync(ctx->d_partials, 0, (uint64_t) plan.n_units * NGSD_TILE_ELEMS * sizeof(double), ctx->stream));
  }
  NGSD_CUDA(ctx, dbg_sync(ctx, "contraction"));
  tick(ctx, 4);
  if (run_k3) {
    NGSD_CUDA(ctx, cudaStreamWaitEvent(ctx->aux_stream, ctx->ev_fork, 0));
    NGSD_CUDA(ctx, cudaEventRecord(ctx->ev[6], ctx->aux_stream));
    NGSD_CUDA(ctx, ngsd_launch_mask_count(ctx, (uint32_t) n_blocks, ctx->aux_stream));
    NGSD_CUDA(ctx, cudaEventRecord(ctx->ev[7], ctx->aux_stream));
    NGSD_CUDA(ctx, cudaEventRecord(ctx->ev_join, ctx->aux_stream));
    NGSD_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_join, 0));
    launches++;
  }
  NGSD_CUDA(ctx, dbg_sync(ctx, "mask count"));
  tick(ctx, 8);
  if (!em_path && ctx->planes == 2) {
    NGSD_CUDA(ctx, ngsd_launch_cvec(ctx, weighted, n_eff));
    launches++;
    if (!ctx->deficit.empty()) {
      int rcd = upload_deficit(ctx);
      if (rcd) return rcd;
      NGSD_CUDA(ctx, ngsd_launch_deficit_fix(ctx, weighted, n_eff));
      launches++;
    }
  }
  if (em_path) {
    NGSD_CUDA(ctx, ngsd_launch_epilogue_em(ctx, em_splits, n_eff, do_count));
    launches++;
  } else {
    ngsd_epilogue_args ea;
    ea.n_splits = plan.n_splits;
    ea.const_cnt = n_eff;
    ea.use_cnt = do_count;
    NGSD_CUDA(ctx, ngsd_launch_epilogue(ctx, ea));
    launches += 2;
  }
  NGSD_CUDA(ctx, dbg_sync(ctx, "epilogue"));
  tick(ctx, 5);
  job->count_timed = cnt_on_tc || run_k3;
  ctx->timing.launches = launches;
  ctx->timing.dist_ctas = plan.grid;
  // DMMAs executed per K4 step (ctx->k4 steps per chunk): 256 per full tile, 136 per diagonal tile, 16 per real 8-column block of an edge tile
  const uint64_t dmma_step = (uint64_t) (ctx->n_tiles - ctx->n_diag_tiles - ctx->n_edge_tiles) * 256ull + (uint64_t) ctx->n_diag_tiles * 136ull +
                             (uint64_t) ctx->n_edge_tiles * 16ull * ngsd_edge_c8(ctx->n_ind);
  ctx->timing.dist_dmma = (em_path || (use_cache && !build_cache)) ? 0 : (uint64_t) plan.n_chunks * ctx->k4 * dmma_step;
  ctx->timing.active_sites = active_sites;
  ctx->timing.block_cache = use_cache ? (build_cache ? 1 : 2) : 0;
  if (use_cache) {
    ctx->cache_valid = true;
    ctx->cache_blocks = n_blocks;
    ctx->cache_bs = block_size;
  }
  ctx->cur_partials = ctx->d_partials;
  ctx->cur_split_w = nullptr;
  ctx->cur_cnt_cache = nullptr;
  job->timing = ctx->timing;
  return NGSD_OK;
}

// Device times of an enqueued matrix into job->timing (waits for its epilogue).
static int distances_collect(ngsd_ctx *ctx, dist_job *job) {
  if (job->copied) return NGSD_OK;
  cudaEvent_t *ev = job->ev;
  NGSD_CUDA(ctx, cudaEventSynchronize(ev[5]));
  float ms;
  ngsd_timing &t = job->timing;
  t.count_ms = 0;
  if (job->count_timed) { cudaEventElapsedTime(&ms, ev[6], ev[7]); t.count_ms = ms; }   // K3 overlaps dist_ms; the tensor-core count precedes it
  cudaEventElapsedTime(&ms, ev[3], ev[4]); t.dist_ms = ms;
  cudaEventElapsedTime(&ms, ev[8], ev[5]); t.epilogue_ms = ms;
  cudaEventElapsedTime(&ms, ev[2], ev[5]); t.total_ms = ms;
  return NGSD_OK;
}

int ngsd_distances(ngsd_ctx *ctx, const uint32_t *block_counts, uint64_t n_blocks, uint64_t block_size, double *out,
                   double *num_opt, uint64_t *cnt_opt) {
  if (!ctx) return NGSD_ERR_ARG;
  if (!ctx->kids.empty()) return ngsd_group_distances(ctx, block_counts, n_blocks, block_size, out, num_opt, cnt_opt);
  dist_job job;
  int rc = distances_enqueue(ctx, block_counts, n_blocks, block_size, out, num_opt, cnt_opt, &job);
  if (rc || job.copied) return rc;
  rc = copy_out(ctx, out, num_opt, cnt_opt);
  if (rc) return rc;
  rc = distances_collect(ctx, &job);
  ctx->timing = job.timing;
  return rc;
}

// The single-GPU replicate loop.  Replicate r + 1 is enqueued -- its host bookkeeping included -- before replicate r is
// collected, so the device runs the replicates back to back instead of waiting for each result copy and for the host to
// build the next replicate's lists.  The matrices alternate between d_out and d_out_alt and reach the host on
// copy_stream; replicate r + 2 waits for the copy of r before it overwrites that buffer.
static int distances_pipelined(ngsd_ctx *ctx, const uint32_t *block_counts, uint64_t n_rep, uint64_t n_blocks, uint64_t block_size,
                               double *out, ngsd_timing *sum) {
  const uint64_t n2 = ctx->n_ind * ctx->n_ind;
  if (n_rep > 1) {
    int rc = ensure_dist_buffers(ctx, 1);
    if (rc) return rc;
    if (!ctx->d_out_alt) NGSD_CUDA(ctx, dev_alloc(&ctx->d_out_alt, n2));
  }
  double *buf[2] = {ctx->d_out, ctx->d_out_alt};
  dist_job job[2];
  auto collect = [&](uint64_t r) -> int {
    dist_job &j = job[r & 1];
    if (!j.copied) {
      NGSD_CUDA(ctx, cudaStreamWaitEvent(ctx->copy_stream, j.ev[5], 0));
      NGSD_CUDA(ctx, cudaMemcpyAsync(out + r * n2, buf[r & 1], n2 * sizeof(double), cudaMemcpyDeviceToHost, ctx->copy_stream));
      NGSD_CUDA(ctx, cudaEventRecord(ctx->ev_copied[r & 1], ctx->copy_stream));
      int rc = distances_collect(ctx, &j);
      if (rc) return rc;
    }
    const ngsd_timing &t = j.timing;
    sum->count_ms += t.count_ms; sum->dist_ms += t.dist_ms; sum->epilogue_ms += t.epilogue_ms;
    sum->total_ms += t.total_ms; sum->launches += t.launches; sum->dist_dmma += t.dist_dmma;
    sum->dist_imma += t.dist_imma; sum->active_sites += t.active_sites;
    sum->dist_ctas = t.dist_ctas; sum->block_cache = t.block_cache;
    return NGSD_OK;
  };
  int rc = NGSD_OK;
  for (uint64_t r = 0; r < n_rep && !rc; r++) {
    if (r >= 2 && cudaStreamWaitEvent(ctx->stream, ctx->ev_copied[r & 1], 0) != cudaSuccess) {
      ngsd_set_error(ctx, "CUDA error: cannot order replicate %llu after a result copy", (unsigned long long) r);
      rc = NGSD_ERR_CUDA;
      break;
    }
    ctx->d_out = buf[r & 1];
    ctx->ev = ctx->ev_sets[r & 1];
    rc = distances_enqueue(ctx, block_counts + r * n_blocks, n_blocks, block_size, out + r * n2, nullptr, nullptr, &job[r & 1]);
    buf[r & 1] = ctx->d_out;   // (allocated by the first enqueue when n_rep == 1)
    if (job[r & 1].copied) job[r & 1].timing = ctx->timing;
    if (!rc && r >= 1) rc = collect(r - 1);
    if (!rc && r + 1 == n_rep) rc = collect(r);
  }
  // d_out keeps the last matrix (ngsd_device_results, ngsd_finish), d_out_alt the other buffer; set 0 times the pushes
  ctx->d_out_alt = ctx->d_out == buf[0] ? buf[1] : buf[0];
  ctx->ev = ctx->ev_sets[0];
  const cudaError_t e = cudaStreamSynchronize(ctx->copy_stream);
  if (rc) return rc;
  NGSD_CUDA(ctx, e);
  return NGSD_OK;
}

// The bootstrap loop of main() (ngsDist.cpp:217-238) in one call.  One GPU: distances_pipelined; groups and
// communicators deal the replicates out (comm.cu).
int ngsd_distances_batch(ngsd_ctx *ctx, const uint32_t *block_counts, uint64_t n_rep, uint64_t n_blocks, uint64_t block_size, double *out) {
  if (!ctx) return NGSD_ERR_ARG;
  if (!block_counts && n_rep) { ngsd_set_error(ctx, "null block_counts"); return NGSD_ERR_ARG; }
  if (!ctx->kids.empty() || ctx->comm) return ngsd_group_distances_batch(ctx, block_counts, n_rep, n_blocks, block_size, out);
  if (!out && n_rep) { ngsd_set_error(ctx, "null output"); return NGSD_ERR_ARG; }
  NGSD_CUDA(ctx, cudaSetDevice(ctx->device));
  ngsd_timing sum = ngsd_timing();
  int rc = distances_pipelined(ctx, block_counts, n_rep, n_blocks, block_size, out, &sum);
  if (rc) return rc;
  ctx->timing = sum;
  return NGSD_OK;
}

// ---------------------------------------------------------------------------------------------- multi-GPU ----

int ngsd_set_tile_shard(ngsd_ctx *ctx, uint32_t rank, uint32_t world) {
  if (!ctx) return NGSD_ERR_ARG;
  if (!ctx->kids.empty()) { ngsd_set_error(ctx, "a multi-GPU context deals the tiles to its GPUs itself"); return NGSD_ERR_ARG; }
  if (world == 0 || rank >= world) { ngsd_set_error(ctx, "invalid tile shard %u of %u", rank, world); return NGSD_ERR_ARG; }
  NGSD_CUDA(ctx, cudaSetDevice(ctx->device));
  // the unit of ownership is a PAIR of neighbouring tiles of one row block (the odd tile of a row alone): dist_umma.cu
  // contracts such pairs with one shared A operand, so a shard keeps them together
  // (dealt in list order, each unit to the rank holding the fewest tiles so far, lowest rank first: tile counts differ by <= 2)
  std::vector<ngsd_tile> all = make_tiles((uint32_t) ctx->RB), mine;
  std::vector<uint32_t> held(world, 0);
  for (size_t t = 0; t < all.size();) {
    const size_t len = (t + 1 < all.size() && all[t + 1].ti == all[t].ti) ? 2 : 1;
    const uint32_t to = (uint32_t) (std::min_element(held.begin(), held.end()) - held.begin());
    held[to] += (uint32_t) len;
    if (to == rank)
      for (size_t k = 0; k < len; k++) mine.push_back(all[t + k]);
    t += len;
  }
  NGSD_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  ctx->n_tiles = (uint32_t) mine.size();
  ctx->n_diag_tiles = 0;
  ctx->n_edge_tiles = 0;
  for (auto &t : mine) {
    ctx->n_diag_tiles += (t.ti == t.tj);
    ctx->n_edge_tiles += ngsd_is_edge_tile(t, ctx->n_ind, ctx->RB);
  }
  if (!mine.empty()) NGSD_CUDA(ctx, copy_sync(ctx, ctx->d_tiles, mine.data(), mine.size() * sizeof(ngsd_tile), cudaMemcpyHostToDevice));
  NGSD_CUDA(ctx, upload_tile_index(ctx, mine));
  if (!ctx->cfg.indep_geno) NGSD_CUDA(ctx, upload_em_tiles(ctx, mine));   // the EM path contracts the 64 x 64 tiles inside them
  ctx->shard_rank = rank;
  ctx->shard_world = world;
  ctx->cache_valid = false;
  return NGSD_OK;
}

int ngsd_device_results(ngsd_ctx *ctx, double **out_dev, double **num_dev, uint64_t **cnt_dev) {
  if (!ctx) return NGSD_ERR_ARG;
  if (!ctx->kids.empty()) ctx = ctx->kids[0];   // the root GPU of a group holds the assembled / reduced matrices
  if (!ctx->d_out) { ngsd_set_error(ctx, "no results yet: call ngsd_distances first"); return NGSD_ERR_STATE; }
  if (out_dev) *out_dev = ctx->d_out;
  if (num_dev) *num_dev = ctx->d_num;
  if (cnt_dev) *cnt_dev = ctx->d_cntout;
  return NGSD_OK;
}

int ngsd_finish(ngsd_ctx *ctx, double *out_host) {
  if (!ctx) return NGSD_ERR_ARG;
  if (!ctx->kids.empty()) ctx = ctx->kids[0];
  if (!ctx->d_out) { ngsd_set_error(ctx, "no results yet: call ngsd_distances first"); return NGSD_ERR_STATE; }
  NGSD_CUDA(ctx, cudaSetDevice(ctx->device));
  NGSD_CUDA(ctx, ngsd_launch_finish(ctx));
  return copy_out(ctx, out_host, nullptr, nullptr);
}

// ------------------------------------------------------------------------------------------- bootstrap RNG ----
// gsl_rng_taus (GSL rng/taus.c semantics; SURVEY App. B): the reference seeds it at ngsDist.cpp:179-180 and draws
// n_blocks uniforms per replicate in rnd_map_data (ngsDist.cpp:421-423) through draw_rnd (gen_func.cpp:117-119).

static inline uint32_t taus_step(uint32_t *s) {
#define NGSD_TAUS(x, a, b, c, d) ((((x) & (c)) << (d)) ^ ((((x) << (a)) ^ (x)) >> (b)))
  s[0] = NGSD_TAUS(s[0], 13, 19, 4294967294u, 12);
  s[1] = NGSD_TAUS(s[1], 2, 25, 4294967288u, 4);
  s[2] = NGSD_TAUS(s[2], 3, 11, 4294967280u, 17);
#undef NGSD_TAUS
  return s[0] ^ s[1] ^ s[2];
}

void ngsd_taus_seed(uint32_t state[3], uint32_t seed) {
  if (seed == 0) seed = 1;
  state[0] = 69069u * seed;
  state[1] = 69069u * state[0];
  state[2] = 69069u * state[1];
  for (int i = 0; i < 6; i++) taus_step(state);
}

uint32_t ngsd_taus_get(uint32_t state[3]) { return taus_step(state); }

void ngsd_boot_block_counts(uint32_t state[3], uint64_t n_blocks, uint32_t *counts) {
  memset(counts, 0, n_blocks * sizeof(uint32_t));
  for (uint64_t b = 0; b < n_blocks; b++) {
    const double u = taus_step(state) / 4294967296.0;
    const uint64_t rb = (uint64_t) floor(0.0 + u * (double) n_blocks);
    counts[rb]++;
  }
}

// ------------------------------------------------------------------------------------------- measurement ----

int ngsd_synth_raw_device(ngsd_ctx *ctx, double *raw_dev, uint64_t seed, double miss_rate, uint64_t site0, uint64_t n) {
  if (!ctx || !raw_dev) return NGSD_ERR_ARG;
  if (!ctx->kids.empty()) { ngsd_set_error(ctx, "synthetic device input needs a single-GPU context"); return NGSD_ERR_ARG; }
  NGSD_CUDA(ctx, cudaSetDevice(ctx->device));
  NGSD_CUDA(ctx, ngsd_launch_synth(ctx, raw_dev, seed, miss_rate, site0, n));
  NGSD_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return NGSD_OK;
}

int ngsd_get_timing(const ngsd_ctx *ctx, ngsd_timing *t) {
  if (!ctx || !t) return NGSD_ERR_ARG;
  ngsd_ctx *c = const_cast<ngsd_ctx *>(ctx);
  if (!c->kids.empty()) return ngsd_group_get_timing(c, t);
  if (c->timing.total_ms < 0) {   // a push: events 0..1
    if (cudaEventSynchronize(c->ev[1]) != cudaSuccess) return NGSD_ERR_CUDA;
    float ms = 0;
    cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]);
    c->timing.frontend_ms = ms;
    c->timing.total_ms = ms;
  }
  *t = c->timing;
  return NGSD_OK;
}

int ngsd_deferred_stats(const ngsd_ctx *ctx, uint64_t *host_evaluated) {
  if (!ctx || !host_evaluated) return NGSD_ERR_ARG;
  uint64_t n = ctx->deferred_total;
  for (const ngsd_ctx *k : ctx->kids) n += k->deferred_total;
  *host_evaluated = n;
  return NGSD_OK;
}

void *ngsd_stream(ngsd_ctx *ctx) { return ctx ? (void *) (ctx->kids.empty() ? ctx->stream : ctx->kids[0]->stream) : nullptr; }

void *ngsd_host_alloc(uint64_t bytes) {
  void *p = nullptr;
  if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) return nullptr;
  return p;
}

void ngsd_host_free(void *p) {
  if (p) cudaFreeHost(p);
}

}  // extern "C"
