// K2 dist_dmma: the per-pair, per-site loop of gen_dist with indep_geno (ngsDist.cpp:333-364) as a weighted
// FP64 tensor-core contraction
//     num(i,j) = sum_s w_s * sum_g p_i(s,g) * (score . p_j(s))_g          (K = 3 * n_sites)
// on DMMA.8x8x4 (mma.sync.m8n8k4.f64; the only FP64 tensor instruction on sm_100a -- tcgen05 has no kind::f64).
//
// Structure (one persistent CTA per SM):
//   warp 8        producer: one elected lane stages (A tile, B tile[, 8 weights]) of one 8-site chunk per pipeline
//                 step with cp.async.bulk (TMA bulk copy, SASS UBLKCP) completing on an mbarrier; 4 stages x 48 KiB
//                 (three planes, K4 = 6 k4-groups per chunk) or 4 stages x 32 KiB (pdel two-plane mode, K4 = 4; a
//                 6-stage ring measured the same at C3 on a B200).
//   warps 0..7    consumers, 2 (M) x 4 (N): each owns a 64 x 32 sub-tile = 8 x 4 DMMA accumulators (128 registers);
//                 fragments come straight from the packed layout with conflict-free 256-byte LDS.64.
//                 Diagonal tiles (upper triangle only) and edge tiles (real columns only) have their own warp layouts.
// Work units are (K-split q, upper-triangle tile t), ordered split-major so that the CTAs resident at any moment
// sweep the same site range of neighbouring tiles (operand tiles are shared through L2); CTA c takes units
// c, c+grid, ...  Each unit writes its 128 x 128 partial in fragment order to a workspace slot; K4 (epilogue.cu)
// reduces the splits in a fixed order (deterministic) and applies the normalisation + evolutionary model.
// Bootstrap replicates (ngsDist.cpp:235-238,416-437) run as block-multiplicity weights: the chunk list skips chunks whose
// 8 weights are all zero and B fragments are scaled in registers (exact: weights are small integers).
#include "ngsd_internal.h"

namespace {

constexpr int kConsumerWarps = 8;
constexpr int kThreads = (kConsumerWarps + 1) * 32;

// Pipeline geometry for K4 k4-groups per chunk (6: three planes or the 12-site two-plane layout; 4: pdel two-plane mode)
template <int K4>
struct Ring {
  static constexpr int kTileDoubles = K4 * NGSD_K4_DOUBLES;
  static constexpr int kTileBytes = kTileDoubles * 8;
  static constexpr int kStages = 4;
  static constexpr int kStageBytes = 2 * kTileBytes + 128;   // A + B + up to 12 per-site weights
  static constexpr size_t kSmemBytes = (size_t) kStages * kStageBytes + 2 * kStages * sizeof(uint64_t) + kStages * 2 * sizeof(uint32_t) + 128;
};

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t) __cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {}
}
// TMA bulk copy global -> shared, completion counted in bytes on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void dmma884(double &c0, double &c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

struct DistArgs {
  const double *Apack, *Bpack;
  const double *weights;        // [NC*8] or nullptr
  const uint32_t *chunk_ids;    // [n_chunks] or nullptr (identity)
  const ngsd_tile *tiles;
  const uint32_t *split_begin;  // [n_splits + 1] chunk-list boundaries of the K splits
  const double *split_scale;    // [n_splits] weight common to all chunks of the split, or nullptr (= 1)
  uint32_t *sched;              // dynamic scheduler: next unit to hand out (zeroed before launch)
  double *partials;             // [n_units][16384]
  uint64_t NC;                  // chunk stride of the packed planes
  uint32_t n_tiles, n_units;
  uint32_t edge_tj;             // last row block when n_ind % 128 != 0 (its off-diagonal tiles are edge tiles), else ~0
  uint32_t edge_c8;             // 8-column blocks of the last row block that hold individuals (1..15)
};

enum : uint32_t { kFirst = 1u, kLast = 2u, kDiag = 4u, kExit = 8u, kEdge = 16u };

// One K4 step of a full (off-diagonal) tile for one consumer warp: 64 x 32 sub-tile, 12 LDS.64 + 32 DMMA.
__device__ __forceinline__ void step_full(double (&acc)[64], const double *As, const double *Bs, double w) {
  double af[8], bf[4];
#pragma unroll
  for (int mi = 0; mi < 8; mi++) af[mi] = As[mi * 32];
#pragma unroll
  for (int ni = 0; ni < 4; ni++) bf[ni] = Bs[ni * 32] * w;
#pragma unroll
  for (int mi = 0; mi < 8; mi++)
#pragma unroll
    for (int ni = 0; ni < 4; ni++) dmma884(acc[(mi * 4 + ni) * 2], acc[(mi * 4 + ni) * 2 + 1], af[mi], bf[ni]);
}

// One chunk (6 K4 steps) of a DIAGONAL tile: only the upper triangle of the 16 x 16 grid of 8x8 blocks is needed
// (136 of 256).  Warp W owns block-rows W and 15-W (17 blocks, the same for every warp, so the four SMSPs stay
// balanced): acc[0..31] = row W, columns 0..15; acc[32..63] = row 15-W.  Specialised per warp at compile time:
// predicated-off DMMAs still cost issue slots on the FP64 tensor pipe, so each warp runs straight-line code with
// exactly its 17 DMMA + (18 - W) LDS.64 per K4 step.
template <int W, int PLANES, int K4>
__device__ __forceinline__ void chunk_diag(double (&acc)[64], const double *As, const double *Bs, const double (&wv)[3]) {
#pragma unroll
  for (int k4 = 0; k4 < K4; k4++) {
    const double *Ak = As + k4 * 512, *Bk = Bs + k4 * 512;
    const double w = wv[PLANES == 3 ? (k4 & 1) : (k4 % 3)];
    const double a0 = Ak[W * 32], a1 = Ak[(15 - W) * 32];
    double bf[16];
#pragma unroll
    for (int c = W; c < 16; c++) bf[c] = Bk[c * 32] * w;
#pragma unroll
    for (int c = W; c < 16; c++) dmma884(acc[c * 2], acc[c * 2 + 1], a0, bf[c]);
#pragma unroll
    for (int c = 15 - W; c < 16; c++) dmma884(acc[32 + c * 2], acc[32 + c * 2 + 1], a1, bf[c]);
  }
}

template <int W>
__device__ __forceinline__ void store_diag(const double (&acc)[64], double2 *dst) {
#pragma unroll
  for (int c = W; c < 16; c++) dst[c * 32] = make_double2(acc[c * 2], acc[c * 2 + 1]);
#pragma unroll
  for (int c = 15 - W; c < 16; c++) dst[(16 + c) * 32] = make_double2(acc[32 + c * 2], acc[32 + c * 2 + 1]);
}

// One chunk of an EDGE tile: off-diagonal, with the last row block as its column block, whose real individuals fill only
// C8 of the 16 8-column blocks.  Warp W owns block-rows W and W + 8 x the C8 real block-columns: 2 * C8 DMMA + (2 + C8)
// LDS.64 per K4 step on every warp (the full-tile layout would leave the padding columns on SMSPs 2 and 3 and keep them
// the busiest).  acc[0 .. 2*C8) = row W, acc[2*C8 .. 4*C8) = row W + 8.  Each 8x8 block takes the same fragments, the
// same weight product and the same DMMA sequence as in step_full, so its sums are bit-identical.
template <int C8, int PLANES, int K4>
__device__ __forceinline__ void chunk_edge(double (&acc)[64], const double *As, const double *Bs, const double (&wv)[3]) {
#pragma unroll
  for (int k4 = 0; k4 < K4; k4++) {
    const double *Ak = As + k4 * 512, *Bk = Bs + k4 * 512;
    const double w = wv[PLANES == 3 ? (k4 & 1) : (k4 % 3)];
    const double a0 = Ak[0], a1 = Ak[8 * 32];
    double bf[C8];
#pragma unroll
    for (int c = 0; c < C8; c++) bf[c] = Bk[c * 32] * w;
#pragma unroll
    for (int c = 0; c < C8; c++) dmma884(acc[c * 2], acc[c * 2 + 1], a0, bf[c]);
#pragma unroll
    for (int c = 0; c < C8; c++) dmma884(acc[(C8 + c) * 2], acc[(C8 + c) * 2 + 1], a1, bf[c]);
  }
}

// Edge-tile partial in the full-tile fragment order (block (R, C) -> warp (R/8)*4 + C/4, frag (R%8)*4 + C%4), so that
// k_epilogue decodes it like a full tile; the padding blocks are not written (the epilogue reads no column >= n_ind).
template <int C8>
__device__ __forceinline__ void store_edge(const double (&acc)[64], double2 *tile, int W) {
#pragma unroll
  for (int h = 0; h < 2; h++)
#pragma unroll
    for (int c = 0; c < C8; c++)
      tile[((h * 4 + c / 4) * 32 + W * 4 + (c & 3)) * 32] = make_double2(acc[(h * C8 + c) * 2], acc[(h * C8 + c) * 2 + 1]);
}

// PLANES = 3: chunk of 8 sites, k4-group = g*2 + h;  PLANES = 2: chunk of 12 sites, k4-group = g*3 + h (ngsd_internal.h).
// The only place the two differ inside the kernel is which per-site weight a k4-group takes.  K4 = k4-groups per chunk:
// 6, or 4 in pdel two-plane mode (8-site chunks, PLANES = 3 weight indexing, g = 0..1).
template <bool WEIGHTED, int PLANES, int K4>
__global__ void __launch_bounds__(kThreads, 1) k_dist_dmma(DistArgs a) {
  constexpr int kStages = Ring<K4>::kStages, kStageBytes = Ring<K4>::kStageBytes, kTileBytes = Ring<K4>::kTileBytes;
  constexpr int kTileDoubles = Ring<K4>::kTileDoubles;
  extern __shared__ __align__(128) unsigned char smem[];
  uint64_t *full = reinterpret_cast<uint64_t *>(smem + (size_t) kStages * kStageBytes);
  uint64_t *empty = full + kStages;
  uint32_t *meta = reinterpret_cast<uint32_t *>(empty + kStages);   // [kStages][2] = {unit, flags}
  auto stageA = [&](int s) { return reinterpret_cast<double *>(smem + (size_t) s * kStageBytes); };
  auto stageB = [&](int s) { return reinterpret_cast<double *>(smem + (size_t) s * kStageBytes + kTileBytes); };
  auto stageW = [&](int s) { return reinterpret_cast<double *>(smem + (size_t) s * kStageBytes + 2 * kTileBytes); };

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; s++) { mbar_init(&full[s], 1); mbar_init(&empty[s], kConsumerWarps); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  int stage = 0;
  uint32_t phase = 0;

  if (warp == kConsumerWarps) {
    // ===== producer: one lane pulls units from the global counter and streams their chunks =====
    if (lane == 0) {
      for (;;) {
        const uint32_t u = atomicAdd(a.sched, 1u);
        if (u >= a.n_units) break;
        const uint32_t q = u / a.n_tiles, t = u - q * a.n_tiles;
        const ngsd_tile tl = a.tiles[t];
        const uint32_t c0 = a.split_begin[q], c1 = a.split_begin[q + 1];
        const double *Ab = a.Apack + (uint64_t) tl.ti * a.NC * kTileDoubles;
        const double *Bb = a.Bpack + (uint64_t) tl.tj * a.NC * kTileDoubles;
        const uint32_t fl = tl.ti == tl.tj ? kDiag : (tl.tj == a.edge_tj ? kEdge : 0u);
        for (uint32_t c = c0; c < c1; c++) {
          const uint64_t chunk = a.chunk_ids ? a.chunk_ids[c] : c;
          mbar_wait(&empty[stage], phase ^ 1);
          meta[stage * 2] = u;
          meta[stage * 2 + 1] = fl | (c == c0 ? kFirst : 0u) | (c + 1 == c1 ? kLast : 0u);
          constexpr int kSites = PLANES == 3 ? NGSD_SC : NGSD_SC2;
          mbar_expect_tx(&full[stage], 2 * kTileBytes + (WEIGHTED ? kSites * 8 : 0));
          bulk_g2s(stageA(stage), Ab + chunk * kTileDoubles, kTileBytes, &full[stage]);
          bulk_g2s(stageB(stage), Bb + chunk * kTileDoubles, kTileBytes, &full[stage]);
          if (WEIGHTED) bulk_g2s(stageW(stage), a.weights + chunk * kSites, kSites * 8, &full[stage]);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
      mbar_wait(&empty[stage], phase ^ 1);
      meta[stage * 2 + 1] = kExit;
      mbar_arrive(&full[stage]);
    }
    return;
  }

  // ===== consumers =====
  const int wm = warp >> 2, wn = warp & 3;            // full tiles: 2 x 4 warps, warp tile 64 (rows) x 32 (cols)
  double acc[64];
  for (;;) {
    mbar_wait(&full[stage], phase);
    const uint32_t u = meta[stage * 2], fl = meta[stage * 2 + 1];
    if (fl & kExit) break;
    if (fl & kFirst) {
#pragma unroll
      for (int k = 0; k < 64; k++) acc[k] = 0.0;
    }
    double wv[3] = {1.0, 1.0, 1.0};              // weight of this lane's site in each 4-site group of the chunk
    if (WEIGHTED) {
      const double *Ws = stageW(stage);
      wv[0] = Ws[lane & 3];
      wv[1] = Ws[4 + (lane & 3)];
      if (PLANES == 2) wv[2] = Ws[8 + (lane & 3)];
    }
    const double w0 = wv[0], w1 = wv[1];
    (void) w0; (void) w1;
    if (fl & kDiag) {
      const double *As = stageA(stage) + lane, *Bs = stageB(stage) + lane;
      switch (warp) {       // warp-uniform: no divergence
        case 0: chunk_diag<0, PLANES, K4>(acc, As, Bs, wv); break;
        case 1: chunk_diag<1, PLANES, K4>(acc, As, Bs, wv); break;
        case 2: chunk_diag<2, PLANES, K4>(acc, As, Bs, wv); break;
        case 3: chunk_diag<3, PLANES, K4>(acc, As, Bs, wv); break;
        case 4: chunk_diag<4, PLANES, K4>(acc, As, Bs, wv); break;
        case 5: chunk_diag<5, PLANES, K4>(acc, As, Bs, wv); break;
        case 6: chunk_diag<6, PLANES, K4>(acc, As, Bs, wv); break;
        default: chunk_diag<7, PLANES, K4>(acc, As, Bs, wv); break;
      }
    } else if (fl & kEdge) {
      const double *As = stageA(stage) + warp * 32 + lane, *Bs = stageB(stage) + lane;
      switch (a.edge_c8) {  // kernel-uniform
#define NGSD_EDGE_CASE(C) case C: chunk_edge<C, PLANES, K4>(acc, As, Bs, wv); break;
        NGSD_EDGE_CASE(1) NGSD_EDGE_CASE(2) NGSD_EDGE_CASE(3) NGSD_EDGE_CASE(4) NGSD_EDGE_CASE(5)
        NGSD_EDGE_CASE(6) NGSD_EDGE_CASE(7) NGSD_EDGE_CASE(8) NGSD_EDGE_CASE(9) NGSD_EDGE_CASE(10)
        NGSD_EDGE_CASE(11) NGSD_EDGE_CASE(12) NGSD_EDGE_CASE(13) NGSD_EDGE_CASE(14) default: chunk_edge<15, PLANES, K4>(acc, As, Bs, wv); break;
#undef NGSD_EDGE_CASE
      }
    } else {
      const double *As = stageA(stage) + (wm * 8) * 32 + lane, *Bs = stageB(stage) + (wn * 4) * 32 + lane;
#pragma unroll
      for (int k4 = 0; k4 < K4; k4++) step_full(acc, As + k4 * 512, Bs + k4 * 512, wv[PLANES == 3 ? (k4 & 1) : (k4 % 3)]);
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty[stage]);
    if (++stage == kStages) { stage = 0; phase ^= 1; }
    if (fl & kLast) {
      // partial tile in fragment order: [warp][32 accumulator pairs][lane] double2 (decoded in epilogue.cu)
      double2 *tile = reinterpret_cast<double2 *>(a.partials + (uint64_t) u * NGSD_TILE_ELEMS) + lane;
      double2 *dst = tile + (warp * 32) * 32;
      if (a.split_scale) {      // bootstrap multiplicity shared by every chunk of this split (block_size % 8 == 0)
        const double sc = a.split_scale[u / a.n_tiles];
        if (sc != 1.0) {
#pragma unroll
          for (int k = 0; k < 64; k++) acc[k] *= sc;
        }
      }
      if (fl & kDiag) {
        switch (warp) {
          case 0: store_diag<0>(acc, dst); break;
          case 1: store_diag<1>(acc, dst); break;
          case 2: store_diag<2>(acc, dst); break;
          case 3: store_diag<3>(acc, dst); break;
          case 4: store_diag<4>(acc, dst); break;
          case 5: store_diag<5>(acc, dst); break;
          case 6: store_diag<6>(acc, dst); break;
          default: store_diag<7>(acc, dst); break;
        }
      } else if (fl & kEdge) {
        switch (a.edge_c8) {
#define NGSD_EDGE_CASE(C) case C: store_edge<C>(acc, tile, warp); break;
          NGSD_EDGE_CASE(1) NGSD_EDGE_CASE(2) NGSD_EDGE_CASE(3) NGSD_EDGE_CASE(4) NGSD_EDGE_CASE(5)
          NGSD_EDGE_CASE(6) NGSD_EDGE_CASE(7) NGSD_EDGE_CASE(8) NGSD_EDGE_CASE(9) NGSD_EDGE_CASE(10)
          NGSD_EDGE_CASE(11) NGSD_EDGE_CASE(12) NGSD_EDGE_CASE(13) NGSD_EDGE_CASE(14) default: store_edge<15>(acc, tile, warp); break;
#undef NGSD_EDGE_CASE
        }
      } else {
#pragma unroll
        for (int f = 0; f < 32; f++) dst[f * 32] = make_double2(acc[f * 2], acc[f * 2 + 1]);
      }
    }
  }
}

// register-only DMMA loop: the FP64-tensor issue-rate ceiling used as roofline denominator
__global__ void k_dmma_peak(double *out, int iters) {
  double c[8][2];
#pragma unroll
  for (int i = 0; i < 8; i++) c[i][0] = c[i][1] = 0;
  double x = 1.0 + threadIdx.x, y = 2.0 - threadIdx.x;
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int i = 0; i < 8; i++) dmma884(c[i][0], c[i][1], x, y);
  }
  double s = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) s += c[i][0] + c[i][1];
  if (s == 12345.678) out[0] = s;
}

}  // namespace

size_t ngsd_dist_smem_bytes() { return std::max(Ring<NGSD_K4_3>::kSmemBytes, Ring<NGSD_K4_PD2>::kSmemBytes); }

cudaError_t ngsd_launch_dist_dmma(ngsd_ctx *ctx, const ngsd_dist_plan &p) {
  static bool attr_set[64] = {};
  if (!attr_set[ctx->device & 63]) {
    const void *fns[5] = {(const void *) k_dist_dmma<false, 3, NGSD_K4_3>, (const void *) k_dist_dmma<true, 3, NGSD_K4_3>,
                          (const void *) k_dist_dmma<true, 2, NGSD_K4_3>, (const void *) k_dist_dmma<false, 3, NGSD_K4_PD2>,
                          (const void *) k_dist_dmma<true, 3, NGSD_K4_PD2>};
    const size_t smem[5] = {Ring<NGSD_K4_3>::kSmemBytes, Ring<NGSD_K4_3>::kSmemBytes, Ring<NGSD_K4_3>::kSmemBytes,
                            Ring<NGSD_K4_PD2>::kSmemBytes, Ring<NGSD_K4_PD2>::kSmemBytes};
    for (int k = 0; k < 5; k++) {
      const void *f = fns[k];
      cudaError_t e = cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem[k]);
      if (e != cudaSuccess) return e;
      e = cudaFuncSetAttribute(f, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
      if (e != cudaSuccess) return e;
    }
    attr_set[ctx->device & 63] = true;
  }
  DistArgs a;
  a.Apack = ctx->Apack;
  a.Bpack = ctx->Bpack;
  a.weights = (p.weighted && !p.uniform_scale) ? ctx->d_weights : nullptr;
  a.chunk_ids = p.weighted ? ctx->d_chunk_ids : nullptr;
  a.tiles = ctx->d_tiles;
  a.split_begin = ctx->d_split_begin;
  a.split_scale = p.uniform_scale ? ctx->d_split_scale : nullptr;
  a.sched = ctx->d_sched;
  a.partials = ctx->cur_partials;
  a.NC = ctx->NC;
  a.n_tiles = ctx->n_tiles;
  a.n_units = p.n_units;
  const uint32_t c8 = ngsd_edge_c8(ctx->n_ind);
  a.edge_tj = c8 ? (uint32_t) ctx->RB - 1 : 0xFFFFFFFFu;
  a.edge_c8 = c8;
  cudaError_t e = cudaMemsetAsync(ctx->d_sched, 0, sizeof(uint32_t), ctx->stream);
  if (e != cudaSuccess) return e;
  constexpr size_t smem3 = Ring<NGSD_K4_3>::kSmemBytes, smem2 = Ring<NGSD_K4_PD2>::kSmemBytes;
  const bool per_site = p.weighted && !p.uniform_scale;
  if (ctx->pdel2) {
    if (per_site)
      k_dist_dmma<true, 3, NGSD_K4_PD2><<<p.grid, kThreads, smem2, ctx->stream>>>(a);
    else
      k_dist_dmma<false, 3, NGSD_K4_PD2><<<p.grid, kThreads, smem2, ctx->stream>>>(a);
  } else if (per_site) {
    if (ctx->planes == 3)
      k_dist_dmma<true, 3, NGSD_K4_3><<<p.grid, kThreads, smem3, ctx->stream>>>(a);
    else
      k_dist_dmma<true, 2, NGSD_K4_3><<<p.grid, kThreads, smem3, ctx->stream>>>(a);
  } else {
    k_dist_dmma<false, 3, NGSD_K4_3><<<p.grid, kThreads, smem3, ctx->stream>>>(a);   // unweighted: plane count is irrelevant
  }
  return cudaGetLastError();
}

extern "C" int ngsd_probe_fp64_tflops(int device, double *dmma_tflops) {
  if (cudaSetDevice(device) != cudaSuccess) return NGSD_ERR_CUDA;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return NGSD_ERR_CUDA;
  double *d = nullptr;
  if (cudaMalloc(&d, 64) != cudaSuccess) return NGSD_ERR_CUDA;
  const int iters = 8192, warps = 16, nsm = prop.multiProcessorCount;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  float best = 1e30f;
  for (int r = 0; r < 4; r++) {
    cudaEventRecord(e0);
    k_dmma_peak<<<nsm, warps * 32>>>(d, iters);
    cudaEventRecord(e1);
    if (cudaEventSynchronize(e1) != cudaSuccess) { cudaFree(d); return NGSD_ERR_CUDA; }
    float ms;
    cudaEventElapsedTime(&ms, e0, e1);
    if (r > 0 && ms < best) best = ms;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(d);
  *dmma_tflops = (double) nsm * warps * iters * 8 * 512.0 / (best * 1e-3) * 1e-12;
  return NGSD_OK;
}
