// K4 epilogue: deterministic reduction of the K-split partial tiles + the tail of gen_dist (ngsDist.cpp:372-401):
//   cnt <- tot_sites override; d = num / (double) cnt; model 0: d, 1: -log(1-d), 2: -log(1-(d*4/3))*3/4;
// symmetric write of both triangles as gen_dist_slave does (ngsDist.cpp:408-412), 0.0 diagonal (ngsDist.cpp:200).
// k_epilogue reduces the FP64 partials of dist_dmma.cu, k_epilogue_int the exact int32 partials of dist_umma.cu.
#include "ngsd_internal.h"

namespace {

struct EpiArgs {
  const double *partials;     // [n_splits][n_tiles][16384] fragment order (dist_dmma.cu)
  const double *split_w;      // [n_splits] weight of each split (bootstrap block cache) or nullptr
  const ngsd_tile *tiles;
  const uint32_t *cnt;        // [n_pad][n_pad] or nullptr
  const uint32_t *cnt_cache;  // per-block counts [n_splits][n_tiles][4][64][64] (bootstrap block cache) or nullptr
  const double *cvec;         // [n_pad] 2-plane mode: weighted row sums of the B_2 plane, added for column j; or nullptr
  const double *fix;          // [n_ind][n_ind] 2-plane mode: correction for row triples that do not sum to one; or nullptr
  double kappa;               // pdel two-plane mode: num += kappa * cnt (the mask term of ngsd_internal.h); else 0
  double *out, *num;          // [n_ind][n_ind]
  uint64_t *cntout;
  uint64_t n_ind, n_pad, const_cnt, tot_sites;
  uint32_t n_splits, n_tiles;
  int evol_model;
};

// grid (n_tiles, 32); block 256: one thread per double2 slot of the tile (8192 slots), splits summed in a fixed order
__global__ void __launch_bounds__(256) k_epilogue(EpiArgs a) {
  const uint32_t t = blockIdx.x;
  const ngsd_tile tl = a.tiles[t];
  const uint32_t e = blockIdx.y * 256 + threadIdx.x;     // double2 index inside the tile: (warp*32 + frag)*32 + lane
  const int lane = e & 31, frag = (e >> 5) & 31, warp = e >> 10;
  // decode the slot -> (row, first column) inside the tile; layouts written by dist_dmma.cu
  int row, col0;
  if (tl.ti == tl.tj) {     // diagonal tile: warp owns 8x8 block-rows `warp` (frags 0..15) and 15-warp (frags 16..31)
    const int R = (frag < 16) ? warp : 15 - warp, c = frag & 15;
    if (c < R) return;      // below the diagonal: never computed, never stored
    row = R * 8 + (lane >> 2);
    col0 = c * 8 + 2 * (lane & 3);
  } else {                  // full tile: 2 x 4 warps of 64 x 32, frag = mi*4 + ni
    const int wm = warp >> 2, wn = warp & 3, mi = frag >> 2, ni = frag & 3;
    row = wm * 64 + mi * 8 + (lane >> 2);
    col0 = wn * 32 + ni * 8 + 2 * (lane & 3);
  }
  const uint64_t i = (uint64_t) tl.ti * NGSD_TILE + row;
  const uint64_t j0 = (uint64_t) tl.tj * NGSD_TILE + col0;
  if (i >= a.n_ind || j0 >= a.n_ind) return;   // padding rows / columns
  const double2 *src = reinterpret_cast<const double2 *>(a.partials + (uint64_t) t * NGSD_TILE_ELEMS) + e;
  const uint64_t stride = (uint64_t) a.n_tiles * (NGSD_TILE_ELEMS / 2);   // in double2
  double s0 = 0, s1 = 0;
  uint32_t q = 0;
  if (a.split_w) {                                       // per-block partials x block multiplicities, in block order
    for (; q < a.n_splits; q++) {
      const double w = a.split_w[q];
      if (w == 0.0) continue;                            // block not drawn in this replicate: its partial is not even read
      const double2 v = src[(uint64_t) q * stride];
      s0 += w * v.x;
      s1 += w * v.y;
    }
  }
  for (; q + 8 <= a.n_splits; q += 8) {                  // 8 independent loads in flight, adds in split order
    double2 v[8];
#pragma unroll
    for (int k = 0; k < 8; k++) v[k] = src[(uint64_t) (q + k) * stride];
#pragma unroll
    for (int k = 0; k < 8; k++) { s0 += v[k].x; s1 += v[k].y; }
  }
  for (; q < a.n_splits; q++) {
    const double2 v = src[(uint64_t) q * stride];
    s0 += v.x;
    s1 += v.y;
  }
#pragma unroll
  for (int c = 0; c < 2; c++) {
    const uint64_t j = j0 + c;
    if (i >= j || j >= a.n_ind) continue;
    double num = (c ? s1 : s0) + (a.cvec ? a.cvec[j] : 0.0);
    if (a.fix) num += a.fix[i * a.n_ind + j];
    uint64_t cnt = a.cnt ? (uint64_t) a.cnt[i * a.n_pad + j] : a.const_cnt;
    if (a.cnt_cache) {        // sum_b c[b] * cnt_b(i,j): integers, exact
      const int rr = row, cc = col0 + c;
      const uint32_t *pc = a.cnt_cache + ((uint64_t) t * 4 + (rr >> 6) * 2 + (cc >> 6)) * 4096 + (rr & 63) * 64 + (cc & 63);
      const uint64_t cstride = (uint64_t) a.n_tiles * 4 * 4096;
      cnt = 0;
      for (uint32_t q2 = 0; q2 < a.n_splits; q2++) {
        const double w = a.split_w[q2];
        if (w != 0.0) cnt += (uint64_t) w * (uint64_t) pc[(uint64_t) q2 * cstride];
      }
    }
    if (a.kappa != 0.0) num += a.kappa * (double) cnt;   // the weighted shared-site count, before the tot_sites override
    if (a.num) a.num[i * a.n_ind + j] = a.num[j * a.n_ind + i] = num;
    if (a.cntout) a.cntout[i * a.n_ind + j] = a.cntout[j * a.n_ind + i] = cnt;
    if (a.tot_sites > 0) cnt = a.tot_sites;
    double d = num / (double) cnt;
    if (a.evol_model == 1) d = -log(1 - d);
    else if (a.evol_model == 2) d = -log(1 - (d * 4 / 3)) * 3 / 4;
    a.out[i * a.n_ind + j] = a.out[j * a.n_ind + i] = d;
  }
}

struct EpiIntArgs {
  const int32_t *partials;    // [n_splits][n_tiles][pstride] row-major tiles of dist_umma.cu (sum tile, then count tile when in_kernel_cnt)
  const double *split_w;      // [n_splits] integer weight of each split (bootstrap block cache) or nullptr
  uint32_t pstride;
  int in_kernel_cnt;
  const ngsd_tile *tiles;
  double *out, *num;
  uint64_t *cntout;
  uint64_t n_ind, const_cnt, tot_sites;
  uint32_t n_splits, n_tiles;
  int evol_model;
  double scale;               // S
};

// Integer path (dist_umma.cu): grid (n_tiles, 16); block 256: one thread per 4 elements of the tile (rows row0 and
// row0 + 8, columns col0 and col0 + 1); splits summed in int64 (order-free, exact), then num = acc / S
__global__ void __launch_bounds__(256) k_epilogue_int(EpiIntArgs a) {
  const uint32_t t = blockIdx.x;
  const ngsd_tile tl = a.tiles[t];
  const uint32_t e = blockIdx.y * 256 + threadIdx.x;
  const int lane = e & 31, frag = (e >> 5) & 15, warp = e >> 9;
  const int wm = warp >> 2, wn = warp & 3, mi = frag >> 2, ni = frag & 3;
  const int row0 = wm * 64 + mi * 16 + (lane >> 2), col0 = wn * 32 + ni * 8 + 2 * (lane & 3);
  const int32_t *src = a.partials + (uint64_t) t * a.pstride + row0 * NGSD_TILE + col0;
  const uint64_t stride = (uint64_t) a.n_tiles * a.pstride;
  long long s[4] = {0, 0, 0, 0}, c[4] = {0, 0, 0, 0};
  for (uint32_t q = 0; q < a.n_splits; q++) {
    long long m = 1;
    if (a.split_w) {                     // per-block partials x block multiplicities: integers, exact
      m = (long long) a.split_w[q];
      if (m == 0) continue;
    }
    const int32_t *p = src + (uint64_t) q * stride;
    const int2 lo = *reinterpret_cast<const int2 *>(p), hi = *reinterpret_cast<const int2 *>(p + 8 * NGSD_TILE);
    s[0] += m * lo.x; s[1] += m * lo.y; s[2] += m * hi.x; s[3] += m * hi.y;
    if (a.in_kernel_cnt) {
      const int2 clo = *reinterpret_cast<const int2 *>(p + NGSD_TILE_ELEMS), chi = *reinterpret_cast<const int2 *>(p + NGSD_TILE_ELEMS + 8 * NGSD_TILE);
      c[0] += m * clo.x; c[1] += m * clo.y; c[2] += m * chi.x; c[3] += m * chi.y;
    }
  }
#pragma unroll
  for (int k = 0; k < 4; k++) {
    const uint64_t i = (uint64_t) tl.ti * NGSD_TILE + row0 + (k >> 1) * 8, j = (uint64_t) tl.tj * NGSD_TILE + col0 + (k & 1);
    if (i >= j || j >= a.n_ind) continue;
    const double num = (double) s[k] / a.scale;
    uint64_t cnt = a.in_kernel_cnt ? (uint64_t) c[k] : a.const_cnt;
    if (a.num) a.num[i * a.n_ind + j] = a.num[j * a.n_ind + i] = num;
    if (a.cntout) a.cntout[i * a.n_ind + j] = a.cntout[j * a.n_ind + i] = cnt;
    if (a.tot_sites > 0) cnt = a.tot_sites;
    double d = num / (double) cnt;
    if (a.evol_model == 1) d = -log(1 - d);
    else if (a.evol_model == 2) d = -log(1 - (d * 4 / 3)) * 3 / 4;
    a.out[i * a.n_ind + j] = a.out[j * a.n_ind + i] = d;
  }
}

__global__ void k_zero_diag(double *out, double *num, uint64_t *cnt, uint64_t n) {
  const uint64_t i = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  out[i * n + i] = 0.0;
  if (num) num[i * n + i] = 0.0;
  if (cnt) cnt[i * n + i] = 0;
}

// ngsd_finish: the tail of gen_dist on already reduced raw sums (site-sharded runs): out = model(num / cnt)
__global__ void k_finish(const double *__restrict__ num, uint64_t *__restrict__ cnt, double *__restrict__ out, uint64_t n,
                         uint64_t tot_sites, int evol_model, uint64_t const_cnt) {
  const uint64_t idx = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n * n) return;
  const uint64_t i = idx / n, j = idx % n;
  if (i == j) { out[idx] = 0.0; return; }
  if (const_cnt) cnt[idx] = const_cnt;      // no --pairwise_del: every pair counted every site (ngsDist.cpp:362)
  uint64_t c = cnt[idx];
  if (tot_sites > 0) c = tot_sites;
  double d = num[idx] / (double) c;
  if (evol_model == 1) d = -log(1 - d);
  else if (evol_model == 2) d = -log(1 - (d * 4 / 3)) * 3 / 4;
  out[idx] = d;
}

// 2-plane mode: c_j = sum_s w_s * C[j][s] (C = B_2 plane, stored [64-site word][n_pad][64]); one block per individual,
// fixed-order tree reduction
__global__ void __launch_bounds__(256) k_cvec(const double *__restrict__ C, uint64_t n_pad, const double *__restrict__ w, uint64_t n_eff,
                                             double *__restrict__ cvec) {
  __shared__ double red[256];
  const double *row = C + (uint64_t) blockIdx.x * 64;
  double s = 0;
  for (uint64_t k = threadIdx.x; k < n_eff; k += 256) {
    const double v = row[(k >> 6) * n_pad * 64 + (k & 63)];
    s += w ? w[k] * v : v;
  }
  red[threadIdx.x] = s;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int) threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) cvec[blockIdx.x] = red[0];
}

// 2-plane mode, rows holding a triple with p0 + p1 + p2 = 1 + delta: the contraction used p2 = 1 - p0 - p1, so
// delta * w_s * B_2(j, s) is missing from num(i, j) for every j > i.  One block per such row, entries in (site) order.
__global__ void __launch_bounds__(256) k_deficit_fix(const uint32_t *__restrict__ row_ptr, const uint32_t *__restrict__ row_ind,
                                                    const uint64_t *__restrict__ site, const double *__restrict__ delta,
                                                    const double *__restrict__ w, uint64_t n_eff, const double *__restrict__ C, uint64_t n_pad,
                                                    uint64_t n_ind, double *__restrict__ fix) {
  const uint64_t i = row_ind[blockIdx.x];
  const uint32_t e0 = row_ptr[blockIdx.x], e1 = row_ptr[blockIdx.x + 1];
  for (uint64_t j = i + 1 + threadIdx.x; j < n_ind; j += blockDim.x) {
    double acc = 0;
    for (uint32_t e = e0; e < e1; e++) {
      const uint64_t s = site[e];
      if (s >= n_eff) continue;
      const double ws = w ? w[s] : 1.0;
      acc += delta[e] * ws * C[((s >> 6) * n_pad + j) * 64 + (s & 63)];
    }
    fix[i * n_ind + j] = acc;
  }
}

// Entries (i, j) and (j, i) whose 128 x 128 tile a tile shard does not own -> 0, the diagonal of such tiles included.
__global__ void k_clear_unowned(const uint32_t *__restrict__ tile_index, uint64_t RB, double *out, double *num, uint64_t *cnt, uint64_t n) {
  const uint64_t idx = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n * n) return;
  const uint64_t i = idx / n, j = idx - i * n, lo = (i < j ? i : j) / NGSD_TILE, hi = (i < j ? j : i) / NGSD_TILE;
  if (tile_index[lo * RB + hi] != 0xFFFFFFFFu) return;
  out[idx] = 0.0;
  num[idx] = 0.0;
  cnt[idx] = 0;
}

}  // namespace

// Before an epilogue: zero the diagonal, and with a tile shard every entry, since the tiles of other ranks must read as
// 0 (ngsd_set_tile_shard).
cudaError_t ngsd_clear_outputs(ngsd_ctx *ctx) {
  if (ctx->shard_world > 1) {
    const uint64_t n2 = ctx->n_ind * ctx->n_ind;
    cudaError_t e = cudaMemsetAsync(ctx->d_out, 0, n2 * sizeof(double), ctx->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(ctx->d_num, 0, n2 * sizeof(double), ctx->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(ctx->d_cntout, 0, n2 * sizeof(uint64_t), ctx->stream);
    if (e != cudaSuccess) return e;
  }
  k_zero_diag<<<(unsigned) ((ctx->n_ind + 255) / 256), 256, 0, ctx->stream>>>(ctx->d_out, ctx->d_num, ctx->d_cntout, ctx->n_ind);
  return cudaGetLastError();
}

// After a result that was written for every pair (the early-outs of ngsd_distances): with a tile shard, keep only the
// tiles this context owns, so that the sum over the ranks is the whole-matrix result.
cudaError_t ngsd_clear_unowned(ngsd_ctx *ctx) {
  if (ctx->shard_world <= 1) return cudaSuccess;
  const uint64_t n2 = ctx->n_ind * ctx->n_ind;
  k_clear_unowned<<<(unsigned) ((n2 + 255) / 256), 256, 0, ctx->stream>>>(ctx->d_tile_index, ctx->RB, ctx->d_out, ctx->d_num, ctx->d_cntout, ctx->n_ind);
  return cudaGetLastError();
}

cudaError_t ngsd_launch_deficit_fix(ngsd_ctx *ctx, bool weighted, uint64_t n_eff) {
  cudaError_t e = cudaMemsetAsync(ctx->d_fix, 0, ctx->n_ind * ctx->n_ind * sizeof(double), ctx->stream);
  if (e != cudaSuccess) return e;
  k_deficit_fix<<<ctx->def_rows, 256, 0, ctx->stream>>>(ctx->d_def_rowptr, ctx->d_def_rowind, ctx->d_def_site, ctx->d_def_delta,
                                                       weighted ? ctx->d_weights : nullptr, n_eff, ctx->Cplane, ctx->n_pad, ctx->n_ind, ctx->d_fix);
  return cudaGetLastError();
}

cudaError_t ngsd_launch_cvec(ngsd_ctx *ctx, bool weighted, uint64_t n_eff) {
  k_cvec<<<(unsigned) ctx->n_pad, 256, 0, ctx->stream>>>(ctx->Cplane, ctx->ldc, weighted ? ctx->d_weights : nullptr, n_eff, ctx->d_cvec);
  return cudaGetLastError();
}

cudaError_t ngsd_launch_finish(ngsd_ctx *ctx, uint64_t const_cnt) {
  const uint64_t n2 = ctx->n_ind * ctx->n_ind;
  k_finish<<<(unsigned) ((n2 + 255) / 256), 256, 0, ctx->stream>>>(ctx->d_num, ctx->d_cntout, ctx->d_out, ctx->n_ind, ctx->cfg.tot_sites,
                                                                 ctx->cfg.evol_model, const_cnt);
  return cudaGetLastError();
}

cudaError_t ngsd_launch_epilogue(ngsd_ctx *ctx, const ngsd_epilogue_args &e) {
  EpiArgs a;
  a.partials = ctx->cur_partials;
  a.split_w = ctx->cur_split_w;
  a.tiles = ctx->d_tiles;
  a.cnt = (e.use_cnt && !ctx->cur_cnt_cache) ? ctx->d_cnt : nullptr;
  a.cnt_cache = e.use_cnt ? ctx->cur_cnt_cache : nullptr;
  a.cvec = ctx->planes == 2 ? ctx->d_cvec : nullptr;
  a.fix = (ctx->planes == 2 && ctx->def_rows) ? ctx->d_fix : nullptr;
  a.kappa = ctx->pdel2 ? ctx->pd_kappa : 0.0;         // pdel2 implies --pairwise_del: cnt is the real count
  a.out = ctx->d_out;
  a.num = ctx->d_num;
  a.cntout = ctx->d_cntout;
  a.n_ind = ctx->n_ind;
  a.n_pad = ctx->n_pad;
  a.const_cnt = e.const_cnt;
  a.tot_sites = ctx->cfg.tot_sites;
  a.n_splits = e.n_splits;
  a.n_tiles = ctx->n_tiles;
  a.evol_model = ctx->cfg.evol_model;
  cudaError_t err = ngsd_clear_outputs(ctx);
  if (err != cudaSuccess) return err;
  k_epilogue<<<dim3(ctx->n_tiles, 32), 256, 0, ctx->stream>>>(a);
  return cudaGetLastError();
}

cudaError_t ngsd_launch_epilogue_int(ngsd_ctx *ctx, uint32_t n_splits, uint64_t const_cnt, bool in_kernel_cnt) {
  EpiIntArgs a;
  a.partials = reinterpret_cast<const int32_t *>(ctx->cur_partials);
  a.split_w = ctx->cur_split_w;
  a.pstride = in_kernel_cnt ? 2 * NGSD_TILE_ELEMS : NGSD_TILE_ELEMS;
  a.in_kernel_cnt = in_kernel_cnt ? 1 : 0;
  a.tiles = ctx->d_tiles;
  a.out = ctx->d_out;
  a.num = ctx->d_num;
  a.cntout = ctx->d_cntout;
  a.n_ind = ctx->n_ind;
  a.const_cnt = const_cnt;
  a.tot_sites = ctx->cfg.tot_sites;
  a.n_splits = n_splits;
  a.n_tiles = ctx->n_tiles;
  a.evol_model = ctx->cfg.evol_model;
  a.scale = ctx->int_scale;
  cudaError_t err = ngsd_clear_outputs(ctx);
  if (err != cudaSuccess) return err;
  k_epilogue_int<<<dim3(ctx->n_tiles, 16), 256, 0, ctx->stream>>>(a);
  return cudaGetLastError();
}
