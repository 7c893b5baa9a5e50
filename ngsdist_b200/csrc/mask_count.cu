// K3 mask_count: the per-block shared-site counts of the bootstrap block cache under --pairwise_del, bit-exact.
//   cnt_b(i,j) = sum_{s in block b} m_i(s) * m_j(s)        m = !miss_data (gen_func.cpp:862-868; skip at ngsDist.cpp:335-338,362)
// as an integer AND+POPC "mask GEMM" over 64-site words (1-bit MMA is emulated on sm_100a, SURVEY App. D, so the
// CUDA-core LOP3+POPC path is the native one).  The host lists the sites of every block as (word index, mask word)
// entries -- a block need not start or end on a word -- and split y of the grid counts block y.  The counts are kept
// next to the per-block partial sums, and every replicate takes sum_b c[b] * cnt_b (epilogue.cu, dist_em.cu).  The
// counts of a matrix without the cache come from the int8 tensor cores instead (dist_umma.cu, ngsd_launch_count_umma).
#include "ngsd_internal.h"

namespace {

constexpr int kEB = 8;   // entries per shared-memory batch

struct CountArgs {
  const uint64_t *mask;       // [RB][NW][128]
  const uint32_t *ent_word;
  const uint64_t *ent_mask;
  const ngsd_tile *tiles;
  uint64_t NW;
  // split y = source block y, entries [ent_begin[y], ent_begin[y+1]); the per-block counts are stored (no atomics) to
  // cache[((y * n_tiles + tile) * 4 + quadrant) * 4096 + row * 64 + col]
  const uint32_t *ent_begin;
  uint32_t *cache;
  uint32_t n_tiles;
};

// grid (4 * n_tiles, n_blocks): a CTA owns the 64 x 64 quadrant `blockIdx.x & 3` of tile `blockIdx.x >> 2`.
// block 128 = 8 x 16 threads, each 8 x 4 pairs (rows r*8+ty, cols c*16+tx).  Sized (4 warps x 64 registers, 8 KiB
// shared memory) so that a CTA fits on an SM NEXT TO the persistent k_dist_dmma CTA (9 warps x 168 registers): the
// counts run on the XU/ALU pipes in the shadow of the FP64 tensor contraction (api.cu launches K3 on a second stream
// right after K2).
__global__ void __launch_bounds__(128, 8) k_mask_count(CountArgs a) {
  __shared__ uint64_t sa[kEB][64];
  __shared__ uint64_t sb[kEB][64];
  const ngsd_tile tl = a.tiles[blockIdx.x >> 2];
  const int qr = (blockIdx.x >> 1) & 1, qc = blockIdx.x & 1;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const uint64_t e0 = a.ent_begin[blockIdx.y], e1 = a.ent_begin[blockIdx.y + 1];
  const uint64_t *ma = a.mask + (uint64_t) tl.ti * a.NW * 128 + qr * 64;
  const uint64_t *mb = a.mask + (uint64_t) tl.tj * a.NW * 128 + qc * 64;
  uint32_t acc[8][4];
#pragma unroll
  for (int r = 0; r < 8; r++)
#pragma unroll
    for (int c = 0; c < 4; c++) acc[r][c] = 0;

  for (uint64_t eb = e0; eb < e1; eb += kEB) {
    const int nb = (int) ((e1 - eb) < kEB ? (e1 - eb) : kEB);
    __syncthreads();
#pragma unroll
    for (int k = 0; k < kEB * 64 / 128; k++) {
      const int idx = k * 128 + tid, e = idx >> 6, r = idx & 63;
      uint64_t va = 0, vb = 0;
      if (e < nb) {
        const uint64_t w = a.ent_word[eb + e];
        va = ma[w * 128 + r];
        vb = mb[w * 128 + r] & a.ent_mask[eb + e];
      }
      sa[e][r] = va;
      sb[e][r] = vb;
    }
    __syncthreads();
#pragma unroll 2
    for (int e = 0; e < kEB; e++) {
      uint64_t bv[4];
#pragma unroll
      for (int c = 0; c < 4; c++) bv[c] = sb[e][c * 16 + tx];
#pragma unroll
      for (int r = 0; r < 8; r++) {
        const uint64_t av = sa[e][r * 8 + ty];
#pragma unroll
        for (int c = 0; c < 4; c++) acc[r][c] += __popcll(av & bv[c]);
      }
    }
  }
  uint32_t *dst = a.cache + ((uint64_t) blockIdx.y * a.n_tiles * 4 + blockIdx.x) * 4096;
#pragma unroll
  for (int r = 0; r < 8; r++)
#pragma unroll
    for (int c = 0; c < 4; c++) dst[(r * 8 + ty) * 64 + c * 16 + tx] = acc[r][c];
}

}  // namespace

// one split per source block (gridDim.y <= 65535: checked by the caller)
cudaError_t ngsd_launch_mask_count(ngsd_ctx *ctx, uint32_t n_blocks, cudaStream_t stream) {
  // same shared-memory carveout as k_dist_dmma, otherwise the SMs would have to drain before K3 could be placed on them
  cudaError_t e = cudaFuncSetAttribute(k_mask_count, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  if (e != cudaSuccess) return e;
  CountArgs a;
  a.mask = ctx->mask;
  a.ent_word = ctx->d_ent_word;
  a.ent_mask = ctx->d_ent_mask;
  a.tiles = ctx->d_tiles;
  a.NW = ctx->NW;
  a.ent_begin = ctx->d_ent_begin;
  a.cache = ctx->d_cnt_cache;
  a.n_tiles = ctx->n_tiles;
  k_mask_count<<<dim3(4 * ctx->n_tiles, n_blocks), 128, 0, stream>>>(a);
  return cudaGetLastError();
}
