// Internal declarations shared by the .cu files of libngsdist_b200.so (not part of the ABI).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <string>
#include <thread>
#include <vector>

#include "../../include/ngsdist_b200.h"

// ---------------------------------------------------------------------------------------------
// Geometry of the packed operand planes (DESIGN.md "Data layout in HBM")
//
//   row block  : 128 individuals           (n_pad = ceil(n_ind/128)*128, RB = n_pad/128)
//   site chunk : 8 sites                   (NC = ceil(n_sites/8))
//   one (row block, chunk) tile of an operand = 6 k4-groups x 16 row-groups x 32 doubles = 24 KiB, contiguous
//   (ngsd_ctx::k4 / tile_doubles: 4 k4-groups = 16 KiB in pdel two-plane mode, below):
//       k4-group  kg = g*2 + h     genotype plane g in 0..2, half h in 0..1 (sites chunk*8 + h*4 .. +3)
//       row-group r8               8 consecutive individuals
//       32 doubles in DMMA.8x8x4 fragment order: lane = (ind&7)*4 + (site&3)
//   so a warp reads one A or B fragment of mma.m8n8k4.f64 with a single conflict-free 256-byte LDS.64, and the
//   producer stages a whole pipeline step with ONE cp.async.bulk (TMA) copy per operand.
//   A planes hold p_g (zeroed where --pairwise_del drops the individual-site),
//   B planes hold (score . p)_g, also zeroed there; bootstrap weights scale B fragments in registers.
//
// Two-plane mode (planes == 2; used when nothing masks individual-sites: indep_geno && !pairwise_del).  Posteriors sum to
// one, so  sum_g p_g B_g = B_2 + p_0 (B_0 - B_2) + p_1 (B_1 - B_2):  the contraction needs only K = 2 per site,
//   A planes = (p_0, p_1), B planes = (B_0 - B_2, B_1 - B_2), chunk = 12 sites (k4-group = g*3 + h, h = 0..2: the tile
//   stays 6 k4-groups = 24 KiB), plus the plane C[ind][site] = B_2 whose (weighted) row sums c_j are added in the epilogue.
//   One third fewer DMMAs and 8 bytes less per individual-site; exact for one-hot posteriors, ~1e-16 absolute otherwise.
//
// Pdel two-plane mode (ngsd_ctx::pdel2; indep_geno && pairwise_del, FP64 path, well-conditioned score).  With Z the
// zero-sum directions [[1,0],[0,1],[-1,-1]], V = Z^T S Z and the shifts l, r (api.cu pdel2_coefficients), a present
// triple p (sum one) and a missing one (zero) satisfy  p_i^T S p_j = q_i^T V q_j + kappa * m_i m_j  exactly, so
//   A planes = m (p_0 + l_0, p_1 + l_1), B planes = m V (p_0 + r_0, p_1 + r_1)        (m = presence bit)
// and the epilogue adds kappa * cnt(i, j) (the exact shared-site count of --pairwise_del).  Chunks stay 8 sites with
// k4-group kg = g*2 + h, g = 0..1: the three-plane layout without its third plane, 4 k4-groups = 16 KiB per tile.
// One third fewer DMMAs and 16 bytes less per individual-site; exact for one-hot posteriors and dyadic coefficients
// (default score), ~1e-16 absolute per site otherwise.
// ---------------------------------------------------------------------------------------------
constexpr int NGSD_TILE = 128;                 // individuals per row block / CTA tile edge
constexpr int NGSD_SC = 8;                     // sites per chunk (= one pipeline stage), 3-plane and pdel two-plane modes
constexpr int NGSD_SC2 = 12;                   // sites per chunk, 2-plane mode
constexpr int NGSD_SC_MAX = 12;
constexpr int NGSD_K4_DOUBLES = 16 * 32;       // one k4-group of a tile: 16 row-groups x 32 doubles = 4 KiB
constexpr int NGSD_K4_3 = 6;                   // k4-groups per chunk: 3 planes x 2 halves (also 2 planes x 3 thirds, planes == 2)
constexpr int NGSD_K4_PD2 = 4;                 // k4-groups per chunk in pdel two-plane mode: 2 planes x 2 halves
// Pdel two-plane mode is taken for matrices of at least 2^30 pair-sites (n_ind (n_ind - 1) / 2 * n_sites).  Below that a
// three-plane contraction takes under 0.2 ms on a B200 and launch, count pass and epilogue set the matrix time, so the
// exact three-plane form is kept: per-site products without the shifted cancellation of the two-plane form, exact
// ngsd_get_posteriors, and the same sums as the three-plane contraction for every small data set.
constexpr uint64_t NGSD_PDEL2_MIN_PAIR_SITES = 1ull << 30;
constexpr int NGSD_TILE_ELEMS = NGSD_TILE * NGSD_TILE;           // accumulator elements per tile

struct ngsd_tile { uint16_t ti, tj; };

// 8-column blocks of the last row block that hold individuals (1..15), or 0 when all 16 do (n_ind % 128 == 0 or > 120).
// k_dist_dmma contracts only these columns in the off-diagonal tiles of that block ("edge tiles").
inline uint32_t ngsd_edge_c8(uint64_t n_ind) {
  const uint32_t c8 = (uint32_t) ((n_ind % NGSD_TILE + 7) / 8);
  return c8 < 16 ? c8 : 0u;
}
inline bool ngsd_is_edge_tile(const ngsd_tile &t, uint64_t n_ind, uint64_t RB) {
  return ngsd_edge_c8(n_ind) && t.ti != t.tj && t.tj == RB - 1;
}

// A triple whose outcome hangs on the last ulp of log / exp (a comparison of the reference within 1e-11 of flipping):
// the front-end kernels append it here and the host re-evaluates it with its own libm -- the reference's -- before
// anything is contracted (api.cu resolve_deferred, frontend.cu k_patch).
struct ngsd_deferred {
  uint64_t site;
  uint32_t ind;
  uint32_t flags;      // after the host pass: bit 0 miss_data(), bits 8..9 genotype code (integer path)
  double x[3];         // raw values as pushed; after the host pass the normal-space posterior
};

struct ngsd_ctx {
  ngsd_cfg cfg;
  int device = 0;
  int n_sm = 0;
  cudaStream_t stream = nullptr;      // compute stream (all kernels)
  cudaStream_t copy_stream = nullptr; // H2D staging
  cudaStream_t aux_stream = nullptr;  // K3 mask count, concurrent with K2
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  uint64_t n_ind = 0, n_pad = 0, RB = 0, n_sites = 0, NC = 0, NW = 0;
  int planes = 3, sc = NGSD_SC;                // operand planes per site (3, or 2 with the sum-to-one reduction) / sites per chunk
  // pdel two-plane mode (see above): planes stays 3 (8-site chunks, no C plane), k4 = 4
  bool pdel2 = false;
  double pd_l[2] = {0, 0}, pd_r[2] = {0, 0}, pd_V[4] = {0, 0, 0, 0}, pd_kappa = 0;   // V row-major
  int k4 = NGSD_K4_3;                          // k4-groups per chunk
  uint64_t tile_doubles = NGSD_K4_3 * NGSD_K4_DOUBLES;   // doubles per (row block, chunk) tile of Apack / Bpack
  double *Cplane = nullptr;                    // [NW][n_pad][64] B_2 plane (2-plane mode); ldc = n_pad
  uint64_t ldc = 0;
  double *d_cvec = nullptr;                    // [n_pad] weighted row sums of Cplane for the current matrix
  double *Apack = nullptr, *Bpack = nullptr;   // [RB][NC][tile_doubles]
  uint64_t *mask = nullptr;                    // [RB][NW][128] presence bits (1 = data present)
  // called-genotype integer path (dist_umma.cu): 2-bit codes instead of FP64 planes
  bool int_path = false;
  uint32_t *codes = nullptr;                   // [RB][NW][4][128] 16 sites per word, code 3 = missing
  uint32_t *codes4 = nullptr;                  // [RB][NW][8][128] the same codes as PRMT selector nibbles, 8 sites per word (k_dist_umma)
  uint8_t *d_wsite = nullptr; uint64_t wsite_cap = 0;        // [layers][NW*64] per-site weights
  uint32_t *d_word_layer = nullptr; uint64_t word_cap = 0;   // weight layer of each word-list entry (ids live in d_chunk_ids)
  uint32_t *d_word_ids = nullptr;
  uint32_t int_lut[4] = {0, 0, 0, 0};
  double int_scale = 1.0;
  int int_max_byte = 0;
  int *d_err = nullptr;                        // device error flags (bit0 NaN, bit1 bad genotype code, bit2 blank site seen, bit3 deferred list full)
  ngsd_deferred *d_defer = nullptr; unsigned *d_defer_n = nullptr; unsigned defer_cap = 0;   // knife-edge triples for the host
  uint64_t deferred_total = 0, deferred_changed = 0;   // statistics: triples re-evaluated by the host / whose outcome differed
  uint64_t *d_blank = nullptr;                 // [NW] sites that were empty text lines (read_data.cpp:58-59)
  std::vector<uint64_t> h_blank;               // host copy (empty: none), fetched by ngsd_frontend
  bool any_blank = false;
  // 2-plane mode rests on p0 + p1 + p2 == 1.  The one triple the reference produces that breaks it (all-zero binary
  // likelihoods -> exp(-1.125) three times, SURVEY App. E-11) is kept here with its deficit; ngsd_distances adds
  // deficit * w_s * B_2(j, s) for the pairs whose row individual holds it (epilogue.cu k_deficit_fix).
  struct deficit_entry { uint32_t ind; uint64_t site; double delta; };
  std::vector<deficit_entry> deficit;
  bool deficit_dirty = false;
  uint32_t *d_def_rowptr = nullptr, *d_def_rowind = nullptr; uint64_t *d_def_site = nullptr; double *d_def_delta = nullptr;
  uint32_t def_rows = 0; uint64_t def_cap = 0;
  double *d_fix = nullptr;                     // [n_ind][n_ind] correction of the current matrix (allocated on first use)
  bool deferred_nan = false;                   // a host-evaluated triple produced the NaN that is fatal on the binary path
  // push state
  std::vector<uint8_t> pushed;                 // per 64-site word: pushed?
  uint64_t words_pushed = 0;
  bool frontend_done = false;
  double *stage_dev[2] = {nullptr, nullptr};   // device staging for host pushes
  cudaEvent_t stage_free[2] = {nullptr, nullptr};
  cudaEvent_t stage_ready[2] = {nullptr, nullptr};
  uint64_t stage_sites = 0;
  uint64_t stage_bps = 0;                      // bytes per site the staging slots were sized for (packed genotype pushes)
  int stage_next = 0;
  // distance workspaces (allocated lazily)
  ngsd_tile *d_tiles = nullptr; uint32_t n_tiles = 0;
  uint32_t *d_tile_index = nullptr;            // [RB][RB] position of tile (ti, tj) in d_tiles (0xFFFFFFFF: not owned)
  // the per pair-site EM path (dist_em.cu) works on 64 x 64 tiles: the owned ones (those inside an owned 128 x 128 tile)
  uint32_t *d_em_tiles = nullptr; uint32_t em_n_tiles = 0;   // [em_n_tiles][2] (ti, tj) in upper-triangle order
  uint32_t *d_em_slot = nullptr;               // [n64][n64] position of 64-tile (ti, tj) in d_em_tiles (0xFFFFFFFF: not owned)
  uint32_t *d_pairs = nullptr; uint32_t n_pairs = 0;   // [n_pairs][2] positions of two tiles of one row block (second 0xFFFFFFFF: single); dist_umma.cu
  double *d_partials = nullptr; uint64_t partial_slots = 0;
  // what the contraction launchers write and the epilogues read: d_partials, or the per-block cache below
  double *cur_partials = nullptr;
  const double *cur_split_w = nullptr;         // per-split weights applied by the epilogue (block multiplicities) or nullptr
  // bootstrap block cache: per-block partial sums, computed once; every replicate is then a weighted sum of them
  double *d_cache = nullptr; uint64_t cache_doubles = 0, cache_blocks = 0, cache_bs = 0;
  bool cache_valid = false;
  uint32_t *d_cnt_cache = nullptr; uint64_t cnt_cache_elems = 0;   // per-block shared-site counts [block][tile][4][64][64]
  uint32_t *d_ent_begin = nullptr; uint64_t ent_begin_cap = 0;
  const uint32_t *cur_cnt_cache = nullptr;     // set while the epilogue should take cnt from the block cache
  double *d_weights = nullptr;                 // [NC*8] per-site bootstrap weights
  uint32_t *d_chunk_ids = nullptr;             // [NC] active chunk list
  uint32_t *d_split_begin = nullptr; uint32_t split_cap = 0;
  double *d_split_scale = nullptr;   // K-split boundaries in the chunk list
  uint32_t *d_sched = nullptr;                 // dynamic unit counter of k_dist_dmma
  uint32_t n_diag_tiles = 0;
  uint32_t n_edge_tiles = 0;                   // owned off-diagonal tiles of the last row block when n_ind % 128 != 0 (ngsd_edge_c8)
  uint32_t shard_rank = 0, shard_world = 1;   // output-tile sharding
  uint32_t *d_ent_word = nullptr; uint64_t *d_ent_mask = nullptr; uint64_t ent_cap = 0;   // mask-count entries
  uint32_t *d_cnt = nullptr;                   // [n_pad][n_pad] shared-site counts
  double *d_out = nullptr, *d_num = nullptr; uint64_t *d_cntout = nullptr;   // [n_ind][n_ind]
  double *d_out_alt = nullptr;                 // second result buffer of the single-GPU replicate loop (ngsd_distances_batch)
  cudaEvent_t ev_copied[2] = {nullptr, nullptr};   // copy_stream: the matrix in d_out / d_out_alt has reached the host
  void *h_pin = nullptr; uint64_t h_pin_bytes = 0;    // pinned scratch for weights / lists / results
  void *h_pin2 = nullptr; uint64_t h_pin2_bytes = 0;  // pinned scratch of the tensor-core count pass of the FP64 path
  void *h_lists = nullptr; uint64_t h_lists_bytes = 0, h_lists_used = 0;   // pinned staging of small host lists (K splits, scales)
  cudaEvent_t ev_pin = nullptr;                // ctx->stream: the uploads of the last enqueued matrix have read h_pin, h_pin2 and h_lists
  uint32_t *d_cs_begin = nullptr; uint32_t cs_cap = 0;          // its K-split boundaries
  int32_t *d_cnt_part = nullptr; uint64_t cnt_part_ints = 0;    // its partial count tiles
  // ---- multi-GPU (comm.cu) ----
  void *comm = nullptr;                        // ncclComm_t of this context's rank (ngsd_comm_attach, or the group's ncclCommInitAll)
  uint32_t comm_rank = 0, comm_world = 1;
  double *d_tri = nullptr; uint64_t tri_cap = 0;        // packed upper triangle of num / cnt for the site-shard reduce
  double *d_gather = nullptr; uint64_t gather_cap = 0;  // root side: matrices received from the other ranks (batched replicates)
  uint64_t comm_bytes = 0; float comm_ms = 0.f;         // last collective: bytes over NVLink (sent + received), device time
  cudaEvent_t ev_comm[2] = {nullptr, nullptr};
  // in-process group (ngsd_cfg.n_gpus > 1): the parent owns no device memory, only its per-GPU contexts
  std::vector<ngsd_ctx *> kids;
  ngsd_ctx *parent = nullptr;
  int shard_mode = 0;                          // ngsd_shard_mode the group resolved to
  std::vector<uint64_t> site_begin;            // [n_gpus + 1] first site of every kid
  bool kids_tile_sharded = false;
  // timing
  // events 0..1 time a push (set 0); 2..8 time one distance matrix.  The single-GPU replicate loop keeps two matrices in
  // flight and alternates the sets, so `ev` points at the set of the matrix being enqueued.
  cudaEvent_t ev_sets[2][10] = {};
  cudaEvent_t *ev = ev_sets[0];
  ngsd_timing timing = {};
  char err[512] = {0};
};

#define NGSD_CUDA(ctx, call)                                                                                  \
  do {                                                                                                        \
    cudaError_t e_ = (call);                                                                                  \
    if (e_ != cudaSuccess) {                                                                                  \
      ngsd_set_error((ctx), "CUDA error: %s (%s:%d: %s)", cudaGetErrorString(e_), __FILE__, __LINE__, #call); \
      return NGSD_ERR_CUDA;                                                                                   \
    }                                                                                                         \
  } while (0)

void ngsd_set_error(ngsd_ctx *ctx, const char *fmt, ...);

// ---- kernel launchers (each .cu file owns its kernels) ----
struct ngsd_frontend_args {
  const double *raw;        // [n][n_ind][3] device, or nullptr for genotype codes
  const int8_t *codes;      // [n][n_ind] device, or nullptr
  uint64_t site0, n;
};
cudaError_t ngsd_launch_frontend(ngsd_ctx *ctx, const ngsd_frontend_args &a);
cudaError_t ngsd_launch_unpack(ngsd_ctx *ctx, double *P_dev /*[ind][site][3]*/, uint8_t *miss_dev /*[ind][site]*/);
cudaError_t ngsd_launch_unpack_2bit(ngsd_ctx *ctx, const uint8_t *packed_dev, uint64_t row_stride, uint32_t code_of_field, uint64_t n,
                                    int8_t *codes_dev);   // packed fields -> [site][ind] int8 codes
cudaError_t ngsd_launch_widen(ngsd_ctx *ctx, const void *src_dev, int format, double denom, uint64_t n, double *raw_dev);
cudaError_t ngsd_launch_patch(ngsd_ctx *ctx, const ngsd_deferred *list_dev, unsigned n);
cudaError_t ngsd_launch_synth(ngsd_ctx *ctx, double *raw_dev, uint64_t seed, double miss_rate, uint64_t site0, uint64_t n);

struct ngsd_dist_plan {
  uint32_t n_chunks;        // active chunks L
  uint32_t n_splits;        // S
  uint32_t n_units;         // S * n_tiles
  bool weighted;
  bool uniform_scale;       // weighted, but every chunk has one weight: splits carry it, no per-site scaling in the loop
  int grid;
};
cudaError_t ngsd_launch_dist_dmma(ngsd_ctx *ctx, const ngsd_dist_plan &p);
cudaError_t ngsd_launch_mask_count(ngsd_ctx *ctx, uint32_t n_blocks, cudaStream_t stream);   // per-block counts of the block cache
struct ngsd_epilogue_args {
  uint32_t n_splits;
  uint64_t const_cnt;       // used when !pairwise_del
  bool use_cnt;             // pairwise_del
};
cudaError_t ngsd_launch_epilogue(ngsd_ctx *ctx, const ngsd_epilogue_args &a);
size_t ngsd_dist_smem_bytes();
// K2b: per pair-site EM path (indep_geno == 0)
constexpr int NGSD_EM_EDGE = 64;               // pair tile edge of k_dist_em3
uint32_t ngsd_em_splits(const ngsd_ctx *ctx, uint32_t n_chunks);
uint64_t ngsd_em_split_doubles(const ngsd_ctx *ctx);   // EM partials of one K split: one 64 x 64 slot per owned tile
cudaError_t ngsd_launch_dist_em(ngsd_ctx *ctx, uint32_t n_chunks, uint32_t n_splits, bool weighted);
cudaError_t ngsd_launch_finish(ngsd_ctx *ctx, uint64_t const_cnt = 0);   // const_cnt > 0: cnt is that constant (no --pairwise_del)
cudaError_t ngsd_launch_cvec(ngsd_ctx *ctx, bool weighted, uint64_t n_eff);
cudaError_t ngsd_launch_deficit_fix(ngsd_ctx *ctx, bool weighted, uint64_t n_eff);
cudaError_t ngsd_launch_epilogue_em(ngsd_ctx *ctx, uint32_t n_splits, uint64_t const_cnt, bool use_cnt);
cudaError_t ngsd_clear_outputs(ngsd_ctx *ctx);       // epilogue.cu: zero diagonal; with a tile shard, every entry
cudaError_t ngsd_clear_unowned(ngsd_ctx *ctx);       // epilogue.cu: with a tile shard, zero every entry of a tile it does not own
// K2c: called genotypes on the int8 tensor cores (dist_umma.cu, tcgen05)
bool ngsd_int_lut(const double *score, bool pairwise_del, uint32_t lut[4], double *scale, int *max_byte);
uint32_t ngsd_int_weight_cap(const ngsd_ctx *ctx);   // largest site weight per weight layer of the integer path
cudaError_t ngsd_launch_dist_umma(ngsd_ctx *ctx, uint32_t n_units, int grid, uint32_t pstride, bool count);
struct ngsd_count_umma_args {
  const uint32_t *split_begin;   // [n_splits + 1] positions in the word list
  uint32_t n_splits;
  int32_t *partials;             // [n_splits][n_tiles][128][128]
  const uint8_t *wsite;          // [layers][NW * 64] per-site weight bytes
  const uint32_t *word_ids, *word_layer;
};
cudaError_t ngsd_launch_count_umma(ngsd_ctx *ctx, const ngsd_count_umma_args &c);   // dist_umma.cu: --pairwise_del counts of the FP64 path
cudaError_t ngsd_launch_epilogue_int(ngsd_ctx *ctx, uint32_t n_splits, uint64_t const_cnt, bool in_kernel_cnt);   // epilogue.cu

// ---- N4 trees (nj.cu, bme.cu) ----
// join t merged the subtrees in slots i < j with limb lengths li, lj; the new node takes slot i, slot j retires
struct NjJoin { uint32_t i, j; double li, lj; };
// the three slots left after the joins (in increasing order) and their distances d(a,b), d(a,c), d(b,c)
struct NjLast { uint32_t rem[3], pad; double d3[3]; };
// the neighbour-joining results of one chunk of matrices
struct NjBatch {
  uint32_t n = 0, count = 0;
  std::vector<NjJoin> joins;    // [count][n - 2]: the n - 3 joins of every matrix
  std::vector<NjLast> last;     // [count]
  std::vector<int> bad;         // [count]: the matrix holds non-finite values (no tree)
};
// Trees of n_mat matrices on ctx's GPU (nj.cu), in chunks sized from the free device memory: dist_host [n_mat][n][n], or
// the single device matrix dist_dev.  out[k], n_nni[k] and status[k] (NGSD_ERR_ARG: non-finite, out[k] empty) per matrix.
// method: NGSD_TREE_NJ / NGSD_TREE_BME.  ngsd_nj_tree, ngsd_bme_tree and ngsd_trees_batch all run through it.
int ngsd_trees_run(ngsd_ctx *ctx, const double *dist_host, const double *dist_dev, uint64_t n_mat, int method, const char *const *labels,
                   std::string *out, uint64_t *n_nni, int32_t *status);
// BME refinement of the NJ trees of one chunk (bme.cu): D the chunk's input matrices (device, stride dstride), R NJ's
// working copies, reused for the prefix sums (n (n + 1) doubles each, stride rstride); skips the matrices nj marks bad
int ngsd_bme_chunk(ngsd_ctx *ctx, const double *D, uint64_t dstride, double *R, uint64_t rstride, const NjBatch &nj, const char *const *labels,
                   std::string *out, uint64_t *n_nni);
uint64_t ngsd_bme_bytes(uint64_t n);   // device bytes of one matrix in ngsd_bme_chunk besides D and R

// fn(0) .. fn(count - 1) on up to one host thread per core (inline for a single item); every item is independent
template <typename F>
void ngsd_parallel_for(uint64_t count, F fn) {
  const uint64_t T = std::min<uint64_t>({count, (uint64_t) std::max(1u, std::thread::hardware_concurrency()), 64});
  if (T <= 1) {
    for (uint64_t k = 0; k < count; k++) fn(k);
    return;
  }
  std::atomic<uint64_t> next{0};
  auto work = [&]() { for (uint64_t k; (k = next.fetch_add(1)) < count;) fn(k); };
  std::vector<std::thread> th;
  for (uint64_t t = 1; t < T; t++) th.emplace_back(work);
  work();
  for (auto &x : th) x.join();
}

// ---- multi-GPU (comm.cu) ----
extern "C" int ngsd_frontend_resolve(ngsd_ctx *ctx);      // api.cu: knife-edge triples -> host libm -> k_patch
extern "C" int ngsd_frontend_flags(ngsd_ctx *ctx);        // api.cu: the deferred error flags of the front end, without the completeness check
extern "C" void ngsd_mark_all_pushed(ngsd_ctx *ctx);      // api.cu: after an all-gather every site is resident
void ngsd_comm_release(ngsd_ctx *ctx);         // comm.cu: communicator + staging buffers of one context
int ngsd_group_create(const ngsd_cfg *cfg, ngsd_ctx **out);
int ngsd_group_destroy(ngsd_ctx *ctx);
int ngsd_group_push(ngsd_ctx *ctx, int what /*0 sites host, 1 genotypes, 2 packed genotypes, 3 sites device*/, const void *ptr,
                    uint64_t bytes_per_site, uint64_t row_stride, const int8_t *code_of_field, uint64_t site0, uint64_t n);
int ngsd_group_frontend(ngsd_ctx *ctx);
int ngsd_group_distances(ngsd_ctx *ctx, const uint32_t *block_counts, uint64_t n_blocks, uint64_t block_size, double *out, double *num_opt,
                         uint64_t *cnt_opt);
int ngsd_group_distances_batch(ngsd_ctx *ctx, const uint32_t *block_counts, uint64_t n_rep, uint64_t n_blocks, uint64_t block_size, double *out);
int ngsd_group_get_posteriors(ngsd_ctx *ctx, double *P_host, uint8_t *miss_host);
int ngsd_group_get_timing(ngsd_ctx *ctx, ngsd_timing *t);
int ngsd_group_trees(ngsd_ctx *ctx, const double *dist_host, uint64_t n_mat, int method, const char *const *labels, std::string *out,
                     uint64_t *n_nni, int32_t *status);   // contiguous slices of the batch, one per GPU, through ngsd_trees_run
