/* ngsdist_b200.h -- C ABI of the B200-native ngsDist pairwise-distance hot path.
 *
 * ngsDist has no plugin / FFI interface; its only internal seam is the code between
 * "read_geno returned" (ngsDist.cpp:156) and "print matrix" (ngsDist.cpp:282-287):
 *   - the per-individual-site front end      ngsDist.cpp:161-174 (+ the normalisation half that lives in the
 *                                             reader, shared/read_data.cpp:37-45,83-99)
 *   - the pair dispatch + gen_dist()          ngsDist.cpp:197-269, 325-412
 *   - the bootstrap re-mapping                ngsDist.cpp:235-238, 416-437 (RNG stays on the host)
 * This library replaces exactly that code.  A maintainer keeps parse_args.cpp, the readers and the writer and
 * calls the entry points below instead (INTEGRATION.md shows the patch).
 *
 * Conventions: plain pointers and sizes, no C++/torch types; every function returns 0 on success or a
 * negative ngsd_status and records a message retrievable with ngsd_last_error() -- the host turns it into the
 * reference's error(__FUNCTION__, msg) (shared/gen_func.cpp:12-18).  No CPU fallback exists: without a CUDA
 * device ngsd_create fails with NGSD_ERR_CUDA.  One host thread drives one context; contexts are independent
 * (one per GPU / per rank).
 */
#ifndef NGSDIST_B200_H
#define NGSDIST_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NGSD_ABI_VERSION 2

#if defined(__GNUC__)
#define NGSD_API __attribute__((visibility("default")))
#else
#define NGSD_API
#endif

typedef enum {
  NGSD_OK = 0,
  NGSD_ERR_ARG = -1,       /* invalid argument / configuration                                    */
  NGSD_ERR_CUDA = -2,      /* CUDA runtime failure (including "no device")                        */
  NGSD_ERR_NAN = -3,       /* "NaN found! Is the file format correct?"   (read_data.cpp:42-45)    */
  NGSD_ERR_THRESH = -4,    /* "missing data threshold must be smaller than calling genotype
                              threshold!"                                (gen_func.cpp:887-888)   */
  NGSD_ERR_MODEL = -5,     /* evol_model 3..6 "not yet supported" / invalid (ngsDist.cpp:387-401) */
  NGSD_ERR_STATE = -6,     /* call order violated (e.g. distances before all sites were pushed)   */
  NGSD_ERR_GENO = -7,      /* "Genotypes must be coded as {-1,0,1,2} !"  (read_data.cpp:91-92)    */
  NGSD_ERR_COMM = -8       /* NCCL failure / communicator misuse (multi-GPU entry points)         */
} ngsd_status;

/* How a multi-GPU context (ngsd_cfg.n_gpus > 1) places the data set on its GPUs (SURVEY §8e). */
typedef enum {
  NGSD_SHARD_AUTO = 0,        /* REPLICATED when the packed operands of all sites fit one GPU, else SITES            */
  NGSD_SHARD_REPLICATED = 1,  /* every GPU ends up with all sites (site-sharded front end + NCCL all-gather of the packed
                                 operands): bootstrap replicates (ngsd_distances_batch) and output-triangle tiles
                                 (ngsd_distances) are dealt to the GPUs, no reduction on the data path                */
  NGSD_SHARD_SITES = 2        /* GPU g holds a contiguous site range: partial sums, ONE ncclReduce of the upper triangle
                                 of num (+ cnt under --pairwise_del), epilogue after the reduction                    */
} ngsd_shard_mode;

/* How raw values were read; selects the reader-side half of the front end (H2 in SURVEY §8a). */
typedef enum {
  NGSD_INPUT_BINARY_GL = 0,  /* read_data.cpp:29-47: log() unless log scale, -inf -> -1e15, normalise, NaN is fatal */
  NGSD_INPUT_TEXT_GL = 1,    /* read_data.cpp:83-87,98: log() unless log scale, no clamp, normalise                 */
  NGSD_INPUT_GENOTYPES = 2   /* read_data.cpp:88-95,98: codes {-1,0,1,2}; pushed with ngsd_push_genotypes          */
} ngsd_input_kind;

/* Mirrors the fields of `params` (ngsDist.hpp:11-44) that the hot path reads. */
typedef struct {
  uint64_t n_ind;            /* params.n_ind                                                        */
  uint64_t n_sites;          /* params.n_sites (all sites of the data set)                          */
  uint64_t tot_sites;        /* params.tot_sites; > 0 overrides the per-pair count (ngsDist.cpp:372) */
  double score[9];           /* params.score[g1][g2], row-major (parse_args.cpp:25-27,134-137); g1 is the genotype of
                                the lower-index individual of the pair, g2 of the higher (i1 < i2, ngsDist.cpp:351-353).
                                Need not be symmetric                                                 */
  int32_t evol_model;        /* 0 raw p-distance, 1 -log(1-d), 2 JC69 (ngsDist.cpp:378-386)         */
  int32_t pairwise_del;      /* params.pairwise_del                                                  */
  int32_t indep_geno;        /* params.indep_geno AFTER the forcing rules of ngsDist.cpp:55-62      */
  int32_t call_geno;         /* params.call_geno                                                     */
  double N_thresh;           /* params.N_thresh                                                      */
  double call_thresh;        /* params.call_thresh                                                   */
  int32_t input_is_log;      /* params.in_logscale as given on the command line                     */
  int32_t input_kind;        /* ngsd_input_kind                                                      */
  int32_t device;            /* CUDA device ordinal this context owns                                */
  int32_t reserved;          /* flags: bit 0 = keep all three operand planes (disables the sum-to-one reduction that is
                                used when indep_geno && !pairwise_del; for inspection through ngsd_get_posteriors);
                                bit 1 = do not use the integer (int8 tensor core) path for called genotypes, i.e. run
                                them through the FP64 contraction like soft posteriors (A/B testing);
                                bit 2 = contract every bootstrap replicate directly (weighted contraction) instead of
                                reusing per-block partial sums (the bootstrap block cache)                          */
  int32_t n_gpus;            /* 0 / 1: one GPU (`device`).  N > 1: the context drives devices device .. device+N-1 from one
                                host thread per GPU inside the library (replaces the pthread pool of ngsDist.cpp:197-269
                                at box level); every entry point below takes such a context unchanged                 */
  int32_t shard;             /* ngsd_shard_mode (n_gpus > 1 only)                                                     */
  uint64_t boot_block_size;  /* params.boot_block_size when bootstrap replicates will follow (0 / 1: none): site shards
                                are aligned to whole blocks (ngsDist.cpp:416-437)                                     */
} ngsd_cfg;

/* An empty text line consumes a site and leaves the reference's values at their -1e15 fill without normalisation
 * (read_data.cpp:58-59): after exp() every individual has (0,0,0) there -- or plain missing data under --call_geno.
 * A host reader reproduces that by filling the site, for every individual, with this quiet-NaN bit pattern (all three
 * doubles) or, for genotype input, with the code NGSD_BLANK_SITE_CODE. */
#define NGSD_BLANK_SITE_BITS 0x7FF84E4753444231ull
#define NGSD_BLANK_SITE_CODE (-128)

typedef struct ngsd_ctx ngsd_ctx;

/* Per-call device timings of the last ngsd_distances()/ngsd_push_* call, milliseconds, measured with CUDA
 * events on the context's stream.  launches = number of this library's kernels launched by that call. */
typedef struct {
  float frontend_ms;         /* K1 front-end kernel(s)                                   */
  float count_ms;            /* K3 mask-count kernel                                     */
  float dist_ms;             /* K2 DMMA contraction / K2b pair-site EM / K2c int8 contraction kernel */
  float epilogue_ms;         /* K4 split reduction + epilogue kernel                     */
  float total_ms;            /* first launch to last launch of the call                  */
  int32_t launches;
  int32_t dist_ctas;         /* grid size of the distance kernel                         */
  uint64_t dist_dmma;        /* warp-level DMMA.8x8x4 instructions the K2 launch issued  */
  uint64_t active_sites;     /* sites with non-zero weight in the call                   */
  uint64_t dist_imma;        /* K2c work of the called-genotype integer path, in IMMA-equivalents of 4096 int8 MAC */
  int32_t block_cache;       /* bootstrap block cache: 0 not used, 1 built by this call, 2 reused (no contraction launched) */
  int32_t pad_;
} ngsd_timing;

NGSD_API void ngsd_default_cfg(ngsd_cfg *cfg);   /* init_pars (parse_args.cpp:6-37) for the fields above */

/* Creates a context: validates cfg (NGSD_ERR_THRESH when N_thresh > call_thresh with call_geno, NGSD_ERR_MODEL for
 * evol_model outside 0..2, NGSD_ERR_ARG for tot_sites with pairwise_del as parse_args.cpp:209-210), selects the device
 * and allocates the packed operand planes for n_ind x n_sites.  The library owns all device memory. */
NGSD_API int ngsd_create(const ngsd_cfg *cfg, ngsd_ctx **out);
NGSD_API int ngsd_destroy(ngsd_ctx *ctx);
NGSD_API const char *ngsd_last_error(const ngsd_ctx *ctx);   /* ctx may be NULL: last error of ngsd_create */

/* Front end (H2+H3+H4).  `raw` holds n sites starting at site0 exactly as the reader obtained them, binary layout
 * [site][ind][3] doubles (read_data.cpp:28-31), un-normalised.  Replaces read_data.cpp:37-45 / :83-99 (normalisation)
 * and ngsDist.cpp:165-174 (call_geno + exp).  site0 must be a multiple of 64 (chunks are independent, so the host reader
 * never holds the whole data set).  The host variant copies asynchronously from `raw` (pinned memory recommended) and
 * returns when the copy has been consumed; the device variant reads a device pointer in place. */
NGSD_API int ngsd_push_sites(ngsd_ctx *ctx, const double *raw_host, uint64_t site0, uint64_t n);
NGSD_API int ngsd_push_sites_device(ngsd_ctx *ctx, const double *raw_dev, uint64_t site0, uint64_t n);
/* Transport tiers for likelihoods / posteriors (SURVEY §8f N3): the same front end fed from narrower host values, for
 * hosts where the 24 B per individual-site of the binary layout (read_data.cpp:28-31) make PCIe the bottleneck.  The
 * values are widened to double on the device and then take exactly the path of ngsd_push_sites.
 *   NGSD_XFER_F32   [site][ind][3] float:   12 B.  Rounds every input to 24 bits; measured effect on distances in DESIGN §4.
 *   NGSD_XFER_U32   [site][ind][3] uint32:  12 B.  value = q / denom (IEEE division): EXACTLY the double strtod gives a decimal
 *                                           with <= 9 significant digits when denom is the matching power of ten.
 *   NGSD_XFER_U20X3 [site][ind] uint64:      8 B.  q0 | q1 << 20 | q2 << 40, value = q / denom: exact for the 6-decimal
 *                                           posteriors the reference's text inputs hold (ANGSD -doGeno 8), denom = 1e6.
 * denom is ignored for NGSD_XFER_F32.  Normal-scale and log-scale contexts alike (fixed point: normal scale only). */
typedef enum { NGSD_XFER_F32 = 1, NGSD_XFER_U32 = 2, NGSD_XFER_U20X3 = 3 } ngsd_xfer_format;
NGSD_API int ngsd_push_sites_packed(ngsd_ctx *ctx, const void *host, int32_t format, double denom, uint64_t site0, uint64_t n);
/* Genotype input (no --probs): codes [site][ind] in {-1,0,1,2}; NGSD_ERR_GENO for anything > 2. */
NGSD_API int ngsd_push_genotypes(ngsd_ctx *ctx, const int8_t *codes_host, uint64_t site0, uint64_t n);
/* The same genotype input, four individuals per byte (SURVEY §8f N3: the 1 B -- or as text 2-3 B -- per individual-site
 * of read_data.cpp:88-95 is what makes the 5 000 x 5 000 000 configuration expensive to store and to move).  Site-major:
 * individual i of site s is the 2-bit field (packed[s * row_stride + i / 4] >> 2 * (i % 4)) & 3, row_stride >= ceil(n_ind / 4);
 * code_of_field[f] in {-1,0,1,2} is the reference's code for field value f (NULL: {0,1,2,-1}).  A variant-major PLINK .bed
 * body (after its 3 magic bytes) is exactly this layout with code_of_field = {0,-1,1,2} and row_stride = ceil(n_ind / 4).
 * Results are bit-identical to ngsd_push_genotypes of the unpacked codes. */
NGSD_API int ngsd_push_packed_genotypes(ngsd_ctx *ctx, const uint8_t *packed_host, uint64_t row_stride, const int8_t *code_of_field,
                                        uint64_t site0, uint64_t n);
/* Completes the front end: checks that every site was pushed and raises the deferred NGSD_ERR_NAN. */
NGSD_API int ngsd_frontend(ngsd_ctx *ctx);

/* One distance matrix = one pass of ngsDist.cpp:244-269 (all pairs through gen_dist).
 *   block_counts == NULL : replicate 0, all n_sites sites, weight 1.
 *   block_counts != NULL : a bootstrap replicate.  block_counts[b] = how many times source block b was drawn by
 *                          rnd_map_data (ngsDist.cpp:416-437) for this replicate; n_blocks * block_size sites are
 *                          used (the persistent truncation of ngsDist.cpp:236).  The RNG stays on the host.
 *   out      : n_ind x n_ind row-major, symmetric, 0.0 diagonal (ngsDist.cpp:200,411), model-transformed distances.
 *   num_opt  : optional, same shape: the raw accumulator `dist` before normalisation (the --verbose 3 value, :366-367).
 *   cnt_opt  : optional, same shape: the number of valid sites per pair BEFORE the tot_sites override.
 * All three are host pointers (may be pageable). */
NGSD_API int ngsd_distances(ngsd_ctx *ctx, const uint32_t *block_counts, uint64_t n_blocks, uint64_t block_size,
                   double *out, double *num_opt, uint64_t *cnt_opt);

/* The bootstrap loop of main() in one call (ngsDist.cpp:217-238 for rep = 1 .. n_rep): block_counts[r][b] as for
 * ngsd_distances, out[r] = the n_ind x n_ind matrix of replicate r (host).  With one GPU the replicates run back to back;
 * a multi-GPU context (REPLICATED) or a communicator (ngsd_comm_attach) deals replicate r to GPU / rank r % N -- no
 * data-path collective, every GPU writes its matrices to the host through its own PCIe link; with a communicator the
 * matrices are gathered on rank 0 (NCCL send/recv) and `out` may be NULL on the other ranks.  SITES contexts run the
 * replicates one after the other, each on all GPUs. */
NGSD_API int ngsd_distances_batch(ngsd_ctx *ctx, const uint32_t *block_counts, uint64_t n_rep, uint64_t n_blocks, uint64_t block_size,
                                  double *out);

/* ---- multi-GPU support (one context per GPU / process; SURVEY §8e) -------------------------------------------------
 * Bootstrap replicates shard by simply calling ngsd_distances for different replicates on different contexts.
 *
 * Output-triangle tiles: after ngsd_set_tile_shard(rank, world) the context computes only the 128 x 128 upper-triangle
 * tiles dealt to `rank` (pairs of neighbouring tiles of one row block, each to the rank holding the fewest so far); every entry it does not own is written as 0 in out / num /
 * cnt, so an element-wise SUM over the ranks assembles the full matrices exactly (x + 0 == x).  On the per pair-site EM
 * path (indep_geno == 0) the context contracts the 64 x 64 tiles inside the 128 x 128 tiles it owns; its bootstrap
 * block cache then holds only those tiles.
 *
 * Sites: each rank creates its context for its own contiguous, block-aligned site range, calls ngsd_distances with
 * out == NULL (raw sums stay on the device), all-reduces the buffers returned by ngsd_device_results (num: FP64 sum,
 * cnt: uint64 sum -- e.g. ncclAllReduce over NVLink) and then calls ngsd_finish, which applies the tail of gen_dist
 * (ngsDist.cpp:372-401: tot_sites override, division, evolutionary model) to the reduced sums: the epilogue is
 * non-linear, so it must run after the reduction. */
NGSD_API int ngsd_set_tile_shard(ngsd_ctx *ctx, uint32_t rank, uint32_t world);
NGSD_API int ngsd_device_results(ngsd_ctx *ctx, double **out_dev, double **num_dev, uint64_t **cnt_dev);   /* n_ind x n_ind each */
NGSD_API int ngsd_finish(ngsd_ctx *ctx, double *out_host);

/* ---- one process per GPU: NCCL communicator over the contexts of all ranks (SURVEY §5 "distributed communication
 * backend", §2.1 rows C1 / C2).  The library links NCCL itself; the host only has to carry 128 bytes from rank 0 to
 * the other ranks (a file, MPI, torch.distributed -- anything).  All calls below are collective: every rank makes
 * them in the same order.  The reference has no counterpart (ngsDist.cpp:197-269 is one shared-memory pool). */
#define NGSD_COMM_ID_BYTES 128
NGSD_API int ngsd_comm_unique_id(uint8_t id[NGSD_COMM_ID_BYTES]);                           /* ncclGetUniqueId, on rank 0 */
NGSD_API int ngsd_comm_attach(ngsd_ctx *ctx, const uint8_t id[NGSD_COMM_ID_BYTES], uint32_t rank, uint32_t world);
/* REPLICATED data from a site-sharded front end: rank g pushed only sites [site_begin[g], site_begin[g+1]) (multiples
 * of 64; 192 when the context contracts two planes) of a context created for ALL sites; one grouped NCCL all-gather of
 * the packed operands, masks and codes makes every rank hold every site (row C2). */
NGSD_API int ngsd_comm_allgather_operands(ngsd_ctx *ctx, const uint64_t *site_begin /* [world + 1] */);
/* Site shards (row C1): after ngsd_distances(out == NULL) on every rank, ONE ncclReduce of the packed upper triangle of
 * num (FP64) -- and of cnt (uint64) only under --pairwise_del, otherwise cnt is the constant n_eff_total -- onto `root`,
 * which then runs the tail of gen_dist (ngsDist.cpp:372-401) and returns the matrix in out_host (NULL elsewhere). */
NGSD_API int ngsd_comm_reduce_sites(ngsd_ctx *ctx, uint32_t root, uint64_t n_eff_total, double *out_host);
/* Tile shards (ngsd_set_tile_shard(rank, world) on every rank), on every contraction path including the per pair-site
 * EM: after ngsd_distances(out == NULL), the matrices are assembled on `root` by an NCCL sum (entries a rank does not
 * own are exact zeros; a NaN matrix of the EM path keeps its NaNs only on the owned entries).  with_num_cnt (the same value on
 * every rank) also assembles the raw sums and counts; the host pointers are only read on `root`. */
NGSD_API int ngsd_comm_reduce_tiles(ngsd_ctx *ctx, uint32_t root, int32_t with_num_cnt, double *out_host, double *num_host, uint64_t *cnt_host);
NGSD_API int ngsd_comm_barrier(ngsd_ctx *ctx);
/* bytes moved over NVLink by the last collective of this rank (sent + received) and its device time in ms */
NGSD_API int ngsd_comm_stats(const ngsd_ctx *ctx, uint64_t *bytes, float *ms);

/* Host placement (VERDICT r1: 8 ranks pushing from pinned buffers that all sit on one NUMA node): binds the calling
 * thread to the CPUs local to `device` (sysfs local_cpulist of its PCI function) and prefers that node for the pages
 * it touches afterwards -- call before ngsd_host_alloc.  Returns the NUMA node, -1 when the platform exposes none. */
NGSD_API int ngsd_bind_host_to_device(int device);

/* Downstream of the matrices (SURVEY §8f N4; the workflow of README.md:83-98 hands the .dist file to FastME for one tree
 * per matrix): a neighbour-joining tree (Saitou & Nei 1987 / Studier & Keppler 1988; ties: smallest i, then j) computed on
 * the device.  dist_host == NULL: from the matrix the last ngsd_distances / ngsd_finish left on the device (as transformed
 * by cfg.evol_model); otherwise from the given n_ind x n_ind host matrix (e.g. after the host's own -log / JC69 tail).
 * labels: n_ind C strings or NULL ("Ind_<i>", ngsDist.cpp:118-124).  Writes Newick with "%.10f" branch lengths and a
 * trifurcating root into `newick` (NUL-terminated) and its length into *newick_len; NGSD_ERR_ARG with the needed size in
 * *newick_len when newick_cap is too small, or when the matrix holds non-finite values.  The reference has no
 * counterpart: parity is against a CPU restatement of the same rules (oracle/nj_oracle.py). */
NGSD_API int ngsd_nj_tree(ngsd_ctx *ctx, const double *dist_host, const char *const *labels, char *newick, uint64_t newick_cap,
                          uint64_t *newick_len);

/* The criterion FastME optimises: a balanced minimum-evolution tree (BME; Desper & Gascuel 2002, Pauplin's length
 * L(T) = sum_{i<j} 2^(1 - tau_ij) d_ij, tau_ij the number of edges between leaves i and j).  Starts from the tree of
 * ngsd_nj_tree, applies the BME nearest-neighbour interchange of largest gain (ties: smallest internal node id, then the
 * swap with the child of the smaller individual index) while its gain exceeds 1e-12 M, M = sum_{i<j} 2^(1 - tau_ij) |d_ij|
 * (M = L when no distance is negative), and writes the tree with balanced branch lengths (they sum to L; negative lengths
 * are written as computed).  Every applied interchange lowers L, so the call returns for every finite matrix, negative
 * entries included.  Every round is O(n^2) work on the device; the matrix is read in place (dist_host: one upload).  Same arguments, matrix source, labels and errors as ngsd_nj_tree; the Newick is rooted as a trifurcation at the
 * neighbour of individual 0, "(Ind_0:l,(...):l,(...):l);", every node's children in order of their smallest individual
 * index.  n_nni (may be NULL) receives the number of interchanges applied.  Parity is against a CPU restatement of the
 * same rules (oracle/bme_oracle.py); DESIGN §3 N4 states them. */
NGSD_API int ngsd_bme_tree(ngsd_ctx *ctx, const double *dist_host, const char *const *labels, char *newick, uint64_t newick_cap,
                           uint64_t *newick_len, uint64_t *n_nni);

/* The trees of a whole batch of matrices -- e.g. every bootstrap replicate -- in one pass per GPU: one launch of each
 * kernel serves every matrix of a chunk, so a batch pays the launches of one tree while the device work grows with it.
 * dist_host: n_mat x n_ind x n_ind host matrices (required when n_mat > 0); method NGSD_TREE_NJ (ngsd_nj_tree) or
 * NGSD_TREE_BME (ngsd_bme_tree).  Tree k is byte-identical to what that call gives for matrix k alone; it is the
 * NUL-terminated string at newicks + offsets[k] (offsets has n_mat + 1 entries; offsets[n_mat] = bytes used).
 * status[k] is NGSD_OK, or NGSD_ERR_ARG for a matrix with non-finite entries, whose tree is then the empty string -- the
 * other trees are still built.  n_nni (may be NULL) receives the interchanges applied per tree (0 for NJ).  When cap is too
 * small the call returns NGSD_ERR_ARG with the bytes needed in offsets[n_mat].  n_mat == 0 does nothing.
 * The matrices are processed in chunks sized from the free device memory at call time; chunking changes no result.
 * A multi-GPU context (ngsd_cfg.n_gpus > 1) deals contiguous slices of the batch to its GPUs, each uploading only its own
 * matrices; results come back in input order.  A context with a communicator (ngsd_comm_attach) builds trees on its own GPU
 * only: each rank passes its own matrices. */
#define NGSD_TREE_NJ 0
#define NGSD_TREE_BME 1
NGSD_API int ngsd_trees_batch(ngsd_ctx *ctx, const double *dist_host /* n_mat x n_ind x n_ind */, uint64_t n_mat, int32_t method,
                              const char *const *labels, char *newicks, uint64_t cap, uint64_t *offsets /* n_mat + 1 */,
                              uint64_t *n_nni /* n_mat, may be NULL */, int32_t *status /* n_mat */);

/* Bootstrap support of a tree -- the last step of the reference's workflow (README.md:83-98: `raxmlHPC -f b -t main -z
 * boots` on FastME's trees).  HOST code only, no context: for every internal edge of `main_newick`, the number of trees among
 * `rep_newicks[n_reps]` that hold the same bipartition of the leaf labels is written as the node's label
 * ("(A:0.1,B:0.2)87:0.05"); percent != 0 gives RAxML's integer percentages (int)(0.5 + 100 c / n), else the raw counts.
 * Replicates given as "NA" (the CLI's marker for a matrix without a tree) are skipped.  Branch lengths are copied as
 * written.  NGSD_ERR_ARG for malformed Newick, leaf sets that differ, or when out_cap is too small (*out_len = bytes
 * needed, without the NUL).  No reference code exists for this step: parity is against tests/ restating the definition. */
NGSD_API int ngsd_tree_support(const char *main_newick, const char *const *rep_newicks, uint64_t n_reps, int percent, char *out,
                               uint64_t out_cap, uint64_t *out_len);

/* Host-side helper with the reference's RNG semantics (gsl_rng_taus; ngsDist.cpp:179-180, gen_func.cpp:117-119):
 * state[3] is seeded by ngsd_taus_seed and advanced by n_blocks draws per call of ngsd_boot_block_counts, which
 * fills counts[n_blocks] for one replicate exactly as rnd_map_data would have re-pointed the blocks. */
NGSD_API void ngsd_taus_seed(uint32_t state[3], uint32_t seed);
NGSD_API uint32_t ngsd_taus_get(uint32_t state[3]);
NGSD_API void ngsd_boot_block_counts(uint32_t state[3], uint64_t n_blocks, uint32_t *counts);

/* Inspection (tests, --verbose): copy the front-end results back in the reference's own shapes.
 *   P    : [ind][site][3] normal-space posteriors as gen_dist would read them (params.geno_lkl).
 *   miss : [ind][site] 1 where miss_data() is true (gen_func.cpp:862-868). */
NGSD_API int ngsd_get_posteriors(ngsd_ctx *ctx, double *P_host, uint8_t *miss_host);
/* How many individual-sites sat within 1e-11 of one of the reference's comparisons (miss_data's EPSILON, N_thresh,
 * call_thresh, a tie of the two largest values) and were therefore evaluated by the HOST's libm -- the reference's own
 * log / exp -- instead of the device's (front end, DESIGN §4). */
NGSD_API int ngsd_deferred_stats(const ngsd_ctx *ctx, uint64_t *host_evaluated);

/* Measurement support (bench.py): device-side synthetic raw GLs (SURVEY §8(d) generator, bit-identical to the CPU
 * restatement), timings of the last call, the context's stream, and an FP64 DMMA issue-rate probe used as the
 * roofline denominator when MEASURED_PEAKS.json has no FP64 figure. */
NGSD_API int ngsd_synth_raw_device(ngsd_ctx *ctx, double *raw_dev, uint64_t seed, double miss_rate, uint64_t site0, uint64_t n);
NGSD_API int ngsd_get_timing(const ngsd_ctx *ctx, ngsd_timing *t);
NGSD_API void *ngsd_stream(ngsd_ctx *ctx);                       /* cudaStream_t */
NGSD_API int ngsd_probe_fp64_tflops(int device, double *dmma_tflops);
NGSD_API int ngsd_probe_int8_tmacs(int device, double *imma_tmacs);   /* mma.sync int8 (IMMA.16832) issue-rate ceiling, 1e12 MAC/s */
NGSD_API int ngsd_probe_umma_tmacs(int device, double *umma_tmacs);   /* tcgen05.mma kind::i8 (UTCIMMA) issue-rate ceiling, 1e12 MAC/s */
NGSD_API void *ngsd_host_alloc(uint64_t bytes);                  /* pinned host memory for push/out buffers */
NGSD_API void ngsd_host_free(void *p);
NGSD_API int ngsd_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* NGSDIST_B200_H */
