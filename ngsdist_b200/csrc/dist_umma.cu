// K2c dist_umma: the pair loop of gen_dist (ngsDist.cpp:333-364) for CALLED genotypes as an exact integer contraction on
// the 5th-generation tensor cores: tcgen05.mma kind::i8 (SASS UTCIMMA), A operand and int32 accumulators in tensor
// memory, B operand in shared memory.
//
// When every individual-site is either a hard call or missing -- genotype input (read_data.cpp:88-95) or --call_geno with
// N_thresh == call_thresh (gen_func.cpp:903-913; the default 0/0) -- its posterior triple is one of four states:
// one-hot(0), one-hot(1), one-hot(2) or the uniform triple of a missing entry (code 3).  The site term
// sum_{g1,g2} score[g1][g2] p_i[g1] p_j[g2] (ngsDist.cpp:351-353) then only depends on the two codes: a 4 x 4 table
// f(c_i, c_j).  HBM holds 2 bits per individual-site (plus the same codes as 4-bit selectors) instead of FP64 planes.
//
// The arithmetic.  With S = 2 (--pairwise_del) or 18 (otherwise: the uniform 1/3 makes f a multiple of 1/18) and w_s the
// bootstrap multiplicity of the site (ngsDist.cpp:416-437; 1 for replicate 0, 0 for padding):
// acc(i,j) = S sum_s w_s f(c_i(s), c_j(s)) as an int8 GEMM with exact int32 accumulation and THREE K bytes per site:
//     A_i[s][k] = w_s (m [c_i = k] + [c_i = 3] t),     B_j[s][k] = (S / m) f(k, c_j),     k = 0, 1, 2
// with (m, t) = (1, 0) with --pairwise_del (row and column 3 of f are zero) and (3, 1) without (a missing genotype is the
// uniform triple, gen_func.cpp:895-899, so its row of f is the mean of the other three) -- the same S f(c_i, c_j) exactly,
// a quarter fewer operand bytes, MMAs and expansion instructions than one K byte per code value.  Weights above
// ngsd_int_weight_cap go into further weight layers (api.cu).  k_epilogue_int (epilogue.cu) sums the splits in int64 and
// applies num = acc / S and the tail of gen_dist: num, cnt and the model-0 distances are bit-exact whenever the
// reference's own sum is exact (no missing data, or --pairwise_del).  UMMA runs the int8 GEMM
// 4x faster than mma.sync (probe: 2.3e15 vs 5.7e14 MAC/s) but cannot take operands from registers, so the expansion of the
// 2-bit codes is written out every stage.  A CTA is a four-role pipeline connected by mbarrier rings:
//
//   warp 0      producer   cp.async.bulk of the packed codes (3 x 4 KiB of selector nibbles + 64 weight bytes per 64-site stage)
//   warps 2-17  expanders  codes -> int8 operands.  B (48 KiB per stage) goes to shared memory in the K-major, no-swizzle
//                          UMMA layout (8-row x 16-byte core matrices; one STS.128 = 16 K bytes of one row, fence.proxy.async);
//                          A (128 rows x 192 bytes per stage) goes to TENSOR MEMORY with tcgen05.st (row = lane, 4 K bytes
//                          per 32-bit column) -- the MMA reads it from there, which takes a third of the operand traffic
//                          off the shared-memory pipe.  The warps work in kGroups groups on alternate stages (below)
//   warp 1      MMA        one lane issues 6 x tcgen05.mma (128 x 256 x 32, A from TMEM) per stage, tcgen05.commit frees the stage
//   warps 18-21 epilogue   tcgen05.ld of a finished unit's 128 x 256 accumulator, int32 partial tiles written row-major
//                          (TMEM: 256 accumulator columns + kExp x 64 A columns)
//
// A unit is a PAIR of output tiles of one row block (api.cu: d_pairs): they share the A operand, so one stage expands
// 3 x 128 rows for 128 x 256 pairs instead of 2 x 128 rows for 128 x 128 (the odd tile of a row runs alone, N = 128).
#include <math.h>
#include <stdlib.h>

#include <algorithm>

#include "ngsd_internal.h"

namespace {

#ifndef NGSD_UMMA_KRAW
#define NGSD_UMMA_KRAW 4
#endif
#ifndef NGSD_UMMA_KEXP
#define NGSD_UMMA_KEXP 3
#endif
// The expander warps work in kGroups groups on ALTERNATE stages.  A stage costs a warp a fixed chain of latencies (barrier
// wake-up, LDS, tcgen05.wait::st, fence.proxy.async, arrive) that does not shrink with the work: with every warp in every
// stage the stage rate was one warp's latency, whatever the instruction count.  Measured at 5 000 x 100 000 (groups, raw
// stages, expanded stages): (1, 4, 3) 3.08 ms, (2, 4, 3) 2.77 ms, (2, 2, 4) 2.75 ms, (2, 6, 3) 2.76 ms; with --pairwise_del
// 4.74 / 4.45 / 4.55 / 4.44 ms.  What bounds a stage now is the shared-memory pipe: 48 KiB of B written + 48 KiB read back
// by the tensor core + 12 KiB of codes written by the bulk copies + 12 KiB read = 120 KiB at 128 B/clk = 940 cycles
// (measured 1 250; the 6 MMAs need 770).  A group is kExpWarps / kGroups warps (a multiple of 4: a warp reaches only the TMEM lanes of quadrant warp % 4)
// and a thread expands kGroups site quads of each code word of its row.
#ifndef NGSD_UMMA_GROUPS
#define NGSD_UMMA_GROUPS 2
#endif
constexpr int kRaw = NGSD_UMMA_KRAW;              // raw (packed codes) stages
constexpr int kExp = NGSD_UMMA_KEXP;              // expanded operand stages
constexpr int kGroups = NGSD_UMMA_GROUPS;
constexpr int kExpWarps = 16, kEpiWarps = 4;
constexpr int kGroupWarps = kExpWarps / kGroups;
static_assert(kGroups == 1 || kGroups == 2 || kGroups == 4, "expander groups");
// mbarrier waits tell phases apart by parity only.  A raw slot must always belong to the same group (else a group could wait
// for phase k of a slot whose phase k - 1, another group's, has not landed yet -- bulk copies complete out of order), and a
// group runs at most kGroups + kExp stages ahead of the MMA, which must stay below two phases of an expanded slot
// (kGroups = 4 with kExp = 3 hung on the GPU for exactly that reason).
static_assert(kRaw % kGroups == 0 && kGroups <= kExp, "expander groups vs ring depths");
constexpr int kThreads = (2 + kExpWarps + kEpiWarps) * 32;
constexpr int kCodeBytes = 8 * 128 * 4;           // [8 words][128 rows] uint32 of selector nibbles (codes4), one operand of one 64-site stage
constexpr int kMaskBytes = 128 * 8;               // presence bits of one operand of one 64-site word (count pass)
constexpr int kRawBytes = 3 * kCodeBytes + 128;   // A codes, B codes of the two tiles, 64 site weights; a multiple of 128
constexpr int kBChunk = 4096;                     // B: bytes between 16-byte K chunks (32 row groups x 8 rows x 16 B)
constexpr int kChunks = 12;                       // 16-byte K chunks per stage: 64 sites x 3 planes (count pass: 192 sites x 1 byte)
constexpr int kMmas = kChunks / 2;                // K = 32 bytes per tcgen05.mma
constexpr int kExpBytes = kChunks * kBChunk;      // expanded B of one stage: 48 KiB
constexpr uint32_t kAccCols = 256, kACols = 64;   // TMEM columns: accumulator, one stage of A (48 in use)
constexpr int kCntGroup = 3;                      // count pass: word-list entries (64 sites, one byte each) per stage
constexpr int kCntEntry = 3 * kMaskBytes;         // count pass raw stage: kCntGroup x {A, B, B' masks} then kCntGroup x 64 weights
constexpr int kCntRawBytes = (kCntGroup * (kCntEntry + 64) + 127) / 128 * 128;
static_assert(kCntRawBytes <= kRawBytes, "count-pass raw stages live in the code ring");
constexpr int kRingBytes = kRaw * kRawBytes;
constexpr int kNBar = 2 * kRaw + 2 * kExp + 4;
constexpr size_t kSmemBytes = (size_t) kRingBytes + (size_t) kExp * kExpBytes + kNBar * 8 + (kRaw + kExp + 2) * 8 + 16 + 64 + 1024;
static_assert(kSmemBytes <= 232448, "k_dist_umma shared memory");
static_assert(kAccCols + kExp * kACols <= 512, "k_dist_umma tensor memory");

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
__device__ __forceinline__ void mbar_wait_sleep(uint64_t *bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) __nanosleep(100);
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
// tcgen05.commit: the mbarrier gets one arrival when every tcgen05.mma issued so far by this thread has completed
__device__ __forceinline__ void umma_commit(uint64_t *bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// K-major, SWIZZLE_NONE shared-memory matrix descriptor: start >> 4 [0,14), K-direction (leading) byte offset >> 4
// [16,30), M/N-direction (stride, between 8-row groups) byte offset >> 4 [32,46), version 1 [46,48), layout 0 [61,64)
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return (uint64_t) ((saddr & 0x3FFFF) >> 4) | ((uint64_t) ((lbo_bytes >> 4) & 0x3FFF) << 16) | ((uint64_t) ((sbo_bytes >> 4) & 0x3FFF) << 32) |
         ((uint64_t) 1 << 46);
}
__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "l"(da), "l"(db), "r"(idesc), "r"(accumulate), "r"(0u)
      : "memory");
}

// the same with the A operand in tensor memory (row = lane, K bytes along the columns)
__device__ __forceinline__ void umma_i8_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t db, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], [%1], %2, %3, {%5, %5, %5, %5}, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "r"(tmem_a), "l"(db), "r"(idesc), "r"(accumulate), "r"(0u)
      : "memory");
}
// 4 consecutive 32-bit columns of this thread's TMEM lane (lane quadrant = warp % 4)
__device__ __forceinline__ void tmem_st4(uint32_t taddr, uint4 v) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

__device__ __forceinline__ uint32_t pick_half(uint32_t word, uint32_t pick) { return __byte_perm(word, 0u, pick); }

struct UmmaArgs {
  const uint32_t *codes;        // codes4 [RB][NW][8][128]: selector nibbles, 8 sites per word
  const uint64_t *mask;         // [RB][NW][128] presence bits (count pass)
  const uint32_t *pairs;        // [n_pairs][2] tile positions of a unit (second 0xFFFFFFFF: single tile)
  const uint8_t *wsite;         // [n_layers][NW * 64]
  const uint32_t *word_ids, *word_layer;
  const ngsd_tile *tiles;
  const uint32_t *split_begin;
  uint32_t *sched;
  int32_t *partials;            // [n_units][pstride], sum tile row-major [128][128]
  uint64_t NW;
  uint32_t n_tiles, n_pairs, n_units, pstride;   // n_units = splits x n_pairs
  uint32_t cnt_off;             // count pass: offset of the count tile inside a unit's slot (ints)
  uint32_t rowk[3];             // B table: byte c of rowk[k] = (S / m) f(k, c)
  uint32_t tA[3];               // A table for unit weights: byte c of tA[k] = m [c = k] + t [c = 3]
  uint32_t t3, amul;            // weighted A: selector table of the missing code (0xFF000000 or 0), m
};

enum : uint32_t { kFirst = 1u, kLast = 2u, kPair = 4u, kExit = 8u, kUnitW = 16u, kEntriesShift = 8u };   // count pass: entries of the stage in bits 8..10

// Expansion of one 64-site stage of the sum pass by thread (row r, site quads qb .. qb + kGroups - 1 of each of the 4 code
// words): A row -> tensor memory, B rows -> shared memory.  The K order inside a stage is free as long as both operands use
// it: the 4 codes of a site quad arrive as the 4 selector nibbles of one 16-bit half word (codes4, spread once by the front
// end), and PRMT(T_k, sel) picks byte c_j of the table T_k for site j -- one instruction builds plane k of 4 sites, no table
// loads.  Word n = 3 i + k of site quad q0 (sites 16 i + 4 q0 .. + 3, plane k) is K word 12 q0 + n of the row in BOTH
// operands.  The code words are read into registers first and the raw stage is handed back to the producer BEFORE the wait
// for a free expanded stage, so the next codes travel while this stage is built.
template <bool UNITW>
__device__ __forceinline__ void expand_stage(const unsigned char *rawS, int r, int qb, int lane, bool paired, unsigned char *eB, uint32_t ta,
                                             const UmmaArgs &a, uint64_t *raw_empty_bar, uint64_t *exp_empty_bar, uint32_t exp_parity) {
  constexpr int kWG = kGroups >= 2 ? kGroups / 2 : 1;               // nibble words per 16 sites this thread reads (two site quads each)
  const uint32_t *cw = reinterpret_cast<const uint32_t *>(rawS) + r;
  uint32_t wa[kWG][4], wb[kWG][4], wc[kWG][4], wt[kGroups][4];
#pragma unroll
  for (int g = 0; g < kWG; g++) {
    const int w0 = ((qb >> 1) + g) * 128;
#pragma unroll
    for (int i = 0; i < 4; i++) {
      wa[g][i] = cw[i * 256 + w0];
      wb[g][i] = cw[kCodeBytes / 4 + i * 256 + w0];
      wc[g][i] = paired ? cw[2 * (kCodeBytes / 4) + i * 256 + w0] : 0u;
    }
  }
  if (!UNITW) {
    const uint32_t *W32 = reinterpret_cast<const uint32_t *>(rawS + 3 * kCodeBytes);
#pragma unroll
    for (int q = 0; q < kGroups; q++)
#pragma unroll
      for (int i = 0; i < 4; i++) wt[q][i] = W32[4 * i + qb + q];
  }
  __syncwarp();
  if (lane == 0) mbar_arrive(raw_empty_bar);                        // (release: orders the warp's reads above before the arrival)
  mbar_wait(exp_empty_bar, exp_parity);
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
  for (int q = 0; q < kGroups; q++) {
    const int q0 = qb + q, g = kGroups >= 2 ? q >> 1 : 0;
    const uint32_t pick = (q0 & 1) ? 0x4432u : 0x4410u;             // site quad 4 i + q0 = half (q0 & 1) of nibble word 2 i + (q0 >> 1)
    uint32_t va[12], vb[12];
#pragma unroll
    for (int i = 0; i < 4; i++) {
      const uint32_t sx = pick_half(wa[g][i], pick), sy = pick_half(wb[g][i], pick);
      if (UNITW) {
#pragma unroll
        for (int k = 0; k < 3; k++) va[3 * i + k] = __byte_perm(a.tA[k], 0u, sx);
      } else {
        const uint32_t ww = wt[q][i], wm = ww * a.amul, m3 = __byte_perm(a.t3, 0u, sx) & ww;   // weight bytes <= 42 when amul = 3
#pragma unroll
        for (int k = 0; k < 3; k++) va[3 * i + k] = (__byte_perm(0xFFu << (8 * k), 0u, sx) & wm) | m3;
      }
#pragma unroll
      for (int k = 0; k < 3; k++) vb[3 * i + k] = __byte_perm(a.rowk[k], 0u, sy);
    }
    unsigned char *eq = eB + (uint32_t) (3 * q0) * kBChunk;
#pragma unroll
    for (int m = 0; m < 3; m++) {
      tmem_st4(ta + 12u * q0 + 4u * m, make_uint4(va[4 * m], va[4 * m + 1], va[4 * m + 2], va[4 * m + 3]));
      *reinterpret_cast<uint4 *>(eq + m * kBChunk) = make_uint4(vb[4 * m], vb[4 * m + 1], vb[4 * m + 2], vb[4 * m + 3]);
    }
    if (paired) {                                                   // second tile's rows: row groups 16..31 of B
#pragma unroll
      for (int i = 0; i < 4; i++) {
        const uint32_t sz = pick_half(wc[g][i], pick);
#pragma unroll
        for (int k = 0; k < 3; k++) vb[3 * i + k] = __byte_perm(a.rowk[k], 0u, sz);
      }
#pragma unroll
      for (int m = 0; m < 3; m++)
        *reinterpret_cast<uint4 *>(eq + m * kBChunk + 2048) = make_uint4(vb[4 * m], vb[4 * m + 1], vb[4 * m + 2], vb[4 * m + 3]);
    }
  }
}

// COUNT = true: the same pipeline computes the shared-site counts of --pairwise_del, cnt(i,j) = sum_s w_s m_i(s) m_j(s), as an
// int8 GEMM with ONE byte per site (A' = w_s m_i(s), B' = m_j(s) from the presence masks) and writes them as the second
// tile of the unit's slot.  A stage then holds up to kCntGroup = 3 word-list entries (192 sites), so that it is the same
// 192 K bytes, 6 MMAs and operand layout as a stage of the sum pass.
template <bool COUNT>
__global__ void __launch_bounds__(kThreads, 1) k_dist_umma(const __grid_constant__ UmmaArgs a) {
  constexpr int kOffW = 3 * kCodeBytes;                              // sum pass: weights behind the three code tiles
  constexpr int kRawStage = COUNT ? kCntRawBytes : kRawBytes;        // (both passes use the kRaw slots of the ring)
  extern __shared__ __align__(1024) unsigned char smem[];
  unsigned char *raw = smem;                                         // kRaw x kRawBytes
  unsigned char *exps = smem + (size_t) kRingBytes;                  // kExp x kExpBytes (16-byte aligned: the ring is a multiple of 128)
  uint64_t *bars = reinterpret_cast<uint64_t *>(exps + (size_t) kExp * kExpBytes);
  uint64_t *raw_full = bars, *raw_empty = raw_full + kRaw, *exp_full = raw_empty + kRaw, *exp_empty = exp_full + kExp;
  uint64_t *acc_full = exp_empty + kExp, *acc_empty = acc_full + 2;
  uint32_t *raw_meta = reinterpret_cast<uint32_t *>(bars + kNBar);    // [kRaw][2] = {unit, flags}
  uint32_t *exp_meta = raw_meta + 2 * kRaw;                           // [kExp][2]
  uint32_t *acc_meta = exp_meta + 2 * kExp;                           // {unit, flags} of the finished accumulator (+ 2 spare words)
  uint32_t *tmem_slot = acc_meta + 4;
  uint32_t *lut16 = tmem_slot + 4;                                    // [16] presence nibble -> 0x01 bytes (count pass)

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < kRaw; s++) { mbar_init(&raw_full[s], 1); mbar_init(&raw_empty[s], kGroupWarps); }
    for (int s = 0; s < kExp; s++) { mbar_init(&exp_full[s], kGroupWarps); mbar_init(&exp_empty[s], 1); }
    for (int s = 0; s < 2; s++) { mbar_init(&acc_full[s], 2); mbar_init(&acc_empty[s], kEpiWarps); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (COUNT && threadIdx.x >= 32 && threadIdx.x < 48) {
    const uint32_t n = threadIdx.x - 32;
    lut16[n] = (n & 1u) | ((n & 2u) << 7) | ((n & 4u) << 14) | ((n & 8u) << 21);
  }
  if (warp == 1) {                                  // TMEM: accumulator + kExp stages of A (one CTA per SM)
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = *tmem_slot;

  if (warp == 0) {
    // ===== producer =====
    if (lane == 0) {
      int rs = 0;
      uint32_t rph = 0;
      for (;;) {
        const uint32_t u = atomicAdd(a.sched, 1u);
        if (u >= a.n_units) break;
        const uint32_t q = u / a.n_pairs, p = u - q * a.n_pairs;
        const uint32_t t0 = a.pairs[2 * p], t1 = a.pairs[2 * p + 1];
        const bool paired = t1 != 0xFFFFFFFFu;
        const ngsd_tile tl = a.tiles[t0];
        const uint32_t tj1 = paired ? a.tiles[t1].tj : tl.tj;
        const uint32_t c0 = a.split_begin[q], c1 = a.split_begin[q + 1];
        const uint32_t *Ab = a.codes + (uint64_t) tl.ti * a.NW * 1024;     // codes4: 1024 words per (row block, 64-site word)
        const uint32_t *Bb = a.codes + (uint64_t) tl.tj * a.NW * 1024;
        const uint32_t *B1b = a.codes + (uint64_t) tj1 * a.NW * 1024;
        if (COUNT) {
          for (uint32_t c = c0; c < c1; c += kCntGroup) {
            const uint32_t ne = min((uint32_t) kCntGroup, c1 - c);
            uint32_t words[kCntGroup], layers[kCntGroup], unitw = 1u;
            for (uint32_t e = 0; e < ne; e++) { words[e] = a.word_ids[c + e]; layers[e] = a.word_layer[c + e]; unitw &= layers[e] >> 31; }
            mbar_wait(&raw_empty[rs], rph ^ 1);
            raw_meta[rs * 2] = u;
            raw_meta[rs * 2 + 1] = (c == c0 ? kFirst : 0u) | (c + kCntGroup >= c1 ? kLast : 0u) | (paired ? kPair : 0u) | (unitw ? kUnitW : 0u) | (ne << kEntriesShift);
            mbar_expect_tx(&raw_full[rs], ne * ((paired ? 3 : 2) * kMaskBytes + 64));
            unsigned char *dst = raw + (size_t) rs * kRawStage;
            for (uint32_t e = 0; e < ne; e++) {
              const uint64_t word = words[e];
              unsigned char *de = dst + e * kCntEntry;
              bulk_g2s(de, a.mask + ((uint64_t) tl.ti * a.NW + word) * 128, kMaskBytes, &raw_full[rs]);
              bulk_g2s(de + kMaskBytes, a.mask + ((uint64_t) tl.tj * a.NW + word) * 128, kMaskBytes, &raw_full[rs]);
              if (paired) bulk_g2s(de + 2 * kMaskBytes, a.mask + ((uint64_t) tj1 * a.NW + word) * 128, kMaskBytes, &raw_full[rs]);
              bulk_g2s(dst + kCntGroup * kCntEntry + e * 64, a.wsite + ((uint64_t) (layers[e] & 0x7FFFFFFFu) * a.NW + word) * 64, 64, &raw_full[rs]);
            }
            if (++rs == kRaw) { rs = 0; rph ^= 1; }
          }
          continue;
        }
        uint32_t nword = a.word_ids[c0], nlayer = a.word_layer[c0];
        for (uint32_t c = c0; c < c1; c++) {
          const uint64_t word = nword;
          const uint32_t unitw = nlayer >> 31;                      // api.cu: bit 31 = all 64 site weights of this word are 1
          const uint8_t *wsrc = a.wsite + ((uint64_t) (nlayer & 0x7FFFFFFFu) * a.NW + word) * 64;
          if (c + 1 < c1) { nword = a.word_ids[c + 1]; nlayer = a.word_layer[c + 1]; }   // next entry's loads fly during the wait below
          mbar_wait(&raw_empty[rs], rph ^ 1);
          raw_meta[rs * 2] = u;
          raw_meta[rs * 2 + 1] = (c == c0 ? kFirst : 0u) | (c + 1 == c1 ? kLast : 0u) | (paired ? kPair : 0u) | (unitw ? kUnitW : 0u);
          mbar_expect_tx(&raw_full[rs], (paired ? 3 : 2) * kCodeBytes + 64);
          unsigned char *dst = raw + (size_t) rs * kRawStage;
          bulk_g2s(dst, Ab + word * 1024, kCodeBytes, &raw_full[rs]);
          bulk_g2s(dst + kCodeBytes, Bb + word * 1024, kCodeBytes, &raw_full[rs]);
          if (paired) bulk_g2s(dst + 2 * kCodeBytes, B1b + word * 1024, kCodeBytes, &raw_full[rs]);
          bulk_g2s(dst + kOffW, wsrc, 64, &raw_full[rs]);
          if (++rs == kRaw) { rs = 0; rph ^= 1; }
        }
      }
      for (int g = 0; g < kGroups; g++) {                             // one exit stage per expander group
        mbar_wait_sleep(&raw_empty[rs], rph ^ 1);
        raw_meta[rs * 2 + 1] = kExit;
        mbar_arrive(&raw_full[rs]);
        if (++rs == kRaw) { rs = 0; rph ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issue (one lane) =====
    if (lane == 0) {
      // D = S32 (2 << 4), A = B = INT8 (1 << 7, 1 << 10), both K-major, N (>> 3 at [17,23)), M = 128 (>> 4 at [24,29))
      const uint32_t idesc1 = (2u << 4) | (1u << 7) | (1u << 10) | ((128u >> 3) << 17) | ((128u >> 4) << 24);
      const uint32_t idesc2 = (2u << 4) | (1u << 7) | (1u << 10) | ((256u >> 3) << 17) | ((128u >> 4) << 24);
      int es = 0;
      uint32_t eph = 0, aph = 0;
      for (;;) {
        mbar_wait(&exp_full[es], eph);
        const uint32_t u = exp_meta[es * 2], fl = exp_meta[es * 2 + 1];
        if (fl & kExit) {                                            // (the first exit stage in stage order; the other groups' are never read)
          mbar_wait(&acc_empty[0], aph ^ 1);
          acc_meta[1] = kExit;
          mbar_arrive(&acc_full[0]);
          mbar_arrive(&acc_full[0]);
          break;
        }
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        if (fl & kFirst) {
          mbar_wait(&acc_empty[0], aph ^ 1);                         // the epilogue has drained the accumulator
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        }
        const uint32_t sb = smem_u32(exps + (size_t) es * kExpBytes);
        const uint32_t ta = tmem + kAccCols + (uint32_t) es * kACols;
        const uint32_t idesc = (fl & kPair) ? idesc2 : idesc1;
        const int n_mma = COUNT ? 2 * (int) ((fl >> kEntriesShift) & 7u) : kMmas;   // count pass: 2 per word-list entry of the stage
#pragma unroll
        for (int j = 0; j < kMmas; j++) {                           // K 32 per instruction: 8 TMEM columns of A, two 16-byte chunks of B (4 KiB apart)
          if (j < n_mma) {
            const uint64_t db = umma_desc(sb + j * 2 * kBChunk, kBChunk, 128);
            umma_i8_ts(tmem, ta + 8u * j, db, idesc, ((fl & kFirst) && j == 0) ? 0u : 1u);
          }
        }
        umma_commit(&exp_empty[es]);                                 // stage (B in shared memory, A in TMEM) reusable once these MMAs have read it
        if (fl & kLast) {
          acc_meta[0] = u;
          acc_meta[1] = fl & kPair;
          umma_commit(&acc_full[0]);                                 // accumulator complete ...
          mbar_arrive(&acc_full[0]);                                 // ... and its meta word published
          aph ^= 1;
        }
        if (++es == kExp) { es = 0; eph ^= 1; }
      }
    }
  } else if (warp < 2 + kExpWarps) {
    // ===== expanders: group grp takes stages grp, grp + kGroups, ...; thread -> (row r, site quads qb .. qb + kGroups - 1 of each word) =====
    // (a warp reaches the TMEM lanes of its quadrant warp % 4 only: that fixes which rows it expands)
    const int r = (warp & 3) * 32 + lane;
    const int grp = (warp - 2) / kGroupWarps, qb = (((warp - 2) % kGroupWarps) >> 2) * kGroups;
    const bool lead = (warp - 2) % kGroupWarps == 0 && lane == 0;
    const uint32_t ta_lane = tmem + ((uint32_t) ((warp & 3) * 32) << 16) + kAccCols;
    const uint32_t unit_off = (uint32_t) (r >> 3) * 128 + (uint32_t) (r & 7) * 16;
    for (uint32_t n = (uint32_t) grp;; n += kGroups) {              // stage n: raw slot n % kRaw, expanded slot n % kExp
      const int rs = (int) (n % kRaw), es = (int) (n % kExp);
      const uint32_t rph = (n / kRaw) & 1u, eph = (n / kExp) & 1u;
      mbar_wait(&raw_full[rs], rph);
      const uint32_t u = raw_meta[rs * 2], fl = raw_meta[rs * 2 + 1];
      if (fl & kExit) {
        mbar_wait(&exp_empty[es], eph ^ 1);
        if (lead) exp_meta[es * 2 + 1] = kExit;
        __syncwarp();
        if (lane == 0) mbar_arrive(&exp_full[es]);
        break;
      }
      const unsigned char *rawS = raw + (size_t) rs * kRawStage;
      if (COUNT) {
        // one byte per site: for each word-list entry e of the stage, thread (r, q0) expands the 16 presence bits
        // 16 q0 .. 16 q0 + 15 of its row of each operand into one 16-byte unit (K chunk 4 e + q0); A bytes carry the site weights
        mbar_wait(&exp_empty[es], eph ^ 1);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t ne = (fl >> kEntriesShift) & 7u;
        for (uint32_t eq = 0; eq < ne * kGroups; eq++) {
          const uint32_t e = eq / kGroups;
          const int q0 = qb + (int) (eq % kGroups);
          const unsigned char *re = rawS + e * kCntEntry;
          const uint32_t ma = reinterpret_cast<const uint32_t *>(re)[r * 2 + (q0 >> 1)] >> (16 * (q0 & 1));
          const uint32_t mb = reinterpret_cast<const uint32_t *>(re + kMaskBytes)[r * 2 + (q0 >> 1)] >> (16 * (q0 & 1));
          uint4 va, vb;
          va.x = lut16[ma & 15u];
          va.y = lut16[(ma >> 4) & 15u];
          va.z = lut16[(ma >> 8) & 15u];
          va.w = lut16[(ma >> 12) & 15u];
          if (!(fl & kUnitW)) {
            const uint4 ww = *reinterpret_cast<const uint4 *>(rawS + kCntGroup * kCntEntry + e * 64 + 16 * q0);
            va.x = (va.x * 0xFFu) & ww.x;
            va.y = (va.y * 0xFFu) & ww.y;
            va.z = (va.z * 0xFFu) & ww.z;
            va.w = (va.w * 0xFFu) & ww.w;
          }
          vb.x = lut16[mb & 15u];
          vb.y = lut16[(mb >> 4) & 15u];
          vb.z = lut16[(mb >> 8) & 15u];
          vb.w = lut16[(mb >> 12) & 15u];
          unsigned char *eB = exps + (size_t) es * kExpBytes + unit_off + (4u * e + (uint32_t) q0) * kBChunk;
          tmem_st4(ta_lane + (uint32_t) es * kACols + 16u * e + 4u * q0, va);
          *reinterpret_cast<uint4 *>(eB) = vb;
          if (fl & kPair) {
            const uint32_t mb1 = reinterpret_cast<const uint32_t *>(re + 2 * kMaskBytes)[r * 2 + (q0 >> 1)] >> (16 * (q0 & 1));
            vb.x = lut16[mb1 & 15u];
            vb.y = lut16[(mb1 >> 4) & 15u];
            vb.z = lut16[(mb1 >> 8) & 15u];
            vb.w = lut16[(mb1 >> 12) & 15u];
            *reinterpret_cast<uint4 *>(eB + 2048) = vb;
          }
        }
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        if (lead) { exp_meta[es * 2] = u; exp_meta[es * 2 + 1] = fl; }
        __syncwarp();
        if (lane == 0) { mbar_arrive(&exp_full[es]); mbar_arrive(&raw_empty[rs]); }
        continue;
      }
      unsigned char *eB = exps + (size_t) es * kExpBytes + unit_off;
      const uint32_t ta = ta_lane + (uint32_t) es * kACols;
      const bool paired = (fl & kPair) != 0;
      if (fl & kUnitW)
        expand_stage<true>(rawS, r, qb, lane, paired, eB, ta, a, &raw_empty[rs], &exp_empty[es], eph ^ 1);
      else
        expand_stage<false>(rawS, r, qb, lane, paired, eB, ta, a, &raw_empty[rs], &exp_empty[es], eph ^ 1);
      asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");   // A rows are in tensor memory
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy stores -> visible to the UMMA (async) proxy
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      if (lead) { exp_meta[es * 2] = u; exp_meta[es * 2 + 1] = fl; }
      __syncwarp();
      if (lane == 0) mbar_arrive(&exp_full[es]);
    }
  } else {
    // ===== epilogue: a warp can read the 32 TMEM lanes (= tile rows) of its quadrant warp % 4 =====
    const int qd = warp & 3;
    uint32_t aph = 0;
    for (;;) {
      mbar_wait_sleep(&acc_full[0], aph);                          // (idle for a whole unit: do not compete for issue slots)
      const uint32_t u = acc_meta[0], fl = acc_meta[1];
      if (fl & kExit) break;
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t q = u / a.n_pairs, p = u - q * a.n_pairs;
      const int ncol = (fl & kPair) ? 256 : 128;
#pragma unroll 1
      for (int c0 = 0; c0 < ncol; c0 += 32) {
        const uint32_t t = a.pairs[2 * p + (c0 >> 7)];
        int4 *dst = reinterpret_cast<int4 *>(a.partials + ((uint64_t) q * a.n_tiles + t) * a.pstride + (COUNT ? a.cnt_off : 0u) +
                                             (uint64_t) (qd * 32 + lane) * 128);
        uint32_t v[32];
        const uint32_t taddr = tmem + ((uint32_t) (qd * 32) << 16) + (uint32_t) c0;
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
            : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]),
              "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]),
              "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]),
              "=r"(v[31])
            : "r"(taddr));
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int k = 0; k < 8; k++) dst[(c0 & 127) / 4 + k] = make_int4((int) v[4 * k], (int) v[4 * k + 1], (int) v[4 * k + 2], (int) v[4 * k + 3]);
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty[0]);
      aph ^= 1;
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u) : "memory");
}

// register / smem-resident UMMA loop: the int8 tensor issue-rate ceiling through tcgen05 (roofline denominator of K2c)
__global__ void __launch_bounds__(128, 1) k_umma_peak(int iters) {
  __shared__ __align__(128) unsigned char sA[2 * 16 * 128];
  __shared__ __align__(128) unsigned char sB[2 * 16 * 128];
  __shared__ __align__(8) uint64_t bar;
  __shared__ uint32_t slot;
  const int warp = threadIdx.x >> 5;
  for (int e = threadIdx.x; e < 4096; e += 128) { sA[e] = (unsigned char) (e * 7); sB[e] = (unsigned char) (e * 13); }
  if (threadIdx.x == 0) {
    mbar_init(&bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&slot)), "r"(128u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = slot;
  if (threadIdx.x == 0) {
    const uint64_t da = umma_desc(smem_u32(sA), 2048, 128), db = umma_desc(smem_u32(sB), 2048, 128);
    const uint32_t idesc = (2u << 4) | (1u << 7) | (1u << 10) | ((128u >> 3) << 17) | ((128u >> 4) << 24);
    for (int it = 0; it < iters; it++) umma_i8(tmem, da, db, idesc, it ? 1u : 0u);
    umma_commit(&bar);
  }
  mbar_wait(&bar, 0);
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(128u) : "memory");
}

// register-only loop of the older warp-level int8 MMA (mma.sync, SASS IMMA.16832): its issue-rate ceiling, for comparison
__device__ __forceinline__ void imma16832(int (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k32.row.col.s32.s8.s8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+r"(c[0]), "+r"(c[1]), "+r"(c[2]), "+r"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

__global__ void k_imma_peak(int *out, int iters) {
  int c[8][4];
#pragma unroll
  for (int i = 0; i < 8; i++) c[i][0] = c[i][1] = c[i][2] = c[i][3] = 0;
  const uint32_t a[4] = {threadIdx.x, threadIdx.x * 3u, 7u, 9u};
  const uint32_t b0 = threadIdx.x + 1u, b1 = 5u;
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int i = 0; i < 8; i++) imma16832(c[i], a, b0, b1);
  }
  int s = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) s += c[i][0] + c[i][1] + c[i][2] + c[i][3];
  if (s == 0x12345678) out[0] = s;
}

}  // namespace

extern "C" int ngsd_probe_umma_tmacs(int device, double *umma_tmacs) {
  if (cudaSetDevice(device) != cudaSuccess) return NGSD_ERR_CUDA;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return NGSD_ERR_CUDA;
  const int iters = 1 << 15, nsm = prop.multiProcessorCount;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  float best = 1e30f;
  for (int r = 0; r < 4; r++) {
    cudaEventRecord(e0);
    k_umma_peak<<<nsm, 128>>>(iters);
    cudaEventRecord(e1);
    if (cudaEventSynchronize(e1) != cudaSuccess) return NGSD_ERR_CUDA;
    float ms;
    cudaEventElapsedTime(&ms, e0, e1);
    if (r > 0 && ms < best) best = ms;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  *umma_tmacs = (double) nsm * iters * (128.0 * 128 * 32) / (best * 1e-3) * 1e-12;
  return NGSD_OK;
}

extern "C" int ngsd_probe_int8_tmacs(int device, double *imma_tmacs) {
  if (cudaSetDevice(device) != cudaSuccess) return NGSD_ERR_CUDA;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return NGSD_ERR_CUDA;
  int *d = nullptr;
  if (cudaMalloc(&d, 64) != cudaSuccess) return NGSD_ERR_CUDA;
  const int iters = 8192, warps = 16, nsm = prop.multiProcessorCount;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  float best = 1e30f;
  for (int r = 0; r < 4; r++) {
    cudaEventRecord(e0);
    k_imma_peak<<<nsm, warps * 32>>>(d, iters);
    cudaEventRecord(e1);
    if (cudaEventSynchronize(e1) != cudaSuccess) { cudaFree(d); return NGSD_ERR_CUDA; }
    float ms;
    cudaEventElapsedTime(&ms, e0, e1);
    if (r > 0 && ms < best) best = ms;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(d);
  *imma_tmacs = (double) nsm * warps * iters * 8 * 4096.0 / (best * 1e-3) * 1e-12;
  return NGSD_OK;
}

// f(k, c) * S as int8 bytes; returns false when S * score is not a matrix of exact small integers (-> FP64 path).
// Only then is acc / S the reference's sum: a score that is merely close to k / S (1e-12 x the default, or 0.5 + 3e-11)
// must not be rounded onto the integer grid.  The missing-genotype entries (the uniform triple) are built from those
// integers: S f(k, 3) = sum_c R[k][c] / 3, S f(3, c) = sum_k R[k][c] / 3, S f(3, 3) = sum R / 9, each an exact quotient.
bool ngsd_int_lut(const double *score, bool pairwise_del, uint32_t lut[4], double *scale, int *max_byte) {
  const double S = pairwise_del ? 2.0 : 18.0;
  long long R[4][4] = {};
  for (int k = 0; k < 3; k++)
    for (int c = 0; c < 3; c++) {
      const double v = score[k * 3 + c], r = nearbyint(v * S);
      if (!(fabs(r) <= 127) || fma(v, S, -r) != 0.0) return false;   // NaN, out of range, or S v not exactly the integer r
      R[k][c] = (long long) r;
    }
  if (!pairwise_del) {
    long long tot = 0;
    for (int k = 0; k < 3; k++) {
      const long long rs = R[k][0] + R[k][1] + R[k][2], cs = R[0][k] + R[1][k] + R[2][k];
      if (rs % 3 || cs % 3) return false;
      R[k][3] = rs / 3;
      R[3][k] = cs / 3;
      tot += rs;
    }
    if (tot % 9) return false;
    R[3][3] = tot / 9;
  }
  int mx = 0;
  for (int c = 0; c < 4; c++) {
    uint32_t wv = 0;
    for (int k = 0; k < 4; k++) {
      const long long r = R[k][c];
      if (r < 0 || r > 127) return false;
      if (!pairwise_del && k < 3 && r % 3) return false;   // the three-plane form (header) carries S / 3 on the B side
      wv |= (uint32_t) r << (8 * k);
      if ((int) r > mx) mx = (int) r;
    }
    lut[c] = wv;
  }
  *scale = S;
  *max_byte = mx;
  return true;
}

// largest site weight one weight layer may carry: the A bytes are int8 and hold 3 w without --pairwise_del (header)
uint32_t ngsd_int_weight_cap(const ngsd_ctx *ctx) { return ctx->cfg.pairwise_del ? 127u : 42u; }

cudaError_t ngsd_launch_dist_umma(ngsd_ctx *ctx, uint32_t n_units, int grid, uint32_t pstride, bool count) {
  static bool attr_set[64] = {};
  if (!attr_set[ctx->device & 63]) {
    const void *fns[2] = {(const void *) k_dist_umma<false>, (const void *) k_dist_umma<true>};
    for (const void *f : fns) {
      cudaError_t e = cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) kSmemBytes);
      if (e != cudaSuccess) return e;
    }
    attr_set[ctx->device & 63] = true;
  }
  UmmaArgs a;
  a.codes = ctx->codes4;
  a.mask = ctx->mask;
  a.wsite = ctx->d_wsite;
  a.word_ids = ctx->d_word_ids;
  a.word_layer = ctx->d_word_layer;
  a.tiles = ctx->d_tiles;
  a.split_begin = ctx->d_split_begin;
  a.sched = ctx->d_sched;
  a.partials = reinterpret_cast<int32_t *>(ctx->cur_partials);
  a.NW = ctx->NW;
  a.n_tiles = ctx->n_tiles;
  a.n_pairs = ctx->n_pairs;
  a.pairs = ctx->d_pairs;
  a.n_units = ctx->n_tiles ? n_units / ctx->n_tiles * ctx->n_pairs : 0;     // (split, tile) units -> (split, tile pair) units
  a.pstride = pstride;
  a.cnt_off = NGSD_TILE_ELEMS;
  // ctx->int_lut[c] byte k = S f(k, c) (ngsd_int_lut); the three-plane tables of the header
  const bool third = !ctx->cfg.pairwise_del;                                // missing = the uniform triple
  a.amul = third ? 3u : 1u;
  a.t3 = third ? 0xFF000000u : 0u;
  for (int k = 0; k < 3; k++) {
    a.tA[k] = (a.amul << (8 * k)) | (third ? 0x01000000u : 0u);
    a.rowk[k] = 0;
    for (int c = 0; c < 4; c++) a.rowk[k] |= (((ctx->int_lut[c] >> (8 * k)) & 0xFFu) / a.amul) << (8 * c);
  }
  cudaError_t e = cudaMemsetAsync(ctx->d_sched, 0, sizeof(uint32_t), ctx->stream);
  if (e != cudaSuccess) return e;
  if (count)
    k_dist_umma<true><<<grid, kThreads, kSmemBytes, ctx->stream>>>(a);
  else
    k_dist_umma<false><<<grid, kThreads, kSmemBytes, ctx->stream>>>(a);
  return cudaGetLastError();
}

namespace {

// shared-site counts of the FP64 path: K splits of the int8 count GEMM -> cnt [n_pad][n_pad]
// grid (n_tiles, 16), block 256: one thread per int4 of the 128 x 128 tile
__global__ void __launch_bounds__(256) k_cnt_reduce(const int32_t *__restrict__ partials, uint32_t n_splits, uint32_t n_tiles,
                                                    const ngsd_tile *__restrict__ tiles, uint32_t *__restrict__ cnt, uint64_t n_pad) {
  const uint32_t t = blockIdx.x, e = blockIdx.y * 256 + threadIdx.x;
  const ngsd_tile tl = tiles[t];
  const int4 *src = reinterpret_cast<const int4 *>(partials + (uint64_t) t * NGSD_TILE_ELEMS) + e;
  const uint64_t stride = (uint64_t) n_tiles * (NGSD_TILE_ELEMS / 4);
  int4 s = make_int4(0, 0, 0, 0);
  for (uint32_t q = 0; q < n_splits; q++) {
    const int4 v = src[(uint64_t) q * stride];
    s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
  }
  const uint32_t row = e >> 5, col0 = (e & 31u) * 4u;
  *reinterpret_cast<uint4 *>(cnt + ((uint64_t) tl.ti * NGSD_TILE + row) * n_pad + (uint64_t) tl.tj * NGSD_TILE + col0) =
      make_uint4((uint32_t) s.x, (uint32_t) s.y, (uint32_t) s.z, (uint32_t) s.w);
}

}  // namespace

// --pairwise_del counts of the FP64 path on the int8 tensor cores: cnt(i,j) = sum_s w_s m_i(s) m_j(s) from the presence
// masks (k_dist_umma<true>, one byte per site), K splits reduced into ctx->d_cnt.  Replaces the AND+POPC kernel
// (mask_count.cu) on the per-replicate path: 7x faster alone, and it does not have to share SMs with the contraction.
cudaError_t ngsd_launch_count_umma(ngsd_ctx *ctx, const ngsd_count_umma_args &c) {
  static bool attr_set[64] = {};
  if (!attr_set[ctx->device & 63]) {
    cudaError_t e = cudaFuncSetAttribute((const void *) k_dist_umma<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) kSmemBytes);
    if (e != cudaSuccess) return e;
    attr_set[ctx->device & 63] = true;
  }
  UmmaArgs a;
  a.codes = nullptr;
  a.mask = ctx->mask;
  a.wsite = c.wsite;
  a.word_ids = c.word_ids;
  a.word_layer = c.word_layer;
  a.tiles = ctx->d_tiles;
  a.split_begin = c.split_begin;
  a.sched = ctx->d_sched;
  a.partials = c.partials;
  a.NW = ctx->NW;
  a.n_tiles = ctx->n_tiles;
  a.n_pairs = ctx->n_pairs;
  a.pairs = ctx->d_pairs;
  a.n_units = c.n_splits * ctx->n_pairs;
  a.pstride = NGSD_TILE_ELEMS;
  a.cnt_off = 0;
  for (int k = 0; k < 3; k++) a.rowk[k] = a.tA[k] = 0;
  a.t3 = 0;
  a.amul = 1;
  cudaError_t e = cudaMemsetAsync(ctx->d_sched, 0, sizeof(uint32_t), ctx->stream);
  if (e != cudaSuccess) return e;
  const int grid = (int) std::min<uint64_t>((uint64_t) ctx->n_sm, std::max<uint32_t>(a.n_units, 1u));
  k_dist_umma<true><<<grid, kThreads, kSmemBytes, ctx->stream>>>(a);
  e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  k_cnt_reduce<<<dim3(ctx->n_tiles, 16), 256, 0, ctx->stream>>>(c.partials, c.n_splits, ctx->n_tiles, ctx->d_tiles, ctx->d_cnt, ctx->n_pad);
  return cudaGetLastError();
}
