// tcgen05.mma kind::i8 (SASS UTCIMMA) probe on sm_100a: one 128 x N x 32 int8 MMA per instruction, operands in shared
// memory (K-major, no swizzle: 8-row x 16-byte core matrices), int32 accumulators in TMEM.
//   1. correctness of the descriptor / layout conventions against a CPU product on random int8 data;
//   2. issue rate of back-to-back accumulating MMAs (one CTA per SM) -> int8 tensor peak through the UMMA path,
//      to compare with the 570 TMAC/s of mma.sync IMMA.16832 that the first K2c kernel (k_dist_imma, mma.sync; since removed) ran on.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o tools/probe_utcimma tools/probe_utcimma.cu
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <vector>
#include <cuda_runtime.h>

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); return 1; } } while (0)

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t) __cvta_generic_to_shared(p); }

// K-major, SWIZZLE_NONE shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start >> 4 in [0,14), leading
// (K-direction) byte offset >> 4 in [16,30), stride (M/N-direction, 8-row groups) byte offset >> 4 in [32,46),
// version 1 in [46,48), layout type 0 in [61,64).
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t) ((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t) ((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t) ((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t) 1 << 46;
  return d;
}

template <int N>
__global__ void __launch_bounds__(128, 1) k_probe(const int8_t *A /*[128][32]*/, const int8_t *B /*[N][32]*/, int *D /*[128][N]*/, int iters,
                                                  int check) {
  // operand tiles: [k-chunk 0..1][row group][8 rows][16 bytes]
  __shared__ __align__(128) unsigned char sA[2 * 16 * 128];
  __shared__ __align__(128) unsigned char sB[2 * (N / 8) * 128];
  __shared__ __align__(8) uint64_t mbar;
  __shared__ uint32_t tmem_base_s;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // fill: element (row r, k) -> chunk k/16, group r/8, row-in-group r%8, byte k%16
  for (int e = tid; e < 128 * 32; e += 128) {
    const int r = e / 32, k = e % 32;
    sA[(k / 16) * (16 * 128) + (r / 8) * 128 + (r % 8) * 16 + (k % 16)] = (unsigned char) A[r * 32 + k];
  }
  for (int e = tid; e < N * 32; e += 128) {
    const int r = e / 32, k = e % 32;
    sB[(k / 16) * ((N / 8) * 128) + (r / 8) * 128 + (r % 8) * 16 + (k % 16)] = (unsigned char) B[r * 32 + k];
  }
  if (tid == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&mbar)));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");    // generic-proxy stores -> visible to the async (UMMA) proxy
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"((uint32_t) (N < 32 ? 32 : N)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = tmem_base_s;

  if (tid == 0) {
    const uint64_t da = make_desc(smem_u32(sA), 16 * 128, 128);
    const uint64_t db = make_desc(smem_u32(sB), (N / 8) * 128, 128);
    // instruction descriptor (cute::UMMA::InstrDescriptor): D = S32 (2 << 4), A = B = INT8 (1 << 7, 1 << 10), K-major both,
    // N >> 3 at [17,23), M >> 4 at [24,29)
    const uint32_t idesc = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t) (N >> 3) << 17) | ((128u >> 4) << 24);
    for (int it = 0; it < iters; it++) {
      const uint32_t acc = it ? 1u : 0u;
      asm volatile(
          "{\n\t"
          ".reg .pred p;\n\t"
          "setp.ne.b32 p, %4, 0;\n\t"
          "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t"
          "}\n" ::"r"(tmem),
          "l"(da), "l"(db), "r"(idesc), "r"(acc), "r"(0u)
          : "memory");
    }
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(&mbar)) : "memory");
  }
  // everyone waits for the MMAs
  {
    uint32_t ok = 0;
    while (!ok) {
      asm volatile(
          "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
          : "=r"(ok)
          : "r"(smem_u32(&mbar)), "r"(0u)
          : "memory");
    }
  }
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  if (check) {
    // warp w owns TMEM lanes 32w..32w+31 (= rows of D); 32 columns per load
    for (int c0 = 0; c0 < N; c0 += 32) {
      uint32_t v[32];
      const uint32_t taddr = tmem + ((uint32_t) (warp * 32) << 16) + (uint32_t) c0;
      asm volatile(
          "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
          : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]),
            "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]),
            "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]),
            "=r"(v[31])
          : "r"(taddr));
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
      for (int k = 0; k < 32; k++) D[(warp * 32 + lane) * N + c0 + k] = (int) v[k];
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"((uint32_t) (N < 32 ? 32 : N)) : "memory");
}

template <int N>
int run(int nsm, int clock_khz) {
  std::vector<int8_t> hA(128 * 32), hB(N * 32);
  srand(7);
  for (auto &x : hA) x = (int8_t) (rand() % 255 - 127);
  for (auto &x : hB) x = (int8_t) (rand() % 255 - 127);
  int8_t *dA, *dB;
  int *dD;
  CK(cudaMalloc(&dA, hA.size()));
  CK(cudaMalloc(&dB, hB.size()));
  CK(cudaMalloc(&dD, 128 * N * 4));
  CK(cudaMemcpy(dA, hA.data(), hA.size(), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dB, hB.data(), hB.size(), cudaMemcpyHostToDevice));
  k_probe<N><<<1, 128>>>(dA, dB, dD, 3, 1);      // 3 accumulating MMAs: D = 3 * A B^T
  CK(cudaDeviceSynchronize());
  std::vector<int> hD(128 * N);
  CK(cudaMemcpy(hD.data(), dD, hD.size() * 4, cudaMemcpyDeviceToHost));
  long bad = 0;
  for (int m = 0; m < 128; m++)
    for (int n = 0; n < N; n++) {
      int s = 0;
      for (int k = 0; k < 32; k++) s += (int) hA[m * 32 + k] * (int) hB[n * 32 + k];
      if (hD[m * N + n] != 3 * s) { if (bad < 5) printf("  mismatch m=%d n=%d got %d want %d\n", m, n, hD[m * N + n], 3 * s); bad++; }
    }
  printf("tcgen05.mma kind::i8 M=128 N=%d K=32: %ld mismatches of %d\n", N, bad, 128 * N);
  if (bad) return 1;
  const int iters = 1 << 16;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  float best = 1e30f;
  for (int r = 0; r < 4; r++) {
    cudaEventRecord(e0);
    k_probe<N><<<nsm, 128>>>(dA, dB, dD, iters, 0);
    cudaEventRecord(e1);
    CK(cudaEventSynchronize(e1));
    float ms;
    cudaEventElapsedTime(&ms, e0, e1);
    if (r && ms < best) best = ms;
  }
  const double macs = (double) nsm * iters * 128.0 * N * 32;
  printf("  rate: %.3f ms for %d MMAs per SM -> %.1f TMAC/s (%.0f MAC/clk/SM at %d MHz)\n", best, iters, macs / best * 1e-9,
         macs / (best * 1e-3) / nsm / (clock_khz * 1e3), clock_khz / 1000);
  cudaFree(dA); cudaFree(dB); cudaFree(dD);
  return 0;
}

int main() {
  cudaDeviceProp p;
  CK(cudaGetDeviceProperties(&p, 0));
  int rc = run<128>(p.multiProcessorCount, p.clockRate);
  if (!rc) rc = run<256>(p.multiProcessorCount, p.clockRate);
  return rc;
}
