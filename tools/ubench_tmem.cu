// ubench_tmem.cu -- can tensor memory feed operand bytes to the SSV row loop next to shared memory?
// One persistent CTA of 16 warps per SM sweeps "rows" the way ssv_rows<32> does: a warp-uniform residue picks a row,
// each lane reads NX consecutive TMEM columns of its own lane with tcgen05.ld.32x32b.xNX and NLDS conflict-free LDS.128
// (row + g*512 + lane*16), and folds the words into one register (LOP3, so the ALU pipe is not the limit).
// Rates are bytes per SM clock from clock64() inside the CTA, so they do not depend on the clock the card runs at.
// Build: nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -o ubench_tmem tools/ubench_tmem.cu
#include <cstdio>
#include <cstdint>
#include <cuda_runtime.h>
#define CHECK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("CUDA error %s at %d\n", cudaGetErrorString(e), __LINE__); return 1; } } while (0)

constexpr int WARPS = 16, KROWS = 30, ROW_BYTES = 4096, TMEM_COLS = 512;

__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}

template <int NX> __device__ __forceinline__ void tmem_ld(uint32_t taddr, uint32_t (&r)[16]) {
  if constexpr (NX == 4)
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(taddr));
  else if constexpr (NX == 8)
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]) : "r"(taddr));
  else if constexpr (NX == 16)
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(taddr));
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// NX TMEM words + NLDS LDS.128 per row; B rows per tcgen05.wait::ld
template <int NX, int NLDS, int B>
__global__ void __launch_bounds__(WARPS * 32, 1) k(unsigned *out, long long *cycles, int iters) {
  extern __shared__ __align__(128) uint8_t smem[];
  __shared__ uint32_t s_taddr;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < KROWS * ROW_BYTES / 4; i += blockDim.x) reinterpret_cast<uint32_t *>(smem)[i] = i * 2654435761u;
  if (NX > 0 && warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(&s_taddr)), "r"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tbase = (NX > 0) ? s_taddr + ((uint32_t)(32 * (warp & 3)) << 16) : 0u;
  const uint32_t lane_off = (uint32_t)__cvta_generic_to_shared(smem) + lane * 16;
  uint32_t acc = tid, st = 12345u + warp;
  long long t0 = 0;
  __syncthreads();
  if (tid == 0) t0 = clock64();
  for (int i = 0; i < iters; ++i) {
    uint32_t r[B][16];
    uint32_t xs[B];
#pragma unroll
    for (int b = 0; b < B; ++b) {
      st = st * 1664525u + 1013904223u;
      xs[b] = ((st >> 16) * KROWS) >> 16;                      // warp-uniform residue 0..29
      if (NX > 0) tmem_ld<NX>(tbase + xs[b] * NX, r[b]);
    }
#pragma unroll
    for (int b = 0; b < B; ++b) {
      const uint32_t row = lane_off + xs[b] * ROW_BYTES;
#pragma unroll
      for (int g = 0; g < NLDS; ++g) {
        const uint4 v = lds128(row + g * 512);
        acc ^= v.x ^ v.y ^ v.z ^ v.w;
      }
    }
    if (NX > 0) {
      tmem_wait_ld();
#pragma unroll
      for (int b = 0; b < B; ++b)
#pragma unroll
        for (int j = 0; j < NX; ++j) { asm volatile("" : "+r"(r[b][j])); acc ^= r[b][j]; }
    }
  }
  __syncthreads();
  if (tid == 0) cycles[blockIdx.x] = clock64() - t0;
  out[blockIdx.x * blockDim.x + tid] = acc;
  if (NX > 0) {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(s_taddr), "r"(TMEM_COLS) : "memory");
  }
}

template <int NX, int NLDS, int B>
int run(const char *name, int grid) {
  static_assert(NX == 0 || KROWS * NX <= TMEM_COLS, "row does not fit the TMEM allocation");
  const size_t smem = (size_t)KROWS * ROW_BYTES;
  const int iters = 20000 / B;
  unsigned *out; long long *cyc;
  CHECK(cudaMalloc(&out, sizeof(unsigned) * grid * WARPS * 32));
  CHECK(cudaMalloc(&cyc, sizeof(long long) * grid));
  CHECK(cudaFuncSetAttribute(k<NX, NLDS, B>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k<NX, NLDS, B><<<grid, WARPS * 32, smem>>>(out, cyc, 100);
  CHECK(cudaDeviceSynchronize());
  cudaEvent_t a, b; cudaEventCreate(&a); cudaEventCreate(&b);
  cudaEventRecord(a);
  k<NX, NLDS, B><<<grid, WARPS * 32, smem>>>(out, cyc, iters);
  cudaEventRecord(b);
  CHECK(cudaDeviceSynchronize());
  float ms; cudaEventElapsedTime(&ms, a, b);
  long long hc[256]; CHECK(cudaMemcpy(hc, cyc, sizeof(long long) * grid, cudaMemcpyDeviceToHost));
  double cmax = 0, csum = 0;
  for (int i = 0; i < grid; ++i) { csum += hc[i]; cmax = hc[i] > cmax ? hc[i] : cmax; }
  const double rows = (double)iters * B * WARPS;                       // warp-rows per SM
  const double tm_bytes = rows * NX * 128, ld_bytes = rows * NLDS * 512;
  const double c = csum / grid;
  printf("%-30s grid=%3d  %8.3f ms  %6.2f clk/warp-row/SM  TMEM %6.1f B/clk/SM  LDS %6.1f B/clk/SM  total %6.1f B/clk/SM  "
         "(%.2f tcgen05.ld + %.2f LDS.128 warp-instr/clk/SM; max/mean cycles %.3f; %.0f MHz effective)\n",
         name, grid, ms, c / rows, tm_bytes / c, ld_bytes / c, (tm_bytes + ld_bytes) / c, rows * (NX > 0) / c, rows * NLDS / c,
         cmax / c, cmax / (ms * 1e3));
  cudaFree(out); cudaFree(cyc);
  return 0;
}

int main() {
  cudaDeviceProp pr; CHECK(cudaGetDeviceProperties(&pr, 0));
  int clk = 0; cudaDeviceGetAttribute(&clk, cudaDevAttrClockRate, 0);
  printf("# %s, %d SMs, %.0f MHz max SM clock; 16 warps x 1 CTA per SM; a warp-row is 32 lanes x (NX words + 4*NLDS words)\n",
         pr.name, pr.multiProcessorCount, clk / 1e3);
  for (int grid : {1, pr.multiProcessorCount}) {
    int rc = 0;
    rc |= run<4, 0, 4>("(a) tcgen05.ld x4", grid);
    rc |= run<8, 0, 4>("(a) tcgen05.ld x8", grid);
    rc |= run<16, 0, 4>("(a) tcgen05.ld x16", grid);
    rc |= run<16, 0, 1>("(a) tcgen05.ld x16, wait/row", grid);
    rc |= run<0, 8, 4>("(b) 8 LDS.128", grid);
    rc |= run<0, 7, 4>("(b) 7 LDS.128 (today's row)", grid);
    rc |= run<0, 4, 4>("(b) 4 LDS.128", grid);
    rc |= run<16, 4, 1>("(c) x16 + 4 LDS.128, wait/row", grid);
    rc |= run<16, 4, 4>("(c) x16 + 4 LDS.128", grid);
    rc |= run<8, 6, 1>("(c) x8 + 6 LDS.128, wait/row", grid);
    rc |= run<8, 6, 4>("(c) x8 + 6 LDS.128", grid);
    if (rc) return 1;
  }
  return 0;
}
