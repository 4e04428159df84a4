// Microbenchmark: sustained TMA (cp.async.bulk.tensor.2d) L2 -> shared memory rate per SM when every CTA streams the SAME
// [512, 512] bf16 weight matrix (512 KB, L2 resident) in boxes of 64 K-columns (128 B, SWIZZLE_128B) x `rows` rows, with
// `slots` boxes in flight per CTA.
#include <cuda.h>
#include <cuda_runtime.h>
#include <cstdio>
#include <cstdint>
#include "../../nf_distillation_b200/csrc/launch_util.h"
#include "../../nf_distillation_b200/csrc/ptx.cuh"
using namespace nfk;

__global__ void __launch_bounds__(64, 1)
bench(const __grid_constant__ CUtensorMap tm, int rows, int slots, int iters, int per, int mode, long long* out) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ uint64_t full[32];
  const int box_bytes = rows * 128 * per;
  if (threadIdx.x == 0) { for (int s = 0; s < slots; ++s) mbar_init(&full[s], 1); fence_mbar_init(); }
  __syncthreads();
  if (threadIdx.x < 32) {
    const int nrow_boxes = 512 / rows;
    const long long t0 = clock64();
    uint32_t ph = 0; int s = 0;
    for (int i = 0; i < iters + slots; ++i) {
      if (i >= slots && mode != 1) { mbar_wait_warp(&full[s], ph); }
      if (i < iters) {
        if (mode == 2) { if (elect_one()) mbar_arrive(&full[s]); }
        else if (mode != 1) mbar_expect_tx_elect(&full[s], box_bytes);
        if (mode != 2) for (int j = 0; j < per; ++j) {
          const int b = (i * per + j + blockIdx.x * 3) & (nrow_boxes * 8 - 1);
          tma_load_2d_elect(smem + s * box_bytes + j * rows * 128, &tm, &full[s], (b & 7) * 64, (b >> 3) * rows);
        }
      }
      if (++s == slots) { s = 0; if (i >= slots) ph ^= 1; }
    }
    if (threadIdx.x == 0) out[blockIdx.x] = clock64() - t0;
  }
}

int main() {
  void* w; cudaMalloc(&w, 512 * 512 * 2); cudaMemset(w, 0, 512 * 512 * 2);
  long long* d; cudaMalloc(&d, 148 * 8);
  cudaFuncSetAttribute(bench, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
  const int iters = 4096;
  for (int grid : {148}) for (int rows : {64}) for (int slots : {4}) for (int per : {1, 2}) for (int mode : {0, 1, 2}) {
    if (rows * 128 * slots * per > 190 * 1024) continue;
    CUtensorMap tm;
    if (make_tmap_2d(&tm, w, 512, 512, 512, rows) != NFK_OK) { printf("tensor map encode failed\n"); return 1; }
    // phase bookkeeping above is simplistic: use iters multiple of slots
    for (int rep = 0; rep < 2; ++rep) {
      bench<<<grid, 64, 200 * 1024>>>(tm, rows, slots, iters, per, mode, d);
      cudaError_t e = cudaDeviceSynchronize();
      if (e != cudaSuccess) { printf("error %s\n", cudaGetErrorString(e)); return 1; }
    }
    long long h[148]; cudaMemcpy(h, d, grid * 8, cudaMemcpyDeviceToHost);
    double s = 0; for (int i = 0; i < grid; ++i) s += h[i];
    printf("mode %d (0 wait+expect+tma, 1 tma only, 2 wait+arrive only) grid %3d box %3d rows (%5d B) x %d per barrier x %2d slots: %6.1f B/clk per SM, %6.1f cycles per request\n", mode, grid, rows, rows * 128, per, slots,
           (double)iters * per * rows * 128 / (s / grid), (s / grid) / ((double)iters * per));
  }
  return 0;
}
