// Host-side launch helpers shared by the .cu files.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>

#include <cstdint>
#include <cstdlib>

#include <mutex>
#include <unordered_map>

#include "../../include/nfk.h"

namespace nfk {

// Row-major [rows, cols] matrix with leading dimension ld (elements), bf16 or (f32) fp32, as a 2-D TMA tensor map:
// boxes of 128 bytes of columns (64 bf16 / 32 fp32) x box_rows rows, SWIZZLE_128B, L2_256B promotion. The driver's
// encoder is looked up once; returns NFK_ERR_ALIGN for a pointer or row stride that is not 16-byte aligned.
inline int make_tmap_2d(CUtensorMap* m, const void* ptr, uint64_t cols, uint64_t rows, uint64_t ld, uint32_t box_rows,
                        bool f32 = false) {
  using EncodeTiledFn = decltype(&cuTensorMapEncodeTiled);
  static const EncodeTiledFn enc = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      return static_cast<EncodeTiledFn>(nullptr);
    return reinterpret_cast<EncodeTiledFn>(p);
  }();
  if (!enc) return NFK_ERR_DRIVER;
  const uint64_t es = f32 ? 4 : 2;
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) || (ld * es) % 16) return NFK_ERR_ALIGN;
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {ld * es};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(128 / es), box_rows};
  cuuint32_t estr[2] = {1, 1};
  const CUresult r = enc(m, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2,
                         const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? NFK_OK : NFK_ERR_DRIVER;
}

// SM count of the current device (148, a B200's, if the query fails), cached per device ordinal so that launches —
// including those made while a CUDA graph is being captured — issue no attribute query after the first.
inline int num_sms() {
  int dev = 0;
  cudaGetDevice(&dev);
  static std::mutex mu;
  static std::unordered_map<int, int> cache;
  std::lock_guard<std::mutex> lock(mu);
  auto it = cache.find(dev);
  if (it != cache.end()) return it->second;
  int n = 0;
  if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
  cache[dev] = n;
  return n;
}

// Opt a kernel in to > 48 KB of dynamic shared memory exactly once (keyed by the kernel's address), so later launches
// — including launches made while a CUDA graph is being captured — issue no attribute call.
inline int ensure_dyn_smem(const void* kernel, int bytes) {
  if (bytes <= 48 * 1024) return NFK_OK;
  if (bytes > 227 * 1024) return NFK_ERR_SHAPE;
  static std::mutex mu;
  static std::unordered_map<const void*, bool> done;
  std::lock_guard<std::mutex> lock(mu);
  auto it = done.find(kernel);
  if (it != done.end()) return NFK_OK;
  if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess)
    return NFK_ERR_LAUNCH;
  done[kernel] = true;
  return NFK_OK;
}

// Launch with programmatic dependent launch allowed (see ptx.cuh: pdl_wait / pdl_launch_dependents). NFK_PDL=0 in the
// environment turns the attribute off (the kernels' griddepcontrol instructions are then no-ops).
inline bool pdl_enabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("NFK_PDL");
    v = (e && e[0] == '0') ? 0 : 1;
  }
  return v == 1;
}

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                              Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = pdl_enabled() ? 1 : 0;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

}  // namespace nfk
