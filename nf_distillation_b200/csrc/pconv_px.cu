// Conv2dZeros + affine coupling for the 4x4-map levels (C = 48, C = 96): the per-tap products with the PIXELS on the MMA's
// M axis.
// (reference: models/layers.py:231-260 Conv2dZeros, models/flows.py:150-171 normal_flow / :173-190 reverse_flow)
//
// pconv_coupling_kernel<48> keeps the weights on M (432 rows = four 128-row blocks) and a tile of 64 pixels on N: sixteen
// N = 64 MMAs per k-block, each paying the ~70-cycle issue floor of an instruction a quarter that size, and 442 KB of
// weights streamed per 64 pixels -- 33 us for a launch whose h2 read is 34 MB (0.18 of the HBM roofline). Here
//
//     P[pixel, tap*48 + co] = sum_k h2[pixel, k] * B3[tap*48 + co, k]        M = 128 pixels (8 images), K = 512
//
// runs as passes of whole taps per tile -- C = 48: N = 240 (taps 0-4) and N = 192 (taps 5-8); C = 96 (CelebA's top level,
// which the weight-major kernel cannot hold: 864 weight rows): four passes of two taps (N = 192) and one of N = 96 --
// the weights streamed once per 128 pixels, and consecutive passes alternate over two accumulators (TMEM columns [0,256)
// and [256,512)) = the two pipeline stages: the next pass runs while the taps of this one are gathered. With pixels on the TMEM lanes
// and 16-pixel images, an image is half a warp of the epilogue: the col2im gather
//     out[p, c] = bias[c] + sum_tap P[p + off(tap), tap*48 + c]
// needs no shared memory at all -- a tcgen05.ld of the tap's 16 columns, then one __shfl_sync per value from the
// neighbour's lane (same tap order as the other kernels: bit-identical results). 12 epilogue warps: lane quadrant x
// channel third; each thread finishes C/6 (shift, logit) pairs of one pixel and applies the coupling in place.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdlib>

#include "../../include/nfk.h"
#include "launch_util.h"
#include "ptx.cuh"

namespace nfk {

constexpr int PX_EPI = 384;
constexpr int PX_THREADS = 64 + PX_EPI;
constexpr int PX_STAGES = 3;
constexpr int PX_H_BYTES = 128 * 128;          // h2 k-block: 128 pixels x 64 K (bf16)
constexpr int PX_W_BYTES = 256 * 128;          // room for the largest weight k-block (240 rows x 128 B)
constexpr int PX_STAGE = PX_H_BYTES + PX_W_BYTES;
constexpr int PX_SMEM = PX_STAGES * PX_STAGE + 1024;

template <int C> struct PxCfg {
  static constexpr int TP = C == 48 ? 5 : 2;               // taps per (full) pass
  static constexpr int NP = (9 + TP - 1) / TP;             // passes per tile
  static constexpr int NA = TP * C;                        // weight rows (= MMA N) of a full pass
  static constexpr int NB = (9 - (NP - 1) * TP) * C;       // ... of the last pass
  static constexpr int CG = C / 3;                         // channels per epilogue warp third
  static_assert(NA <= 256 && NA % 16 == 0 && NB % 16 == 0 && CG % 16 == 0, "pass shapes");
};

struct PxArgs {
  long long M;          // pixels = B * 16
  int num_kb;           // hid / 64
  const float* bias3;   // [C] folded Conv2dZeros bias
  float* y;             // [B, C, 4, 4] fp32: channels C/2.. are updated in place
  float* hsave;         // optional [M, C] fp32: conv output (shift, logit pairs) kept for the backward pass
  float* ld;            // optional [B] log-det, accumulated
  int reverse;
};

template <int C>
__global__ void __launch_bounds__(PX_THREADS, 1)
pconv_px_kernel(const __grid_constant__ CUtensorMap tmH, const __grid_constant__ CUtensorMap tmWA,
                const __grid_constant__ CUtensorMap tmWB, const PxArgs g) {
  using Cfg = PxCfg<C>;
  constexpr int TP = Cfg::TP, NP = Cfg::NP, NA = Cfg::NA, NB = Cfg::NB, CG = Cfg::CG, J = C / 2;
  extern __shared__ __align__(1024) uint8_t smem[];
  pdl_launch_dependents();
  if (smem_u32(smem) & 1023u) __trap();
  const int warp = static_cast<int>(uniform_u32(threadIdx.x >> 5)), lane = threadIdx.x & 31;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + PX_STAGES * PX_STAGE);
  uint64_t* empty = full + PX_STAGES;
  uint64_t* tmem_full = empty + PX_STAGES;   // [2]: pass A / pass B accumulator complete
  uint64_t* tmem_empty = tmem_full + 2;      // [2]: drained by the 12 epilogue warps
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);
  float* bias_s = reinterpret_cast<float*>(tmem_slot + 4);   // [C]

  const int num_tiles = static_cast<int>((g.M + 127) / 128);
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmH); tma_prefetch_desc(&tmWA); tma_prefetch_desc(&tmWB);
    for (int s = 0; s < PX_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(&tmem_full[a], 1); mbar_init(&tmem_empty[a], PX_EPI / 32); }
    fence_mbar_init();
  }
  if (warp == 1) { tmem_alloc(tmem_slot, 512); tmem_relinquish(); }
  pdl_wait();      // barrier init / TMEM allocation above overlap the previous kernel's tail
  if (threadIdx.x < C) bias_s[threadIdx.x] = g.bias3[threadIdx.x];
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = uniform_u32(*tmem_slot);

  if (warp == 0) {
    // ===================================================== TMA producer (whole warp, uniform control flow: ptx.cuh)
    int s = 0;
    uint32_t ph = 0;
    for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
      for (int pass = 0; pass < NP; ++pass) {
        const bool last = pass == NP - 1;
        for (int kb = 0; kb < g.num_kb; ++kb) {
          mbar_wait_warp(&empty[s], ph ^ 1);
          uint8_t* sa = smem + s * PX_STAGE;
          mbar_expect_tx_elect(&full[s], static_cast<uint32_t>(PX_H_BYTES + (last ? NB : NA) * 128));
          tma_load_2d_elect(sa, &tmH, &full[s], kb * 64, t * 128);
          tma_load_2d_elect(sa + PX_H_BYTES, last ? &tmWB : &tmWA, &full[s], kb * 64, pass * NA);
          if (++s == PX_STAGES) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================================================== MMA issuer (whole warp, uniform control flow)
    const uint32_t idescA = umma_idesc_bf16(128, NA, false, false);
    const uint32_t idescB = umma_idesc_bf16(128, NB, false, false);
    int s = 0;
    uint32_t ph = 0, nuse0 = 0, nuse1 = 0;     // uses of accumulator 0 / 1 so far
    for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
      for (int pass = 0; pass < NP; ++pass) {
        const int a = pass & 1;
        const uint32_t n = a ? nuse1 : nuse0;
        mbar_wait_warp(&tmem_empty[a], (n & 1) ^ 1);          // the epilogue has read this accumulator's previous use
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + a * 256;
        const uint32_t idesc = pass == NP - 1 ? idescB : idescA;
        for (int kb = 0; kb < g.num_kb; ++kb) {
          mbar_wait_warp(&full[s], ph);
          tc_fence_after();
          const uint32_t a_addr = smem_u32(smem + s * PX_STAGE);
          const uint32_t b_addr = a_addr + PX_H_BYTES;
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_f16_elect(tmem_d, umma_desc_sw128(a_addr + k * 32, 16, 1024), umma_desc_sw128(b_addr + k * 32, 16, 1024),
                           idesc, (kb > 0 || k > 0) ? 1u : 0u);
          umma_commit_elect(&empty[s]);
          if (++s == PX_STAGES) { s = 0; ph ^= 1; }
        }
        umma_commit_elect(&tmem_full[a]);
        if (a) ++nuse1; else ++nuse0;
      }
    }
  } else {
    // ===================================================== epilogue: 12 warps = TMEM lane quadrant x channel third
    const int q = warp & 3;                    // pixels q*32 .. q*32+31 of the tile (two images)
    const int w3 = (warp - 2) >> 2;            // channels CG*w3 .. CG*w3+CG-1 = (shift, logit) pairs (CG/2)*w3 ..
    const uint32_t lane_off = static_cast<uint32_t>(q * 32) << 16;
    const int r = lane & 15, yy = r >> 2, xx = r & 3;          // pixel inside its 4x4 image
    uint32_t nuse0 = 0, nuse1 = 0;             // uses of accumulator 0 / 1 so far
    for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
      const long long m = static_cast<long long>(t) * 128 + q * 32 + lane;
      const bool live = m < g.M;
      const long long b = m >> 4;
      // this thread's z2 values: requested before the waits for the MMAs
      float z2v[CG / 2];
      float* yp = g.y + ((b * C + J + (CG / 2) * w3) << 4) + r;
#pragma unroll
      for (int jj = 0; jj < CG / 2; ++jj) z2v[jj] = live ? yp[jj << 4] : 0.f;
      float acc[CG];
#pragma unroll
      for (int c = 0; c < CG; ++c) acc[c] = bias_s[CG * w3 + c];
#pragma unroll
      for (int tap = 0; tap < 9; ++tap) {
        constexpr int dummy = 0; (void)dummy;
        const int pass = tap / TP, ti = tap % TP, a = pass & 1;
        if (ti == 0) {   // first tap of a pass: its accumulator must be complete
          mbar_wait(&tmem_full[a], (a ? nuse1 : nuse0) & 1);
          tc_fence_after();
        }
        const uint32_t col = static_cast<uint32_t>(a * 256 + ti * C + CG * w3);
        uint32_t R[CG];
#pragma unroll
        for (int i = 0; i < CG / 16; ++i)
          tmem_ld16(tmem_base + lane_off + col + 16 * i, *reinterpret_cast<uint32_t(*)[16]>(&R[16 * i]));
        tmem_ld_wait();
        if (ti == TP - 1 || tap == 8) {   // last read of that accumulator: back to the MMA issuer
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&tmem_empty[a]);
          if (a) ++nuse1; else ++nuse0;
        }
        const int dy = tap / 3 - 1, dx = tap % 3 - 1;
        const bool valid = (yy + dy >= 0) && (yy + dy < 4) && (xx + dx >= 0) && (xx + dx < 4);
        const int src = (lane + dy * 4 + dx) & 31;     // the neighbour pixel's lane (same image when valid)
#pragma unroll
        for (int c = 0; c < CG; ++c) {
          const float v = __uint_as_float(__shfl_sync(0xffffffffu, R[c], src));
          if (valid) acc[c] += v;
        }
      }
      float lsum = 0.f;
#pragma unroll
      for (int jj = 0; jj < CG / 2; ++jj) {
        const float sh = acc[2 * jj], lg = acc[2 * jj + 1];
        if (live) {
          if (g.hsave) *reinterpret_cast<float2*>(g.hsave + m * C + 2 * ((CG / 2) * w3 + jj)) = make_float2(sh, lg);
          // sigmoid / log-sigmoid of (logit + 2), stable on both sides
          const float tt = lg + 2.f;
          const float e = expf(-fabsf(tt));
          const float l1p = log1pf(e);
          float sg, lsv;
          if (tt >= 0.f) { sg = 1.f / (1.f + e); lsv = -l1p; }
          else { sg = e / (1.f + e); lsv = tt - l1p; }
          yp[jj << 4] = g.reverse ? (z2v[jj] / sg - sh) : (z2v[jj] + sh) * sg;
          lsum += g.reverse ? -lsv : lsv;
        }
      }
      if (g.ld) {   // the 16 lanes of an image (all inside or all outside the batch) reduce; their first lane adds
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) lsum += __shfl_xor_sync(0xffffffffu, lsum, o);
        if (r == 0 && live) atomicAdd(g.ld + b, lsum);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

// C = 48 or 96, 4x4 maps, K3p >= 9 C rows of B3 [K3p, hid]. Returns NFK_ERR_SHAPE when the shape is not this kernel's.
template <int C>
static int px_launch(const void* h2, const void* B3, int K3p, const float* bias3, float* y, float* hsave, float* ld,
                     int B, int hid, int reverse, cudaStream_t st) {
  using Cfg = PxCfg<C>;
  if (K3p < 9 * C || hid % 64 || hid <= 0 || B <= 0) return NFK_ERR_SHAPE;
  PxArgs g{static_cast<long long>(B) * 16, hid / 64, bias3, y, hsave, ld, reverse};
  CUtensorMap tmH, tmWA, tmWB;
  int rc;
  if ((rc = make_tmap_2d(&tmH, h2, hid, static_cast<uint64_t>(g.M), hid, 128))) return rc;
  if ((rc = make_tmap_2d(&tmWA, B3, hid, K3p, hid, Cfg::NA))) return rc;
  if ((rc = make_tmap_2d(&tmWB, B3, hid, K3p, hid, Cfg::NB))) return rc;
  if ((rc = ensure_dyn_smem(reinterpret_cast<const void*>(pconv_px_kernel<C>), PX_SMEM))) return rc;
  const int sms = num_sms();
  const int tiles = static_cast<int>((g.M + 127) / 128);
  const cudaError_t le = launch_pdl(pconv_px_kernel<C>, dim3(tiles < sms ? tiles : sms), dim3(PX_THREADS), PX_SMEM, st,
                                    tmH, tmWA, tmWB, g);
  return (le == cudaSuccess && cudaGetLastError() == cudaSuccess) ? NFK_OK : NFK_ERR_LAUNCH;
}

int pconv_px_launch(const void* h2, const void* B3, int K3p, const float* bias3, float* y, float* hsave, float* ld,
                    int B, int C, int hid, int reverse, cudaStream_t st) {
  if (C == 48) return px_launch<48>(h2, B3, K3p, bias3, y, hsave, ld, B, hid, reverse, st);
  if (C == 96) return px_launch<96>(h2, B3, K3p, bias3, y, hsave, ld, B, hid, reverse, st);
  return NFK_ERR_SHAPE;
}

}  // namespace nfk
