// Input gradient of the coupling net's first conv (3x3, pad 1) fused with its col2im and the backward of the fused
// ActNorm o invertible 1x1 conv (reference: models/layers.py:101-142,404-421, models/flows.py:142-171).
//
// The backward mirror of pconv_coupling.cu. The per-tap products of the conv#1 dgrad
//     P^T[tap*CH + ci, pixel] = sum_k B1T[tap*CH + ci, k] * dpre1[pixel, k]
// run on tcgen05 with the small weight matrix as the M operand (9*CH <= 128 rows per accumulator block) and a tile of
// whole images as the N operand. The accumulator never goes to HBM: the epilogue drains TMEM into shared memory and,
// per tile, does what affine1x1_bwd_kernel (zpath.cu) does with the fp32 dcol it reads back from HBM:
//     dys[ci] = dy[ci] + sum_tap P^T[tap*CH + ci][pixel - off(tap)]   on the y1 half (dys = dy on the y2 half),
//     dx = W'^T dys,   dW' += dys x^T,   db' += sum dys.
// The tap sum, the dy + col2im add and the fmaf chain of dx run in the same order as col2im_gather and
// affine1x1_bwd_kernel, and the products are the same tcgen05 products as the gemm_nt dgrad's, so dx is bit-identical
// to that pair of kernels; dW' and db' are per-CTA register / shared sums flushed with one global atomic per entry.
// HBM traffic: dpre1 (bf16) read once, dy and x read, dx written. The fp32 dcol [M, K1p] is never materialised.
//
// Warp roles (320 threads): warp 0 TMA producer, warp 1 MMA issuer (+ TMEM allocation), warps 2-9 epilogue.
// Two TMEM accumulator stages: the epilogue of tile i overlaps the MMAs of tile i+1.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <cstdint>

#include "../../include/nfk.h"
#include "launch_util.h"
#include "ptx.cuh"

namespace nfk {

constexpr int DG_EPI = 256;                 // epilogue threads: 8 warps, two per TMEM lane quadrant
constexpr int DG_THREADS = 64 + DG_EPI;
constexpr int DG_BK = 64;

template <int C> struct DgCfg;
// NPIX pixels per tile (whole images), MB accumulator blocks of 128 rows (K1p = 64, 128, 256). The full tile's P^T,
// the dy / x tiles and the operand ring share the 227 KB of shared memory; that sets NPIX and STAGES.
template <> struct DgCfg<12> { static constexpr int NPIX = 256, MB = 1, STAGES = 3; };   // one 16x16 image
template <> struct DgCfg<24> { static constexpr int NPIX = 128, MB = 1, STAGES = 4; };   // two 8x8 images
template <> struct DgCfg<48> { static constexpr int NPIX = 64, MB = 2, STAGES = 3; };    // four 4x4 images

struct DgArgs {
  int B, lgHW, lgW, H, W;
  int num_kb;            // hid / 64
  int a_box_rows;        // rows of B1T per 128-row block the TMA loads: min(128, K1p)
  const float* dy;       // [B, C, H, W] gradient at the coupling's input (coupling_bwd's output)
  const float* x;        // [B, C, H, W] the step's input
  const float* Wf;       // [C, C] fused affine
  float* dx;             // [B, C, H, W]
  float* dWf;            // [C, C] accumulated
  float* dbf;            // [C] accumulated
};

template <int C>
struct DgSmem {
  using Cfg = DgCfg<C>;
  static constexpr int a_bytes = Cfg::MB * 128 * 128;          // B1T k-block: MB x (128 rows x 128 B)
  static constexpr int b_bytes = Cfg::NPIX * 128;              // dpre1 k-block: NPIX pixels x 128 B
  static constexpr int stage_bytes = a_bytes + b_bytes;
  static constexpr int pitch = Cfg::NPIX + 1;                  // odd: a warp's 32 drained rows hit 32 banks
  static constexpr int s_bytes = ((9 * (C / 2) * pitch * 4 + 15) / 16) * 16;
  static constexpr int t_bytes = C * pitch * 4;                // one [C][NPIX] fp32 tile (dys or xs)
  static constexpr int off_s = Cfg::STAGES * stage_bytes;
  static constexpr int off_dys = off_s + s_bytes;
  static constexpr int off_xs = off_dys + t_bytes;
  static constexpr int off_wt = off_xs + t_bytes;              // W'^T [C][C]
  static constexpr int off_acc = off_wt + C * C * 4;           // db' [C]
  static constexpr int off_bar = off_acc + ((C * 4 + 15) / 16) * 16;
  static constexpr int total = off_bar + 128;
  static_assert(total <= 227 * 1024, "shared memory budget");
};

template <int C>
__global__ void __launch_bounds__(DG_THREADS, 1)
conv1_dgrad_affine_bwd_kernel(const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmD,
                              const DgArgs g) {
  using Cfg = DgCfg<C>;
  using Sm = DgSmem<C>;
  constexpr int NPIX = Cfg::NPIX, MB = Cfg::MB, STAGES = Cfg::STAGES;
  constexpr int CH = C / 2, K1 = 9 * CH;
  constexpr int ACC_COLS = MB * NPIX;                // TMEM columns of one accumulator stage
  constexpr int TMEM_COLS = 2 * ACC_COLS;            // 512 or 256: a power of two
  constexpr int ldp = Sm::pitch;
  extern __shared__ __align__(1024) uint8_t smem[];
  pdl_launch_dependents();
  if (smem_u32(smem) & 1023u) __trap();
  const int warp = static_cast<int>(uniform_u32(threadIdx.x >> 5)), lane = threadIdx.x & 31;
  float* S = reinterpret_cast<float*>(smem + Sm::off_s);
  float* dys = reinterpret_cast<float*>(smem + Sm::off_dys);
  float* xs = reinterpret_cast<float*>(smem + Sm::off_xs);
  float* WT = reinterpret_cast<float*>(smem + Sm::off_wt);
  float* acc = reinterpret_cast<float*>(smem + Sm::off_acc);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + Sm::off_bar);
  uint64_t* empty = full + STAGES;
  uint64_t* tmem_full = empty + STAGES;   // [2]
  uint64_t* tmem_empty = tmem_full + 2;   // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);

  const int ipt = NPIX >> g.lgHW;                    // images per tile
  const int num_tiles = (g.B + ipt - 1) / ipt;
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmW);
    tma_prefetch_desc(&tmD);
    for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(&tmem_full[a], 1); mbar_init(&tmem_empty[a], 8); }
    fence_mbar_init();
  }
  if (warp == 1) { tmem_alloc(tmem_slot, TMEM_COLS); tmem_relinquish(); }
  pdl_wait();      // barrier init / TMEM allocation above overlap the previous kernel's tail
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = uniform_u32(*tmem_slot);

  if (warp == 0) {
    {   // whole warp, uniform control flow: single-thread instructions are elected inside the asm (ptx.cuh)
      // C = 12: only the 64 rows of B1T are loaded; rows 64-127 of the A block hold stale data, which only reaches
      // accumulator rows >= 64 that the epilogue never reads (an MMA row depends on its own A row alone)
      const uint32_t tx = MB * g.a_box_rows * 128 + Sm::b_bytes;
      int s = 0;
      uint32_t ph = 0;
      for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
        for (int kb = 0; kb < g.num_kb; ++kb) {
          mbar_wait_warp(&empty[s], ph ^ 1);
          uint8_t* sa = smem + s * Sm::stage_bytes;
          mbar_expect_tx_elect(&full[s], tx);
#pragma unroll
          for (int mb = 0; mb < MB; ++mb) tma_load_2d_elect(sa + mb * 128 * 128, &tmW, &full[s], kb * DG_BK, mb * 128);
          tma_load_2d_elect(sa + Sm::a_bytes, &tmD, &full[s], kb * DG_BK, t * NPIX);
          if (++s == STAGES) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    {   // whole warp, uniform control flow: single-thread instructions are elected inside the asm (ptx.cuh)
      const uint32_t idesc = umma_idesc_bf16(128, NPIX, false, false);
      int s = 0, it = 0;
      uint32_t ph = 0;
      for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++it) {
        const int ac = it & 1;
        mbar_wait_warp(&tmem_empty[ac], ((it >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + ac * ACC_COLS;
        for (int kb = 0; kb < g.num_kb; ++kb) {
          mbar_wait_warp(&full[s], ph);
          tc_fence_after();
          const uint32_t a_addr = smem_u32(smem + s * Sm::stage_bytes);
          const uint32_t b_addr = a_addr + Sm::a_bytes;
#pragma unroll
          for (int k = 0; k < DG_BK / 16; ++k) {
            const uint64_t bd = umma_desc_sw128(b_addr + k * 32, 16, 1024);
#pragma unroll
            for (int mb = 0; mb < MB; ++mb) {
              const uint64_t ad = umma_desc_sw128(a_addr + mb * 128 * 128 + k * 32, 16, 1024);
              umma_f16_elect(tmem_d + mb * NPIX, ad, bd, idesc, (kb > 0 || k > 0) ? 1u : 0u);
            }
          }
          umma_commit_elect(&empty[s]);
          if (++s == STAGES) { s = 0; ph ^= 1; }
        }
        umma_commit_elect(&tmem_full[ac]);
      }
    }
  } else {
    // ---- epilogue: 8 warps; for the drain, warp w owns TMEM lanes (w % 4) * 32.. and half (w - 2) / 4 of the columns.
    const int q = warp & 3, half = (warp - 2) >> 2;
    const int et = threadIdx.x - 64;   // 0..255
    const int HW = 1 << g.lgHW, HWm = HW - 1, Wm = g.W - 1;
    for (int i = et; i < C * C; i += DG_EPI) {
      const int o = i / C, c = i - o * C;
      WT[c * C + o] = g.Wf[i];
    }
    for (int i = et; i < C; i += DG_EPI) acc[i] = 0.f;
    constexpr int NBK = (C / 4) * (C / 4);              // 4x4 blocks of dW'
    constexpr int SL = NBK >= DG_EPI ? 1 : DG_EPI / NBK;   // pixel slices per block
    static_assert(NBK <= DG_EPI, "one dW' block per thread");
    float wacc[4][4] = {};
    constexpr int PARTS = DG_EPI / NPIX;                // dx: threads per pixel, each C / PARTS outputs
    static_assert(DG_EPI % NPIX == 0 && C % (4 * PARTS) == 0, "dx split");
    constexpr int ITEMS = CH * NPIX / DG_EPI;           // col2im (ci, pixel) items per thread
    static_assert(CH * NPIX % DG_EPI == 0, "col2im items divide over the epilogue threads");
    constexpr int TLD = C * NPIX / DG_EPI;              // dy / x tile elements per thread
    static_assert(C * NPIX % DG_EPI == 0, "tile loads divide over the epilogue threads");

    // dy and x of a tile's images: one contiguous [nimg, C, HW] block each. The next tile's block is requested right
    // after this tile's is staged, so its HBM latency hides behind this tile's drain, col2im, dx and dW' work.
    float xv[TLD], dv[TLD];
    auto load_tile = [&](int t) {
      const int b0 = t * ipt;
      const int nel = (min(ipt, g.B - b0) * C) << g.lgHW;
      const long long base = static_cast<long long>(b0) * C << g.lgHW;
#pragma unroll
      for (int u = 0; u < TLD; ++u) {
        const int i = et + u * DG_EPI;
        xv[u] = i < nel ? __ldg(g.x + base + i) : 0.f;
        dv[u] = i < nel ? __ldg(g.dy + base + i) : 0.f;
      }
    };
    if (static_cast<int>(blockIdx.x) < num_tiles) load_tile(blockIdx.x);

    int it = 0;
    for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++it) {
      const int ac = it & 1;
      const int b0 = t * ipt;
      const int npix = min(ipt, g.B - b0) << g.lgHW;
      // (1) stage this tile's dy and x (xs / dys are free: end-of-tile barrier), request the next tile's
#pragma unroll
      for (int u = 0; u < TLD; ++u) {
        const int i = et + u * DG_EPI;
        const int ic = i >> g.lgHW, img = ic / C, c = ic - img * C;
        const int so = c * ldp + (img << g.lgHW) + (i & HWm);
        xs[so] = xv[u];
        dys[so] = dv[u];
      }
      if (t + static_cast<int>(gridDim.x) < num_tiles) load_tile(t + gridDim.x);
      // (2) drain the accumulator P^T [K1, NPIX] into S; the two warps of a lane quadrant split the columns
      mbar_wait(&tmem_full[ac], (it >> 1) & 1);
      tc_fence_after();
      {
        constexpr int HCOLS = NPIX / 2;
        static_assert(HCOLS % 32 == 0, "column halves are drained 32 columns at a time");
#pragma unroll
        for (int mb = 0; mb < MB; ++mb) {
          const int row = mb * 128 + q * 32 + lane;
          const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + ac * ACC_COLS + mb * NPIX +
                                 half * HCOLS;
          float* srow = S + row * ldp + half * HCOLS;
          if (mb * 128 + q * 32 < K1) {   // warp-uniform: this block of 32 rows holds real taps
#pragma unroll 1
            for (int c = 0; c < HCOLS; c += 32) {
              uint32_t r0[16], r1[16];
              tmem_ld16(taddr + c, r0);
              tmem_ld16(taddr + c + 16, r1);
              tmem_ld_wait();
              if (row < K1) {
#pragma unroll
                for (int k = 0; k < 16; ++k) srow[c + k] = __uint_as_float(r0[k]);
#pragma unroll
                for (int k = 0; k < 16; ++k) srow[c + 16 + k] = __uint_as_float(r1[k]);
              }
            }
          }
        }
        tc_fence_before();   // last TMEM read of this tile: accumulator stage back to the MMA warp
        __syncwarp();
        if (lane == 0) mbar_arrive(&tmem_empty[ac]);
      }
      asm volatile("bar.sync 1, %0;" ::"n"(DG_EPI) : "memory");
      // (3) col2im onto the y1 half: item (ci, pixel), pixel fastest (conflict-free rows of S); the tap sum in
      // col2im_gather's order, then dys = dy + sum
#pragma unroll
      for (int u = 0; u < ITEMS; ++u) {
        const int i = et + u * DG_EPI;
        const int ci = i / NPIX, pl = i % NPIX;
        if (pl < npix) {
          const int rem = pl & HWm;
          const int yy = rem >> g.lgW, xx = rem & Wm;
          const float* sp = S + ci * ldp + pl;
          float a = 0.f;
#pragma unroll
          for (int tap = 0; tap < 9; ++tap) {
            const int ddy = tap / 3 - 1, ddx = tap % 3 - 1;
            const int ny = yy - ddy, nx = xx - ddx;
            a += (ny >= 0 && ny < g.H && nx >= 0 && nx < g.W) ? sp[tap * CH * ldp - ddy * g.W - ddx] : 0.f;
          }
          dys[ci * ldp + pl] += a;
        }
      }
      asm volatile("bar.sync 1, %0;" ::"n"(DG_EPI) : "memory");
      // (4) dx = W'^T dys: thread = (pixel, part), the same fmaf chain over o as affine1x1_bwd_kernel
      {
        const int pl = et % NPIX, part = et / NPIX;
        if (pl < npix) {
          const int img = pl >> g.lgHW, rem = pl & HWm;
          float dv[C];
#pragma unroll
          for (int o = 0; o < C; ++o) dv[o] = dys[o * ldp + pl];
          float* dxp = g.dx + ((static_cast<long long>(b0 + img) * C) << g.lgHW) + rem;
#pragma unroll 2
          for (int ii = 0; ii < C / PARTS; ++ii) {
            const int i = part * (C / PARTS) + ii;
            float a = 0.f;
            const float4* wr = reinterpret_cast<const float4*>(WT + i * C);
#pragma unroll
            for (int o = 0; o < C / 4; ++o) {
              const float4 w = wr[o];
              a = fmaf(w.x, dv[4 * o], a);
              a = fmaf(w.y, dv[4 * o + 1], a);
              a = fmaf(w.z, dv[4 * o + 2], a);
              a = fmaf(w.w, dv[4 * o + 3], a);
            }
            dxp[static_cast<long long>(i) << g.lgHW] = a;
          }
        }
      }
      // (5) dW'[o][i] += sum_p dys[o][p] x[i][p]: 4x4 register blocks, pixel range split over SL thread slices; the
      // partial sums stay in registers across all tiles of this CTA
      {
        const int blk = et % NBK, slice = et / NBK;
        if (slice < SL) {
          const int to = blk / (C / 4), ti = blk % (C / 4);
#pragma unroll 4
          for (int p = slice; p < npix; p += SL) {
            float dw[4], xw[4];
#pragma unroll
            for (int qq = 0; qq < 4; ++qq) {
              dw[qq] = dys[(4 * to + qq) * ldp + p];
              xw[qq] = xs[(4 * ti + qq) * ldp + p];
            }
#pragma unroll
            for (int qq = 0; qq < 4; ++qq)
#pragma unroll
              for (int r = 0; r < 4; ++r) wacc[qq][r] = fmaf(dw[qq], xw[r], wacc[qq][r]);
          }
        }
      }
      // (6) db'[o] += sum_p dys[o][p]: one warp per channel
      {
        const int ew = et >> 5;
        for (int o = ew; o < C; o += DG_EPI / 32) {
          float a = 0.f;
          for (int p = lane; p < npix; p += 32) a += dys[o * ldp + p];
          for (int sft = 16; sft > 0; sft >>= 1) a += __shfl_xor_sync(0xffffffffu, a, sft);
          if (lane == 0) acc[o] += a;
        }
      }
      asm volatile("bar.sync 1, %0;" ::"n"(DG_EPI) : "memory");   // S, dys and xs are free for the next tile
    }
    // the pixel slices of a block meet through a scratch tile (S is dead now), then one global atomic per entry
    static_assert(SL * C * C * 4 <= Sm::s_bytes, "slice scratch fits in S");
    {
      const int blk = et % NBK, slice = et / NBK;
      if (slice < SL) {
        const int to = blk / (C / 4), ti = blk % (C / 4);
#pragma unroll
        for (int qq = 0; qq < 4; ++qq)
#pragma unroll
          for (int r = 0; r < 4; ++r) S[slice * C * C + (4 * to + qq) * C + 4 * ti + r] = wacc[qq][r];
      }
    }
    asm volatile("bar.sync 1, %0;" ::"n"(DG_EPI) : "memory");
    for (int i = et; i < C * C; i += DG_EPI) {
      float a = 0.f;
      for (int sl2 = 0; sl2 < SL; ++sl2) a += S[sl2 * C * C + i];
      atomicAdd(g.dWf + i, a);
    }
    for (int i = et; i < C; i += DG_EPI) atomicAdd(g.dbf + i, acc[i]);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, TMEM_COLS);
}

template <int C>
static int dg_launch(const void* dpre1, const void* B1T, int K1p, int hid, DgArgs g, cudaStream_t st) {
  using Cfg = DgCfg<C>;
  CUtensorMap tmW, tmD;
  int rc;
  g.a_box_rows = K1p < 128 ? K1p : 128;
  const long long M = static_cast<long long>(g.B) << g.lgHW;
  if ((rc = make_tmap_2d(&tmW, B1T, hid, K1p, hid, g.a_box_rows))) return rc;
  if ((rc = make_tmap_2d(&tmD, dpre1, hid, static_cast<uint64_t>(M), hid, Cfg::NPIX))) return rc;
  if ((rc = ensure_dyn_smem(reinterpret_cast<const void*>(conv1_dgrad_affine_bwd_kernel<C>), DgSmem<C>::total)))
    return rc;
  const int sms = num_sms();
  const int ipt = Cfg::NPIX >> g.lgHW;
  const int tiles = (g.B + ipt - 1) / ipt;
  const cudaError_t le = launch_pdl(conv1_dgrad_affine_bwd_kernel<C>, dim3(tiles < sms ? tiles : sms),
                                    dim3(DG_THREADS), DgSmem<C>::total, st, tmW, tmD, g);
  return (le == cudaSuccess && cudaGetLastError() == cudaSuccess) ? NFK_OK : NFK_ERR_LAUNCH;
}

}  // namespace nfk

using namespace nfk;

extern "C" int nfk_conv1_dgrad_affine_bwd_supported(int C, int H, int W, int hid) {
  if (hid <= 0 || hid % 64) return 0;
  if (H <= 0 || W <= 0 || (H & (H - 1)) || (W & (W - 1))) return 0;
  const int HW = H * W;
  switch (C) {   // whole images per tile: the col2im needs no halo from a neighbouring tile
    case 12: return HW <= DgCfg<12>::NPIX;
    case 24: return HW <= DgCfg<24>::NPIX;
    case 48: return HW <= DgCfg<48>::NPIX;
    default: return 0;
  }
}

extern "C" int nfk_conv1_dgrad_affine_bwd(const void* dpre1, const void* B1T, int K1p, const float* dy,
                                          const float* x, const float* Wf, float* dx, float* dWf, float* dbf, int B,
                                          int C, int H, int W, int hid, void* stream) {
  if (B <= 0 || !nfk_conv1_dgrad_affine_bwd_supported(C, H, W, hid)) return NFK_ERR_SHAPE;
  if (K1p != (9 * (C / 2) + 63) / 64 * 64) return NFK_ERR_SHAPE;
  if (!dpre1 || !B1T || !dy || !x || !Wf || !dx || !dWf || !dbf) return NFK_ERR_ARG;
  DgArgs g{};
  g.B = B; g.H = H; g.W = W;
  g.lgW = 0; while ((1 << g.lgW) < W) ++g.lgW;
  g.lgHW = 0; while ((1 << g.lgHW) < H * W) ++g.lgHW;
  g.num_kb = hid / 64;
  g.dy = dy; g.x = x; g.Wf = Wf; g.dx = dx; g.dWf = dWf; g.dbf = dbf;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (C == 12) return dg_launch<12>(dpre1, B1T, K1p, hid, g, st);
  if (C == 24) return dg_launch<24>(dpre1, B1T, K1p, hid, g, st);
  return dg_launch<48>(dpre1, B1T, K1p, hid, g, st);
}
