// Last convolution of the coupling net fused with the affine coupling itself (reference: models/layers.py:231-260
// Conv2dZeros, models/flows.py:150-171 normal_flow / :173-190 reverse_flow).
//
// The 3x3 Conv2dZeros is computed as per-tap products  P^T[tap*C + c, pixel] = sum_k B3[tap*C + c, k] * h2[pixel, k]
// on tcgen05 -- the small weight matrix is the M operand (9C <= 128 rows per accumulator block), a tile of whole
// images is the N operand (256 pixels for C = 12, 128 for C = 24), so every MMA runs at the full 128 x N shape --
// and the accumulator never goes to HBM: the epilogue drains TMEM into shared memory, sums the nine shifted
// taps per output pixel (col2im), adds the bias, and applies the coupling
//     z2 <- (z2 + shift) * sigmoid(logit + 2),   logdet += sum log sigmoid(logit + 2)          (or its inverse)
// in place on the fp32 NCHW map. What used to be a GEMM writing P [M, 9C] fp32, and a second kernel reading it back,
// is one kernel whose HBM traffic is the bf16 h2 read plus the z2 update.
//
// Warp roles (448 threads): warp 0 TMA producer, warp 1 MMA issuer (+ TMEM allocation), warps 2-13 epilogue (the
// col2im + coupling gather is what bounds the C = 24 kernel: twelve warps share it, eight of them drain TMEM).
// Two TMEM accumulator stages: the epilogue of tile i overlaps the MMAs of tile i+1.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdlib>

#include "../../include/nfk.h"
#include "launch_util.h"
#include "ptx.cuh"

namespace nfk {

constexpr int PC_EPI = 384;            // epilogue threads: 12 warps (8 of them also drain TMEM, all 12 gather)
constexpr int PC_THREADS = 64 + PC_EPI;
constexpr int PC_BK = 64;

template <int C> struct PcCfg;
// NPIX pixels per tile (whole images), MB accumulator blocks of 128 rows; the epilogue handles the tile in two halves
// of NPIX/2 output pixels, each staging a window of WIN source pixels (the half plus one image row + 1 of halo when
// the image is larger than the half), so the staging buffer leaves room for a 3-stage operand ring.
template <> struct PcCfg<12> { static constexpr int NPIX = 256, MB = 1, WIN = 160, STAGES = 3; };  // one 16x16 image
template <> struct PcCfg<24> { static constexpr int NPIX = 128, MB = 2, WIN = 64, STAGES = 3; };   // two 8x8 images
template <> struct PcCfg<48> { static constexpr int NPIX = 64, MB = 4, WIN = 32, STAGES = 2; };    // four 4x4 images

struct PcArgs {
  long long M;          // pixels = B * H * W
  int num_kb;           // hid / 64
  int B, H, W, lgHW, lgW;
  const float* bias3;   // [C] folded Conv2dZeros bias
  float* y;             // [B, C, H, W] fp32: channels C/2.. are updated in place
  float* hsave;         // optional [M, C] fp32: conv output (shift, logit pairs) kept for the backward pass
  float* ld;            // optional [B] log-det, accumulated
  int reverse;
  // band mode (maps larger than a tile, W * 8 == NPIX): a tile is 8 image rows = rb output rows + one halo row above and
  // below; nb bands per image. banded == 0: tiles are NPIX consecutive pixels = whole images.
  int banded, nb, rb;
};

// First pixel (global index, may be negative for the halo above the very first image) of tile t.
template <int NPIX>
__device__ __forceinline__ long long pc_tile_pix0(const PcArgs& g, int t) {
  if (!g.banded) return static_cast<long long>(t) * NPIX;
  const int img = t / g.nb, band = t - img * g.nb;
  return (static_cast<long long>(img) << g.lgHW) + static_cast<long long>(band * g.rb - 1) * g.W;
}

template <int C>
struct PcSmem {
  using Cfg = PcCfg<C>;
  static constexpr int a_bytes = Cfg::MB * 128 * 128;          // B3 k-block: MB x (128 rows x 128 B)
  static constexpr int b_bytes = Cfg::NPIX * 128;              // h2 k-block: NPIX pixels x 128 B
  static constexpr int stage_bytes = a_bytes + b_bytes;
  static constexpr int pitch = Cfg::WIN + 1;                   // odd: a warp's 32 rows hit 32 banks
  static constexpr int s_bytes = ((9 * C * pitch * 4 + 15) / 16) * 16;
  static constexpr int off_s = Cfg::STAGES * stage_bytes;
  static constexpr int off_bar = off_s + s_bytes;
  static constexpr int off_bias = off_bar + 128;               // [C] floats
  static constexpr int total = off_bias + 128;
};

template <int C>
__global__ void __launch_bounds__(PC_THREADS, 1)
pconv_coupling_kernel(const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmH,
                      const PcArgs g) {
  using Cfg = PcCfg<C>;
  using Sm = PcSmem<C>;
  constexpr int NPIX = Cfg::NPIX, MB = Cfg::MB, WIN = Cfg::WIN, HALF = NPIX / 2, PC_STAGES = Cfg::STAGES;
  constexpr int K3 = 9 * C, J = C / 2;
  constexpr int ACC_COLS = MB * NPIX;   // TMEM columns of one accumulator stage
  extern __shared__ __align__(1024) uint8_t smem[];
  pdl_launch_dependents();
  if (smem_u32(smem) & 1023u) __trap();
  const int warp = static_cast<int>(uniform_u32(threadIdx.x >> 5)), lane = threadIdx.x & 31;
  float* S = reinterpret_cast<float*>(smem + Sm::off_s);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + Sm::off_bar);
  uint64_t* empty = full + PC_STAGES;
  uint64_t* tmem_full = empty + PC_STAGES;   // [2]
  uint64_t* tmem_empty = tmem_full + 2;      // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);
  float* bias_s = reinterpret_cast<float*>(smem + Sm::off_bias);

  const int num_tiles = g.banded ? g.B * g.nb : static_cast<int>((g.M + NPIX - 1) / NPIX);
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmW);
    tma_prefetch_desc(&tmH);
    for (int s = 0; s < PC_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(&tmem_full[a], 1); mbar_init(&tmem_empty[a], 8); }
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
    {   // whole warp, uniform control flow: single-thread instructions are elected inside the asm (ptx.cuh)
      int s = 0;
      uint32_t ph = 0;
      for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
        for (int kb = 0; kb < g.num_kb; ++kb) {
          mbar_wait_warp(&empty[s], ph ^ 1);
          uint8_t* sa = smem + s * Sm::stage_bytes;
          mbar_expect_tx_elect(&full[s], Sm::stage_bytes);
#pragma unroll
          for (int mb = 0; mb < MB; ++mb) tma_load_2d_elect(sa + mb * 128 * 128, &tmW, &full[s], kb * PC_BK, mb * 128);
          tma_load_2d_elect(sa + Sm::a_bytes, &tmH, &full[s], kb * PC_BK, static_cast<int>(pc_tile_pix0<NPIX>(g, t)));
          if (++s == PC_STAGES) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    {   // whole warp, uniform control flow: single-thread instructions are elected inside the asm (ptx.cuh)
      const uint32_t idesc = umma_idesc_bf16(128, NPIX, false, false);
      int s = 0, it = 0;
      uint32_t ph = 0;
      for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++it) {
        const int acc = it & 1;
        mbar_wait_warp(&tmem_empty[acc], ((it >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + acc * ACC_COLS;
        for (int kb = 0; kb < g.num_kb; ++kb) {
          mbar_wait_warp(&full[s], ph);
          tc_fence_after();
          const uint32_t a_addr = smem_u32(smem + s * Sm::stage_bytes);
          const uint32_t b_addr = a_addr + Sm::a_bytes;
#pragma unroll
          for (int k = 0; k < PC_BK / 16; ++k) {
            const uint64_t bd = umma_desc_sw128(b_addr + k * 32, 16, 1024);
#pragma unroll
            for (int mb = 0; mb < MB; ++mb) {
              const uint64_t ad = umma_desc_sw128(a_addr + mb * 128 * 128 + k * 32, 16, 1024);
              umma_f16_elect(tmem_d + mb * NPIX, ad, bd, idesc, (kb > 0 || k > 0) ? 1u : 0u);
            }
          }
          umma_commit_elect(&empty[s]);
          if (++s == PC_STAGES) { s = 0; ph ^= 1; }
        }
        umma_commit_elect(&tmem_full[acc]);
      }
    }
  } else {
    // ---- epilogue: 12 warps; for the drain, warp w < 10 owns TMEM lanes (w % 4) * 32.. and half (w - 2) / 4 of the
    // window's columns (warps 10-13 only gather).
    // Per tile: (1) prefetch this thread's z2 values (their HBM latency hides behind the wait for the MMAs and the
    // drain), (2) drain the whole accumulator P^T [9C, NPIX] into shared memory, (3) per (pixel, channel pair): sum
    // the nine shifted taps, bias, coupling, in-place z2 update, log-det partial sums.
    const int q = warp & 3, half = (warp - 2) >> 2;
    const int et = threadIdx.x - 64;   // 0..383
    const bool drains = half < 2;
    const bool banded = (C == 12) && g.banded;   // only the C = 12 kernel has a band mode: elsewhere OH folds to HALF
    const int HW = g.H * g.W, HWm = HW - 1, Wm = g.W - 1;
    constexpr int ITEMS = J * NPIX / PC_EPI;    // (pixel, j) items per thread: item i = et + PC_EPI k, pixel fastest
    static_assert(J * NPIX % (2 * PC_EPI) == 0, "each half's items must divide over the epilogue threads");
    // output pixels of one half: HALF consecutive pixels, or in band mode rb/2 image rows after the halo row
    const int OH = banded ? (g.rb >> 1) * g.W : HALF;
    int it = 0;
    for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++it) {
      const int acc = it & 1;
      const long long tile_base = pc_tile_pix0<NPIX>(g, t);
      const int row0 = banded ? (t % g.nb) * g.rb - 1 : 0;                   // band mode: image row of tile row 0
      const int row_end = banded ? min(g.H, row0 + 1 + g.rb) : 0;            //            first image row not owned
      // item ih of half hf -> (channel pair j, tile-local pixel pl, global pixel m); live = it exists and is ours
      auto decode = [&](int hf, int ih, int& j, int& pl, long long& m) -> bool {
        j = ih / OH;
        pl = (banded ? g.W : 0) + hf * OH + (ih - j * OH);
        m = tile_base + pl;
        if (j >= J) return false;
        if (!banded) return m < g.M;
        return row0 + (pl >> g.lgW) < row_end;   // (rows past the image end would alias the next image's first rows)
      };
      float z2v[ITEMS];
#pragma unroll
      for (int k = 0; k < ITEMS; ++k) {   // same (half, j, pixel) mapping as the gather below
        const int hf = k / (ITEMS / 2);
        int j, pl;
        long long m;
        const bool live = decode(hf, et + PC_EPI * (k - hf * (ITEMS / 2)), j, pl, m);
        const int b = static_cast<int>(m >> g.lgHW), rem = static_cast<int>(m) & HWm;
        z2v[k] = live ? g.y[((static_cast<long long>(b) * C + J + j) << g.lgHW) + rem] : 0.f;
      }
      mbar_wait(&tmem_full[acc], (it >> 1) & 1);
      tc_fence_after();
#pragma unroll
      for (int hf = 0; hf < 2; ++hf) {
        // source window of this half's outputs: the half itself when it holds whole images, else grown by the halo
        // and clipped to the tile (= the image)
        const int w0 = (WIN == HALF) ? hf * HALF : (hf == 0 ? 0 : NPIX - WIN);
        if (hf == 1) asm volatile("bar.sync 1, %0;" ::"n"(PC_EPI) : "memory");   // first half's gather is done with S
        // drain: TMEM [row][w0 .. w0+WIN) -> S[row][0 .. WIN); the two warps of a lane quadrant split the columns
        constexpr int HCOLS = WIN / 2;
        static_assert(HCOLS % 16 == 0, "window halves are drained 16 columns at a time");
#pragma unroll
        for (int mb = 0; mb < MB; ++mb) {
          const int row = mb * 128 + q * 32 + lane;
          const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * ACC_COLS + mb * NPIX + w0 +
                                 half * HCOLS;
          float* srow = S + row * Sm::pitch + half * HCOLS;
          if (drains && mb * 128 + q * 32 < K3) {   // warp-uniform: this block of 32 rows holds real taps
#pragma unroll 1
            for (int c = 0; c < HCOLS; c += 32) {
              uint32_t r0[16], r1[16];
              const bool two = c + 16 < HCOLS;
              tmem_ld16(taddr + c, r0);
              if (two) tmem_ld16(taddr + c + 16, r1);
              tmem_ld_wait();
              if (row < K3) {
#pragma unroll
                for (int k = 0; k < 16; ++k) srow[c + k] = __uint_as_float(r0[k]);
                if (two) {
#pragma unroll
                  for (int k = 0; k < 16; ++k) srow[c + 16 + k] = __uint_as_float(r1[k]);
                }
              }
            }
          }
        }
        if (hf == 1 && drains) {   // last TMEM read of this tile: accumulator stage back to the MMA warp
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&tmem_empty[acc]);
        }
        asm volatile("bar.sync 1, %0;" ::"n"(PC_EPI) : "memory");
#pragma unroll
        for (int kk = 0; kk < ITEMS / 2; ++kk) {
          const int k = hf * (ITEMS / 2) + kk;
          int j, pl;                                        // item inside this half: (j, pixel), pixel fastest
          long long m;
          const bool live = decode(hf, et + PC_EPI * kk, j, pl, m);
          const int b = static_cast<int>(m >> g.lgHW);
          float lsum = 0.f;
          if (live) {
            const int rem = static_cast<int>(m) & HWm;
            const int yy = rem >> g.lgW, xx = rem & Wm;
            float sh = bias_s[2 * j], lg = bias_s[2 * j + 1];
            const float* sp = S + (2 * j) * Sm::pitch + (pl - w0);
#pragma unroll
            for (int tap = 0; tap < 9; ++tap) {
              const int dy = tap / 3 - 1, dx = tap % 3 - 1;
              const int ny = yy + dy, nx = xx + dx;
              if (ny >= 0 && ny < g.H && nx >= 0 && nx < g.W) {
                const float* p = sp + tap * C * Sm::pitch + dy * g.W + dx;
                sh += p[0];
                lg += p[Sm::pitch];
              }
            }
            if (g.hsave) *reinterpret_cast<float2*>(g.hsave + m * C + 2 * j) = make_float2(sh, lg);
            // sigmoid / log-sigmoid of (logit + 2), stable on both sides
            const float tt = lg + 2.f;
            const float e = expf(-fabsf(tt));
            const float l1p = log1pf(e);
            float sg, lsv;
            if (tt >= 0.f) { sg = 1.f / (1.f + e); lsv = -l1p; }
            else { sg = e / (1.f + e); lsv = tt - l1p; }
            g.y[((static_cast<long long>(b) * C + J + j) << g.lgHW) + rem] =
                g.reverse ? (z2v[k] / sg - sh) : (z2v[k] + sh) * sg;
            lsum = g.reverse ? -lsv : lsv;
          }
          if (g.ld) {
            // pixel-fastest items: min(32, HW) consecutive lanes belong to one image (all inside or all outside the
            // batch); reduce inside those segments, the first lane of each adds
            const int seg = HW < 32 ? HW : 32;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
              const float v = __shfl_xor_sync(0xffffffffu, lsum, o);
              if (o < seg) lsum += v;
            }
            if ((lane & (seg - 1)) == 0 && live) atomicAdd(g.ld + b, lsum);
          }
        }
      }
      asm volatile("bar.sync 1, %0;" ::"n"(PC_EPI) : "memory");   // S is free for the next tile
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

template <int C>
static int pc_launch(const void* h2, const void* B3, int K3p, const PcArgs& g, int hid, cudaStream_t st) {
  using Cfg = PcCfg<C>;
  CUtensorMap tmW, tmH;
  int rc;
  if ((rc = make_tmap_2d(&tmW, B3, hid, K3p, hid, 128))) return rc;
  if ((rc = make_tmap_2d(&tmH, h2, hid, static_cast<uint64_t>(g.M), hid, Cfg::NPIX))) return rc;
  if ((rc = ensure_dyn_smem(reinterpret_cast<const void*>(pconv_coupling_kernel<C>), PcSmem<C>::total))) return rc;
  const int sms = num_sms();
  const int tiles = g.banded ? g.B * g.nb : static_cast<int>((g.M + Cfg::NPIX - 1) / Cfg::NPIX);
  const cudaError_t le = launch_pdl(pconv_coupling_kernel<C>, dim3(tiles < sms ? tiles : sms), dim3(PC_THREADS),
                                    PcSmem<C>::total, st, tmW, tmH, g);
  return (le == cudaSuccess && cudaGetLastError() == cudaSuccess) ? NFK_OK : NFK_ERR_LAUNCH;
}

// pconv_px.cu: the 4x4-map levels (C = 48, 96) with the pixels on the MMA's M axis; NFK_PCONV_PX=0 keeps
// pconv_coupling_kernel<48> (and leaves C = 96 to the per-tap GEMM + coupling_fwd path)
int pconv_px_launch(const void* h2, const void* B3, int K3p, const float* bias3, float* y, float* hsave, float* ld,
                    int B, int C, int hid, int reverse, cudaStream_t st);
static bool pconv_use_px() {
  static const bool v = [] { const char* e = getenv("NFK_PCONV_PX"); return !(e && e[0] == '0'); }();
  return v;
}

}  // namespace nfk

using namespace nfk;

extern "C" int nfk_pconv_coupling_supported(int C, int H, int W, int hid) {
  if (hid <= 0 || hid % 64) return 0;
  const int HW = H * W;
  if (HW < 4 || (HW & (HW - 1)) || (W & (W - 1))) return 0;
  // whole images per tile half: no halo between tiles (C = 12 may also split one image over the two halves)
  if (C == 12) {
    // whole images per half; or one image split over the two halves with its halo (W + 1 pixels) inside the staging
    // window; or band mode: 8 image rows per tile (6 output rows + a halo row either side), any H
    if (HW <= PcCfg<12>::NPIX / 2) return 1;
    if (HW == PcCfg<12>::NPIX && W + 1 <= PcCfg<12>::WIN - PcCfg<12>::NPIX / 2) return 1;
    return W * 8 == PcCfg<12>::NPIX && 3 * W + W + 1 <= PcCfg<12>::WIN + 1;
  }
  if (C == 24) return HW <= PcCfg<24>::NPIX / 2 && HW >= 4;
  if (C == 48) return HW <= PcCfg<48>::NPIX / 2 && HW >= 4;
  if (C == 96) return H == 4 && W == 4 && pconv_use_px();      // pixel-major kernel only (pconv_px.cu)
  return 0;
}

extern "C" int nfk_pconv_coupling_fwd(const void* h2, const void* B3, int K3p, const float* bias3, float* y,
                                      float* hsave, float* ld, int B, int C, int H, int W, int hid, int reverse,
                                      void* stream) {
  if (B <= 0 || !nfk_pconv_coupling_supported(C, H, W, hid)) return NFK_ERR_SHAPE;
  if (K3p % 64 || K3p < 9 * C || K3p > 128 * ((9 * C + 127) / 128)) return NFK_ERR_SHAPE;
  if (!h2 || !B3 || !bias3 || !y) return NFK_ERR_ARG;
  PcArgs g{};
  g.M = static_cast<long long>(B) * H * W;
  g.num_kb = hid / 64;
  g.B = B; g.H = H; g.W = W;
  g.lgW = 0; while ((1 << g.lgW) < W) ++g.lgW;
  g.lgHW = 0; while ((1 << g.lgHW) < H * W) ++g.lgHW;
  g.bias3 = bias3; g.y = y; g.hsave = hsave; g.ld = ld; g.reverse = reverse;
  if (C == 12 && H * W > PcCfg<12>::NPIX / 2 && !(H * W == PcCfg<12>::NPIX && W + 1 <= 32)) {
    g.banded = 1;
    g.rb = PcCfg<12>::NPIX / W - 2;          // 6 output rows per 8-row tile
    g.nb = (H + g.rb - 1) / g.rb;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if ((C == 48 || C == 96) && H == 4 && W == 4 && pconv_use_px())
    return pconv_px_launch(h2, B3, K3p, bias3, y, hsave, ld, B, C, hid, reverse, st);
  if (C == 12) return pc_launch<12>(h2, B3, K3p, g, hid, st);
  if (C == 24) return pc_launch<24>(h2, B3, K3p, g, hid, st);
  return pc_launch<48>(h2, B3, K3p, g, hid, st);
}
