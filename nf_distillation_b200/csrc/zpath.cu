// fp32 "z path" kernels of a 2-D FlowStep (reference: models/flows.py:142-202, models/layers.py:101-142,404-421).
// All tensors are contiguous NCHW fp32; HBM-bound, coalesced along the pixel axis.
//
//  affine1x1_fwd   y = W' x + b' per pixel (ActNorm folded into the invertible 1x1 conv), logdet += pixels*sl,
//                  and the bf16 im2col matrix of y1 = y[:, :C/2] that feeds the first coupling conv (3x3, pad 1).
//  coupling_fwd    col2im of the last conv's per-tap products P, + folded bias, then the affine coupling
//                  z2 = (z2 + shift) * sigmoid(s + 2)  (or its inverse), log-det reduced per sample.
//  coupling_bwd    gradient of the coupling wrt (z2, h) and the im2col matrix of dh for the dgrad / wgrad GEMMs; the
//                  same kernel with INV = true is the backward of the inverse coupling (coupling_inv_bwd).
//  affine1x1_bwd   col2im of the first conv's input gradient, dx = W'^T dy, dW' and db' reductions.
//  col2im_add      dz1 += col2im of the first conv's input gradient (inverse pass: the conv reads z1 directly).
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <cstdint>

#include "../../include/nfk.h"
#include "launch_util.h"
#include "ptx.cuh"

namespace nfk {

constexpr int ZT = 256;  // threads per CTA

__device__ __forceinline__ uint32_t bf2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}

// log(sigmoid(t)) and sigmoid(t), stable for both signs.
__device__ __forceinline__ void sigmoid_logsigmoid(float t, float& s, float& ls) {
  const float e = expf(-fabsf(t));
  const float l1p = log1pf(e);
  if (t >= 0.f) {
    s = 1.f / (1.f + e);
    ls = -l1p;
  } else {
    s = e / (1.f + e);
    ls = t - l1p;
  }
}

struct Geo {
  int B, HW, W, H;
  int ipc;     // images per CTA
  int pixt;    // ipc * HW
  int og;      // affine1x1_fwd: output-channel groups per pixel (more threads for small images)
  int lgHW, lgW;  // H, W are powers of two for the forward kernels
};

// Staging tile (rows of r16 16-byte chunks, row stride rs16) -> global rows of r16 chunks, consecutive threads on
// consecutive chunks. r16 = K/8 is a power of two for every shipped width except K = 448, so a thread's chunk column is
// fixed and its row advances by ZT / r16 per pass (no per-element division).
__device__ __forceinline__ void copy_out_rows(uint4* __restrict__ out4, const uint4* __restrict__ cst, int npix,
                                              int r16, int rs16, int tid) {
  if ((r16 & (r16 - 1)) == 0 && r16 <= ZT) {
    const int lg = __ffs(r16) - 1;
    const int c4 = tid & (r16 - 1), step = ZT >> lg;
    for (int pl = tid >> lg; pl < npix; pl += step) out4[(pl << lg) + c4] = cst[pl * rs16 + c4];
  } else {
    for (int i = tid; i < npix * r16; i += ZT) {
      const int pl = i / r16, c4 = i - pl * r16;
      out4[i] = cst[pl * rs16 + c4];
    }
  }
}

// ------------------------------------------------------------------------------------------ affine1x1 fwd
// One CTA = `ipc` whole images (the 3x3 im2col needs their halo). H, W are powers of two (shifts, no divisions).
// Phase 1: thread = (pixel, output group): y = W'x + b' with x in registers, W' broadcast from smem (LDS.128).
// Phase 2: thread = (tap, pixel): one bounds test per tap, C/2 conflict-free smem reads of y1, bf16x2 packs into a
//          row-per-pixel staging tile (odd word stride -> conflict-free). Phase 3: coalesced 16-byte copy-out.
// smem: Ws[C*C] bs[C] | y1s[(C/2) * (pixt+1)] | cst[pixt * (K1p/8 + 1)] 16-byte chunks
template <int C>
__global__ void __launch_bounds__(ZT)
affine1x1_fwd_kernel(const float* __restrict__ x, const float* __restrict__ Wf, const float* __restrict__ bf,
                     const float* __restrict__ sl, float* __restrict__ y, __nv_bfloat16* __restrict__ col,
                     const float* __restrict__ ld_in, float* __restrict__ ld_out, Geo g, int K1p) {
  pdl_launch_dependents();
  pdl_wait();   // (reads global memory from its first instruction: only the launch latency overlaps)
  extern __shared__ float sm[];
  constexpr int CH = C / 2;
  float* Ws = sm;
  float* bs = Ws + C * C;
  float* y1s = bs + C;
  // staging tile starts 16-byte aligned after the y1 tile
  float* cst_raw = y1s + ((CH * (g.pixt + 1) + 3) & ~3);
  const int tid = threadIdx.x;
  const int b0 = blockIdx.x * g.ipc;
  const int nimg = min(g.ipc, g.B - b0);
  const int npix = nimg << g.lgHW;
  const int ldp = g.pixt + 1;
  const int HWm = g.HW - 1, Wm = g.W - 1;

  const int pixb = ZT / g.og;            // pixels per pass; lanes = consecutive pixels, output groups across warps
  const int og = tid / pixb;
  const int opg = C / g.og;              // outputs per group
  // narrow steps: the first pass's inputs are requested before the weights, so the two global round trips overlap
  // (wide ones would carry C live registers across the barrier and lose a resident CTA)
  constexpr bool PREFETCH_X = C <= 24;
  float xv[C];
  if (PREFETCH_X) {
    const int pl = tid % pixb;
    if (pl < npix && og < g.og) {
      const float* xp = x + (static_cast<long long>(b0 + (pl >> g.lgHW)) * C << g.lgHW) + (pl & HWm);
#pragma unroll
      for (int i = 0; i < C; ++i) xv[i] = __ldg(xp + (static_cast<long long>(i) << g.lgHW));
    }
  }
  if (Wf) {
    // C*C/4 float4 weights: all of a thread's loads first, then its stores (C*C is a multiple of 4; cudaMalloc'd)
    constexpr int W4 = C * C / 4, WPT = (W4 + ZT - 1) / ZT;
    float4 wreg[WPT];
#pragma unroll
    for (int k = 0; k < WPT; ++k) {
      const int i = tid + k * ZT;
      if (i < W4) wreg[k] = __ldg(reinterpret_cast<const float4*>(Wf) + i);
    }
#pragma unroll
    for (int k = 0; k < WPT; ++k) {
      const int i = tid + k * ZT;
      if (i < W4) reinterpret_cast<float4*>(Ws)[i] = wreg[k];
    }
    for (int i = tid; i < C; i += ZT) bs[i] = bf[i];
  }
  if (ld_out && tid < nimg) ld_out[b0 + tid] = ld_in[b0 + tid] + sl[0] * static_cast<float>(g.HW);
  __syncthreads();

  for (int pl = tid % pixb; pl < npix && og < g.og; pl += pixb) {
    const int img = pl >> g.lgHW, p = pl & HWm;
    const float* xp = x + (static_cast<long long>(b0 + img) * C << g.lgHW) + p;
    if (!PREFETCH_X || pl >= pixb) {   // later passes (the first one was prefetched above)
#pragma unroll
      for (int i = 0; i < C; ++i) xv[i] = __ldg(xp + (static_cast<long long>(i) << g.lgHW));
    }
    if (Wf) {
      float* yp = y + (static_cast<long long>(b0 + img) * C << g.lgHW) + p;
      for (int o = og * opg; o < (og + 1) * opg; ++o) {
        float acc = bs[o];
        const float4* wr = reinterpret_cast<const float4*>(Ws + o * C);
#pragma unroll
        for (int i = 0; i < C / 4; ++i) {
          const float4 w = wr[i];
          acc = fmaf(w.x, xv[4 * i], acc);
          acc = fmaf(w.y, xv[4 * i + 1], acc);
          acc = fmaf(w.z, xv[4 * i + 2], acc);
          acc = fmaf(w.w, xv[4 * i + 3], acc);
        }
        yp[static_cast<long long>(o) << g.lgHW] = acc;
        if (col && o < CH) y1s[o * ldp + pl] = acc;
      }
    } else if (col) {
#pragma unroll
      for (int o = 0; o < CH; ++o)   // static register indices (a runtime xv[o] would push xv to local memory)
        if (o >= og * opg && o < (og + 1) * opg) y1s[o * ldp + pl] = xv[o];
    }
  }
  if (!col) return;
  __syncthreads();
  // Phase 2: thread = pixel. All (tap, channel) positions of a 16-byte chunk are compile-time constants, so a chunk is
  // eight predicated conflict-free smem reads + four bf16x2 packs + one STS.128 into the staging tile.
  constexpr int K1 = 9 * CH;
  constexpr int NCH = (K1 + 7) / 8;      // chunks holding data; chunks >= NCH are zero padding
  const int r16 = K1p / 8;               // 16-byte chunks per im2col row
  const int rs16 = r16 + 1;              // staging row stride in chunks (odd -> conflict-free 16-byte accesses)
  uint4* cst = reinterpret_cast<uint4*>(cst_raw);
  int noff[9];
#pragma unroll
  for (int tap = 0; tap < 9; ++tap) noff[tap] = (tap / 3 - 1) * g.W + (tap % 3 - 1);
  // small tiles: GR threads share a pixel, thread gid takes the chunks c4 with c4 % GR == gid (pixt is a power of two)
  const int GR = g.pixt >= ZT ? 1 : ZT / g.pixt;
  const int gid = tid / g.pixt;          // 0 when GR == 1 (then tid < pixt may not hold: handled by the loop below)
  for (int pl = GR > 1 ? (tid & (g.pixt - 1)) : tid; pl < npix; pl += (GR > 1 ? g.pixt : ZT)) {
    const int rem = pl & HWm;
    const int yy = rem >> g.lgW, xx = rem & Wm;
    uint32_t vmask = 0;
#pragma unroll
    for (int tap = 0; tap < 9; ++tap) {
      const int ny = yy + tap / 3 - 1, nx = xx + tap % 3 - 1;
      vmask |= (ny >= 0 && ny < g.H && nx >= 0 && nx < g.W) ? (1u << tap) : 0u;
    }
    const float* yb = y1s + pl;
    uint4* drow = cst + pl * rs16;
#pragma unroll
    for (int c4 = 0; c4 < NCH; ++c4) {
      if (GR > 1 && (c4 & (GR - 1)) != gid) continue;
      float v[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        constexpr int dummy = 0; (void)dummy;
        const int k = c4 * 8 + e;
        if (k < K1) {
          const int tap = k / CH, ci = k % CH;
          v[e] = ((vmask >> tap) & 1u) ? yb[ci * ldp + noff[tap]] : 0.f;
        } else {
          v[e] = 0.f;
        }
      }
      drow[c4] = make_uint4(bf2(v[0], v[1]), bf2(v[2], v[3]), bf2(v[4], v[5]), bf2(v[6], v[7]));
    }
    for (int c4 = NCH; c4 < r16; ++c4)
      if (GR == 1 || (c4 & (GR - 1)) == gid) drow[c4] = make_uint4(0u, 0u, 0u, 0u);
  }
  __syncthreads();
  // Phase 3: coalesced copy-out, 16 bytes per thread, consecutive threads -> consecutive chunks of the same row
  uint4* out4 = reinterpret_cast<uint4*>(col + (static_cast<long long>(b0) << g.lgHW) * K1p);
  copy_out_rows(out4, cst, npix, r16, rs16, tid);
}

// col2im of the first conv's input gradient, UN (pixel, channel) items per thread at a time: item i0 + u*ZT is
// (pixel pl = i / CH, channel ci = i % CH) of the pixel range starting at global pixel m0, channel fastest so that the
// CH lanes of a pixel read one contiguous segment of a dcol row per tap. out[u] = sum_tap dcol[m - off(tap), tap*CH+ci]
// (0 for items >= nitems); all 9*UN loads of the (HBM-resident) dcol rows are in flight before the first add.
template <int CH, int UN>
__device__ __forceinline__ void col2im_gather(const float* __restrict__ dcol, int K1p, const Geo& g, long long m0,
                                              int i0, int nitems, float (&out)[UN]) {
  const int HWm = g.HW - 1, Wm = g.W - 1;
  float v[UN][9];
#pragma unroll
  for (int u = 0; u < UN; ++u) {
    const int i = i0 + u * ZT;
    const bool live = i < nitems;
    const int pl = live ? i / CH : 0, ci = live ? i - pl * CH : 0;
    const long long m = m0 + pl;
    const int rem = static_cast<int>(m & HWm);
    const int yy = rem >> g.lgW, xx = rem & Wm;
#pragma unroll
    for (int tap = 0; tap < 9; ++tap) {
      const int ddy = tap / 3 - 1, ddx = tap % 3 - 1;
      const int ny = yy - ddy, nx = xx - ddx;
      v[u][tap] = (live && ny >= 0 && ny < g.H && nx >= 0 && nx < g.W)
                      ? __ldg(dcol + (m - ddy * g.W - ddx) * K1p + tap * CH + ci) : 0.f;
    }
  }
#pragma unroll
  for (int u = 0; u < UN; ++u) {
    float a = 0.f;
#pragma unroll
    for (int tap = 0; tap < 9; ++tap) a += v[u][tap];
    out[u] = a;
  }
}

// ------------------------------------------------------------------------------------------ coupling fwd / inv
// No shared memory. Thread = (pixel, channel pair j), j fastest: the J lanes of a pixel read one contiguous C*4-byte
// segment of that pixel's P row per tap (few 128-byte lines per warp request — the L1 wavefront count, not HBM, was
// the limit of a thread-per-pixel mapping), and the z accesses touch J channel planes x ~32/J consecutive pixels.
// log-det: segmented warp reduction over the (ordered) sample index, one atomicAdd per segment.
template <int C>
__global__ void __launch_bounds__(ZT)
coupling_fwd_kernel(const float* __restrict__ P, int K3p, const float* __restrict__ bias3, float* __restrict__ y,
                    float* __restrict__ hsave, float* __restrict__ ld, Geo g, int reverse) {
  constexpr int J = C / 2;
  const long long M = static_cast<long long>(g.B) << g.lgHW;
  const long long item = static_cast<long long>(blockIdx.x) * ZT + threadIdx.x;
  const long long m = item / J;
  const int j = static_cast<int>(item - m * J);
  const bool live = m < M;
  const int lane = threadIdx.x & 31;
  float lsum = 0.f;
  int b = -1;
  if (live) {
    b = static_cast<int>(m >> g.lgHW);
    const int rem = static_cast<int>(m) & (g.HW - 1);
    const int yy = rem >> g.lgW, xx = rem & (g.W - 1);
    float sh = __ldg(bias3 + 2 * j), lg = __ldg(bias3 + 2 * j + 1);
    const float* prow = P + m * K3p + 2 * j;
#pragma unroll
    for (int tap = 0; tap < 9; ++tap) {
      const int dy = tap / 3 - 1, dx = tap % 3 - 1;
      const int ny = yy + dy, nx = xx + dx;
      if (ny >= 0 && ny < g.H && nx >= 0 && nx < g.W) {
        const float2 v = __ldg(reinterpret_cast<const float2*>(prow + static_cast<long long>(dy * g.W + dx) * K3p +
                                                               tap * C));
        sh += v.x;
        lg += v.y;
      }
    }
    if (hsave) *reinterpret_cast<float2*>(hsave + m * C + 2 * j) = make_float2(sh, lg);
    float s, lsv;
    sigmoid_logsigmoid(lg + 2.f, s, lsv);
    float* yp = y + ((static_cast<long long>(b) * C + J + j) << g.lgHW) + rem;
    const float z2 = *yp;
    *yp = reverse ? (z2 / s - sh) : (z2 + sh) * s;
    lsum = reverse ? -lsv : lsv;
  }
  if (ld) {
    // samples are non-decreasing along the warp: segmented suffix sums, then the first lane of each segment adds
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const float v = __shfl_down_sync(0xffffffffu, lsum, o);
      const int bb = __shfl_down_sync(0xffffffffu, b, o);
      if (lane + o < 32 && bb == b) lsum += v;
    }
    const int bp = __shfl_up_sync(0xffffffffu, b, 1);
    if (live && (lane == 0 || bp != b)) atomicAdd(ld + b, lsum);
  }
}

// ------------------------------------------------------------------------------------------ coupling bwd
// Persistent CTAs walk groups of `ipc` whole images, or -- when one image's staging tile does not fit (32x32 and
// larger) -- bands of `brows` image rows with a one-row halo on either side (the halo's dh is recomputed, its side
// effects are not repeated). Phase 1 (thread = (channel pair, pixel), pixel fastest): gradient of the affine coupling
// wrt (z2, shift, logit) from the saved h; dh goes to a smem tile. Phase 2 (thread = pixel): the im2col matrix of dh
// for the dgrad / wgrad GEMMs with compile-time (tap, channel) positions, staged and copied out in 16-byte coalesced
// chunks. Bias-gradient sums stay in smem across groups: one global atomic per channel and CTA.
// INV = true: backward of the INVERSE coupling zc2 = z2 / s - shift, ld -= sum log s (g_out = dL/dzc, z_out = zc):
// dz2 = dzc2 / s, dshift = -dzc2, dlogit = -(dzc2 * (zc2 + shift) + g_ld) * (1 - s)   (z2 / s = zc2 + shift).
// smem: dhs[C*ldp] dbs[C] | cst[tile * (K3p/8 + 1)] 16-byte chunks,  ldp = tile + 2*halo + 1
template <int C, bool INV>
__global__ void __launch_bounds__(ZT)
coupling_bwd_kernel(const float* __restrict__ g_out, const float* __restrict__ g_ld, const float* __restrict__ z_out,
                    const float* __restrict__ hsave, float* __restrict__ dy, __nv_bfloat16* __restrict__ dhcol,
                    int K3p, float* __restrict__ dbias3, Geo g, int brows) {
  pdl_launch_dependents();
  pdl_wait();   // (reads global memory from its first instruction: only the launch latency overlaps)
  extern __shared__ float sm[];
  constexpr int J = C / 2;
  const int bands = g.H / brows;               // > 1 only with ipc == 1
  const bool banded = bands > 1;
  const int halo = banded ? g.W : 0;
  const int tile = banded ? brows * g.W : g.pixt;
  const int ldp = tile + 2 * halo + 1;
  float* dhs = sm;
  float* dbs = dhs + C * ldp;
  uint4* cst = reinterpret_cast<uint4*>(dbs + ((C + 3) & ~3));
  const int tid = threadIdx.x;
  const int HWm = g.HW - 1, Wm = g.W - 1;
  const int ngroups = banded ? g.B * bands : (g.B + g.ipc - 1) / g.ipc;
  constexpr int K3 = 9 * C;
  constexpr int NCH = (K3 + 7) / 8;
  const int r16 = K3p / 8, rs16 = r16 + 1;
  int noff[9];
#pragma unroll
  for (int tap = 0; tap < 9; ++tap) noff[tap] = -((tap / 3 - 1) * g.W + (tap % 3 - 1));   // P[m'] fed pixel m' - off
  for (int i = tid; i < C; i += ZT) dbs[i] = 0.f;

  for (int grp = blockIdx.x; grp < ngroups; grp += gridDim.x) {
    const int b0 = banded ? grp / bands : grp * g.ipc;
    const int p0 = banded ? (grp - b0 * bands) * tile : 0;   // first pixel of the band inside its image
    const int nimg = banded ? 1 : min(g.ipc, g.B - b0);
    const int npix = banded ? tile : nimg << g.lgHW;
    const int np2 = npix + 2 * halo;
    __syncthreads();   // previous group's tiles are free (also orders the dbs zeroing)
    // ---- phase 1: UN items per thread at a time, every global load of the batch in flight before the first use
    constexpr int UN = 4;
    for (int i0 = tid; i0 < J * np2; i0 += UN * ZT) {
      float g1[UN], g2[UN], o2[UN], glv[UN];
      float2 hh[UN];
      long long lo[UN];
      int pqv[UN], jjv[UN];
      bool inr[UN], ownv[UN];
#pragma unroll
      for (int u = 0; u < UN; ++u) {
        const int i = i0 + u * ZT;
        const int jj = i / np2, pq = i - jj * np2;     // pixel fastest (np2 is a multiple of 32 or the whole tile)
        const int pl = pq - halo;
        const int img = banded ? 0 : pl >> g.lgHW;
        const int rem = banded ? p0 + pl : pl & HWm;
        jjv[u] = jj; pqv[u] = pq;
        ownv[u] = i < J * np2 && pl >= 0 && pl < npix;
        inr[u] = i < J * np2 && rem >= 0 && rem < g.HW;
        g1[u] = g2[u] = o2[u] = glv[u] = 0.f;
        hh[u] = make_float2(0.f, 0.f);
        lo[u] = 0;
        if (inr[u]) {
          lo[u] = ((static_cast<long long>(b0 + img) * C + jj) << g.lgHW) + rem;
          const long long hi = lo[u] + (static_cast<long long>(J) << g.lgHW);
          const long long m = (static_cast<long long>(b0 + img) << g.lgHW) + rem;
          g2[u] = g_out[hi];
          o2[u] = z_out[hi];
          hh[u] = *reinterpret_cast<const float2*>(hsave + m * C + 2 * jj);
          glv[u] = g_ld[b0 + img];
          if (ownv[u]) g1[u] = g_out[lo[u]];
        }
      }
#pragma unroll
      for (int u = 0; u < UN; ++u) {
        if (i0 + u * ZT >= J * np2) continue;   // warp-uniform: J * np2 is a multiple of 32 whenever shuffles are used
        float dsh = 0.f, dlg = 0.f;
        if (inr[u]) {
          float sg, lsv;
          sigmoid_logsigmoid(hh[u].y + 2.f, sg, lsv);
          dsh = INV ? -g2[u] : g2[u] * sg;
          dlg = INV ? -(g2[u] * (o2[u] + hh[u].x) + glv[u]) * (1.f - sg) : (g2[u] * o2[u] + glv[u]) * (1.f - sg);
          if (ownv[u]) {
            // z1 passes through; the coupling-net gradient is added by affine1x1_bwd (col2im_add in the inverse pass)
            dy[lo[u]] = g1[u];
            dy[lo[u] + (static_cast<long long>(J) << g.lgHW)] = INV ? g2[u] / sg : dsh;   // dL/dy2 (dL/dz2)
          }
        }
        const int jj = jjv[u];
        dhs[(2 * jj) * ldp + pqv[u]] = dsh;
        dhs[(2 * jj + 1) * ldp + pqv[u]] = dlg;
        // bias gradient: a warp's 32 items share jj whenever np2 % 32 == 0 (always for >= 2 images of >= 16 pixels)
        float a = ownv[u] ? dsh : 0.f, bsum = ownv[u] ? dlg : 0.f;
        if ((np2 & 31) == 0) {
          for (int o = 16; o > 0; o >>= 1) {
            a += __shfl_xor_sync(0xffffffffu, a, o);
            bsum += __shfl_xor_sync(0xffffffffu, bsum, o);
          }
          if ((tid & 31) == 0) { atomicAdd(&dbs[2 * jj], a); atomicAdd(&dbs[2 * jj + 1], bsum); }
        } else {
          atomicAdd(&dbs[2 * jj], a);
          atomicAdd(&dbs[2 * jj + 1], bsum);
        }
      }
    }
    __syncthreads();
    // ---- phase 2: im2col rows of dh (thread = pixel, small tiles share a pixel between GR threads)
    const int GR = tile >= ZT ? 1 : ZT / tile;
    const int gid = tid / tile;
    for (int pl = GR > 1 ? (tid & (tile - 1)) : tid; pl < npix; pl += (GR > 1 ? tile : ZT)) {
      const int rem = banded ? p0 + pl : pl & HWm;
      const int yy = rem >> g.lgW, xx = rem & Wm;
      uint32_t vmask = 0;
#pragma unroll
      for (int tap = 0; tap < 9; ++tap) {
        const int ny = yy - (tap / 3 - 1), nx = xx - (tap % 3 - 1);
        vmask |= (ny >= 0 && ny < g.H && nx >= 0 && nx < g.W) ? (1u << tap) : 0u;
      }
      const float* db = dhs + halo + pl;
      uint4* drow = cst + pl * rs16;
#pragma unroll
      for (int c4 = 0; c4 < NCH; ++c4) {
        if (GR > 1 && (c4 & (GR - 1)) != gid) continue;
        float v[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const int k = c4 * 8 + e;
          if (k < K3) {
            const int tap = k / C, co = k % C;
            v[e] = ((vmask >> tap) & 1u) ? db[co * ldp + noff[tap]] : 0.f;
          } else {
            v[e] = 0.f;
          }
        }
        drow[c4] = make_uint4(bf2(v[0], v[1]), bf2(v[2], v[3]), bf2(v[4], v[5]), bf2(v[6], v[7]));
      }
      for (int c4 = NCH; c4 < r16; ++c4)
        if (GR == 1 || (c4 & (GR - 1)) == gid) drow[c4] = make_uint4(0u, 0u, 0u, 0u);
    }
    __syncthreads();
    uint4* out4 = reinterpret_cast<uint4*>(dhcol + ((static_cast<long long>(b0) << g.lgHW) + p0) * K3p);
    copy_out_rows(out4, cst, npix, r16, rs16, tid);
  }
  __syncthreads();
  for (int i = tid; i < C; i += ZT) atomicAdd(dbias3 + i, dbs[i]);
}

// ------------------------------------------------------------------------------------------ affine1x1 bwd
// Persistent CTAs over groups of whole images. col2im of the first conv's input gradient straight from global
// (thread = (pixel, channel), channel fastest: the CH lanes of a pixel read one contiguous segment per tap),
// dx = W'^T dy, and dW' / db' accumulated in shared memory across all groups of the CTA (4x4 register blocks),
// flushed with one global atomic per entry and CTA.
// smem: WT[C*C] | dys[C*ldp] | xs[C*ldp] | acc[C*C + C]
template <int C>
__global__ void __launch_bounds__(ZT)
affine1x1_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ dcol, int K1p,
                     const float* __restrict__ x, const float* __restrict__ Wf, float* __restrict__ dx,
                     float* __restrict__ dWf, float* __restrict__ dbf, Geo g, int tile_floats) {
  pdl_launch_dependents();
  pdl_wait();   // (reads global memory from its first instruction: only the launch latency overlaps)
  extern __shared__ float sm[];
  constexpr int CH = C / 2;
  const int ldp = g.pixt + 1;
  float* WT = sm;
  float* dys = WT + C * C;
  float* xs = dys + C * ldp;
  float* acc = dys + tile_floats;   // tile_floats >= 2*C*ldp, and >= the slice-reduction scratch at the end
  const int tid = threadIdx.x;
  const int HWm = g.HW - 1;
  const int ngroups = (g.B + g.ipc - 1) / g.ipc;

  for (int i = tid; i < C * C; i += ZT) {
    const int o = i / C, c = i % C;
    WT[c * C + o] = Wf[i];
  }
  for (int i = tid; i < C * C + C; i += ZT) acc[i] = 0.f;
  constexpr int NBK = (C / 4) * (C / 4);              // 4x4 blocks of dW'
  constexpr int SL = NBK >= ZT ? 1 : ZT / NBK;        // pixel slices per block
  constexpr int RB = (NBK + ZT - 1) / ZT;             // blocks per thread
  float wacc[RB][4][4] = {};

  for (int grp = blockIdx.x; grp < ngroups; grp += gridDim.x) {
    const int b0 = grp * g.ipc;
    const int nimg = min(g.ipc, g.B - b0);
    const int npix = nimg << g.lgHW;
    __syncthreads();
    // coalesced tile loads (pixel fastest), four (x, dy) pairs per thread in flight at a time
    {
      constexpr int UL = 4;
      const int total = C * npix;
      for (int i0 = tid; i0 < total; i0 += UL * ZT) {
        float xv[UL], dv[UL];
        int so[UL];
#pragma unroll
        for (int u = 0; u < UL; ++u) {
          const int i = i0 + u * ZT;
          xv[u] = dv[u] = 0.f;
          so[u] = -1;
          if (i < total) {
            const int c = i / npix, pl = i - c * npix;
            const int img = pl >> g.lgHW, rem = pl & HWm;
            const long long gi = ((static_cast<long long>(b0 + img) * C + c) << g.lgHW) + rem;
            xv[u] = x[gi];
            dv[u] = dy[gi];
            so[u] = c * ldp + pl;
          }
        }
#pragma unroll
        for (int u = 0; u < UL; ++u)
          if (so[u] >= 0) { xs[so[u]] = xv[u]; dys[so[u]] = dv[u]; }
      }
    }
    __syncthreads();
    if (dcol) {
      // dy1[ci, m] += sum_tap dcol[m - off(tap), tap*CH + ci], three items per thread at a time
      constexpr int UN = 3;
      for (int i0 = tid; i0 < CH * npix; i0 += UN * ZT) {
        float a[UN];
        col2im_gather<CH, UN>(dcol, K1p, g, static_cast<long long>(b0) << g.lgHW, i0, CH * npix, a);
#pragma unroll
        for (int u = 0; u < UN; ++u) {
          const int i = i0 + u * ZT;
          if (i < CH * npix) {
            const int pl = i / CH, ci = i - pl * CH;
            dys[ci * ldp + pl] += a[u];
          }
        }
      }
      __syncthreads();
    }
    // dx = W'^T dy
    for (int pl = tid; pl < npix; pl += ZT) {
      const int img = pl >> g.lgHW, rem = pl & HWm;
      float dv[C];
#pragma unroll
      for (int o = 0; o < C; ++o) dv[o] = dys[o * ldp + pl];
      float* dxp = dx + ((static_cast<long long>(b0 + img) * C) << g.lgHW) + rem;
#pragma unroll 4
      for (int i = 0; i < C; ++i) {
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
    // dW'[o][i] += sum_p dy[o][p] x[i][p]: 4x4 register blocks, pixel range split over thread slices; the partial
    // sums stay in registers across all groups of this CTA
#pragma unroll
    for (int rb = 0; rb < RB; ++rb) {
      const int blk = (NBK < ZT ? tid % NBK : tid) + rb * ZT;
      const int slice = NBK < ZT ? tid / NBK : 0;
      if (blk >= NBK || slice >= SL) continue;
      const int to = blk / (C / 4), ti = blk % (C / 4);
      for (int p = slice; p < npix; p += SL) {
        float dv[4], xv[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          dv[q] = dys[(4 * to + q) * ldp + p];
          xv[q] = xs[(4 * ti + q) * ldp + p];
        }
#pragma unroll
        for (int q = 0; q < 4; ++q)
#pragma unroll
          for (int r = 0; r < 4; ++r) wacc[rb][q][r] = fmaf(dv[q], xv[r], wacc[rb][q][r]);
      }
    }
    // db'[o] += sum_p dy[o][p]: one warp per channel
    {
      const int warp = tid >> 5, lane = tid & 31;
      for (int o = warp; o < C; o += ZT / 32) {
        float a = 0.f;
        for (int p = lane; p < npix; p += 32) a += dys[o * ldp + p];
        for (int sft = 16; sft > 0; sft >>= 1) a += __shfl_xor_sync(0xffffffffu, a, sft);
        if (lane == 0) acc[C * C + o] += a;
      }
    }
  }
  // the pixel slices of a block meet through a scratch tile (the x / dy tiles are dead now): shared-memory float
  // atomics are CAS loops, and up to 28 slices would fight over each entry
  __syncthreads();
  float* scratch = dys;   // dys and xs are contiguous: 2*C*ldp floats >= SL * C * C for every supported shape
#pragma unroll
  for (int rb = 0; rb < RB; ++rb) {
    const int blk = (NBK < ZT ? tid % NBK : tid) + rb * ZT;
    const int slice = NBK < ZT ? tid / NBK : 0;
    if (blk >= NBK || slice >= SL) continue;
    const int to = blk / (C / 4), ti = blk % (C / 4);
#pragma unroll
    for (int q = 0; q < 4; ++q)
#pragma unroll
      for (int r = 0; r < 4; ++r) scratch[slice * C * C + (4 * to + q) * C + 4 * ti + r] = wacc[rb][q][r];
  }
  __syncthreads();
  for (int i = tid; i < C * C; i += ZT) {
    float a = 0.f;
    for (int sl2 = 0; sl2 < SL; ++sl2) a += scratch[sl2 * C * C + i];
    acc[i] += a;
  }
  __syncthreads();
  for (int i = tid; i < C * C; i += ZT) atomicAdd(dWf + i, acc[i]);
  for (int i = tid; i < C; i += ZT) atomicAdd(dbf + i, acc[C * C + i]);
}

// ------------------------------------------------------------------------------------------ col2im add
// dz[:, :C/2] += col2im(dcol) in place. CTA = C2I_UN * ZT / CH consecutive pixels x CH channels = C2I_UN * ZT items,
// one col2im_gather per thread; no shared memory. Reads dcol once (HBM-bound), read-modify-writes the z1 half of dz.
constexpr int C2I_UN = 3;
template <int C>
__global__ void __launch_bounds__(ZT)
col2im_add_kernel(const float* __restrict__ dcol, int K1p, float* __restrict__ dz, Geo g) {
  pdl_launch_dependents();
  pdl_wait();
  constexpr int CH = C / 2;
  constexpr int PPC = C2I_UN * ZT / CH;   // pixels per CTA (C2I_UN * ZT is a multiple of every CH)
  const long long M = static_cast<long long>(g.B) << g.lgHW;
  const long long m0 = static_cast<long long>(blockIdx.x) * PPC;
  const int nitems = static_cast<int>(min(static_cast<long long>(PPC), M - m0)) * CH;
  float a[C2I_UN];
  col2im_gather<CH, C2I_UN>(dcol, K1p, g, m0, threadIdx.x, nitems, a);
#pragma unroll
  for (int u = 0; u < C2I_UN; ++u) {
    const int i = threadIdx.x + u * ZT;
    if (i < nitems) {
      const int pl = i / CH, ci = i - pl * CH;
      const long long m = m0 + pl;
      dz[((((m >> g.lgHW) * C) + ci) << g.lgHW) + (m & (g.HW - 1))] += a[u];
    }
  }
}

static Geo make_geo(int B, int C, int H, int W, bool heavy) {
  Geo g;
  g.B = B; g.H = H; g.W = W; g.HW = H * W;
  int target = heavy ? (C <= 24 ? 256 : (C <= 48 ? 128 : 64)) : 256;
  g.ipc = g.HW >= target ? 1 : target / g.HW;
  if (g.ipc > B) g.ipc = B;
  // small images: prefer >= 2 CTAs per SM over fat CTAs (these kernels are latency-bound when the grid is small)
  while (g.ipc > 1 && (B + g.ipc - 1) / g.ipc < 2 * 148) g.ipc >>= 1;
  g.pixt = g.ipc * g.HW;
  g.og = 1;
  g.lgW = 0; while ((1 << g.lgW) < W) ++g.lgW;
  g.lgHW = 0; while ((1 << g.lgHW) < g.HW) ++g.lgHW;
  return g;
}

static bool pow2(int v) { return v > 0 && (v & (v - 1)) == 0; }

template <typename K>
static int ensure_smem(K kernel, int bytes) {
  return ensure_dyn_smem(reinterpret_cast<const void*>(kernel), bytes);
}

#define NFK_DISPATCH_C(C_, ...)                             \
  switch (C_) {                                             \
    case 12: { constexpr int CC = 12; __VA_ARGS__; } break; \
    case 24: { constexpr int CC = 24; __VA_ARGS__; } break; \
    case 48: { constexpr int CC = 48; __VA_ARGS__; } break; \
    case 96: { constexpr int CC = 96; __VA_ARGS__; } break; \
    default: return NFK_ERR_SHAPE;                          \
  }

}  // namespace nfk

using namespace nfk;

extern "C" int nfk_affine1x1_fwd(const float* x, const float* Wf, const float* bf, const float* sl, float* y,
                                 void* col, int K1p, const float* ld_in, float* ld_out, int B, int C, int H, int W,
                                 void* stream) {
  if (B <= 0 || H <= 0 || W <= 0 || H * W > 4096 || !pow2(H) || !pow2(W)) return NFK_ERR_SHAPE;
  if (!x || (!Wf && !col) || (Wf && (!bf || !y)) || (ld_out && (!ld_in || !sl))) return NFK_ERR_ARG;
  if (col && (K1p % 64 || K1p < 9 * (C / 2))) return NFK_ERR_SHAPE;
  Geo g = make_geo(B, C, H, W, false);
  if (col) {
    // keep the im2col staging tile (pixt rows of K1p bf16) under ~64 KB
    while (g.ipc > 1 && static_cast<long long>(g.pixt) * (K1p * 2 + 16) > 64 * 1024) { g.ipc >>= 1; g.pixt = g.ipc * g.HW; }
  }
  {
    // few pixels in flight -> split the C outputs of a pixel over 2 or 4 threads
    const long long M = static_cast<long long>(B) * H * W;
    g.og = M >= 131072 ? 1 : (M >= 32768 ? 2 : (M >= 8192 && C < 48 ? 4 : 8));
    while (g.og > 1 && (C % g.og || (C / g.og) % 2)) g.og >>= 1;
  }
  // 4x4 maps: a CTA of 4 images (64 pixels) leaves half of the threads idle in every phase; twice the images per CTA
  // measured 23.8 -> 15.2 us at B = 2048 (tools/aff_sweep.py) as long as every SM still gets a CTA
  if (col && g.HW <= 16)
    while (g.pixt < 128 && 2 * g.ipc <= B && (B + 2 * g.ipc - 1) / (2 * g.ipc) >= 148) { g.ipc <<= 1; g.pixt = g.ipc * g.HW; }
  const int smem = (C * C + C + (col ? (C / 2) * (g.pixt + 1) + 4 + g.pixt * (K1p / 8 + 1) * 4 : 0)) * 4;
  const int grid = (B + g.ipc - 1) / g.ipc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  NFK_DISPATCH_C(C, {
    int rc = ensure_smem(affine1x1_fwd_kernel<CC>, smem);
    if (rc) return rc;
    if (launch_pdl(affine1x1_fwd_kernel<CC>, dim3(grid), dim3(ZT), smem, st, x, Wf, bf, sl, y,
                   static_cast<__nv_bfloat16*>(col), ld_in, ld_out, g, K1p) != cudaSuccess)
      return NFK_ERR_LAUNCH;
  });
  return cudaGetLastError() == cudaSuccess ? NFK_OK : NFK_ERR_LAUNCH;
}

extern "C" int nfk_coupling_fwd(const float* P, int K3p, const float* bias3, float* y, float* hsave, float* ld,
                                int B, int C, int H, int W, int reverse, void* stream) {
  if (B <= 0 || H <= 0 || W <= 0 || H * W > 4096 || K3p < 9 * C || K3p % 2 || !pow2(H) || !pow2(W))
    return NFK_ERR_SHAPE;
  if (!P || !bias3 || !y) return NFK_ERR_ARG;
  Geo g = make_geo(B, C, H, W, false);
  const long long items = static_cast<long long>(B) * H * W * (C / 2);
  const unsigned grid = static_cast<unsigned>((items + ZT - 1) / ZT);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  NFK_DISPATCH_C(C, { coupling_fwd_kernel<CC><<<grid, ZT, 0, st>>>(P, K3p, bias3, y, hsave, ld, g, reverse); });
  return cudaGetLastError() == cudaSuccess ? NFK_OK : NFK_ERR_LAUNCH;
}

namespace nfk {
// Launch of coupling_bwd_kernel in either direction (the two entry points below share the shape limits and sizing).
template <bool INV>
static int coupling_bwd_launch(const float* g_out, const float* g_ld, const float* z_out, const float* hsave,
                               float* dy, void* dhcol, int K3p, float* dbias3, int B, int C, int H, int W,
                               void* stream) {
  if (B <= 0 || H <= 0 || W <= 0 || H * W > 4096 || K3p % 64 || K3p < 9 * C || !pow2(H) || !pow2(W))
    return NFK_ERR_SHAPE;
  if (!g_out || !g_ld || !z_out || !hsave || !dy || !dhcol || !dbias3) return NFK_ERR_ARG;
  Geo g = make_geo(B, C, H, W, true);
  // keep the dh tile + the im2col staging under ~100 KB so two CTAs fit per SM: fewer images per group first, then
  // bands of image rows (with a one-row halo) once a single image is too large
  auto bytes = [&](int tile, int halo) {
    return static_cast<long long>(C * (tile + 2 * halo + 1) + ((C + 3) & ~3)) * 4 +
           static_cast<long long>(tile) * (K3p / 8 + 1) * 16 + 16;
  };
  while (g.ipc > 1 && bytes(g.pixt, 0) > 100 * 1024) { g.ipc >>= 1; g.pixt = g.ipc * g.HW; }
  int brows = H;
  if (g.ipc == 1)
    while (brows > 1 && bytes(brows * W, brows < H ? W : 0) > 100 * 1024) brows >>= 1;
  const bool banded = brows < H;
  const int smem = static_cast<int>(bytes(banded ? brows * W : g.pixt, banded ? W : 0));
  const int groups = banded ? B * (H / brows) : (B + g.ipc - 1) / g.ipc;
  const int grid = groups < 4 * 148 ? groups : 4 * 148;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  NFK_DISPATCH_C(C, {
    int rc = ensure_smem(coupling_bwd_kernel<CC, INV>, smem);
    if (rc) return rc;
    if (launch_pdl(coupling_bwd_kernel<CC, INV>, dim3(grid), dim3(ZT), smem, st, g_out, g_ld, z_out, hsave, dy,
                   static_cast<__nv_bfloat16*>(dhcol), K3p, dbias3, g, brows) != cudaSuccess)
      return NFK_ERR_LAUNCH;
  });
  return cudaGetLastError() == cudaSuccess ? NFK_OK : NFK_ERR_LAUNCH;
}
}  // namespace nfk

extern "C" int nfk_coupling_bwd(const float* g_out, const float* g_ld, const float* z_out, const float* hsave,
                                float* dy, void* dhcol, int K3p, float* dbias3, int B, int C, int H, int W,
                                void* stream) {
  return coupling_bwd_launch<false>(g_out, g_ld, z_out, hsave, dy, dhcol, K3p, dbias3, B, C, H, W, stream);
}

extern "C" int nfk_coupling_inv_bwd(const float* g_zc, const float* g_ld, const float* zc, const float* hsave,
                                    float* dz, void* dhcol, int K3p, float* dbias3, int B, int C, int H, int W,
                                    void* stream) {
  return coupling_bwd_launch<true>(g_zc, g_ld, zc, hsave, dz, dhcol, K3p, dbias3, B, C, H, W, stream);
}

extern "C" int nfk_affine1x1_bwd(const float* dy, const float* dcol, int K1p, const float* x, const float* Wf,
                                 float* dx, float* dWf, float* dbf, int B, int C, int H, int W, void* stream) {
  if (B <= 0 || H <= 0 || W <= 0 || H * W > 4096 || !pow2(H) || !pow2(W)) return NFK_ERR_SHAPE;
  if (!dy || !x || !Wf || !dx || !dWf || !dbf) return NFK_ERR_ARG;
  Geo g = make_geo(B, C, H, W, true);
  const int nbk = (C / 4) * (C / 4);
  const int slices = nbk >= ZT ? 1 : ZT / nbk;
  int tile_floats = 2 * C * (g.pixt + 1);
  if (tile_floats < slices * C * C) tile_floats = slices * C * C;   // scratch of the final slice reduction
  const int smem = (C * C + tile_floats + C * C + C) * 4;
  const int groups = (B + g.ipc - 1) / g.ipc;
  const int grid = groups < 4 * 148 ? groups : 4 * 148;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  NFK_DISPATCH_C(C, {
    int rc = ensure_smem(affine1x1_bwd_kernel<CC>, smem);
    if (rc) return rc;
    if (launch_pdl(affine1x1_bwd_kernel<CC>, dim3(grid), dim3(ZT), smem, st, dy, dcol, K1p, x, Wf, dx, dWf, dbf, g,
                   tile_floats) != cudaSuccess)
      return NFK_ERR_LAUNCH;
  });
  return cudaGetLastError() == cudaSuccess ? NFK_OK : NFK_ERR_LAUNCH;
}

extern "C" int nfk_col2im_add(const float* dcol, int K1p, float* dz, int B, int C, int H, int W, void* stream) {
  if (B <= 0 || H <= 0 || W <= 0 || H * W > 4096 || !pow2(H) || !pow2(W) || K1p < 9 * (C / 2)) return NFK_ERR_SHAPE;
  if (!dcol || !dz) return NFK_ERR_ARG;
  Geo g = make_geo(B, C, H, W, false);
  const long long M = static_cast<long long>(B) * H * W;
  const long long ppc = C2I_UN * ZT / (C / 2);
  const unsigned grid = static_cast<unsigned>((M + ppc - 1) / ppc);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  NFK_DISPATCH_C(C, {
    if (launch_pdl(col2im_add_kernel<CC>, dim3(grid), dim3(ZT), 0, st, dcol, K1p, dz, g) != cudaSuccess)
      return NFK_ERR_LAUNCH;
  });
  return cudaGetLastError() == cudaSuccess ? NFK_OK : NFK_ERR_LAUNCH;
}
