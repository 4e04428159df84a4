// MAF / MADE support kernels. The reference repository lists MAF in its README but ships no code for it
// (SURVEY.md §0.2), so these follow Papamakarios et al. 2017 (MAF) / Germain et al. 2015 (MADE):
//   (mu, alpha) = MADE(x),  u_i = (x_i - mu_i) * exp(-alpha_i),  log|det| = -sum_i alpha_i,
// with mu_i, alpha_i depending on x_{<i} only. The three masked linears run on the tcgen05 GEMM tiles
// (nfk_gemm_nt_bf16_ranged skips the structurally-zero k-blocks of the degree-sorted hidden mask); this file holds
// the weight masking / packing and the HBM-bound elementwise transforms around them.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <cstdint>

#include "../../include/nfk.h"

namespace nfk {

// masks: m1[o][i] = deg1[o] >= i+1 ; m2[o][k] = deg2[o] >= deg1[k] ; m3[r][k] = (r % D) + 1 > deg2[k]
__global__ void made_prep_kernel(const float* __restrict__ w1, const float* __restrict__ w2,
                                 const float* __restrict__ w3, const int* __restrict__ deg1,
                                 const int* __restrict__ deg2, int D, int H, int Dp, int N3p,
                                 __nv_bfloat16* __restrict__ B1, __nv_bfloat16* __restrict__ B1T,
                                 __nv_bfloat16* __restrict__ B2, __nv_bfloat16* __restrict__ B2T,
                                 __nv_bfloat16* __restrict__ B3, __nv_bfloat16* __restrict__ B3T, int with_t) {
  const long long n1 = static_cast<long long>(H) * Dp, n2 = static_cast<long long>(H) * H,
                  n3 = static_cast<long long>(N3p) * H;
  for (long long e = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; e < n1 + n2 + n3;
       e += static_cast<long long>(gridDim.x) * blockDim.x) {
    if (e < n1) {
      const int o = static_cast<int>(e / Dp), i = static_cast<int>(e % Dp);
      const float v = (i < D && deg1[o] >= i + 1) ? w1[o * D + i] : 0.f;
      const __nv_bfloat16 h = __float2bfloat16_rn(v);
      B1[e] = h;
      if (with_t) B1T[static_cast<long long>(i) * H + o] = h;
    } else if (e < n1 + n2) {
      const long long q = e - n1;
      const int o = static_cast<int>(q / H), k = static_cast<int>(q % H);
      const __nv_bfloat16 h = __float2bfloat16_rn(deg2[o] >= deg1[k] ? w2[q] : 0.f);
      B2[q] = h;
      if (with_t) B2T[static_cast<long long>(k) * H + o] = h;
    } else {
      const long long q = e - n1 - n2;
      const int r = static_cast<int>(q / H), k = static_cast<int>(q % H);
      const float v = (r < 2 * D && (r % D) + 1 > deg2[k]) ? w3[static_cast<long long>(r) * H + k] : 0.f;
      const __nv_bfloat16 h = __float2bfloat16_rn(v);
      B3[q] = h;
      if (with_t) B3T[static_cast<long long>(k) * N3p + r] = h;
    }
  }
}

__global__ void made_prep_bwd_kernel(const float* __restrict__ dB1, const float* __restrict__ dB2,
                                     const float* __restrict__ dB3, const int* __restrict__ deg1,
                                     const int* __restrict__ deg2, int D, int H, int Dp, float* __restrict__ dw1,
                                     float* __restrict__ dw2, float* __restrict__ dw3) {
  const long long n1 = static_cast<long long>(H) * D, n2 = static_cast<long long>(H) * H,
                  n3 = 2LL * D * H;
  for (long long e = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; e < n1 + n2 + n3;
       e += static_cast<long long>(gridDim.x) * blockDim.x) {
    if (e < n1) {
      const int o = static_cast<int>(e / D), i = static_cast<int>(e % D);
      dw1[e] = deg1[o] >= i + 1 ? dB1[static_cast<long long>(o) * Dp + i] : 0.f;
    } else if (e < n1 + n2) {
      const long long q = e - n1;
      const int o = static_cast<int>(q / H), k = static_cast<int>(q % H);
      dw2[q] = deg2[o] >= deg1[k] ? dB2[q] : 0.f;
    } else {
      const long long q = e - n1 - n2;
      const int r = static_cast<int>(q / H), k = static_cast<int>(q % H);
      dw3[q] = (r % D) + 1 > deg2[k] ? dB3[q] : 0.f;
    }
  }
}

// x [B, D] fp32 -> xb [B, Dp] bf16 (zero padded); one thread per (row, 8-column chunk)
__global__ void rows_to_bf16_kernel(const float* __restrict__ x, int B, int D, int Dp,
                                    __nv_bfloat16* __restrict__ xb) {
  const long long total = static_cast<long long>(B) * Dp;
  for (long long e = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; e < total;
       e += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long r = e / Dp;
    const int c = static_cast<int>(e - r * Dp);
    xb[e] = __float2bfloat16_rn(c < D ? x[r * D + c] : 0.f);
  }
}

// One warp per sample. out = [mu | alpha] (+bias3 already added by the GEMM epilogue), row stride N3p.
// u = (x - mu) exp(-alpha) written flipped (next layer sees the reversed ordering) when flip != 0, plus its bf16 copy.
__global__ void made_affine_fwd_kernel(const float* __restrict__ x, const float* __restrict__ out, int N3p,
                                       float* __restrict__ u, __nv_bfloat16* __restrict__ ub, int Dp,
                                       const float* __restrict__ ld_in, float* __restrict__ ld_out, int B, int D,
                                       int flip) {
  const int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (b >= B) return;
  const float* xr = x + static_cast<long long>(b) * D;
  const float* orow = out + static_cast<long long>(b) * N3p;
  float acc = 0.f;
  for (int i = lane; i < Dp; i += 32) {
    float v = 0.f;
    const int src = flip ? D - 1 - i : i;  // output position i takes element src
    if (i < D) {
      const float mu = orow[src], al = orow[D + src];
      v = (xr[src] - mu) * expf(-al);
      acc -= al;
      u[static_cast<long long>(b) * D + i] = v;
    }
    if (ub) ub[static_cast<long long>(b) * Dp + i] = __float2bfloat16_rn(v);
  }
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0 && ld_out) ld_out[b] = ld_in[b] + acc;
}

// Backward of u = (x - mu) e^{-alpha}, ld -= sum alpha:  dx = g e^{-a}, dmu = -g e^{-a}, dalpha = -g u - g_ld.
// g_u is indexed in OUTPUT order (flipped if flip). dout is bf16 [B, N3p] = [dmu | dalpha | 0...].
__global__ void made_affine_bwd_kernel(const float* __restrict__ x, const float* __restrict__ out, int N3p,
                                       const float* __restrict__ g_u, const float* __restrict__ g_ld,
                                       float* __restrict__ dx, __nv_bfloat16* __restrict__ dout,
                                       float* __restrict__ db3, int B, int D, int flip) {
  extern __shared__ float sacc[];  // [2D]
  for (int i = threadIdx.x; i < 2 * D; i += blockDim.x) sacc[i] = 0.f;
  __syncthreads();
  const int warps = blockDim.x >> 5, w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int b = blockIdx.x * warps + w; b < B; b += gridDim.x * warps) {
    const float* xr = x + static_cast<long long>(b) * D;
    const float* orow = out + static_cast<long long>(b) * N3p;
    const float gl = g_ld ? g_ld[b] : 0.f;
    for (int i = lane; i < N3p; i += 32) {
      float v = 0.f;
      if (i < D) {
        const float mu = orow[i], al = orow[D + i];
        const float e = expf(-al);
        const float g = g_u[static_cast<long long>(b) * D + (flip ? D - 1 - i : i)];
        dx[static_cast<long long>(b) * D + i] = g * e;
        v = -g * e;
        atomicAdd(&sacc[i], v);
        const float da = -g * (xr[i] - mu) * e - gl;
        dout[static_cast<long long>(b) * N3p + D + i] = __float2bfloat16_rn(da);
        atomicAdd(&sacc[D + i], da);
      } else if (i < 2 * D) {
        continue;  // alpha slot, written by the lane that owns i - D
      }
      dout[static_cast<long long>(b) * N3p + i] = __float2bfloat16_rn(v);
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * D; i += blockDim.x) atomicAdd(db3 + i, sacc[i]);
}

// Sequential inverse, pass i: x[:, i] = u_in[:, i] * exp(alpha_i) + mu_i with (mu, alpha) = MADE(current x).
// u_in is in the layer's OUTPUT order (flipped if flip). On the last pass ld_out = ld_in + sum alpha.
__global__ void made_inv_update_kernel(float* __restrict__ x, __nv_bfloat16* __restrict__ xb, int Dp,
                                       const float* __restrict__ u_in, const float* __restrict__ out, int N3p,
                                       const float* __restrict__ ld_in, float* __restrict__ ld_out, int B, int D,
                                       int i, int flip, int last) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const float* orow = out + static_cast<long long>(b) * N3p;
  const float uv = u_in[static_cast<long long>(b) * D + (flip ? D - 1 - i : i)];
  const float v = uv * expf(orow[D + i]) + orow[i];
  x[static_cast<long long>(b) * D + i] = v;
  xb[static_cast<long long>(b) * Dp + i] = __float2bfloat16_rn(v);
  if (last && ld_out) {
    float a = 0.f;
    for (int k = 0; k < D; ++k) a += orow[D + k];
    ld_out[b] = ld_in[b] + a;
  }
}

// Gradients of the sequential inverse, pass d (d = D-1 .. 0; the mirror of made_inv_update): with c = the input
// gradient of the network at x for the dout rows finished so far (c[:, d], NULL = zero),
//   mubar_d = g_x,d + c_d,  v_d = e^{alpha_d} mubar_d,  alphabar_d = v_d u_d + g_ld;  g_u[:, d] = v_d (output order),
// dout[:, d] and dout[:, D + d] = bf16(mubar_d, alphabar_d), db3[d], db3[D + d] += their column sums (fp32 values,
// a fixed order within the block, one atomic per block).
__global__ void made_inv_bwd_update_kernel(const float* __restrict__ c, int ldc, const float* __restrict__ g_x,
                                           const float* __restrict__ g_ld, const float* __restrict__ out, int N3p,
                                           const float* __restrict__ u_in, float* __restrict__ g_u,
                                           __nv_bfloat16* __restrict__ dout, float* __restrict__ db3, int B, int D,
                                           int d, int flip) {
  __shared__ float part[2][8];
  const int b = blockIdx.x * blockDim.x + threadIdx.x, lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  float mub = 0.f, alb = 0.f;
  if (b < B) {
    const long long r = b;
    mub = g_x[r * D + d] + (c ? c[r * ldc + d] : 0.f);
    const float v = expf(out[r * N3p + D + d]) * mub;
    alb = v * u_in[r * D + (flip ? D - 1 - d : d)] + (g_ld ? g_ld[b] : 0.f);
    g_u[r * D + (flip ? D - 1 - d : d)] = v;
    dout[r * N3p + d] = __float2bfloat16_rn(mub);
    dout[r * N3p + D + d] = __float2bfloat16_rn(alb);
  }
  for (int o = 16; o > 0; o >>= 1) {
    mub += __shfl_xor_sync(0xffffffffu, mub, o);
    alb += __shfl_xor_sync(0xffffffffu, alb, o);
  }
  if (lane == 0) {
    part[0][w] = mub;
    part[1][w] = alb;
  }
  __syncthreads();
  if (threadIdx.x < 2) {
    float s = 0.f;
    for (int i = 0; i < (blockDim.x >> 5); ++i) s += part[threadIdx.x][i];
    atomicAdd(db3 + (threadIdx.x ? D + d : d), s);
  }
}

}  // namespace nfk

using namespace nfk;

static inline int grid_for(long long n, int cap = 1184) {
  const long long g = (n + 255) / 256;
  return static_cast<int>(g < cap ? (g < 1 ? 1 : g) : cap);
}

extern "C" int nfk_made_prep(const float* w1, const float* w2, const float* w3, const int* deg1, const int* deg2,
                             int D, int H, int Dp, int N3p, void* B1, void* B1T, void* B2, void* B2T, void* B3,
                             void* B3T, int with_t, void* stream) {
  if (D <= 0 || H <= 0 || H % 64 || Dp % 64 || Dp < D || N3p % 64 || N3p < 2 * D) return NFK_ERR_SHAPE;
  if (!w1 || !w2 || !w3 || !deg1 || !deg2 || !B1 || !B2 || !B3 || (with_t && (!B1T || !B2T || !B3T)))
    return NFK_ERR_ARG;
  const long long n = static_cast<long long>(H) * (Dp + H + N3p);
  made_prep_kernel<<<grid_for(n), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      w1, w2, w3, deg1, deg2, D, H, Dp, N3p, static_cast<__nv_bfloat16*>(B1), static_cast<__nv_bfloat16*>(B1T),
      static_cast<__nv_bfloat16*>(B2), static_cast<__nv_bfloat16*>(B2T), static_cast<__nv_bfloat16*>(B3),
      static_cast<__nv_bfloat16*>(B3T), with_t);
  return cudaGetLastError() == cudaSuccess ? NFK_OK : NFK_ERR_LAUNCH;
}

extern "C" int nfk_made_prep_bwd(const float* dB1, const float* dB2, const float* dB3, const int* deg1,
                                 const int* deg2, int D, int H, int Dp, float* dw1, float* dw2, float* dw3,
                                 void* stream) {
  if (D <= 0 || H <= 0) return NFK_ERR_SHAPE;
  if (!dB1 || !dB2 || !dB3 || !deg1 || !deg2 || !dw1 || !dw2 || !dw3) return NFK_ERR_ARG;
  const long long n = static_cast<long long>(H) * (D + H + 2 * D);
  made_prep_bwd_kernel<<<grid_for(n), 256, 0, static_cast<cudaStream_t>(stream)>>>(dB1, dB2, dB3, deg1, deg2, D, H,
                                                                                  Dp, dw1, dw2, dw3);
  return cudaGetLastError() == cudaSuccess ? NFK_OK : NFK_ERR_LAUNCH;
}

extern "C" int nfk_rows_to_bf16(const float* x, int B, int D, int Dp, void* xb, void* stream) {
  if (B <= 0 || D <= 0 || Dp < D) return NFK_ERR_SHAPE;
  if (!x || !xb) return NFK_ERR_ARG;
  rows_to_bf16_kernel<<<grid_for(static_cast<long long>(B) * Dp), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      x, B, D, Dp, static_cast<__nv_bfloat16*>(xb));
  return cudaGetLastError() == cudaSuccess ? NFK_OK : NFK_ERR_LAUNCH;
}

extern "C" int nfk_made_affine_fwd(const float* x, const float* out, int N3p, float* u, void* ub, int Dp,
                                   const float* ld_in, float* ld_out, int B, int D, int flip, void* stream) {
  if (B <= 0 || D <= 0 || N3p < 2 * D || (ub && Dp < D)) return NFK_ERR_SHAPE;
  if (!x || !out || !u || (ld_out && !ld_in)) return NFK_ERR_ARG;
  const long long threads = static_cast<long long>(B) * 32;
  made_affine_fwd_kernel<<<static_cast<int>((threads + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      x, out, N3p, u, static_cast<__nv_bfloat16*>(ub), ub ? Dp : D, ld_in, ld_out, B, D, flip);
  return cudaGetLastError() == cudaSuccess ? NFK_OK : NFK_ERR_LAUNCH;
}

extern "C" int nfk_made_affine_bwd(const float* x, const float* out, int N3p, const float* g_u, const float* g_ld,
                                   float* dx, void* dout, float* db3, int B, int D, int flip, void* stream) {
  if (B <= 0 || D <= 0 || N3p < 2 * D) return NFK_ERR_SHAPE;
  if (!x || !out || !g_u || !dx || !dout || !db3) return NFK_ERR_ARG;
  const int grid = (B + 7) / 8 < 592 ? (B + 7) / 8 : 592;
  made_affine_bwd_kernel<<<grid, 256, 2 * D * sizeof(float), static_cast<cudaStream_t>(stream)>>>(
      x, out, N3p, g_u, g_ld, dx, static_cast<__nv_bfloat16*>(dout), db3, B, D, flip);
  return cudaGetLastError() == cudaSuccess ? NFK_OK : NFK_ERR_LAUNCH;
}

extern "C" int nfk_made_inv_update(float* x, void* xb, int Dp, const float* u_in, const float* out, int N3p,
                                   const float* ld_in, float* ld_out, int B, int D, int i, int flip, int last,
                                   void* stream) {
  if (B <= 0 || D <= 0 || i < 0 || i >= D || N3p < 2 * D || Dp < D) return NFK_ERR_SHAPE;
  if (!x || !xb || !u_in || !out || (ld_out && !ld_in)) return NFK_ERR_ARG;
  made_inv_update_kernel<<<(B + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      x, static_cast<__nv_bfloat16*>(xb), Dp, u_in, out, N3p, ld_in, ld_out, B, D, i, flip, last);
  return cudaGetLastError() == cudaSuccess ? NFK_OK : NFK_ERR_LAUNCH;
}

extern "C" int nfk_made_inv_bwd_update(const float* c, int ldc, const float* g_x, const float* g_ld, const float* out,
                                       int N3p, const float* u_in, float* g_u, void* dout, float* db3, int B, int D,
                                       int d, int flip, void* stream) {
  if (B <= 0 || D <= 0 || d < 0 || d >= D || N3p < 2 * D || (c && ldc < D)) return NFK_ERR_SHAPE;
  if (!g_x || !out || !u_in || !g_u || !dout || !db3) return NFK_ERR_ARG;
  made_inv_bwd_update_kernel<<<(B + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      c, ldc, g_x, g_ld, out, N3p, u_in, g_u, static_cast<__nv_bfloat16*>(dout), db3, B, D, d, flip);
  return cudaGetLastError() == cudaSuccess ? NFK_OK : NFK_ERR_LAUNCH;
}
