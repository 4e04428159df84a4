// fp32-class arithmetic for the coupling network on the bf16 tensor-core tiles ("bf16x3" precision mode).
//
// The reference runs its convolutions in fp32 (models/layers.py:209,249; models/flows.py:25-34). A bf16 operand keeps 8
// significand bits; writing a = hi + lo with hi = bf16(a), lo = bf16(a - hi) keeps 16, and
//     a * b  ~=  hi_a hi_b + hi_a lo_b + lo_a hi_b          (dropped term lo_a lo_b: 2^-16 relative)
// is three bf16 products accumulated in fp32 — which a tensor-core GEMM computes in ONE pass when the split parts are
// laid side by side along K:   A3 = [hi | hi | lo]  (activations),   B3 = [hi | lo | hi]  (weights),
//     A3 B3^T = hi_a hi_b^T + hi_a lo_b^T + lo_a hi_b^T.
// So the precise mode reuses nfk_gemm_nt_bf16 / nfk_gemm_tn_bf16 unchanged (3x the MMA work) and needs only the
// elementwise kernels below, which produce the split operands: fp32 -> [hi|hi|lo] with the im2col, the ReLU or the ReLU
// mask fused in. Everything here is HBM-bound streaming code (one element per thread, coalesced rows).
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <cstdint>

#include "../../include/nfk.h"

namespace nfk {

constexpr int S3T = 256;

// Operand layouts along K (each block K wide; h = bf16(a), m = bf16(a - h), l = bf16(a - h - m)):
//   pattern 0  A, 3 terms  [h | h | m]              with pattern 1  B, 3 terms  [h | m | h]          -> hh + hm + mh
//   pattern 2  A, 6 terms  [h | h | h | m | m | l]  with pattern 3  B, 6 terms  [h | m | l | h | m | h]
//                                                    -> hh + hm + hl + mh + mm + lh   (2^-24: fp32 level)
// The 6-term forms were built to bring the forward pre-activations (whose signs are the ReLU masks) to fp32 accuracy;
// measured, they are no better than the 3-term forms (2e-6..5e-6 of max|out| against fp64, tools/x3_check.py): the tensor
// core's fp32 accumulation is the floor. precise.py therefore uses the 3-term forms everywhere; 2 / 3 stay for the check.
__device__ __forceinline__ int split_terms(int pattern) { return pattern >= 2 ? 6 : 3; }

__device__ __forceinline__ void emit_split(__nv_bfloat16* o, int K, int k, float v, int pattern) {
  const __nv_bfloat16 h = __float2bfloat16_rn(v);
  const float r1 = v - __bfloat162float(h);
  const __nv_bfloat16 m = __float2bfloat16_rn(r1);
  if (pattern == 0) { o[k] = h; o[K + k] = h; o[2 * K + k] = m; return; }
  if (pattern == 1) { o[k] = h; o[K + k] = m; o[2 * K + k] = h; return; }
  const __nv_bfloat16 l = __float2bfloat16_rn(r1 - __bfloat162float(m));
  if (pattern == 2) { o[k] = h; o[K + k] = h; o[2 * K + k] = h; o[3 * K + k] = m; o[4 * K + k] = m; o[5 * K + k] = l; }
  else { o[k] = h; o[K + k] = m; o[2 * K + k] = l; o[3 * K + k] = h; o[4 * K + k] = m; o[5 * K + k] = h; }
}

__global__ void split3_rows_kernel(const float* __restrict__ src, long long lds, long long rows, int K, int Ksrc,
                                   int pattern, __nv_bfloat16* __restrict__ out) {
  const long long i = blockIdx.x * static_cast<long long>(S3T) + threadIdx.x;
  if (i >= rows * K) return;
  const long long r = i / K;
  const int k = static_cast<int>(i - r * K);
  emit_split(out + r * split_terms(pattern) * K, K, k, k < Ksrc ? src[r * lds + k] : 0.f, pattern);
}

// im2col of a 3x3 'same' convolution, split: out[m, k] for k = tap * Cc + c, tap = (dy+1)*3 + (dx+1), source pixel
// (y + s*dy, x + s*dx) with s = +1 (forward conv input) or -1 (flip: the transposed conv of the input gradient).
// layout 0: src is NCHW [B, Ctot, H, W], channels [c0, c0 + Cc);  layout 1: src is pixel-major [M, Cc].
__global__ void im2col3x3_split3_kernel(const float* __restrict__ src, int layout, int Ctot, int c0, int Cc, int B,
                                        int H, int W, int flip, int Kp, int pattern,
                                        __nv_bfloat16* __restrict__ out) {
  const long long i = blockIdx.x * static_cast<long long>(S3T) + threadIdx.x;
  const long long M = static_cast<long long>(B) * H * W;
  if (i >= M * Kp) return;
  const long long m = i / Kp;
  const int k = static_cast<int>(i - m * Kp);
  float v = 0.f;
  if (k < 9 * Cc) {
    const int tap = k / Cc, c = k - tap * Cc;
    const int b = static_cast<int>(m / (H * W)), rem = static_cast<int>(m - static_cast<long long>(b) * H * W);
    const int yy = rem / W, xx = rem - yy * W;
    const int s = flip ? -1 : 1;
    const int ny = yy + s * (tap / 3 - 1), nx = xx + s * (tap % 3 - 1);
    if (ny >= 0 && ny < H && nx >= 0 && nx < W) {
      v = layout == 0 ? src[((static_cast<long long>(b) * Ctot + c0 + c) * H + ny) * W + nx]
                      : src[(static_cast<long long>(b) * H * W + ny * W + nx) * Cc + c];
    }
  }
  emit_split(out + m * split_terms(pattern) * Kp, Kp, k, v, pattern);
}

// mode 0: v = relu(pre);  mode 1: v = gate > 0 ? pre : 0 (gate = hi part of the forward activation, row stride ldg).
// out3 = [hi | hi | lo] of v;  colsum[n] += sum_m v (fp32, unrounded) when given: one CTA = 32 rows x 256... columns
__global__ void act_split3_kernel(const float* __restrict__ pre, long long M, int N, int mode,
                                  const __nv_bfloat16* __restrict__ gate, long long ldg,
                                  __nv_bfloat16* __restrict__ out, float* __restrict__ colsum, int rows_per_cta,
                                  int pattern) {
  // thread = column (N <= blockDim.x * gridDim.y), loops over this CTA's rows: coalesced along n, one atomic per column
  const int n = blockIdx.y * blockDim.x + threadIdx.x;
  if (n >= N) return;
  const long long m0 = static_cast<long long>(blockIdx.x) * rows_per_cta;
  const long long m1 = m0 + rows_per_cta < M ? m0 + rows_per_cta : M;
  float acc = 0.f;
  for (long long m = m0; m < m1; ++m) {
    float v = pre[m * N + n];
    if (mode == 0) v = fmaxf(v, 0.f);
    else if (!(__bfloat162float(gate[m * ldg + n]) > 0.f)) v = 0.f;
    acc += v;
    emit_split(out + m * split_terms(pattern) * N, N, n, v, pattern);
  }
  if (colsum) atomicAdd(colsum + n, acc);
}

// Backward of the affine coupling (models/flows.py:160-168) in fp32, without the bf16 im2col of csrc/zpath.cu:
//   dy1 = g1, dy2 = g2 * s, dh[m, 2j] = g2 * s (shift), dh[m, 2j+1] = (g2 * z2_out + g_ld) * (1 - s) (logit),
//   s = sigmoid(logit + 2); dbias3[c] += sum_m dh[m, c].
__global__ void coupling_bwd_f32_kernel(const float* __restrict__ g_out, const float* __restrict__ g_ld,
                                        const float* __restrict__ z_out, const float* __restrict__ hsave,
                                        float* __restrict__ dy, float* __restrict__ dh, float* __restrict__ dbias3,
                                        int B, int C, int HW) {
  extern __shared__ float sb[];   // [C]
  const int J = C / 2;
  for (int i = threadIdx.x; i < C; i += blockDim.x) sb[i] = 0.f;
  __syncthreads();
  const long long total = static_cast<long long>(B) * HW * J;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long m = i / J;               // pixel (channel pair fastest: hsave rows are read contiguously)
    const int j = static_cast<int>(i - m * J);
    const int b = static_cast<int>(m / HW), rem = static_cast<int>(m - static_cast<long long>(b) * HW);
    const long long lo = (static_cast<long long>(b) * C + j) * HW + rem, hi = lo + static_cast<long long>(J) * HW;
    const float2 h = *reinterpret_cast<const float2*>(hsave + m * C + 2 * j);
    const float t = h.y + 2.f;
    const float e = expf(-fabsf(t));
    const float sg = t >= 0.f ? 1.f / (1.f + e) : e / (1.f + e);
    const float g2 = g_out[hi];
    const float dsh = g2 * sg;
    const float dlg = (g2 * z_out[hi] + g_ld[b]) * (1.f - sg);
    dy[lo] = g_out[lo];
    dy[hi] = dsh;
    *reinterpret_cast<float2*>(dh + m * C + 2 * j) = make_float2(dsh, dlg);
    atomicAdd(&sb[2 * j], dsh);
    atomicAdd(&sb[2 * j + 1], dlg);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < C; i += blockDim.x) atomicAdd(dbias3 + i, sb[i]);
}

// Backward of the INVERSE affine coupling (models/flows.py:185-193: zc2 = z2 / s - shift, ld -= sum log s) in fp32, the
// mirror of coupling_bwd_f32_kernel (arithmetic of coupling_bwd_kernel<C, INV = true> in zpath.cu); zc = the
// post-coupling tensor, g_zc its gradient:
//   dz1 = g1, dz2 = g2 / s, dh[m, 2j] = -g2 (shift), dh[m, 2j+1] = -(g2 * (zc2 + shift) + g_ld) * (1 - s) (logit),
//   s = sigmoid(logit + 2), z2 / s = zc2 + shift; dbias3[c] += sum_m dh[m, c].
__global__ void coupling_inv_bwd_f32_kernel(const float* __restrict__ g_zc, const float* __restrict__ g_ld,
                                            const float* __restrict__ zc, const float* __restrict__ hsave,
                                            float* __restrict__ dz, float* __restrict__ dh,
                                            float* __restrict__ dbias3, int B, int C, int HW) {
  extern __shared__ float sb[];   // [C]
  const int J = C / 2;
  for (int i = threadIdx.x; i < C; i += blockDim.x) sb[i] = 0.f;
  __syncthreads();
  const long long total = static_cast<long long>(B) * HW * J;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long m = i / J;               // pixel (channel pair fastest: hsave / dh rows are contiguous)
    const int j = static_cast<int>(i - m * J);
    const int b = static_cast<int>(m / HW), rem = static_cast<int>(m - static_cast<long long>(b) * HW);
    const long long lo = (static_cast<long long>(b) * C + j) * HW + rem, hi = lo + static_cast<long long>(J) * HW;
    const float2 h = *reinterpret_cast<const float2*>(hsave + m * C + 2 * j);
    const float t = h.y + 2.f;
    const float e = expf(-fabsf(t));
    const float sg = t >= 0.f ? 1.f / (1.f + e) : e / (1.f + e);
    const float g2 = g_zc[hi];
    const float dsh = -g2;
    const float dlg = -(g2 * (zc[hi] + h.x) + g_ld[b]) * (1.f - sg);
    dz[lo] = g_zc[lo];
    dz[hi] = g2 / sg;
    *reinterpret_cast<float2*>(dh + m * C + 2 * j) = make_float2(dsh, dlg);
    atomicAdd(&sb[2 * j], dsh);
    atomicAdd(&sb[2 * j + 1], dlg);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < C; i += blockDim.x) atomicAdd(dbias3 + i, sb[i]);
}

}  // namespace nfk

using namespace nfk;

extern "C" int nfk_split3_rows(const float* src, long long lds, long long rows, int K, int Ksrc, int pattern,
                               void* out, void* stream) {
  if (rows <= 0 || K <= 0 || K % 8 || Ksrc < 0 || Ksrc > K || lds < Ksrc) return NFK_ERR_SHAPE;
  if (!src || !out || pattern < 0 || pattern > 3) return NFK_ERR_ARG;
  const long long total = rows * K;
  split3_rows_kernel<<<static_cast<unsigned>((total + S3T - 1) / S3T), S3T, 0, static_cast<cudaStream_t>(stream)>>>(
      src, lds, rows, K, Ksrc, pattern, static_cast<__nv_bfloat16*>(out));
  return cudaGetLastError() == cudaSuccess ? NFK_OK : NFK_ERR_LAUNCH;
}

extern "C" int nfk_im2col3x3_split3(const float* src, int layout, int Ctot, int c0, int Cc, int B, int H, int W,
                                    int flip, int Kp, int pattern, void* out, void* stream) {
  if (pattern != 0 && pattern != 2) return NFK_ERR_ARG;
  if (B <= 0 || H <= 0 || W <= 0 || Cc <= 0 || Kp % 64 || Kp < 9 * Cc) return NFK_ERR_SHAPE;
  if (layout == 0 ? (c0 < 0 || c0 + Cc > Ctot) : layout != 1) return NFK_ERR_ARG;
  if (!src || !out) return NFK_ERR_ARG;
  const long long total = static_cast<long long>(B) * H * W * Kp;
  im2col3x3_split3_kernel<<<static_cast<unsigned>((total + S3T - 1) / S3T), S3T, 0,
                            static_cast<cudaStream_t>(stream)>>>(src, layout, Ctot, c0, Cc, B, H, W, flip, Kp, pattern,
                                                                 static_cast<__nv_bfloat16*>(out));
  return cudaGetLastError() == cudaSuccess ? NFK_OK : NFK_ERR_LAUNCH;
}

extern "C" int nfk_act_split3(const float* pre, long long M, int N, int mode, const void* gate, long long ldg,
                              int pattern, void* out, float* colsum, void* stream) {
  if (M <= 0 || N <= 0 || N % 8) return NFK_ERR_SHAPE;
  if (pattern != 0 && pattern != 2) return NFK_ERR_ARG;
  if (!pre || !out || (mode != 0 && mode != 1) || (mode == 1 && (!gate || ldg < N))) return NFK_ERR_ARG;
  const int rows_per_cta = 64;
  dim3 grid(static_cast<unsigned>((M + rows_per_cta - 1) / rows_per_cta), static_cast<unsigned>((N + S3T - 1) / S3T));
  act_split3_kernel<<<grid, S3T, 0, static_cast<cudaStream_t>(stream)>>>(
      pre, M, N, mode, static_cast<const __nv_bfloat16*>(gate), ldg, static_cast<__nv_bfloat16*>(out), colsum,
      rows_per_cta, pattern);
  return cudaGetLastError() == cudaSuccess ? NFK_OK : NFK_ERR_LAUNCH;
}

extern "C" int nfk_coupling_bwd_f32(const float* g_out, const float* g_ld, const float* z_out, const float* hsave,
                                    float* dy, float* dh, float* dbias3, int B, int C, int H, int W, void* stream) {
  if (B <= 0 || H <= 0 || W <= 0 || C <= 0 || C % 2) return NFK_ERR_SHAPE;
  if (!g_out || !g_ld || !z_out || !hsave || !dy || !dh || !dbias3) return NFK_ERR_ARG;
  const long long total = static_cast<long long>(B) * H * W * (C / 2);
  const long long want = (total + S3T - 1) / S3T;
  const unsigned grid = static_cast<unsigned>(want < 4 * 148 ? want : 4 * 148);
  coupling_bwd_f32_kernel<<<grid, S3T, C * sizeof(float), static_cast<cudaStream_t>(stream)>>>(
      g_out, g_ld, z_out, hsave, dy, dh, dbias3, B, C, H * W);
  return cudaGetLastError() == cudaSuccess ? NFK_OK : NFK_ERR_LAUNCH;
}

extern "C" int nfk_coupling_inv_bwd_f32(const float* g_zc, const float* g_ld, const float* zc, const float* hsave,
                                        float* dz, float* dh, float* dbias3, int B, int C, int H, int W,
                                        void* stream) {
  // the channel counts of the z-path kernels that produce zc / hsave (nfk_coupling_fwd, nfk_affine1x1_fwd)
  if (B <= 0 || H <= 0 || W <= 0 || (C != 12 && C != 24 && C != 48 && C != 96)) return NFK_ERR_SHAPE;
  if (!g_zc || !g_ld || !zc || !hsave || !dz || !dh || !dbias3) return NFK_ERR_ARG;
  const long long total = static_cast<long long>(B) * H * W * (C / 2);
  const long long want = (total + S3T - 1) / S3T;
  const unsigned grid = static_cast<unsigned>(want < 4 * 148 ? want : 4 * 148);
  coupling_inv_bwd_f32_kernel<<<grid, S3T, C * sizeof(float), static_cast<cudaStream_t>(stream)>>>(
      g_zc, g_ld, zc, hsave, dz, dh, dbias3, B, C, H * W);
  return cudaGetLastError() == cudaSuccess ? NFK_OK : NFK_ERR_LAUNCH;
}
