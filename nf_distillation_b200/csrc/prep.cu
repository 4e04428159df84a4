// Parameter-space kernels ("K0"): everything that depends only on the weights, once per optimiser step.
//
//  * invconv_prep_kernel: builds the fused ActNorm o InvertibleConv1x1 matrix of a FlowStep from the LU
//    parametrisation (reference: models/layers.py:376-397 get_weight, :101-142 ActNorm) — forward
//    W' = P L U diag(e^logs), b' = W' b, and inverse diag(e^-logs) U^-1 L^-1 P^T via in-SM triangular solves
//    (replaces three torch.inverse calls) — plus log|det| = sum(logs) + sum(log_s). The non-LU branch
//    (:366-375) runs a Gauss-Jordan slogdet/inverse in shared memory.
//  * invconv_prep_bwd_kernel: chain rule from (dW', db') back to actnorm.{bias,logs}, invconv.{lower,upper,log_s}.
//  * coupling_prep_kernel: folds the ActNorm affine of Conv2d (models/layers.py:223-228) and the exp(3*logs)
//    output scale of Conv2dZeros (:257-260) into bf16 GEMM operands laid out for the tcgen05 tiles;
//    coupling_prep_bwd_kernel maps GEMM-operand gradients back to the reference parameters.
// Each kernel takes a batch of items (one CTA, or one grid row of CTAs, per FlowStep): include/nfk.h.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <cstdint>

#include "../../include/nfk.h"
#include "launch_util.h"

namespace nfk {

constexpr int PREP_THREADS = 256;

__device__ __forceinline__ float block_sum(float v, float* red) {
  // red: >= 32 floats of shared memory
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();
  if (l == 0) red[w] = v;
  __syncthreads();
  float t = (threadIdx.x < (blockDim.x >> 5)) ? red[threadIdx.x] : 0.f;
  if (w == 0) {
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (l == 0) red[0] = t;
  }
  __syncthreads();
  t = red[0];
  __syncthreads();
  return t;
}

// Gauss-Jordan with partial pivoting on A (destroyed) producing Inv = A^-1 and sum log|pivot|.
__device__ float gauss_jordan(float* A, float* Inv, int C, int* piv_row, float* red) {
  const int tid = threadIdx.x;
  for (int i = tid; i < C * C; i += blockDim.x) Inv[i] = (i / C == i % C) ? 1.f : 0.f;
  __syncthreads();
  float logabs = 0.f;
  for (int c = 0; c < C; ++c) {
    if (tid == 0) {
      int best = c;
      float bv = fabsf(A[c * C + c]);
      for (int r = c + 1; r < C; ++r) {
        const float v = fabsf(A[r * C + c]);
        if (v > bv) { bv = v; best = r; }
      }
      *piv_row = best;
    }
    __syncthreads();
    const int pr = *piv_row;
    if (pr != c) {
      for (int j = tid; j < C; j += blockDim.x) {
        float t = A[c * C + j]; A[c * C + j] = A[pr * C + j]; A[pr * C + j] = t;
        t = Inv[c * C + j]; Inv[c * C + j] = Inv[pr * C + j]; Inv[pr * C + j] = t;
      }
    }
    __syncthreads();
    const float pv = A[c * C + c];
    logabs += logf(fabsf(pv));
    __syncthreads();
    const float ip = 1.f / pv;
    for (int j = tid; j < C; j += blockDim.x) { A[c * C + j] *= ip; Inv[c * C + j] *= ip; }
    __syncthreads();
    // eliminate column c from every other row; factors are read before any write of column c (saved in red? no:
    // each (r, j) pair needs A[r][c]; process j != c first, then zero column c).
    for (int idx = tid; idx < C * C; idx += blockDim.x) {
      const int r = idx / C, j = idx % C;
      if (r == c) continue;
      const float f = A[r * C + c];
      if (j != c) A[r * C + j] -= f * A[c * C + j];
      Inv[r * C + j] -= f * Inv[c * C + j];
    }
    __syncthreads();
    for (int r = tid; r < C; r += blockDim.x)
      if (r != c) A[r * C + c] = 0.f;
    __syncthreads();
  }
  (void)red;
  return logabs;
}

constexpr int INV_THREADS = 512;
constexpr int INV_MAX_BATCH = 24;  // items per launch (passed by value in the kernel parameter block)

struct InvBatch { nfk_invconv_item it[INV_MAX_BATCH]; };
struct InvBwdBatch { nfk_invconv_bwd_item it[INV_MAX_BATCH]; };

// perm[r] = column of the single 1 in row r of the permutation matrix p (one coalesced pass over p)
__device__ __forceinline__ void load_perm(const float* __restrict__ p, int C, int* perm) {
  for (int i = threadIdx.x; i < C * C; i += blockDim.x)
    if (p[i] > 0.5f) perm[i / C] = i % C;
}

// Lm = strict lower + I, Um = strict upper + diag(sign_s e^{log_s})
__device__ __forceinline__ void load_lu(const nfk_invconv_item& q, int C, float* Lm, float* Um) {
  for (int i = threadIdx.x; i < C * C; i += blockDim.x) {
    const int r = i / C, c = i % C;
    Lm[i] = c < r ? q.lower[i] : (c == r ? 1.f : 0.f);
    Um[i] = c > r ? q.upper[i] : (c == r ? q.sign_s[r] * expf(q.log_s[r]) : 0.f);
  }
}

// X <- L^-1 (unit lower) and Y <- U^-1, both by right-looking sweeps: at step k row k of the inverse is final and
// is eliminated from every remaining row at once (C steps of rank-1 updates, one barrier each) instead of one
// thread per column walking O(C^2) dependent shared-memory FMAs. U is first scaled to unit diagonal (U = D U'),
// U^-1 = U'^-1 D^-1. Threads [0, T/2) sweep L top-down, threads [T/2, T) sweep U' bottom-up.
__device__ void tri_inverses(const float* __restrict__ Lm, const float* __restrict__ Um, float* __restrict__ X,
                             float* __restrict__ Y, int C) {
  const int tid = threadIdx.x, half = blockDim.x >> 1;
  for (int i = tid; i < C * C; i += blockDim.x) {
    const float e = (i / C == i % C) ? 1.f : 0.f;
    X[i] = e;
    Y[i] = e;
  }
  __syncthreads();
  const bool lowerSide = tid < half;
  const int t = lowerSide ? tid : tid - half;
  const int jx = t & 31, i0 = t >> 5, irows = half >> 5;
  for (int s = 0; s + 1 < C; ++s) {
    if (lowerSide) {
      const int k = s;  // X[i][j] -= L[i][k] X[k][j]  for i > k, j <= k
      for (int i = k + 1 + i0; i < C; i += irows) {
        const float l = Lm[i * C + k];
        for (int j = jx; j <= k; j += 32) X[i * C + j] = fmaf(-l, X[k * C + j], X[i * C + j]);
      }
    } else {
      const int k = C - 1 - s;  // Y[i][j] -= U'[i][k] Y[k][j]  for i < k, j >= k
      for (int i = i0; i < k; i += irows) {
        const float u = Um[i * C + k] / Um[i * C + i];
        for (int j = k + jx; j < C; j += 32) Y[i * C + j] = fmaf(-u, Y[k * C + j], Y[i * C + j]);
      }
    }
    __syncthreads();
  }
  for (int i = tid; i < C * C; i += blockDim.x) {
    const int r = i / C, c = i % C;
    if (c >= r) Y[i] /= Um[c * C + c];
  }
  __syncthreads();
}

// smem: Lm, Um, X, Y (C*C each) + red[32] + perm[C] + piv
__device__ void invconv_prep_body(const nfk_invconv_item& q, float* sm) {
  const int C = q.C, reverse = q.reverse, transpose = q.transpose;
  float* Lm = sm;
  float* Um = Lm + C * C;
  float* X = Um + C * C;
  float* Y = X + C * C;
  float* red = Y + C * C;
  int* perm = reinterpret_cast<int*>(red + 32);
  int* piv = perm + C;
  const int tid = threadIdx.x;
  const int CC = C * C;

  float lsum = 0.f;
  for (int i = tid; i < C; i += blockDim.x) lsum += q.an_logs[i] + (q.weight ? 0.f : q.log_s[i]);
  lsum = block_sum(lsum, red);

  float* Wplain = X;  // forward matrix W (reference layout: z_o = sum_i W[o][i] x_i in 2-D)
  float* Winv = Y;
  if (q.weight) {
    for (int i = tid; i < CC; i += blockDim.x) { Lm[i] = q.weight[i]; Wplain[i] = q.weight[i]; }
    __syncthreads();
    if (reverse) {
      lsum += gauss_jordan(Lm, Winv, C, piv, red);
    } else {
      lsum += gauss_jordan(Lm, Um, C, piv, red);  // only the log|det| is needed
    }
  } else {
    load_lu(q, C, Lm, Um);
    load_perm(q.p, C, perm);
    __syncthreads();
    if (!reverse) {
      for (int i = tid; i < CC; i += blockDim.x) {
        const int o = i / C, c = i % C, r = perm[o];
        const int kmax = min(r, c);
        float t = 0.f;
        for (int k = 0; k <= kmax; ++k) t = fmaf(Lm[r * C + k], Um[k * C + c], t);
        Wplain[i] = t;
      }
    } else {
      tri_inverses(Lm, Um, X, Y, C);
      // Lm <- (U^-1 L^-1) P^T : column c of the product goes to column where perm[.] == c
      for (int i = tid; i < CC; i += blockDim.x) {
        const int r = i / C, c = i % C, pc = perm[c];
        float t = 0.f;
        for (int k = max(r, pc); k < C; ++k) t = fmaf(Y[r * C + k], X[k * C + pc], t);
        Lm[i] = t;
      }
      __syncthreads();
      for (int i = tid; i < CC; i += blockDim.x) Winv[i] = Lm[i];
    }
  }
  __syncthreads();
  // fused affine in "out" layout: out[a][b] multiplies input channel b into output channel a
  float* Out = Um;  // reuse
  for (int i = tid; i < CC; i += blockDim.x) {
    const int a = i / C, b = i % C;
    float v;
    if (!reverse) v = (transpose ? Wplain[b * C + a] : Wplain[i]) * expf(q.an_logs[b]);
    else v = (transpose ? Winv[b * C + a] : Winv[i]) * expf(-q.an_logs[a]);
    Out[i] = v;
    q.outW[i] = v;
  }
  __syncthreads();
  // b' = W' bias: one warp per output row
  const int warp = tid >> 5, lane = tid & 31, nwarps = blockDim.x >> 5;
  for (int a = warp; a < C; a += nwarps) {
    if (!reverse) {
      float t = 0.f;
      for (int b = lane; b < C; b += 32) t = fmaf(Out[a * C + b], q.an_bias[b], t);
      for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
      if (lane == 0) q.outb[a] = t;
    } else if (lane == 0) {
      q.outb[a] = -q.an_bias[a];
    }
  }
  if (tid == 0) q.out_sl[0] = reverse ? -lsum : lsum;
}

__global__ void __launch_bounds__(INV_THREADS) invconv_prep_kernel(const __grid_constant__ InvBatch batch) {
  extern __shared__ float sm[];
  invconv_prep_body(batch.it[blockIdx.x], sm);
}

// Backward of the prep (either direction). Wf is the saved outW of the same direction. Outputs are overwritten.
__device__ void invconv_prep_bwd_body(const nfk_invconv_bwd_item& g, float* sm) {
  const nfk_invconv_item& q = g.fwd;
  const int C = q.C, reverse = q.reverse, transpose = q.transpose, ldw = g.dWf_ld;
  const float* __restrict__ Wf = q.outW;
  const float* __restrict__ dWf = g.dWf;
  const float* __restrict__ dbf = g.dbf;
  float* Lm = sm;
  float* Um = Lm + C * C;
  float* G = Um + C * C;   // later dT
  float* dW = G + C * C;
  float* red = dW + C * C;
  int* perm = reinterpret_cast<int*>(red + 32);
  int* piv = perm + C;
  const int tid = threadIdx.x;
  const int CC = C * C;
  const int warp = tid >> 5, lane = tid & 31, nwarps = blockDim.x >> 5;

  float gs = 0.f;
  if (g.g_ld) {
    const int B4 = ((reinterpret_cast<uintptr_t>(g.g_ld) & 15) == 0) ? g.B >> 2 : 0;
    const float4* g4 = reinterpret_cast<const float4*>(g.g_ld);
#pragma unroll 8
    for (int b = tid; b < B4; b += blockDim.x) {
      const float4 v = g4[b];
      gs += (v.x + v.y) + (v.z + v.w);
    }
    for (int b = 4 * B4 + tid; b < g.B; b += blockDim.x) gs += g.g_ld[b];
  }
  float gsum = block_sum(gs, red) * g.pixels;

  if (!reverse) {
    // Wf[a][b] = W*[a][b] e^{logs_b}, bf = Wf bias
    for (int i = tid; i < CC; i += blockDim.x) {
      const int a = i / C, b = i % C;
      G[i] = dWf[a * ldw + b] + dbf[a] * q.an_bias[b];
      Lm[i] = Wf[i];
    }
    __syncthreads();
    for (int b = tid; b < C; b += blockDim.x) {
      float db = 0.f, dl = 0.f;
      for (int a = 0; a < C; ++a) {
        db = fmaf(Lm[a * C + b], dbf[a], db);
        dl = fmaf(G[a * C + b], Lm[a * C + b], dl);
      }
      g.d_bias[b] = db;
      g.d_logs[b] = dl + gsum;
    }
    for (int i = tid; i < CC; i += blockDim.x) {
      const int r = i / C, c = i % C;
      dW[i] = transpose ? G[c * C + r] * expf(q.an_logs[r]) : G[i] * expf(q.an_logs[c]);
    }
    __syncthreads();
  } else {
    // Wf[a][b] = Winv*[a][b] e^{-logs_a}, bf = -bias, log-det enters with a minus sign
    gsum = -gsum;
    for (int a = warp; a < C; a += nwarps) {
      float dl = 0.f;
      for (int b = lane; b < C; b += 32) dl = fmaf(dWf[a * ldw + b], Wf[a * C + b], dl);
      for (int o = 16; o > 0; o >>= 1) dl += __shfl_xor_sync(0xffffffffu, dl, o);
      if (lane == 0) {
        g.d_bias[a] = -dbf[a];
        g.d_logs[a] = -dl + gsum;
      }
    }
    float* Winv = G;      // plain layout
    float* dWinv = dW;    // plain layout
    for (int i = tid; i < CC; i += blockDim.x) {
      const int a = i / C, b = i % C;
      const float e = expf(q.an_logs[a]);
      const int pi = transpose ? b * C + a : i;
      Winv[pi] = Wf[i] * e;
      dWinv[pi] = dWf[a * ldw + b] / e;
    }
    __syncthreads();
    // Lm <- dWinv Winv^T ; Um <- -Winv^T Lm  (= dL/dW)
    for (int i = tid; i < CC; i += blockDim.x) {
      const int r = i / C, c = i % C;
      float t = 0.f;
      for (int k = 0; k < C; ++k) t = fmaf(dWinv[r * C + k], Winv[c * C + k], t);
      Lm[i] = t;
    }
    __syncthreads();
    for (int i = tid; i < CC; i += blockDim.x) {
      const int r = i / C, c = i % C;
      float t = 0.f;
      for (int k = 0; k < C; ++k) t = fmaf(Winv[k * C + r], Lm[k * C + c], t);
      Um[i] = -t;
    }
    __syncthreads();
    for (int i = tid; i < CC; i += blockDim.x) dW[i] = Um[i];
    __syncthreads();
  }
  if (q.weight) {
    // d slogdet / dW = W^-T
    for (int i = tid; i < CC; i += blockDim.x) Lm[i] = q.weight[i];
    __syncthreads();
    gauss_jordan(Lm, Um, C, piv, red);
    for (int i = tid; i < CC; i += blockDim.x) {
      const int r = i / C, c = i % C;
      g.d_weight[i] = dW[i] + gsum * Um[c * C + r];
    }
    return;
  }
  load_lu(q, C, Lm, Um);
  load_perm(q.p, C, perm);
  __syncthreads();
  float* dT = G;  // dT[perm[o]][i] = dW[o][i]
  for (int i = tid; i < CC; i += blockDim.x) {
    const int o = i / C, c = i % C;
    dT[perm[o] * C + c] = dW[i];
  }
  __syncthreads();
  for (int i = tid; i < CC; i += blockDim.x) {
    const int r = i / C, k = i % C;
    // d_lower[r][k] = sum_{c>=k} dT[r][c] Um[k][c]   (k < r)
    float dl = 0.f;
    if (k < r)
      for (int c = k; c < C; ++c) dl = fmaf(dT[r * C + c], Um[k * C + c], dl);
    g.d_lower[i] = dl;
    // dUm[r][k] = sum_{rr>=r} Lm[rr][r] dT[rr][k]   (here (r,k) indexes U)
    float du = 0.f;
    if (k >= r)
      for (int rr = r; rr < C; ++rr) du = fmaf(Lm[rr * C + r], dT[rr * C + k], du);
    g.d_upper[i] = k > r ? du : 0.f;
    if (k == r) g.d_log_s[r] = du * Um[r * C + r] + gsum;
  }
}

__global__ void __launch_bounds__(INV_THREADS)
invconv_prep_bwd_kernel(const __grid_constant__ InvBwdBatch batch) {
  extern __shared__ float sm[];
  invconv_prep_bwd_body(batch.it[blockIdx.x], sm);
}

// ------------------------------------------------------------------------------------------ coupling weights
struct CouplingW {
  const float *w1, *b1, *l1;  // Conv2d #1: [hid, cin, 3, 3], actnorm bias/logs [hid]
  const float *w2, *b2, *l2;  // Conv2d #2: [hid, hid, 1, 1]
  const float *w3, *b3, *l3;  // Conv2dZeros: [cout, hid, 3, 3], bias [cout], logs [cout]
};
struct CouplingOps {
  __nv_bfloat16 *B1, *B1T;  // [hid, K1p], [K1p, hid]     k = tap*cin + ci
  __nv_bfloat16 *B2, *B2T;  // [hid, hid] (co, ci), (ci, co)
  __nv_bfloat16 *B3, *B3T;  // [K3p, hid] rows n = tap*cout + co ; [hid, K3p]
  float *bias1, *bias2, *bias3;  // folded biases
};

struct CouplingItem { CouplingW w; CouplingOps o; int cin, hid, cout, K1p, K3p, with_transposed; };
constexpr int CP_MAX_BATCH = 16;
struct CouplingBatch { CouplingItem it[CP_MAX_BATCH]; };

__global__ void coupling_prep_kernel(const __grid_constant__ CouplingBatch batch) {
  const CouplingItem& q = batch.it[blockIdx.y];
  const CouplingW& w = q.w;
  const CouplingOps& o = q.o;
  const int cin = q.cin, hid = q.hid, cout = q.cout, K1p = q.K1p, K3p = q.K3p, with_transposed = q.with_transposed;
  const long long n1 = static_cast<long long>(hid) * K1p;
  const long long n2 = static_cast<long long>(hid) * hid;
  const long long n3 = static_cast<long long>(K3p) * hid;
  const long long total = n1 + n2 + n3 + 2 * hid + cout;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    if (i < n1) {
      const int co = static_cast<int>(i / K1p), k = static_cast<int>(i % K1p);
      float v = 0.f;
      if (k < 9 * cin) {
        const int tap = k / cin, ci = k % cin;
        v = w.w1[(static_cast<long long>(co) * cin + ci) * 9 + tap] * expf(w.l1[co]);
      }
      const __nv_bfloat16 h = __float2bfloat16_rn(v);
      o.B1[i] = h;
      if (with_transposed) o.B1T[static_cast<long long>(k) * hid + co] = h;
    } else if (i < n1 + n2) {
      const long long j = i - n1;
      const int co = static_cast<int>(j / hid), ci = static_cast<int>(j % hid);
      const __nv_bfloat16 h = __float2bfloat16_rn(w.w2[j] * expf(w.l2[co]));
      o.B2[j] = h;
      if (with_transposed) o.B2T[static_cast<long long>(ci) * hid + co] = h;
    } else if (i < n1 + n2 + n3) {
      const long long j = i - n1 - n2;
      const int n = static_cast<int>(j / hid), ci = static_cast<int>(j % hid);
      float v = 0.f;
      if (n < 9 * cout) {
        const int tap = n / cout, co = n % cout;
        v = w.w3[(static_cast<long long>(co) * hid + ci) * 9 + tap] * expf(3.f * w.l3[co]);
      }
      const __nv_bfloat16 h = __float2bfloat16_rn(v);
      o.B3[j] = h;
      if (with_transposed) o.B3T[static_cast<long long>(ci) * K3p + n] = h;
    } else {
      const int j = static_cast<int>(i - n1 - n2 - n3);
      if (j < hid) o.bias1[j] = w.b1[j] * expf(w.l1[j]);
      else if (j < 2 * hid) o.bias2[j - hid] = w.b2[j - hid] * expf(w.l2[j - hid]);
      else o.bias3[j - 2 * hid] = w.b3[j - 2 * hid] * expf(3.f * w.l3[j - 2 * hid]);
    }
  }
}

struct CouplingGradIn {
  const float *dB1, *dbias1;  // [hid, K1p], [hid]
  const float *dB2, *dbias2;  // [hid, hid], [hid]
  const float *dB3, *dbias3;  // [K3p, hid], [cout]
};
struct CouplingGradOut {
  float *dw1, *db1, *dl1, *dw2, *db2, *dl2, *dw3, *db3, *dl3;
};

struct CouplingBwdItem { CouplingW w; CouplingGradIn gi; CouplingGradOut go; int cin, hid, cout, K1p, K3p; };
constexpr int CPB_MAX_BATCH = 12;
struct CouplingBwdBatch { CouplingBwdItem it[CPB_MAX_BATCH]; };

// One CTA per output channel: rows [0,hid) -> layer 1, [hid,2hid) -> layer 2, [2hid, 2hid+cout) -> layer 3;
// blockIdx.y = step of the batch.
__global__ void __launch_bounds__(PREP_THREADS)
coupling_prep_bwd_kernel(const __grid_constant__ CouplingBwdBatch batch) {
  const CouplingBwdItem& q = batch.it[blockIdx.y];
  const CouplingW& w = q.w;
  const CouplingGradIn& gi = q.gi;
  const CouplingGradOut& go = q.go;
  const int cin = q.cin, hid = q.hid, cout = q.cout, K1p = q.K1p, K3p = q.K3p;
  (void)K3p;
  __shared__ float red[32];
  const int row = blockIdx.x, tid = threadIdx.x;
  if (row >= 2 * hid + cout) return;
  float acc = 0.f;
  if (row < hid) {
    const int co = row;
    const float e = expf(w.l1[co]);
    for (int k = tid; k < 9 * cin; k += blockDim.x) {
      const int tap = k / cin, ci = k % cin;
      const long long wi = (static_cast<long long>(co) * cin + ci) * 9 + tap;
      const float g = gi.dB1[static_cast<long long>(co) * K1p + k];
      go.dw1[wi] = g * e;
      acc = fmaf(g, w.w1[wi] * e, acc);
    }
    acc = block_sum(acc, red);
    if (tid == 0) {
      const float gb = gi.dbias1[co];
      go.db1[co] = gb * e;
      go.dl1[co] = acc + gb * w.b1[co] * e;
    }
  } else if (row < 2 * hid) {
    const int co = row - hid;
    const float e = expf(w.l2[co]);
    for (int ci = tid; ci < hid; ci += blockDim.x) {
      const long long wi = static_cast<long long>(co) * hid + ci;
      const float g = gi.dB2[wi];
      go.dw2[wi] = g * e;
      acc = fmaf(g, w.w2[wi] * e, acc);
    }
    acc = block_sum(acc, red);
    if (tid == 0) {
      const float gb = gi.dbias2[co];
      go.db2[co] = gb * e;
      go.dl2[co] = acc + gb * w.b2[co] * e;
    }
  } else {
    const int co = row - 2 * hid;
    const float e = expf(3.f * w.l3[co]);
    for (int j = tid; j < 9 * hid; j += blockDim.x) {
      const int tap = j / hid, ci = j % hid;
      const long long wi = (static_cast<long long>(co) * hid + ci) * 9 + tap;
      const float g = gi.dB3[static_cast<long long>(tap * cout + co) * hid + ci];
      go.dw3[wi] = g * e;
      acc = fmaf(g, w.w3[wi] * e, acc);
    }
    acc = block_sum(acc, red);
    if (tid == 0) {
      const float gb = gi.dbias3[co];
      go.db3[co] = gb * e;
      go.dl3[co] = 3.f * (acc + gb * w.b3[co] * e);
    }
  }
}

static int prep_smem(int C) { return (4 * C * C + 32 + C + 4) * static_cast<int>(sizeof(float)); }

}  // namespace nfk

using namespace nfk;

static int check_item(const nfk_invconv_item& q) {
  if (q.C <= 0 || q.C > 104) return NFK_ERR_SHAPE;
  if (!q.an_bias || !q.an_logs || !q.outW || !q.outb || !q.out_sl) return NFK_ERR_ARG;
  if (!q.weight && (!q.lower || !q.upper || !q.log_s || !q.p || !q.sign_s)) return NFK_ERR_ARG;
  return NFK_OK;
}

extern "C" int nfk_invconv_prep_batch(int n, const nfk_invconv_item* items, void* stream) {
  if (n < 0) return NFK_ERR_SHAPE;
  if (n && !items) return NFK_ERR_ARG;
  int cmax = 0;
  for (int i = 0; i < n; ++i) {
    if (int rc = check_item(items[i])) return rc;
    cmax = items[i].C > cmax ? items[i].C : cmax;
  }
  const int smem = prep_smem(cmax);
  if (n)
    if (int rc = ensure_dyn_smem(reinterpret_cast<const void*>(invconv_prep_kernel), smem)) return rc;
  for (int i0 = 0; i0 < n; i0 += INV_MAX_BATCH) {
    InvBatch b{};
    const int m = n - i0 < INV_MAX_BATCH ? n - i0 : INV_MAX_BATCH;
    for (int i = 0; i < m; ++i) b.it[i] = items[i0 + i];
    invconv_prep_kernel<<<m, INV_THREADS, smem, static_cast<cudaStream_t>(stream)>>>(b);
    if (cudaGetLastError() != cudaSuccess) return NFK_ERR_LAUNCH;
  }
  return NFK_OK;
}

extern "C" int nfk_invconv_prep_bwd_batch(int n, const nfk_invconv_bwd_item* items, void* stream) {
  if (n < 0) return NFK_ERR_SHAPE;
  if (n && !items) return NFK_ERR_ARG;
  int cmax = 0;
  for (int i = 0; i < n; ++i) {
    const nfk_invconv_bwd_item& g = items[i];
    if (int rc = check_item(g.fwd)) return rc;
    if (g.B <= 0 || g.dWf_ld < g.fwd.C) return NFK_ERR_SHAPE;
    if (!g.dWf || !g.dbf || !g.d_bias || !g.d_logs) return NFK_ERR_ARG;
    if (g.fwd.weight ? !g.d_weight : (!g.d_lower || !g.d_upper || !g.d_log_s)) return NFK_ERR_ARG;
    cmax = g.fwd.C > cmax ? g.fwd.C : cmax;
  }
  const int smem = prep_smem(cmax);
  if (n)
    if (int rc = ensure_dyn_smem(reinterpret_cast<const void*>(invconv_prep_bwd_kernel), smem)) return rc;
  for (int i0 = 0; i0 < n; i0 += INV_MAX_BATCH) {
    InvBwdBatch b{};
    const int m = n - i0 < INV_MAX_BATCH ? n - i0 : INV_MAX_BATCH;
    for (int i = 0; i < m; ++i) b.it[i] = items[i0 + i];
    invconv_prep_bwd_kernel<<<m, INV_THREADS, smem, static_cast<cudaStream_t>(stream)>>>(b);
    if (cudaGetLastError() != cudaSuccess) return NFK_ERR_LAUNCH;
  }
  return NFK_OK;
}

static int coupling_item_check(const nfk_coupling_item& c) {
  if (c.cin <= 0 || c.hid <= 0 || c.cout <= 0 || c.hid % 64 || c.K1p % 64 || c.K3p % 64 || c.K1p < 9 * c.cin ||
      c.K3p < 9 * c.cout)
    return NFK_ERR_SHAPE;
  if (!c.w1 || !c.b1 || !c.l1 || !c.w2 || !c.b2 || !c.l2 || !c.w3 || !c.b3 || !c.l3) return NFK_ERR_ARG;
  return NFK_OK;
}

extern "C" int nfk_coupling_prep_batch(int n, const nfk_coupling_item* items, void* stream) {
  if (n < 0) return NFK_ERR_SHAPE;
  if (n && !items) return NFK_ERR_ARG;
  for (int i = 0; i < n; ++i) {
    const nfk_coupling_item& c = items[i];
    if (int rc = coupling_item_check(c)) return rc;
    if (!c.B1 || !c.B2 || !c.B3 || !c.bias1 || !c.bias2 || !c.bias3) return NFK_ERR_ARG;
    if (c.with_transposed && (!c.B1T || !c.B2T || !c.B3T)) return NFK_ERR_ARG;
  }
  for (int i0 = 0; i0 < n; i0 += CP_MAX_BATCH) {
    CouplingBatch b{};
    const int m = n - i0 < CP_MAX_BATCH ? n - i0 : CP_MAX_BATCH;
    long long tmax = 0;
    for (int i = 0; i < m; ++i) {
      const nfk_coupling_item& c = items[i0 + i];
      CouplingItem& q = b.it[i];
      q.w = CouplingW{c.w1, c.b1, c.l1, c.w2, c.b2, c.l2, c.w3, c.b3, c.l3};
      q.o = CouplingOps{static_cast<__nv_bfloat16*>(c.B1), static_cast<__nv_bfloat16*>(c.B1T),
                        static_cast<__nv_bfloat16*>(c.B2), static_cast<__nv_bfloat16*>(c.B2T),
                        static_cast<__nv_bfloat16*>(c.B3), static_cast<__nv_bfloat16*>(c.B3T), c.bias1, c.bias2, c.bias3};
      q.cin = c.cin; q.hid = c.hid; q.cout = c.cout; q.K1p = c.K1p; q.K3p = c.K3p;
      q.with_transposed = c.with_transposed;
      const long long total = static_cast<long long>(c.hid) * (c.K1p + c.hid + c.K3p) + 2 * c.hid + c.cout;
      tmax = total > tmax ? total : tmax;
    }
    const int blocks = static_cast<int>((tmax + 255) / 256 < 1184 ? (tmax + 255) / 256 : 1184);
    coupling_prep_kernel<<<dim3(blocks, m), 256, 0, static_cast<cudaStream_t>(stream)>>>(b);
    if (cudaGetLastError() != cudaSuccess) return NFK_ERR_LAUNCH;
  }
  return NFK_OK;
}

extern "C" int nfk_coupling_prep_bwd_batch(int n, const nfk_coupling_bwd_item* items, void* stream) {
  if (n < 0) return NFK_ERR_SHAPE;
  if (n && !items) return NFK_ERR_ARG;
  for (int i = 0; i < n; ++i) {
    const nfk_coupling_bwd_item& g = items[i];
    if (int rc = coupling_item_check(g.fwd)) return rc;
    if (!g.dB1 || !g.dbias1 || !g.dB2 || !g.dbias2 || !g.dB3 || !g.dbias3) return NFK_ERR_ARG;
    if (!g.dw1 || !g.db1 || !g.dl1 || !g.dw2 || !g.db2 || !g.dl2 || !g.dw3 || !g.db3 || !g.dl3) return NFK_ERR_ARG;
  }
  for (int i0 = 0; i0 < n; i0 += CPB_MAX_BATCH) {
    CouplingBwdBatch b{};
    const int m = n - i0 < CPB_MAX_BATCH ? n - i0 : CPB_MAX_BATCH;
    int rows = 0;
    for (int i = 0; i < m; ++i) {
      const nfk_coupling_bwd_item& g = items[i0 + i];
      const nfk_coupling_item& c = g.fwd;
      CouplingBwdItem& q = b.it[i];
      q.w = CouplingW{c.w1, c.b1, c.l1, c.w2, c.b2, c.l2, c.w3, c.b3, c.l3};
      q.gi = CouplingGradIn{g.dB1, g.dbias1, g.dB2, g.dbias2, g.dB3, g.dbias3};
      q.go = CouplingGradOut{g.dw1, g.db1, g.dl1, g.dw2, g.db2, g.dl2, g.dw3, g.db3, g.dl3};
      q.cin = c.cin; q.hid = c.hid; q.cout = c.cout; q.K1p = c.K1p; q.K3p = c.K3p;
      const int r = 2 * c.hid + c.cout;
      rows = r > rows ? r : rows;
    }
    coupling_prep_bwd_kernel<<<dim3(rows, m), PREP_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(b);
    if (cudaGetLastError() != cudaSuccess) return NFK_ERR_LAUNCH;
  }
  return NFK_OK;
}
