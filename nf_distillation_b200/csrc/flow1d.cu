// 1-D (tabular) Glow FlowStep, fused end to end in one kernel per direction (reference: the is_1d branches of
// models/flows.py:37-52,142-202 and models/layers.py:76,117,410-411).
//
// A persistent CTA (one per SM) walks tiles of NT samples with every weight of the step resident in shared memory.
// Activations live in shared memory feature-major ([feature][NT+4]); each layer is a small fp32 GEMM over the tile,
// register-blocked 8 outputs x 4 samples per thread (3 LDS.128 per 32 FMAs):
//   y = W' x + b'            (ActNorm1d + x @ W folded by nfk_invconv_prep_batch with transpose=1)
//   h = MLP(y1 [, cond])     Linear-ReLU x4, Linear-Tanh, Linear
//   y2 = (y2 + h[0::2]) * sigmoid(h[1::2] + 2),  logdet += sum log sigmoid          (or the inverse order / formulas)
// The backward kernel reloads the saved MLP activations, walks the chain in reverse with the same tile GEMM for the
// data gradients and an 8x4 register-blocked outer-product GEMM (reduction over the samples) for the weight gradients,
// which accumulate per CTA in shared memory and are added to the global gradient block once.
// fp32 SIMT on purpose: these layers are 16..64 wide and the path's parity bar is 1e-4 on log-det in fp32.
#include <cuda_runtime.h>
#include <cstdint>

#include "../../include/nfk.h"
#include "launch_util.h"

namespace nfk {

constexpr int F1_LAYERS = 7;  // 0: fused affine, 1..6: coupling MLP

struct F1Dims {
  int D, D1, D2, Cc, hid;
  int nin[F1_LAYERS], nout[F1_LAYERS], ninp[F1_LAYERS], noutp[F1_LAYERS];
  int offWT[F1_LAYERS], offB[F1_LAYERS];  // forward block: WT_l [nin][noutp], bias_l [noutp]
  int offW[F1_LAYERS];                    // backward block: W_l [nout][ninp]
  int offG[F1_LAYERS], offGB[F1_LAYERS];  // gradient block: dW_l [nout][ninp], db_l [noutp]
  int total_fwd, total_bwd, total_grad;
  int n_act;                              // saved activations per sample: H1..H5 (5*hid) + O (2*D2)
};

static inline int up8(int x) { return (x + 7) / 8 * 8; }
__host__ __device__ static inline int up8d(int x) { return (x + 7) / 8 * 8; }

static F1Dims f1_dims(int D, int Cc, int hid) {
  F1Dims d{};
  d.D = D; d.D1 = D / 2; d.D2 = D - D / 2; d.Cc = Cc; d.hid = hid;
  const int nin[F1_LAYERS] = {D, d.D1 + Cc, hid, hid, hid, hid, hid};
  const int nout[F1_LAYERS] = {D, hid, hid, hid, hid, hid, 2 * d.D2};
  int of = 0, ob = 0, og = 0;
  for (int l = 0; l < F1_LAYERS; ++l) {
    d.nin[l] = nin[l]; d.nout[l] = nout[l]; d.ninp[l] = up8(nin[l]); d.noutp[l] = up8(nout[l]);
    d.offWT[l] = of; of += nin[l] * d.noutp[l];
    d.offB[l] = of; of += d.noutp[l];
    d.offW[l] = ob; ob += nout[l] * d.ninp[l];
    d.offG[l] = og; og += nout[l] * d.ninp[l];
    d.offGB[l] = og; og += d.noutp[l];
  }
  d.total_fwd = of; d.total_bwd = ob; d.total_grad = og;
  d.n_act = 5 * hid + 2 * d.D2;
  return d;
}

struct F1Weights {
  const float* Wf;     // [D][D] fused affine, out-layout
  const float* bf;     // [D]
  const float* w[6];   // nn.Linear weights [nout][nin]
  const float* b[6];
};

__global__ void flow1d_pack_kernel(F1Weights src, F1Dims d, float* __restrict__ PF, float* __restrict__ PB) {
  const int total = d.total_fwd + (PB ? d.total_bwd : 0);
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
    if (e < d.total_fwd) {
      int l = F1_LAYERS - 1;
      while (e < d.offWT[l]) --l;
      const int r = e - d.offWT[l];
      const float* W = l == 0 ? src.Wf : src.w[l - 1];
      const float* bsrc = l == 0 ? src.bf : src.b[l - 1];
      float v = 0.f;
      if (r < d.nin[l] * d.noutp[l]) {
        const int i = r / d.noutp[l], o = r % d.noutp[l];
        if (o < d.nout[l]) v = W[o * d.nin[l] + i];
      } else {
        const int o = r - d.nin[l] * d.noutp[l];
        if (o < d.nout[l]) v = bsrc[o];
      }
      PF[e] = v;
    } else {
      const int q = e - d.total_fwd;
      int l = F1_LAYERS - 1;
      while (q < d.offW[l]) --l;
      const int r = q - d.offW[l];
      const int o = r / d.ninp[l], i = r % d.ninp[l];
      const float* W = l == 0 ? src.Wf : src.w[l - 1];
      PB[q] = i < d.nin[l] ? W[o * d.nin[l] + i] : 0.f;
    }
  }
}

constexpr int F1_THREADS = 512;

// Per-layer shape of the weight-gradient pass (host-computed, depends on the sample tile NT).
struct F1Wg { int n_ot, n_it, lgks; };
struct F1Run {
  int NT, lgNT, nbuf;   // sample tile, log2, input buffers (2 = next tile prefetched while this one computes)
  F1Wg wg[F1_LAYERS];
};

__device__ __forceinline__ void cp_async4(float* smem_dst, const float* gsrc, bool valid) {
  const unsigned dst = static_cast<unsigned>(__cvta_generic_to_shared(smem_dst));
  const int sz = valid ? 4 : 0;  // src-size 0 zero-fills the destination
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(dst), "l"(gsrc), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async16(float* smem_dst, const float* gsrc) {
  const unsigned dst = static_cast<unsigned>(__cvta_generic_to_shared(smem_dst));
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(gsrc) : "memory");
}
// weights block global -> smem (16-byte copies when the source is aligned); completes with the next wait_all
__device__ __forceinline__ void weights_load_async(const float* __restrict__ g, float* __restrict__ sm, int n) {
  if ((reinterpret_cast<uintptr_t>(g) & 15) == 0) {
    const int n4 = n >> 2;
    for (int e = threadIdx.x; e < n4; e += blockDim.x) cp_async16(sm + 4 * e, g + 4 * e);
    for (int e = 4 * n4 + threadIdx.x; e < n; e += blockDim.x) sm[e] = g[e];
  } else {
    for (int e = threadIdx.x; e < n; e += blockDim.x) sm[e] = g[e];
  }
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// Every layer is a small GEMM over the sample tile: out[o][s] = epi(bias[o] + sum_i WT[i][o] * in[i][s]).
// The CTA shares the tile; a thread owns 8 outputs x 2 consecutive samples (16 accumulators): one LDS.64 of
// activations and two broadcast LDS.128 of weights feed 16 FMAs, and a 128-sample tile of a 32-wide layer still
// spreads over 256 threads. Tiles live feature-major in shared memory with row stride ld = NT + 4 floats.
// MODE: 0 none, 1 relu, 2 tanh (forward epilogues); 3 multiply by relu'(hm), 4 multiply by 1 - hm^2 (dgrad epilogues)
// FROM_TOP hands the items out from the last thread downwards, so a data-gradient layer shares its phase with the
// weight-gradient pass (which fills threads from 0 upwards) instead of queueing behind it.
template <int MODE, bool FROM_TOP = false>
__device__ __forceinline__ void lin_tile(const float* __restrict__ in, int nin, float* __restrict__ out, int nout,
                                         const float* __restrict__ WT, const float* __restrict__ bias, int noutp,
                                         const float* __restrict__ hm, int ld, int lgNT) {
  const int lgnsg = lgNT - 1;
  const int items = (noutp >> 3) << lgnsg;
  const int t0 = FROM_TOP ? F1_THREADS - 1 - static_cast<int>(threadIdx.x) : static_cast<int>(threadIdx.x);
  for (int it = t0; it < items; it += F1_THREADS) {
    const int og = it >> lgnsg, sg = it - (og << lgnsg);
    // acc[jp][s] holds outputs (2jp, 2jp+1) of sample s as one packed pair: the FMAs issue as fma.rn.f32x2
    // (two fp32 FMAs per instruction, each an ordinary fused multiply-add) with the weight pairs straight out of the
    // LDS.128 registers.
    float2 acc[4][2];
    if (bias) {
      const float4 b0 = *reinterpret_cast<const float4*>(bias + og * 8);
      const float4 b1 = *reinterpret_cast<const float4*>(bias + og * 8 + 4);
      acc[0][0] = acc[0][1] = make_float2(b0.x, b0.y);
      acc[1][0] = acc[1][1] = make_float2(b0.z, b0.w);
      acc[2][0] = acc[2][1] = make_float2(b1.x, b1.y);
      acc[3][0] = acc[3][1] = make_float2(b1.z, b1.w);
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[j][0] = acc[j][1] = make_float2(0.f, 0.f);
    }
    const float* wp = WT + og * 8;
    const float* ip = in + 2 * sg;
#pragma unroll 8
    for (int i = 0; i < nin; ++i) {
      const float2 a = *reinterpret_cast<const float2*>(ip + i * ld);
      const float4 w0 = *reinterpret_cast<const float4*>(wp + i * noutp);
      const float4 w1 = *reinterpret_cast<const float4*>(wp + i * noutp + 4);
      const float2 ax = make_float2(a.x, a.x), ay = make_float2(a.y, a.y);
      const float2 ww[4] = {make_float2(w0.x, w0.y), make_float2(w0.z, w0.w), make_float2(w1.x, w1.y),
                            make_float2(w1.z, w1.w)};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        acc[j][0] = __ffma2_rn(ww[j], ax, acc[j][0]);
        acc[j][1] = __ffma2_rn(ww[j], ay, acc[j][1]);
      }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int o = og * 8 + j;
      if (o < nout) {
        float2 v = (j & 1) ? make_float2(acc[j >> 1][0].y, acc[j >> 1][1].y)
                           : make_float2(acc[j >> 1][0].x, acc[j >> 1][1].x);
        if (MODE == 1) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); }
        if (MODE == 2) { v.x = tanhf(v.x); v.y = tanhf(v.y); }
        if (MODE == 3 || MODE == 4) {
          const float2 h = *reinterpret_cast<const float2*>(hm + o * ld + 2 * sg);
          if (MODE == 3) {
            v.x = h.x > 0.f ? v.x : 0.f; v.y = h.y > 0.f ? v.y : 0.f;
          } else {
            v.x *= 1.f - h.x * h.x; v.y *= 1.f - h.y * h.y;
          }
        }
        *reinterpret_cast<float2*>(out + o * ld + 2 * sg) = v;
      }
    }
  }
}

// One reduce-scatter step over lane pairs `sh` apart: each lane keeps the half of its CNT partial sums selected by
// its `bit`, adds the partner's copy of that half, and hands the other half over.
template <int CNT>
__device__ __forceinline__ void rs_step(float* acc, bool bit, int sh) {
#pragma unroll
  for (int k = 0; k < CNT / 2; ++k) {
    const float keep = bit ? acc[k + CNT / 2] : acc[k];
    const float send = bit ? acc[k] : acc[k + CNT / 2];
    acc[k] = keep + __shfl_xor_sync(0xffffffffu, send, sh);
  }
}

struct WgOut { float* gacc; float* gbias; int ot, itl, n_ot, n_it, nout, nin, ninp, pre; };
// Add the CNT sums this lane owns after the reduce-scatter (block-linear indices pre .. pre+CNT-1) into dW / db.
template <int CNT>
__device__ __forceinline__ void wg_writeback(const float* acc, const WgOut& w) {
#pragma unroll
  for (int k = 0; k < CNT; ++k) {
    const int v = w.pre + k, j = v >> 2, m = v & 3;
    const int o = w.ot + j * w.n_ot, i = w.itl + m * w.n_it;
    if (o < w.nout) {
      if (i < w.nin) w.gacc[o * w.ninp + i] += acc[k];
      else if (i == w.nin) w.gbias[o] += acc[k];
    }
  }
}

// Weight gradient of one layer over the sample tile, accumulated into the CTA's shared gradient block:
//   gacc[o*ninp + i] += sum_s dout[o][s] * in[i][s],   gbias[o] += sum_s dout[o][s].
// A thread owns an 8 (o, interleaved) x 4 (i, interleaved) block of dW and walks its share of the samples four at a
// time (12 LDS.128 per 128 FMAs); the bias gradient is the extra input row i == nin whose activation is 1. Small
// layers split the samples over ks = 2^lgks adjacent lanes, which meet in a shuffle reduce-scatter (each lane ends
// up owning 32/ks of the block's sums); every dW element has exactly one writer, so there are no atomics.
__device__ __forceinline__ void wgrad_tile(const float* __restrict__ dout, int nout, const float* __restrict__ in,
                                           int nin, int ninp, float* __restrict__ gacc, float* __restrict__ gbias,
                                           int ld, int lgNT, const F1Wg cfg) {
  const int n_ot = cfg.n_ot, n_it = cfg.n_it, lgks = cfg.lgks;
  const int ntiles = n_ot * n_it;
  const int kq = (1 << (lgNT - 2)) >> lgks;
  const int total = ntiles << lgks;
  const int lane = threadIdx.x & 31;
  for (int base = threadIdx.x - lane; base < total; base += F1_THREADS) {
    const int item = base + lane;
    const bool valid = item < total;
    const int t = valid ? item >> lgks : 0, kp = valid ? item - (t << lgks) : 0;
    const int ot = t / n_it, itl = t - ot * n_it;
    int dp[8], ip[4];  // row offsets (rows past the end are clamped; their results are dropped below)
#pragma unroll
    for (int j = 0; j < 8; ++j) dp[j] = min(ot + j * n_ot, nout - 1) * ld;
#pragma unroll
    for (int m = 0; m < 4; ++m) ip[m] = min(itl + m * n_it, nin - 1) * ld;
    const bool ones3 = itl + 3 * n_it == nin, ones2 = itl + 2 * n_it == nin;
    const bool ones1 = itl + n_it == nin, ones0 = itl == nin;
    float acc[32];
#pragma unroll
    for (int v = 0; v < 32; ++v) acc[v] = 0.f;
#pragma unroll 2
    for (int q = kp * kq; q < (kp + 1) * kq; ++q) {
      float4 a[4];
#pragma unroll
      for (int m = 0; m < 4; ++m) a[m] = *reinterpret_cast<const float4*>(in + ip[m] + 4 * q);
      const float4 one = make_float4(1.f, 1.f, 1.f, 1.f);
      if (ones0) a[0] = one;
      if (ones1) a[1] = one;
      if (ones2) a[2] = one;
      if (ones3) a[3] = one;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 d = *reinterpret_cast<const float4*>(dout + dp[j] + 4 * q);
#pragma unroll
        for (int m = 0; m < 4; ++m) {
          acc[j * 4 + m] = fmaf(d.x, a[m].x, acc[j * 4 + m]);
          acc[j * 4 + m] = fmaf(d.y, a[m].y, acc[j * 4 + m]);
          acc[j * 4 + m] = fmaf(d.z, a[m].z, acc[j * 4 + m]);
          acc[j * 4 + m] = fmaf(d.w, a[m].w, acc[j * 4 + m]);
        }
      }
    }
    // reduce-scatter over the ks lanes of this block: step s pairs lanes 2^s apart and splits on index bit 4-s
    int pre = 0;
    if (lgks > 0) { const bool b = kp & 1; rs_step<32>(acc, b, 1); pre |= b ? 16 : 0; }
    if (lgks > 1) { const bool b = kp & 2; rs_step<16>(acc, b, 2); pre |= b ? 8 : 0; }
    if (lgks > 2) { const bool b = kp & 4; rs_step<8>(acc, b, 4); pre |= b ? 4 : 0; }
    if (lgks > 3) { const bool b = kp & 8; rs_step<4>(acc, b, 8); pre |= b ? 2 : 0; }
    if (lgks > 4) { const bool b = kp & 16; rs_step<2>(acc, b, 16); pre |= b ? 1 : 0; }
    if (valid) {
      const WgOut w{gacc, gbias, ot, itl, n_ot, n_it, nout, nin, ninp, pre};
      if (lgks == 0) wg_writeback<32>(acc, w);
      else if (lgks == 1) wg_writeback<16>(acc, w);
      else if (lgks == 2) wg_writeback<8>(acc, w);
      else if (lgks == 3) wg_writeback<4>(acc, w);
      else if (lgks == 4) wg_writeback<2>(acc, w);
      else wg_writeback<1>(acc, w);
    }
  }
}

__device__ __forceinline__ void f1_sigmoid(float t, float& s, float& ls) {
  const float e = expf(-fabsf(t));
  const float l1p = log1pf(e);
  if (t >= 0.f) { s = 1.f / (1.f + e); ls = -l1p; }
  else { s = e / (1.f + e); ls = t - l1p; }
}

// global [samples][n] row-major  ->  smem [n][ld] (samples past nvalid read as zero), asynchronously: every thread
// queues all of its 4-byte cp.async copies at once (each warp copy is one coalesced row segment); the caller commits,
// waits (cp_async_wait_all) and synchronises before reading the tile.
__device__ __forceinline__ void tile_load_async(const float* __restrict__ g, int n, float* __restrict__ sm, int ld,
                                                long long s0, int nvalid, int NT) {
  const int fx = threadIdx.x & 63, qy = threadIdx.x >> 6;
  const int nsg = NT >> 2;
  for (int q = qy; q < nsg; q += F1_THREADS / 64) {
    const float* gp = g + (s0 + 4 * q) * n;
    const int left = nvalid - 4 * q;
    for (int f = fx; f < n; f += 64) {
      float* dst = sm + f * ld + 4 * q;  // rows past the batch: zero-fill, source clamped to a mapped address
      cp_async4(dst, left > 0 ? gp + f : g, left > 0);
      cp_async4(dst + 1, left > 1 ? gp + n + f : g, left > 1);
      cp_async4(dst + 2, left > 2 ? gp + 2 * n + f : g, left > 2);
      cp_async4(dst + 3, left > 3 ? gp + 3 * n + f : g, left > 3);
    }
  }
}
__device__ __forceinline__ void tile_store(float* __restrict__ g, int n, const float* __restrict__ sm, int ld,
                                           long long s0, int nvalid, int NT) {
  const int fx = threadIdx.x & 63, qy = threadIdx.x >> 6;
  const int nsg = NT >> 2;
  for (int q = qy; q < nsg; q += F1_THREADS / 64) {
    float* gp = g + (s0 + 4 * q) * n;
    const int left = nvalid - 4 * q;
    for (int f = fx; f < n; f += 64) {
      const float4 v = *reinterpret_cast<const float4*>(sm + f * ld + 4 * q);
      if (left > 0) gp[f] = v.x;
      if (left > 1) gp[n + f] = v.y;
      if (left > 2) gp[2 * n + f] = v.z;
      if (left > 3) gp[3 * n + f] = v.w;
    }
  }
}

__host__ __device__ static inline int up4(int x) { return (x + 3) / 4 * 4; }

// smem (floats): PF[total_fwd] | X[nbuf][DP*ld] | Y[DP*ld] | A0[(D1+Cc)*ld if Cc] | Ha[hid*ld] | Hb[hid*ld]  (inference)
//                PF[total_fwd] | X[nbuf][DP*ld] | Y[DP*ld] | A0[...] | ACT[n_act*ld]                          (acts saved)
// with DP = max(D, 2*D2) rows and ld = NT + 4. With nbuf = 2 the next tile's input streams in while this one computes.
__global__ void __launch_bounds__(F1_THREADS, 1)
flow1d_fwd_kernel(const float* __restrict__ x, const float* __restrict__ cond, const float* __restrict__ PF,
                  const float* __restrict__ sl, float* __restrict__ y, const float* __restrict__ ld_in,
                  float* __restrict__ ld_out, float* __restrict__ acts, F1Dims d, int B, int reverse, F1Run run) {
  extern __shared__ __align__(16) float sm[];
  const int NT = run.NT, lgNT = run.lgNT, ld = NT + 4;
  const int DP = max(d.D, 2 * d.D2);
  float* W = sm;
  float* Xb = W + up4(d.total_fwd);
  float* Y = Xb + run.nbuf * DP * ld;
  float* A0 = Y + DP * ld;
  float* Hbase = A0 + (d.Cc ? (d.D1 + d.Cc) * ld : 0);
  const int tiles = (B + NT - 1) / NT;
  if (static_cast<int>(blockIdx.x) < tiles) {
    const long long s0 = static_cast<long long>(blockIdx.x) * NT;
    tile_load_async(x, d.D, Xb, ld, s0, min(NT, B - static_cast<int>(s0)), NT);
  }
  weights_load_async(PF, W, d.total_fwd);
  cp_async_commit();
  const float sl0 = sl ? sl[0] : 0.f;
  int cur = 0;
  for (int t = blockIdx.x; t < tiles; t += gridDim.x) {
    const long long s0 = static_cast<long long>(t) * NT;
    const int nvalid = min(NT, B - static_cast<int>(s0));
    float* X = Xb + cur * DP * ld;
    // this thread's log-det input, fetched now so the load is off the critical path at the end of the tile
    const int ls_s = threadIdx.x >> 2;
    const float ld_prev = (ld_out && (threadIdx.x & 3) == 0 && ls_s < nvalid) ? ld_in[s0 + ls_s] : 0.f;
    cp_async_wait_all();
    __syncthreads();  // this tile's input has landed; every buffer of the previous tile is free
    const int tn = t + gridDim.x;
    if (tn < tiles) {
      const long long sn = static_cast<long long>(tn) * NT;
      if (run.nbuf == 2) {
        tile_load_async(x, d.D, Xb + (cur ^ 1) * DP * ld, ld, sn, min(NT, B - static_cast<int>(sn)), NT);
        cp_async_commit();
      }
    }
    if (d.Cc) {
      tile_load_async(cond, d.Cc, A0 + d.D1 * ld, ld, s0, nvalid, NT);
      cp_async_commit();
      cp_async_wait_all();  // (also waits for the prefetch; conditional models are not the hot case)
      __syncthreads();
    }
    float* Z = X;  // the tensor the coupling acts on
    if (!reverse) {
      lin_tile<0>(X, d.D, Y, d.D, W + d.offWT[0], W + d.offB[0], d.noutp[0], nullptr, ld, lgNT);
      Z = Y;
      __syncthreads();
    }
    const float* a0 = Z;
    if (d.Cc) {
      for (int e = threadIdx.x; e < (d.D1 << lgNT); e += F1_THREADS) {
        const int i = e >> lgNT, s = e - (i << lgNT);
        A0[i * ld + s] = Z[i * ld + s];
      }
      a0 = A0;
      __syncthreads();
    }
    float* H[6];
    if (acts) {
      for (int l = 0; l < 6; ++l) H[l] = Hbase + l * d.hid * ld;
    } else {
      float* Ha = Hbase;
      float* Hb = Hbase + d.hid * ld;
      H[0] = Ha; H[1] = Hb; H[2] = Ha; H[3] = Hb; H[4] = Ha;
      H[5] = reverse ? Y : X;  // forward: X is dead after the affine; reverse: Y is not used yet
    }
    lin_tile<1>(a0, d.nin[1], H[0], d.hid, W + d.offWT[1], W + d.offB[1], d.noutp[1], nullptr, ld, lgNT);
    __syncthreads();
    lin_tile<1>(H[0], d.hid, H[1], d.hid, W + d.offWT[2], W + d.offB[2], d.noutp[2], nullptr, ld, lgNT);
    __syncthreads();
    lin_tile<1>(H[1], d.hid, H[2], d.hid, W + d.offWT[3], W + d.offB[3], d.noutp[3], nullptr, ld, lgNT);
    __syncthreads();
    lin_tile<1>(H[2], d.hid, H[3], d.hid, W + d.offWT[4], W + d.offB[4], d.noutp[4], nullptr, ld, lgNT);
    __syncthreads();
    lin_tile<2>(H[3], d.hid, H[4], d.hid, W + d.offWT[5], W + d.offB[5], d.noutp[5], nullptr, ld, lgNT);
    __syncthreads();
    lin_tile<0>(H[4], d.hid, H[5], 2 * d.D2, W + d.offWT[6], W + d.offB[6], d.noutp[6], nullptr, ld, lgNT);
    __syncthreads();
    // affine coupling + per-sample log-det: four threads per sample (j mod 4), combined by two shuffles
    {
      const float* O = H[5];
      const int s = threadIdx.x >> 2, part = threadIdx.x & 3;
      float ldacc = 0.f;
      if (s < NT) {
        for (int j = part; j < d.D2; j += 4) {
          const float sh = O[(2 * j) * ld + s], lg = O[(2 * j + 1) * ld + s];
          float sg, ls;
          f1_sigmoid(lg + 2.f, sg, ls);
          const float z2 = Z[(d.D1 + j) * ld + s];
          Z[(d.D1 + j) * ld + s] = reverse ? (z2 / sg - sh) : (z2 + sh) * sg;
          ldacc += ls;
        }
      }
      ldacc += __shfl_xor_sync(0xffffffffu, ldacc, 1);
      ldacc += __shfl_xor_sync(0xffffffffu, ldacc, 2);
      if (reverse) ldacc = -ldacc;
      if (ld_out && part == 0 && s < nvalid) ld_out[s0 + s] = ld_prev + sl0 + ldacc;
    }
    __syncthreads();
    float* OUT = Z;
    if (reverse) {
      // inverse affine last; Y is free (it only ever held the MLP output, consumed above)
      lin_tile<0>(X, d.D, Y, d.D, W + d.offWT[0], W + d.offB[0], d.noutp[0], nullptr, ld, lgNT);
      OUT = Y;
      __syncthreads();
    }
    tile_store(y, d.D, OUT, ld, s0, nvalid, NT);
    if (acts) tile_store(acts, d.n_act, Hbase, ld, s0, nvalid, NT);
    if (run.nbuf == 2) {
      cur ^= 1;
    } else if (tn < tiles) {
      __syncthreads();  // single buffer: the next input may only land once this tile's stores have read X / Y
      const long long sn = static_cast<long long>(tn) * NT;
      tile_load_async(x, d.D, Xb, ld, sn, min(NT, B - static_cast<int>(sn)), NT);
      cp_async_commit();
    }
  }
}

// Backward of one 1-D FlowStep (either direction). Reads the saved MLP activations, the incoming gradients and
// (forward direction) the step OUTPUT y_out, whose first D1 features are the MLP input and whose last D2 features are
// (y2 + shift) * scale, or (reverse direction) the step input; writes the input gradient and accumulates the
// parameter gradients into G (global, pre-zeroed).
// smem (floats): PB[total_bwd] | GA[total_grad] | XY[DR*ld] | GZ[gzr*ld] | A0[(D1+Cc)*ld if Cc] | ACT[n_act*ld] |
//                SC[scr*ld] | GL[NT]      DR = D rounded up to 8; scr = hid | D1+Cc (forward direction), DR (reverse)
__global__ void __launch_bounds__(F1_THREADS, 1)
flow1d_bwd_kernel(const float* __restrict__ x_in, const float* __restrict__ cond, const float* __restrict__ acts,
                  const float* __restrict__ PB, const float* __restrict__ y_out, const float* __restrict__ g_out,
                  const float* __restrict__ g_ld, float* __restrict__ dx, float* __restrict__ G, F1Dims d, int B,
                  int reverse, int scr, int gzr, F1Run run) {
  extern __shared__ __align__(16) float sm[];
  const int NT = run.NT, lgNT = run.lgNT, ld = NT + 4;
  const int DR = up8d(d.D);
  float* W = sm;
  float* GA = W + up4(d.total_bwd);
  float* XY = GA + up4(d.total_grad);
  float* GZ = XY + DR * ld;      // gzr rows: D, and in the reverse direction also the MLP scratch (hid | D1+Cc)
  float* A0 = GZ + gzr * ld;
  float* ACT = A0 + (d.Cc ? (d.D1 + d.Cc) * ld : 0);
  float* SC = ACT + d.n_act * ld;
  float* GL = SC + scr * ld;  // [NT] incoming log-det gradient of the tile
  weights_load_async(PB, W, d.total_bwd);   // lands with the first tile's cp.async group
  for (int e = threadIdx.x; e < d.total_grad; e += F1_THREADS) GA[e] = 0.f;
  const int tiles = (B + NT - 1) / NT;
  for (int t = blockIdx.x; t < tiles; t += gridDim.x) {
    const long long s0 = static_cast<long long>(t) * NT;
    const int nvalid = min(NT, B - static_cast<int>(s0));
    __syncthreads();
    tile_load_async(reverse ? x_in : y_out, d.D, XY, ld, s0, nvalid, NT);
    tile_load_async(g_out, d.D, GZ, ld, s0, nvalid, NT);
    tile_load_async(acts, d.n_act, ACT, ld, s0, nvalid, NT);
    if (d.Cc) tile_load_async(cond, d.Cc, A0 + d.D1 * ld, ld, s0, nvalid, NT);
    if (static_cast<int>(threadIdx.x) < NT) {
      const bool ok = g_ld && static_cast<int>(threadIdx.x) < nvalid;
      cp_async4(GL + threadIdx.x, ok ? g_ld + s0 + threadIdx.x : g_out, ok);
    }
    cp_async_commit();
    cp_async_wait_all();
    __syncthreads();
    float* H[5];
    for (int l = 0; l < 5; ++l) H[l] = ACT + l * d.hid * ld;
    float* O = ACT + 5 * d.hid * ld;
    float* gz = GZ;      // gradient wrt the coupling output
    float* scr_buf = SC;  // scratch rows for the MLP backward
    if (reverse) {
      // reverse step = coupling^-1 then x = Wi z' + bi. Rebuild z' in place of the input's second half, take the
      // affine's weight gradient against it and pull g_out through Wi.
      for (int e = threadIdx.x; e < (d.D2 << lgNT); e += F1_THREADS) {
        const int j = e >> lgNT, s = e - (j << lgNT);
        float sg, ls;
        f1_sigmoid(O[(2 * j + 1) * ld + s] + 2.f, sg, ls);
        XY[(d.D1 + j) * ld + s] = XY[(d.D1 + j) * ld + s] / sg - O[(2 * j) * ld + s];
      }
      __syncthreads();
      wgrad_tile(GZ, d.D, XY, d.D, d.ninp[0], GA + d.offG[0], GA + d.offGB[0], ld, lgNT, run.wg[0]);
      lin_tile<0, true>(GZ, d.D, SC, d.D, W + d.offW[0], nullptr, d.ninp[0], nullptr, ld, lgNT);  // dL/dz'
      __syncthreads();
      gz = SC;
      scr_buf = GZ;
    }
    const float* a0 = XY;  // first D1 features: the MLP input in either direction
    if (d.Cc) {
      for (int e = threadIdx.x; e < (d.D1 << lgNT); e += F1_THREADS) {
        const int i = e >> lgNT, s = e - (i << lgNT);
        A0[i * ld + s] = XY[i * ld + s];
      }
      a0 = A0;
    }
    // coupling backward: dO in place over O; gz[D1+j] becomes the gradient wrt the pre-coupling z2
    for (int e = threadIdx.x; e < (d.D2 << lgNT); e += F1_THREADS) {
      const int j = e >> lgNT, s = e - (j << lgNT);
      const float gl = GL[s];
      const float sh = O[(2 * j) * ld + s];
      float sg, ls;
      f1_sigmoid(O[(2 * j + 1) * ld + s] + 2.f, sg, ls);
      const float g2 = gz[(d.D1 + j) * ld + s];
      const float v = XY[(d.D1 + j) * ld + s];  // forward: (y2 + sh) * sg;  reverse: z' = z2 / sg - sh
      float dsh, dlg, dz2;
      if (!reverse) {
        dsh = g2 * sg;
        dlg = (g2 * v + gl) * (1.f - sg);
        dz2 = g2 * sg;
      } else {
        dsh = -g2;
        dlg = -(g2 * (v + sh) + gl) * (1.f - sg);
        dz2 = g2 / sg;
      }
      O[(2 * j) * ld + s] = dsh;
      O[(2 * j + 1) * ld + s] = dlg;
      gz[(d.D1 + j) * ld + s] = dz2;
    }
    __syncthreads();
    // MLP backward, layer 6 .. 1. Gradient slots: layer 6 and layer 1 -> scratch, layers 5..2 -> the (consumed)
    // activation slot of the layer above. Each phase runs the layer's weight gradient (threads from 0 up) next to
    // its data gradient (threads from the top down).
    const float* dcur = O;
    int ncur = 2 * d.D2;
    for (int l = 6; l >= 1; --l) {
      const float* in = (l == 1) ? a0 : H[l - 2];
      const int nin = d.nin[l];
      wgrad_tile(dcur, ncur, in, nin, d.ninp[l], GA + d.offG[l], GA + d.offGB[l], ld, lgNT, run.wg[l]);
      float* dn = (l == 6 || l == 1) ? scr_buf : H[l - 1];
      if (l == 6) lin_tile<4, true>(dcur, ncur, dn, nin, W + d.offW[l], nullptr, d.ninp[l], H[l - 2], ld, lgNT);
      else if (l >= 2) lin_tile<3, true>(dcur, ncur, dn, nin, W + d.offW[l], nullptr, d.ninp[l], H[l - 2], ld, lgNT);
      else lin_tile<0, true>(dcur, ncur, dn, d.D1, W + d.offW[l], nullptr, d.ninp[l], nullptr, ld, lgNT);
      __syncthreads();
      if (l == 6 && !reverse) {
        // dO is dead: its 2*D2 >= D rows take the step input for the affine's weight gradient, streaming in
        // behind the rest of the MLP backward
        tile_load_async(x_in, d.D, O, ld, s0, nvalid, NT);
        cp_async_commit();
      }
      dcur = dn;
      ncur = nin;
    }
    for (int e = threadIdx.x; e < (d.D1 << lgNT); e += F1_THREADS) {
      const int i = e >> lgNT, s = e - (i << lgNT);
      gz[i * ld + s] += dcur[i * ld + s];
    }
    const float* DX = gz;
    if (!reverse) {
      cp_async_wait_all();
      __syncthreads();
      wgrad_tile(gz, d.D, O, d.D, d.ninp[0], GA + d.offG[0], GA + d.offGB[0], ld, lgNT, run.wg[0]);
      lin_tile<0, true>(gz, d.D, XY, d.D, W + d.offW[0], nullptr, d.ninp[0], nullptr, ld, lgNT);  // dx = W'^T dy
      DX = XY;
    }
    __syncthreads();
    tile_store(dx, d.D, DX, ld, s0, nvalid, NT);
  }
  __syncthreads();
  // staggered start so the CTAs do not all hit the same addresses at once
  const int start = static_cast<int>((static_cast<long long>(blockIdx.x) * 997) % d.total_grad);
  for (int k = threadIdx.x; k < d.total_grad; k += F1_THREADS) {
    int e = k + start;
    if (e >= d.total_grad) e -= d.total_grad;
    const float v = GA[e];
    if (v != 0.f) atomicAdd(G + e, v);
  }
}

// Stand-alone per-row affine y = W x + b on [B, D] (ActNorm1d / InvertibleConv1x1 called on their own).
__global__ void affine_rows_kernel(const float* __restrict__ x, const float* __restrict__ Wf,
                                   const float* __restrict__ bf, const float* __restrict__ sl, float* __restrict__ y,
                                   const float* __restrict__ ld_in, float* __restrict__ ld_out, int B, int D,
                                   float pixels) {
  extern __shared__ float sm[];
  float* W = sm;
  float* b = W + D * D;
  for (int e = threadIdx.x; e < D * D; e += blockDim.x) W[e] = Wf[e];
  for (int e = threadIdx.x; e < D; e += blockDim.x) b[e] = bf[e];
  __syncthreads();
  const long long total = static_cast<long long>(B) * D;
  for (long long e = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; e < total;
       e += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long r = e / D;
    const int o = static_cast<int>(e - r * D);
    const float* xr = x + r * D;
    float a = b[o];
    for (int i = 0; i < D; ++i) a = fmaf(W[o * D + i], xr[i], a);
    y[e] = a;
    if (o == 0 && ld_out) ld_out[r] = ld_in[r] + sl[0] * pixels;
  }
}

static int ilog2(int x) { int l = 0; while ((1 << (l + 1)) <= x) ++l; return l; }

static void f1_run_fill(const F1Dims& d, int nt, int nbuf, F1Run* run) {
  run->NT = nt; run->lgNT = ilog2(nt); run->nbuf = nbuf;
  const int nsg = nt >> 2;
  for (int l = 0; l < F1_LAYERS; ++l) {
    F1Wg& w = run->wg[l];
    w.n_ot = (d.nout[l] + 7) >> 3;
    w.n_it = (d.nin[l] + 1 + 3) >> 2;  // + the ones row that carries the bias gradient
    const int ntiles = w.n_ot * w.n_it;
    int lg = 0;  // split the samples over 2^lg lanes while threads are idle and every lane keeps >= 2 steps
    while (lg < 5 && (ntiles << (lg + 1)) <= F1_THREADS && (4 << lg) <= nsg) ++lg;
    w.lgks = lg;
  }
}

// Largest power-of-two sample tile NT whose working set fits (the bank pattern of ld = NT + 4 needs NT % 32 == 0),
// double-buffering the input when there is room.
static int f1_tile_fwd(const F1Dims& d, bool save, int* smem_out, F1Run* run) {
  const int DP = d.D > 2 * d.D2 ? d.D : 2 * d.D2;
  for (int nt = 128; nt >= 32; nt >>= 1) {
    for (int nbuf = 2; nbuf >= 1; --nbuf) {
      const int ld = nt + 4;
      long long fl = up4(d.total_fwd) + (1LL + nbuf) * DP * ld + (d.Cc ? (d.D1 + d.Cc) * ld : 0) +
                     (save ? 1LL * d.n_act * ld : 2LL * d.hid * ld);
      if (fl * 4 <= 225 * 1024) { *smem_out = static_cast<int>(fl * 4); f1_run_fill(d, nt, nbuf, run); return nt; }
    }
  }
  return 0;
}

static int f1_tile_bwd(const F1Dims& d, int scr, int gzr, int* smem_out, F1Run* run) {
  const int DR = up8(d.D);
  for (int nt = 128; nt >= 32; nt >>= 1) {
    const int ld = nt + 4;
    long long fl = up4(d.total_bwd) + up4(d.total_grad) + 1LL * (DR + gzr) * ld + (d.Cc ? (d.D1 + d.Cc) * ld : 0) +
                   1LL * d.n_act * ld + 1LL * scr * ld + nt;
    if (fl * 4 <= 225 * 1024) { *smem_out = static_cast<int>(fl * 4); f1_run_fill(d, nt, 1, run); return nt; }
  }
  return 0;
}

}  // namespace nfk

using namespace nfk;

extern "C" int nfk_flow1d_sizes(int D, int Cc, int hid, int* total_fwd, int* total_bwd, int* total_grad, int* n_act,
                                int* offsets /* [7*4]: offG, offGB, ninp, noutp per layer */) {
  if (D < 2 || hid <= 0 || Cc < 0) return NFK_ERR_SHAPE;
  const F1Dims d = f1_dims(D, Cc, hid);
  if (total_fwd) *total_fwd = d.total_fwd;
  if (total_bwd) *total_bwd = d.total_bwd;
  if (total_grad) *total_grad = d.total_grad;
  if (n_act) *n_act = d.n_act;
  if (offsets)
    for (int l = 0; l < F1_LAYERS; ++l) {
      offsets[4 * l + 0] = d.offG[l]; offsets[4 * l + 1] = d.offGB[l];
      offsets[4 * l + 2] = d.ninp[l]; offsets[4 * l + 3] = d.noutp[l];
    }
  return NFK_OK;
}

extern "C" int nfk_flow1d_supported(int D, int Cc, int hid, int training) {
  // the fused kernels keep every weight of the step in shared memory: 1 when the inference kernel -- and, with
  // training != 0, the activation-saving forward and the backward of both directions -- find a sample tile that fits
  if (D < 2 || hid <= 0 || Cc < 0) return 0;
  const F1Dims d = f1_dims(D, Cc, hid);
  int smem = 0;
  F1Run run{};
  if (!f1_tile_fwd(d, false, &smem, &run)) return 0;
  if (!training) return 1;
  if (!f1_tile_fwd(d, true, &smem, &run)) return 0;
  const int mlp_scr = hid > d.nin[1] ? hid : d.nin[1];
  const int gzr = up8(D) > mlp_scr ? up8(D) : mlp_scr;
  if (!f1_tile_bwd(d, mlp_scr, up8(D), &smem, &run) || !f1_tile_bwd(d, up8(D), gzr, &smem, &run)) return 0;
  return 1;
}

extern "C" int nfk_flow1d_pack(const float* Wf, const float* bf, const float* const* w, const float* const* b, int D,
                               int Cc, int hid, float* PF, float* PB, void* stream) {
  if (D < 2 || hid <= 0 || Cc < 0) return NFK_ERR_SHAPE;
  if (!Wf || !bf || !w || !b || !PF) return NFK_ERR_ARG;
  const F1Dims d = f1_dims(D, Cc, hid);
  F1Weights src{};
  src.Wf = Wf; src.bf = bf;
  for (int l = 0; l < 6; ++l) { src.w[l] = w[l]; src.b[l] = b[l]; if (!w[l] || !b[l]) return NFK_ERR_ARG; }
  const int total = d.total_fwd + (PB ? d.total_bwd : 0);
  flow1d_pack_kernel<<<(total + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(src, d, PF, PB);
  return cudaGetLastError() == cudaSuccess ? NFK_OK : NFK_ERR_LAUNCH;
}

extern "C" int nfk_flow1d_fwd(const float* x, const float* cond, const float* PF, const float* sl, float* y,
                              const float* ld_in, float* ld_out, float* acts, int B, int D, int Cc, int hid,
                              int reverse, void* stream) {
  if (B <= 0 || D < 2 || hid <= 0 || Cc < 0) return NFK_ERR_SHAPE;
  if (!x || !PF || !y || (Cc && !cond) || (ld_out && !ld_in)) return NFK_ERR_ARG;
  const F1Dims d = f1_dims(D, Cc, hid);
  int smem = 0;
  F1Run run{};
  const int nt = f1_tile_fwd(d, acts != nullptr, &smem, &run);
  if (!nt) return NFK_ERR_SHAPE;
  if (int rc = ensure_dyn_smem(reinterpret_cast<const void*>(flow1d_fwd_kernel), smem)) return rc;
  const int tiles = (B + nt - 1) / nt;
  const int grid = tiles < 148 ? tiles : 148;
  flow1d_fwd_kernel<<<grid, F1_THREADS, smem, static_cast<cudaStream_t>(stream)>>>(x, cond, PF, sl, y, ld_in, ld_out,
                                                                                  acts, d, B, reverse, run);
  return cudaGetLastError() == cudaSuccess ? NFK_OK : NFK_ERR_LAUNCH;
}

extern "C" int nfk_flow1d_bwd(const float* x_in, const float* cond, const float* acts, const float* PB,
                              const float* y_out, const float* g_out, const float* g_ld, float* dx, float* G, int B,
                              int D, int Cc, int hid, int reverse, void* stream) {
  if (B <= 0 || D < 2 || hid <= 0 || Cc < 0) return NFK_ERR_SHAPE;
  if (!x_in || !acts || !PB || !g_out || !dx || !G || (Cc && !cond) || (!reverse && !y_out)) return NFK_ERR_ARG;
  const F1Dims d = f1_dims(D, Cc, hid);
  const int mlp_scr = hid > d.nin[1] ? hid : d.nin[1];  // rows the MLP backward needs for its ping-pong buffer
  int scr = mlp_scr, gzr = up8(D);
  if (reverse) {  // dL/dz' lives in SC, the incoming-gradient buffer becomes the MLP scratch
    scr = up8(D);
    gzr = gzr > mlp_scr ? gzr : mlp_scr;
  }
  int smem = 0;
  F1Run run{};
  const int nt = f1_tile_bwd(d, scr, gzr, &smem, &run);
  if (!nt) return NFK_ERR_SHAPE;
  if (int rc = ensure_dyn_smem(reinterpret_cast<const void*>(flow1d_bwd_kernel), smem)) return rc;
  const int tiles = (B + nt - 1) / nt;
  const int grid = tiles < 148 ? tiles : 148;
  flow1d_bwd_kernel<<<grid, F1_THREADS, smem, static_cast<cudaStream_t>(stream)>>>(x_in, cond, acts, PB, y_out, g_out,
                                                                                  g_ld, dx, G, d, B, reverse, scr, gzr, run);
  return cudaGetLastError() == cudaSuccess ? NFK_OK : NFK_ERR_LAUNCH;
}

extern "C" int nfk_affine_rows(const float* x, const float* Wf, const float* bf, const float* sl, float* y,
                               const float* ld_in, float* ld_out, int B, int D, float pixels, void* stream) {
  if (B <= 0 || D <= 0 || D > 160) return NFK_ERR_SHAPE;
  if (!x || !Wf || !bf || !y || (ld_out && (!ld_in || !sl))) return NFK_ERR_ARG;
  const int smem = (D * D + D) * 4;
  if (int rc = ensure_dyn_smem(reinterpret_cast<const void*>(affine_rows_kernel), smem)) return rc;
  const long long total = static_cast<long long>(B) * D;
  const int grid = static_cast<int>((total + 255) / 256 < 1184 ? (total + 255) / 256 : 1184);
  affine_rows_kernel<<<grid, 256, smem, static_cast<cudaStream_t>(stream)>>>(x, Wf, bf, sl, y, ld_in, ld_out, B, D,
                                                                           pixels);
  return cudaGetLastError() == cudaSuccess ? NFK_OK : NFK_ERR_LAUNCH;
}
