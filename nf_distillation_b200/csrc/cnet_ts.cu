// Fused conv#1 -> conv#2 of the coupling network with h1 resident in TENSOR MEMORY (the A operand of conv#2 is read
// by tcgen05.mma straight from TMEM, never from shared memory):
//
//   h1 = relu(col * B1^T + b1)       conv3x3 as im2col GEMM          (reference models/flows.py:27-28)
//   h2 = relu(h1  * B2^T + b2)       conv1x1                         (:29-30)
//
// Why h1 lives in TMEM and not in 128B-swizzled shared-memory panels: with h1 in shared memory as conv#2's A operand the
// kernel is bound by shared-memory bandwidth, not by the tensor pipe — per 256x256x16 MMA each SM reads 4 KB of h1 +
// 4 KB of B2 while TMA refills 4 KB and the epilogue moves ~3 KB: 118 of the 128 B/clk the SM has (measured 153 cycles
// per MMA against 128 in isolation, plus operand waits on a 4-slot ring that 128 KB of h1 panels leave no room to
// deepen). Here the epilogue warps write the bf16 activations back into TMEM (tcgen05.st, two K elements per 32-bit
// column: 256 columns for K = 512) and conv#2 is issued with A = [tmem]: shared memory only carries the weights
// (32 B/clk read + 32 B/clk refill) and the store staging, and the 128 KB the panels would take hold the weight ring.
//
//   TMEM   [0,256) h1 (bf16x2 per column) | [256,384) accumulator 0 | [384,512) accumulator 1
//          -> a tile is 4 + 4 quarter-GEMMs of N = 128 (M = 256 over the CTA pair), ping-pong over the two accumulators
//   smem   A tile of GEMM 1 (kb1 x 16 KB, loaded once per tile, prefetched a tile ahead) | store staging 16 warps x
//          4 KB | weight ring nslots x 8 KB (64 weight rows x 64 K per CTA and slot)
//   warps  0: TMA producer, 1: MMA issuer (leader CTA) + TMEM alloc, 2-17: epilogue (4 per TMEM lane quadrant)
//
// MODE 0: forward (+ optional h1 / 1-bit ReLU mask outputs for training).
// MODE 1: the student's backward chain, the two dgrads of Conv2dZeros input gradient -> ReLU mask of h2 -> conv1x1
//         input gradient -> ReLU mask of h1:  d2 = mask_h2 .* (dhcol B3T^T),  d1 = mask_h1 .* (d2 B2T^T). Both are
//         written out as bf16 (the weight-gradient GEMMs read them), and their column sums are the two bias gradients.
//         Same tiles, same pipeline: d2 takes h1's place in TMEM as the A operand of the second GEMM.
// Results are bit-identical to the two unfused GEMMs of gemm_tc.cu (same bf16 products, same K order in the fp32
// accumulators; the N split does not enter the arithmetic).
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <cstdint>

#include "../../include/nfk.h"
#include "launch_util.h"
#include "ptx.cuh"

namespace nfk {

constexpr int TS_THREADS = 576;      // 18 warps: TMA producer, MMA issuer, 16 epilogue warps
constexpr int TS_HID = 512;
constexpr int TS_BOX = 8192;          // one weight box: this CTA's 64 rows of a 128-row weight tile x 64 K (128 B)
constexpr int TS_SLOT = 2 * TS_BOX;   // ring slot = two consecutive k-blocks of one quarter: ONE barrier round trip per
                                      // 8 MMAs (a single-warp wait + expect_tx + issue loop costs ~280 cycles per
                                      // iteration, tools/micro/tma_bench.cu: at one 8 KB box per iteration the producer
                                      // delivers 29 B/clk against the 32 B/clk the quarter MMAs consume)
constexpr int TS_MAX_SLOTS = 8;
constexpr int TS_COLBLK = 16384;      // 128 rows x 128 B: one k-block of the A tile of GEMM 1
constexpr int TS_STAGE = 4096;        // 32 rows x 128 B store staging panel
constexpr int TS_STAGE_BYTES = 16 * TS_STAGE;   // one panel per epilogue warp
constexpr int TS_BAR_BYTES = 512;
constexpr int TS_BIAS_BYTES = 2 * TS_HID * 4;   // both bias vectors, staged once per CTA (MODE 0)
constexpr uint32_t TS_ACC0 = 256;     // first accumulator column

struct TsArgs {
  int M;
  int kb1;           // K1p / 64
  int nslots;
  const float* bias1;
  const float* bias2;
  uint32_t* mask1;   // 1-bit ReLU masks, word-major [16][ldmask]. MODE 0: optional outputs; MODE 1: the masks applied
  uint32_t* mask2;   // to the outputs of GEMM 1 / GEMM 2
  long long ldmask;
  int store_h1;
  long long* prof;   // diagnostics: [grid][8] cycle counters of the MMA issuer
  // GEMM-2 k-blocks (64 input channels each) that are not structurally zero for output half 0 / 1; 8 = all. MADE's
  // degree-sorted hidden mask is block lower triangular: the low-degree half of the outputs never sees the high-degree
  // inputs, so those B2 tiles are neither loaded nor multiplied (they are exact zeros: the result is bit-identical).
  int kb2_end[2];
  float* colsum1;    // MODE 1: column sums of the masked GEMM 1 / GEMM 2 outputs (the bias gradients), or NULL
  float* colsum2;
};

__device__ __forceinline__ void umma_f16_pair_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc,
                                                 uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n"
      ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// 32 lanes x 16 consecutive 32-bit columns: thread t of the warp writes TMEM lane (base_lane + t)
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&a)[8], const uint32_t (&b)[8]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
      ::"r"(taddr), "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]), "r"(b[0]),
        "r"(b[1]), "r"(b[2]), "r"(b[3]), "r"(b[4]), "r"(b[5]), "r"(b[6]), "r"(b[7])
      : "memory");
}
// {lo, hi} -> bf16x2 word (lo in bits 0-15) with ReLU folded into the conversion
__device__ __forceinline__ uint32_t relu_bf16x2(float lo, float hi) {
  uint32_t d;
  asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
  return d;
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

template <int MODE>
__device__ __forceinline__ void cnet_ts_body(const CUtensorMap& tmCol, const CUtensorMap& tmB1, const CUtensorMap& tmB2,
                                             const CUtensorMap& tmH1, const CUtensorMap& tmH2, const TsArgs& g) {
  extern __shared__ __align__(1024) uint8_t smem[];
  pdl_launch_dependents();
  if (smem_u32(smem) & 1023u) __trap();
  const int warp = static_cast<int>(uniform_u32(threadIdx.x >> 5)), lane = threadIdx.x & 31;
  const uint32_t rank = blockIdx.x & 1;      // == %cluster_ctarank for (2,1,1) clusters on a 1-D grid, provably uniform
  const int pair = blockIdx.x >> 1, num_pairs = gridDim.x >> 1;
  const int num_tiles = (g.M + 255) / 256;
  const int nslots = g.nslots;

  uint8_t* colbuf = smem;
  uint8_t* stage_base = colbuf + g.kb1 * TS_COLBLK;
  uint8_t* ring = stage_base + TS_STAGE_BYTES;
  uint64_t* full = reinterpret_cast<uint64_t*>(ring + nslots * TS_SLOT);   // [8] slot filled (leader)
  uint64_t* empty = full + TS_MAX_SLOTS;                                    // [8] slot consumed (local)
  uint64_t* acc_full = empty + TS_MAX_SLOTS;                                // [2]
  uint64_t* acc_empty = acc_full + 2;                                       // [2] (leader, 16 arrivals)
  uint64_t* h1_full = acc_empty + 2;                                        // [8] per 64 channels of h1 (leader, 8 arrivals)
  uint64_t* h1_empty = h1_full + 8;                                         // GEMM 2 of the tile has finished reading h1
  uint64_t* col_full = h1_empty + 1;                                        // A tile of GEMM 1 landed (leader)
  uint64_t* col_empty = col_full + 1;                                       // GEMM 1 of the tile has finished reading it
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(col_empty + 1);
  float* bias_s = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(full) + TS_BAR_BYTES);   // [2][512]

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmCol); tma_prefetch_desc(&tmB1); tma_prefetch_desc(&tmB2); tma_prefetch_desc(&tmH2);
    for (int s = 0; s < nslots; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(&acc_full[a], 1); mbar_init(&acc_empty[a], 16); }
    for (int p = 0; p < 8; ++p) mbar_init(&h1_full[p], 8);
    mbar_init(h1_empty, 1);
    mbar_init(col_full, 1);
    mbar_init(col_empty, 1);
    fence_mbar_init();
  }
  if (warp == 1) { tmem_alloc_pair(tmem_slot, 512); tmem_relinquish_pair(); }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = uniform_u32(*tmem_slot);
  pdl_wait();      // the prologue above overlapped the previous kernel's tail; global memory only from here on

  if (warp == 0) {
    // ===================================================== TMA producer (both CTAs; bytes land on the leader's barrier)
    // (whole warp in uniform control flow, single-thread instructions elected inside the asm: see ptx.cuh)
    {
      int s = 0; uint32_t ph = 0, col_ph = 0;
      // one slot: k-blocks kb, kb + 1 (< kend) of the weight rows starting at `row`
      auto load = [&](const CUtensorMap* tm, int kb, int kend, int row) {
        const int nkb = kend - kb < 2 ? kend - kb : 2;
        mbar_wait_warp(&empty[s], ph ^ 1);
        if (rank == 0) mbar_expect_tx_elect(&full[s], static_cast<uint32_t>(2 * nkb * TS_BOX));
        for (int j = 0; j < nkb; ++j)
          tma_load_2d_pair_elect(ring + s * TS_SLOT + j * TS_BOX, tm, &full[s], (kb + j) * 64, row);
        if (++s == nslots) { s = 0; ph ^= 1; }
      };
      auto load_col = [&](int t) {
        mbar_wait_warp(col_empty, col_ph ^ 1);
        if (rank == 0) mbar_expect_tx_elect(col_full, static_cast<uint32_t>(2 * g.kb1 * TS_COLBLK));
        const int row0 = t * 256 + static_cast<int>(rank) * 128;
        for (int kb = 0; kb < g.kb1; ++kb)
          tma_load_2d_pair_elect(colbuf + kb * TS_COLBLK, &tmCol, col_full, kb * 64, row0);
        col_ph ^= 1;
      };
      if (pair < num_tiles) load_col(pair);
      for (int t = pair; t < num_tiles; t += num_pairs) {
        const int wrow = static_cast<int>(rank) * 64;
        for (int q = 0; q < 4; ++q)
          for (int kb = 0; kb < g.kb1; kb += 2) load(&tmB1, kb, g.kb1, q * 128 + wrow);
        for (int q = 0; q < 4; ++q) {
          const int qe = q;
          const int kend = qe < 2 ? g.kb2_end[0] : g.kb2_end[1];
          for (int kb = 0; kb < kend; kb += 2) load(&tmB2, kb, kend, qe * 128 + wrow);
          // the next tile's A tile: GEMM 1 of this tile has retired by the time the first GEMM-2 quarter's weights are
          // in flight, so the wait inside load_col does not hold back the weight stream
          if (q == 0 && t + num_pairs < num_tiles) load_col(t + num_pairs);
        }
      }
    }
  } else if (warp == 1) {
    // ===================================================== MMA issuer (leader CTA; whole warp, uniform control flow)
    if (rank == 0) {
      const uint32_t idesc = umma_idesc_bf16(256, 128, false, false);
      const uint32_t ring_addr = smem_u32(ring);
      const uint32_t col_addr = smem_u32(colbuf);
      int s = 0; uint32_t ph = 0;
      uint32_t nacc = 0;          // accumulator uses so far (stage = nacc & 1, phase = (nacc >> 1) & 1)
      uint32_t tile_ph = 0;
      long long w_op = 0, w_acc = 0, w_h1 = 0, w_col = 0, w_b1 = 0, w_q0 = 0;
      const long long t_begin = g.prof ? clock64() : 0;
      auto take = [&]() {
        const long long c0 = g.prof ? clock64() : 0;
        mbar_wait_warp(&full[s], ph);
        if (g.prof) w_op += clock64() - c0;
        tc_fence_after();
        return ring_addr + s * TS_SLOT;
      };
      auto release = [&]() { umma_commit_pair_elect(&empty[s], 3); if (++s == nslots) { s = 0; ph ^= 1; } };
      auto acc_begin = [&]() {
        const uint32_t st = nacc & 1;
        const long long c0 = g.prof ? clock64() : 0;
        mbar_wait_warp(&acc_empty[st], ((nacc >> 1) & 1) ^ 1);
        if (g.prof) w_acc += clock64() - c0;
        tc_fence_after();
        return tmem_base + TS_ACC0 + st * 128;
      };
      auto acc_end = [&]() { umma_commit_pair_elect(&acc_full[nacc & 1], 3); ++nacc; };
#ifdef NFK_CNET_TIMELINE
      auto mstamp = [&](int t, int idx) {
        if (g.prof && blockIdx.x == 0 && t == 6 * num_pairs && lane == 0) g.prof[150 * 8 + idx] = clock64();
      };
#else
      auto mstamp = [](int, int) {};
#endif
      for (int t = pair; t < num_tiles; t += num_pairs) {
        // ---- GEMM 1: four 128-channel quarters, A = the tile's im2col rows in shared memory
        mstamp(t, 0);
        {
          const long long c0 = g.prof ? clock64() : 0;
          mbar_wait_warp(col_full, tile_ph);
          if (g.prof) { w_op += clock64() - c0; w_col += clock64() - c0; }
          tc_fence_after();
        }
        const long long w_op_g1 = w_op;
        for (int q = 0; q < 4; ++q) {
          const uint32_t d = acc_begin();
          if (q == 0) mstamp(t, 1);
          for (int kb = 0; kb < g.kb1; kb += 2) {
            const uint32_t b = take();
            const int nkb = g.kb1 - kb < 2 ? g.kb1 - kb : 2;
            for (int j = 0; j < nkb; ++j) {
#pragma unroll
              for (int k = 0; k < 4; ++k)
                umma_f16_pair_elect(d, umma_desc_sw128(col_addr + (kb + j) * TS_COLBLK + k * 32, 16, 1024),
                                    umma_desc_sw128(b + j * TS_BOX + k * 32, 16, 1024), idesc,
                                    (kb + j > 0 || k > 0) ? 1u : 0u);
            }
            release();
          }
          acc_end();
        }
        umma_commit_pair_elect(col_empty, 3);
        mstamp(t, 2);
        w_b1 += w_op - w_op_g1;
        // ---- GEMM 2: A = h1 in tensor memory (written by the epilogue warps of both CTAs), weights streamed.
        //      k-block kb only needs h1 channels [64 kb, 64 kb + 64), so it starts as soon as those have been written
        int blocks_seen = 0;
        for (int q = 0; q < 4; ++q) {
          const uint32_t d = acc_begin();
          mstamp(t, 3 + q);
          const long long w_op_q = w_op;
          const int kend = q < 2 ? g.kb2_end[0] : g.kb2_end[1];
          for (int kb = 0; kb < kend; kb += 2) {
            const uint32_t b = take();
            const int nkb = kend - kb < 2 ? kend - kb : 2;
            for (int j = 0; j < nkb; ++j) {
              if (kb + j >= blocks_seen) {
                const long long c0 = g.prof ? clock64() : 0;
                mbar_wait_warp(&h1_full[kb + j], tile_ph);
                if (g.prof) w_h1 += clock64() - c0;
                tc_fence_after();
                blocks_seen = kb + j + 1;
              }
#pragma unroll
              for (int k = 0; k < 4; ++k)
                umma_f16_pair_ts_elect(d, tmem_base + static_cast<uint32_t>((kb + j) * 32 + k * 8),
                                       umma_desc_sw128(b + j * TS_BOX + k * 32, 16, 1024), idesc,
                                       (kb + j > 0 || k > 0) ? 1u : 0u);
            }
            release();
          }
          acc_end();
          if (q == 0) w_q0 += w_op - w_op_q;
          if (q == 3) mstamp(t, 7);
        }
        umma_commit_pair_elect(h1_empty, 3);      // h1 is free once every MMA issued so far has retired
        tile_ph ^= 1;
      }
      if (g.prof && lane == 0) {
        long long* o = g.prof + blockIdx.x * 8;
        o[0] = clock64() - t_begin; o[1] = w_op; o[2] = w_acc; o[3] = w_h1; o[4] = w_col; o[5] = w_b1; o[6] = w_q0;
      }
    }
  } else {
    // ===================================================== epilogue warps (16: four per TMEM lane quadrant)
    // Warp set ws = 0 / 1 drains accumulator ws, i.e. the quarters q with (q & 1) == ws of both GEMMs; inside a set, the
    // two warps of a lane quadrant take the two 64-column halves of the quarter. Two quarters are therefore converted
    // at the same time (the GEMM-1 quarters gate GEMM 2 of the tile: the tensor pipe idles while they are converted),
    // and four warps per scheduler hide the tcgen05.ld / fence / barrier round trips of one another.
    const int ew = warp - 2;               // 0..15
    const int qd = warp & 3;               // TMEM lane quadrant
    const int hf = (ew >> 2) & 1;          // which 64-column half of a 128-column accumulator
    const int ws = ew >> 3;                // accumulator stage owned by this warp
    const uint32_t lane_off = static_cast<uint32_t>(qd * 32) << 16;
    const uint32_t sw = static_cast<uint32_t>(lane & 7);
    uint8_t* panel = stage_base + ew * TS_STAGE;
    uint32_t nuse = 0, tile_ph = 0;        // uses of accumulator ws so far
    // 16 accumulator columns -> bias + ReLU -> 8 packed bf16x2 words (+ the 16 ReLU mask bits). Packed arithmetic:
    // add.f32x2, then ONE cvt.rn.relu.bf16x2.f32 per pair (round to nearest even, negatives -> +0: equals rounding the
    // fp32 ReLU, rounding is monotonic and keeps the sign)
    auto epi16 = [&](const uint32_t (&r)[16], const float* bias16, uint32_t (&p)[8], bool want_bits) -> uint32_t {
#pragma unroll
      for (int j = 0; j < 16; j += 4) {
        const float4 b = *reinterpret_cast<const float4*>(bias16 + j);
        const float2 s0 = __fadd2_rn(make_float2(__uint_as_float(r[j]), __uint_as_float(r[j + 1])),
                                     make_float2(b.x, b.y));
        const float2 s1 = __fadd2_rn(make_float2(__uint_as_float(r[j + 2]), __uint_as_float(r[j + 3])),
                                     make_float2(b.z, b.w));
        p[j / 2] = relu_bf16x2(s0.x, s0.y);
        p[j / 2 + 1] = relu_bf16x2(s1.x, s1.y);
      }
      uint32_t bits = 0;
      if (want_bits) {   // value > 0  <=>  the (non-negative) bf16 is not +0
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          bits |= ((p[k] & 0xFFFFu) ? 1u : 0u) << (2 * k);
          bits |= ((p[k] >> 16) ? 1u : 0u) << (2 * k + 1);
        }
      }
      return bits;
    };
    // MODE 1: masked copy of 16 accumulator columns
    auto epi16m = [&](const uint32_t (&r)[16], uint32_t bits16, uint32_t (&p)[8]) {
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const float lo = ((bits16 >> (2 * k)) & 1u) ? __uint_as_float(r[2 * k]) : 0.f;
        const float hi = ((bits16 >> (2 * k + 1)) & 1u) ? __uint_as_float(r[2 * k + 1]) : 0.f;
        __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
        p[k] = *reinterpret_cast<uint32_t*>(&v);
      }
    };
    // this thread's 64 packed columns (P[i] = columns 16 i .. 16 i + 15) -> its 128-byte row of the swizzled panel.
    // The panel is reused: the previous bulk store must have finished reading it.
    auto to_panel = [&](const uint32_t (&P)[4][8]) {
      if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
      __syncwarp();
      uint8_t* dst = panel + lane * 128;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        *reinterpret_cast<uint4*>(dst + ((static_cast<uint32_t>(2 * i) ^ sw) << 4)) =
            make_uint4(P[i][0], P[i][1], P[i][2], P[i][3]);
        *reinterpret_cast<uint4*>(dst + ((static_cast<uint32_t>(2 * i + 1) ^ sw) << 4)) =
            make_uint4(P[i][4], P[i][5], P[i][6], P[i][7]);
      }
      fence_proxy_async();
      __syncwarp();
    };
    // column sums of this warp's 32 x 64 panel, straight from the staged bf16 rows: lane owns the column pair
    // (lane >> 2) * 8 + (lane & 3) * 2 (+1); at row r the 32 lanes read the whole 128-byte row (conflict-free)
    auto panel_colsum = [&](float& s0, float& s1) {
      const uint8_t* pb = panel + (lane & 3) * 4;
      const uint32_t chunk = static_cast<uint32_t>(lane >> 2);
      float a0 = 0.f, a1 = 0.f, b0 = 0.f, b1 = 0.f;
#pragma unroll 8
      for (int r = 0; r < 32; r += 2) {
        const uint32_t w0 = *reinterpret_cast<const uint32_t*>(pb + r * 128 + ((chunk ^ (r & 7)) << 4));
        const uint32_t w1 = *reinterpret_cast<const uint32_t*>(pb + (r + 1) * 128 + ((chunk ^ ((r + 1) & 7)) << 4));
        a0 += __uint_as_float(w0 << 16); a1 += __uint_as_float(w0 & 0xFFFF0000u);
        b0 += __uint_as_float(w1 << 16); b1 += __uint_as_float(w1 & 0xFFFF0000u);
      }
      s0 += a0 + b0; s1 += a1 + b1;
    };
    float cs1[2][2] = {}, cs2[2][2] = {};    // [this warp's quarter][column of the pair]: bias-gradient partial sums
    if constexpr (MODE == 0) {
      // both bias vectors into shared memory (the 16 epilogue warps only: the producer and the MMA issuer are already
      // streaming). Read per use from global memory they sat on the conversion's critical path: the first quarter's
      // conversion of a tile measured ~3 k cycles, ~1 k of arithmetic
      for (int i = threadIdx.x - 64; i < TS_HID; i += TS_THREADS - 64) {
        bias_s[i] = __ldg(g.bias1 + i);
        bias_s[TS_HID + i] = __ldg(g.bias2 + i);
      }
      asm volatile("bar.sync 1, %0;" ::"n"(TS_THREADS - 64) : "memory");
    }

    // timeline probe (diagnostics, compiled in with -DNFK_CNET_TIMELINE): the 7th tile of pair 0, one warp per set
    // writes its event clocks to prof rows 148/149 (tools/cnet_diag.py prints them)
#ifdef NFK_CNET_TIMELINE
    auto stamp = [&](int t, int idx) {
      if (g.prof && blockIdx.x == 0 && t == 6 * num_pairs && lane == 0) {
        if (qd == 0 && hf == 0) g.prof[(148 + ws) * 8 + idx] = clock64();
        g.prof[(152 + ew) * 8 + idx] = clock64();      // every epilogue warp of the leader CTA: rows 152..167
      }
    };
#else
    auto stamp = [](int, int) {};
#endif
    for (int t = pair; t < num_tiles; t += num_pairs) {
      const int row0 = t * 256 + static_cast<int>(rank) * 128 + qd * 32;
      const long long row = row0 + lane;
      const bool row_ok = row < g.M;
      uint32_t mw1[4], mw2[4];     // MODE 1: this thread's ReLU-mask words of the tile (fetched before the waits)
      if constexpr (MODE == 1) {
#pragma unroll
        for (int qq = 0; qq < 2; ++qq) {
          const int c = (2 * qq + ws) * 128 + hf * 64;
          mw1[2 * qq] = row_ok ? __ldg(g.mask1 + static_cast<long long>(c >> 5) * g.ldmask + row) : 0u;
          mw1[2 * qq + 1] = row_ok ? __ldg(g.mask1 + static_cast<long long>((c + 32) >> 5) * g.ldmask + row) : 0u;
          mw2[2 * qq] = row_ok ? __ldg(g.mask2 + static_cast<long long>(c >> 5) * g.ldmask + row) : 0u;
          mw2[2 * qq + 1] = row_ok ? __ldg(g.mask2 + static_cast<long long>((c + 32) >> 5) * g.ldmask + row) : 0u;
        }
      }
      const uint32_t tm = tmem_base + TS_ACC0 + ws * 128 + hf * 64 + lane_off;
      // ---- GEMM 1 quarters -> h1 in tensor memory (+ staged copy -> TMA store when h1 is an output)
#pragma unroll
      for (int qq = 0; qq < 2; ++qq) {
        mbar_wait(&acc_full[ws], nuse & 1);
        stamp(t, qq == 0 ? 0 : 6);
        tc_fence_after();
        uint32_t R[4][16];
#pragma unroll
        for (int i = 0; i < 4; ++i) tmem_ld16(tm + 16 * i, R[i]);
        tmem_ld_wait();
        if (qq == 0) stamp(t, 1);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(&acc_empty[ws], 0);   // the quarter after next may overwrite it
        const int col0 = (2 * qq + ws) * 128 + hf * 64;
        uint32_t P[4][8];
        if constexpr (MODE == 0) {
          const bool wb = g.mask1 != nullptr;
          uint32_t b[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) b[i] = epi16(R[i], bias_s + col0 + 16 * i, P[i], wb);
          if (wb && row_ok) {
            g.mask1[static_cast<long long>(col0 >> 5) * g.ldmask + row] = b[0] | (b[1] << 16);
            g.mask1[static_cast<long long>((col0 + 32) >> 5) * g.ldmask + row] = b[2] | (b[3] << 16);
          }
        } else {
          epi16m(R[0], mw1[2 * qq] & 0xFFFFu, P[0]); epi16m(R[1], mw1[2 * qq] >> 16, P[1]);
          epi16m(R[2], mw1[2 * qq + 1] & 0xFFFFu, P[2]); epi16m(R[3], mw1[2 * qq + 1] >> 16, P[3]);
        }
        if (qq == 0) stamp(t, 2);
        if (qq == 0) {
          // h1 of the previous tile must be dead: its GEMM-2 MMAs have retired
          mbar_wait(h1_empty, tile_ph ^ 1);
          tc_fence_after();
        }
        if (qq == 0) stamp(t, 3);
        const uint32_t th = tmem_base + lane_off + static_cast<uint32_t>(col0 >> 1);
        tmem_st16(th, P[0], P[1]);
        tmem_st16(th + 16, P[2], P[3]);
        tmem_st_wait();
        if (qq == 0) stamp(t, 4);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(&h1_full[2 * (2 * qq + ws) + hf], 0);   // GEMM 2 may read these channels
        stamp(t, qq == 0 ? 5 : 7);
        if (g.store_h1) {     // the copy for HBM comes after the hand-off: it is not on the tensor pipe's critical path
          to_panel(P);
          if constexpr (MODE == 1) {
            float s0 = 0.f, s1 = 0.f;
            panel_colsum(s0, s1);
            cs1[qq][0] += s0; cs1[qq][1] += s1;
          }
          if (lane == 0) {
            if (row0 < g.M) tma_store_2d(panel, &tmH1, col0, row0);
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          }
        }
        ++nuse;
      }
      // ---- GEMM 2 quarters -> staging panel -> TMA store of h2
#pragma unroll
      for (int qq = 0; qq < 2; ++qq) {
        mbar_wait(&acc_full[ws], nuse & 1);
        tc_fence_after();
        uint32_t R[4][16];
#pragma unroll
        for (int i = 0; i < 4; ++i) tmem_ld16(tm + 16 * i, R[i]);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(&acc_empty[ws], 0);
        const int col0 = (2 * qq + ws) * 128 + hf * 64;
        uint32_t P[4][8];
        if constexpr (MODE == 0) {
          const bool wb = g.mask2 != nullptr;
          uint32_t b[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) b[i] = epi16(R[i], bias_s + TS_HID + col0 + 16 * i, P[i], wb);
          if (wb && row_ok) {
            g.mask2[static_cast<long long>(col0 >> 5) * g.ldmask + row] = b[0] | (b[1] << 16);
            g.mask2[static_cast<long long>((col0 + 32) >> 5) * g.ldmask + row] = b[2] | (b[3] << 16);
          }
        } else {
          epi16m(R[0], mw2[2 * qq] & 0xFFFFu, P[0]); epi16m(R[1], mw2[2 * qq] >> 16, P[1]);
          epi16m(R[2], mw2[2 * qq + 1] & 0xFFFFu, P[2]); epi16m(R[3], mw2[2 * qq + 1] >> 16, P[3]);
        }
        to_panel(P);
        if constexpr (MODE == 1) {
          float s0 = 0.f, s1 = 0.f;
          panel_colsum(s0, s1);
          cs2[qq][0] += s0; cs2[qq][1] += s1;
        }
        if (lane == 0) {
          if (row0 < g.M) tma_store_2d(panel, &tmH2, col0, row0);
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
        ++nuse;
      }
      tile_ph ^= 1;
    }
    if constexpr (MODE == 1) {   // one atomic per column, accumulator quarter and CTA
      const int cpair = (lane >> 2) * 8 + (lane & 3) * 2;
#pragma unroll
      for (int qq = 0; qq < 2; ++qq) {
        const int c = (2 * qq + ws) * 128 + hf * 64 + cpair;
        if (g.colsum1) { atomicAdd(g.colsum1 + c, cs1[qq][0]); atomicAdd(g.colsum1 + c + 1, cs1[qq][1]); }
        if (g.colsum2) { atomicAdd(g.colsum2 + c, cs2[qq][0]); atomicAdd(g.colsum2 + c + 1, cs2[qq][1]); }
      }
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  }
  tc_fence_before();
  cluster_sync_all();
  if (warp == 1) tmem_dealloc_pair(tmem_base, 512);
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(TS_THREADS, 1)
cnet_fwd_ts_kernel(const __grid_constant__ CUtensorMap tmCol, const __grid_constant__ CUtensorMap tmB1,
                   const __grid_constant__ CUtensorMap tmB2, const __grid_constant__ CUtensorMap tmH1,
                   const __grid_constant__ CUtensorMap tmH2, const TsArgs g) {
  cnet_ts_body<0>(tmCol, tmB1, tmB2, tmH1, tmH2, g);
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(TS_THREADS, 1)
cnet_bwd_ts_kernel(const __grid_constant__ CUtensorMap tmCol, const __grid_constant__ CUtensorMap tmB1,
                   const __grid_constant__ CUtensorMap tmB2, const __grid_constant__ CUtensorMap tmH1,
                   const __grid_constant__ CUtensorMap tmH2, const TsArgs g) {
  cnet_ts_body<1>(tmCol, tmB1, tmB2, tmH1, tmH2, g);
}

// Shared-memory plan for a GEMM-1 A tile of kb1 k-blocks: the weight ring takes what the A tile, the store staging, the
// barriers and the biases leave of the 227 KB, up to TS_MAX_SLOTS slots. Returns the bytes; *nslots = the ring's slots.
static int ts_smem_plan(int kb1, int* nslots) {
  const int fixed = kb1 * TS_COLBLK + TS_STAGE_BYTES + TS_BAR_BYTES + TS_BIAS_BYTES;
  int n = (227 * 1024 - fixed) / TS_SLOT;
  if (n > TS_MAX_SLOTS) n = TS_MAX_SLOTS;
  *nslots = n;
  return fixed + n * TS_SLOT;
}

// Shared launcher: GEMM 1 = A [M, Ka] x W1 [512, Ka]^T, GEMM 2 = (epilogue of GEMM 1) x W2 [512, 512]^T; out1 (optional
// in MODE 0) / out2 are the bf16 [M, 512] epilogue outputs of the two GEMMs. The shape has passed
// nfk_cnet_fused_supported.
template <int MODE>
static int ts_launch(const void* A, int Ka, const void* W1, const void* W2, void* out1, void* out2, TsArgs g,
                     cudaStream_t stream) {
  int nslots = 0;
  const int smem_bytes = ts_smem_plan(Ka / 64, &nslots);
  g.nslots = nslots;
  CUtensorMap tmA, tmW1, tmW2, tmO1, tmO2;
  int rc;
  if ((rc = make_tmap_2d(&tmA, A, Ka, g.M, Ka, 128))) return rc;
  if ((rc = make_tmap_2d(&tmW1, W1, Ka, TS_HID, Ka, 64))) return rc;
  if ((rc = make_tmap_2d(&tmW2, W2, TS_HID, TS_HID, TS_HID, 64))) return rc;
  if ((rc = make_tmap_2d(&tmO2, out2, TS_HID, g.M, TS_HID, 32))) return rc;
  if (out1) { if ((rc = make_tmap_2d(&tmO1, out1, TS_HID, g.M, TS_HID, 32))) return rc; }
  else tmO1 = tmO2;
  auto kernel = MODE == 0 ? cnet_fwd_ts_kernel : cnet_bwd_ts_kernel;
  if ((rc = ensure_dyn_smem(reinterpret_cast<const void*>(kernel), smem_bytes))) return rc;
  const int sms = num_sms();
  const int tiles = (g.M + 255) / 256;
  const int pairs = tiles < sms / 2 ? tiles : sms / 2;
  const cudaError_t le = launch_pdl(kernel, dim3(2 * pairs), dim3(TS_THREADS), smem_bytes, stream, tmA, tmW1, tmW2,
                                    tmO1, tmO2, g);
  return (le == cudaSuccess && cudaGetLastError() == cudaSuccess) ? NFK_OK : NFK_ERR_LAUNCH;
}

}  // namespace nfk

using namespace nfk;

extern "C" int nfk_cnet_fused_supported(int hid, int K) {
  // (the k-block bound only keeps the plan's byte counts in range: 14 k-blocks alone fill the 227 KB)
  if (hid != TS_HID || K < 64 || K % 64 || K / 64 > 227 * 1024 / TS_COLBLK) return 0;
  int nslots = 0;
  ts_smem_plan(K / 64, &nslots);
  return nslots >= 2;     // K <= 448: at K = 512 the A tile leaves room for one weight slot
}

static long long* g_cnet_prof = nullptr;
extern "C" int nfk_cnet_set_prof(void* buf) {
  g_cnet_prof = static_cast<long long*>(buf);
  return NFK_OK;
}

extern "C" int nfk_cnet_fwd_fused(const void* col, int K1p, const void* B1, const void* B2, const float* bias1,
                                  const float* bias2, void* h1, void* h2, void* mask1, void* mask2,
                                  long long ldmask, int M, int hid, void* stream) {
  return nfk_cnet_fwd_fused_ranged(col, K1p, B1, B2, bias1, bias2, h1, h2, mask1, mask2, ldmask, M, hid, 8, stream);
}

extern "C" int nfk_cnet_fwd_fused_ranged(const void* col, int K1p, const void* B1, const void* B2, const float* bias1,
                                         const float* bias2, void* h1, void* h2, void* mask1, void* mask2,
                                         long long ldmask, int M, int hid, int kb2_end_half0, void* stream) {
  if (M <= 0 || !nfk_cnet_fused_supported(hid, K1p)) return NFK_ERR_SHAPE;
  if (kb2_end_half0 < 1 || kb2_end_half0 > 8) return NFK_ERR_ARG;
  if (!col || !B1 || !B2 || !bias1 || !bias2 || !h2) return NFK_ERR_ARG;
  if ((mask1 || mask2) && ldmask < M) return NFK_ERR_ARG;
  TsArgs g{M, K1p / 64, 0, bias1, bias2, static_cast<uint32_t*>(mask1), static_cast<uint32_t*>(mask2), ldmask,
           h1 ? 1 : 0, g_cnet_prof, {kb2_end_half0, 8}, nullptr, nullptr};
  return ts_launch<0>(col, K1p, B1, B2, h1, h2, g, static_cast<cudaStream_t>(stream));
}

extern "C" int nfk_cnet_bwd_fused(const void* dhcol, int K3p, const void* B3T, const void* B2T, const void* mask_h2,
                                  const void* mask_h1, long long ldmask, void* dpre2, void* dpre1, float* dbias2,
                                  float* dbias1, int M, int hid, void* stream) {
  if (M <= 0 || !nfk_cnet_fused_supported(hid, K3p)) return NFK_ERR_SHAPE;
  if (!dhcol || !B3T || !B2T || !mask_h2 || !mask_h1 || !dpre2 || !dpre1) return NFK_ERR_ARG;
  if (ldmask < M) return NFK_ERR_ARG;
  TsArgs g{M, K3p / 64, 0, nullptr, nullptr, static_cast<uint32_t*>(const_cast<void*>(mask_h2)),
           static_cast<uint32_t*>(const_cast<void*>(mask_h1)), ldmask, 1, nullptr, {8, 8}, dbias2, dbias1};
  return ts_launch<1>(dhcol, K3p, B3T, B2T, dpre2, dpre1, g, static_cast<cudaStream_t>(stream));
}
