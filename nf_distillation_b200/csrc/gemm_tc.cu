// tcgen05 / TMEM / TMA GEMM tiles for the coupling network (reference: models/flows.py:25-34 get_block_2d,
// models/layers.py:190-260 Conv2d / Conv2dZeros). Activations are pixel-major ("NHWC") bf16 matrices
// [pixels, channels]; every convolution of the coupling net (and its dgrad / wgrad) is one of two GEMM forms:
//
//   NT:  out[M, N]   = A[M, K] * B[N, K]^T          (forward convs, dgrads; both operands K-major)
//   TN:  out[Mo, No] += sum_k A[k, Mo] * B[k, No]   (wgrads; both operands MN-major, split-K over pixels)
//
// One CTA = one 128 x BN accumulator tile living in TMEM. Warp 0 streams 128-byte-swizzled operand tiles with
// TMA into a multi-stage smem ring, one thread of warp 1 issues tcgen05.mma, warps 2-5 drain TMEM through the
// fused epilogue (bias+ReLU->bf16, ReLU-mask->bf16 + column sums, fp32 store, or split-K red.add).
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdlib>

#include "../../include/nfk.h"
#include "launch_util.h"
#include "ptx.cuh"

namespace nfk {

constexpr int BM = 128;           // accumulator rows per CTA (= TMEM lanes)
constexpr int BK = 64;            // bf16 elements per 128-byte swizzle row
constexpr int UMMA_K = 16;        // K per tcgen05.mma for 16-bit operands
constexpr int GEMM_THREADS = 320; // warp0 TMA, warp1 MMA(+TMEM alloc), warps 2-9 epilogue (2 per TMEM lane quadrant)
constexpr int TN_THREADS = 192;   // TN kernel: warps 2-5 epilogue

struct GemmArgs {
  int M, N, K;         // NT: out[M,N]; TN: out[M=Mo, N=No], K = pixels
  int BN;              // accumulator tile width (multiple of 16, <= 256)
  int stages;          // smem ring depth
  int n_tiles;         // tiles along N
  int kb_per_split;    // TN: k-blocks per split
  void* out;
  long long ldo;
  const float* bias;   // EPI_BIAS_RELU_BF16 / EPI_F32 (optional)
  uint32_t* mask_out;        // EPI_BIAS_RELU_BF16 (optional): 1 bit per output, (value > 0), word-major
  const uint32_t* mask_in;   // EPI_MASK_BF16: that mask, read back by the dgrad of the same layer
  long long ldmask;          // [N/32][ldmask >= M] words: word (col/32, row) holds columns col..col+31 of that row
  float* colsum;       // EPI_MASK_BF16: per-column sum of the masked gradient (bias gradient)
  int slab_bytes;      // per-epilogue-warp staging slab for the TMA store (0 = direct global stores)
  long long* prof;     // optional [grid][8] cycle counters (diagnostics: where each role waits)
  // MADE masked linears: k-blocks [kb_begin, kb_end) that are not structurally zero for each n-tile (kb_end 0 = all)
  short kb_begin[16];
  short kb_end[16];
};

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}

__device__ __forceinline__ uint32_t tmem_cols_pow2(int n) {
  uint32_t c = 32;
  while (c < static_cast<uint32_t>(n)) c <<= 1;
  return c;
}

// ------------------------------------------------------------------------------------------------ NT kernel
// Persistent: every CTA (or CTA pair) walks tiles t = id, id + stride, ... (n-tile fastest, so CTAs running side by
// side share the A row block through L2). Two TMEM accumulator stages let the epilogue of tile i overlap the MMAs of
// tile i+1. PAIR = cta_group::2: two SMs share one 256 x BN tile, each stages its own 128 rows of A and HALF of the B
// tile; the leader issues the M=256 MMAs, both CTAs run TMA producers and epilogues on their own 128 TMEM lanes.
//
// Epilogue data path: TMEM -> registers (tcgen05.ld) -> fused math -> 128B-swizzled smem slab (one per warp) -> TMA
// store. A thread owns one output ROW, so direct global stores would touch 32 different 128-byte lines per warp
// instruction; staging through smem makes every HBM write a full-line bulk store and frees the LSU.
template <int EPI>
__device__ __forceinline__ void nt_epilogue_16(const GemmArgs& g, const uint32_t (&r)[16], long long row, bool row_ok,
                                               int col, int cl, int sc, const float* bias_s, int lane,
                                               uint32_t bits16, uint8_t* slab, bool want_bits, uint32_t& relu_bits) {
  // cl: column inside the tile (bias index), sc: column inside this warp's staging slab
  const uint32_t sw = static_cast<uint32_t>(lane & 7);
  if constexpr (EPI == NFK_EPI_F32) {
    float4 v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      v[j].x = __uint_as_float(r[4 * j + 0]); v[j].y = __uint_as_float(r[4 * j + 1]);
      v[j].z = __uint_as_float(r[4 * j + 2]); v[j].w = __uint_as_float(r[4 * j + 3]);
      if (g.bias) {
        const float4 b = *reinterpret_cast<const float4*>(bias_s + cl + 4 * j);
        v[j].x += b.x; v[j].y += b.y; v[j].z += b.z; v[j].w += b.w;
      }
    }
    if (slab) {
      uint8_t* base = slab + lane * 128;
      const uint32_t cc = static_cast<uint32_t>(sc & 31) >> 2;
#pragma unroll
      for (int j = 0; j < 4; ++j) *reinterpret_cast<float4*>(base + (((cc + j) ^ sw) << 4)) = v[j];
    } else if (row_ok) {
      float* o = static_cast<float*>(g.out) + row * g.ldo + col;
#pragma unroll
      for (int j = 0; j < 4; ++j) *reinterpret_cast<float4*>(o + 4 * j) = v[j];
    }
  } else {
    float v[16];
    if constexpr (EPI == NFK_EPI_BIAS_RELU_BF16) {
#pragma unroll
      for (int j = 0; j < 16; j += 4) {
        const float4 b = *reinterpret_cast<const float4*>(bias_s + cl + j);
        v[j] = fmaxf(__uint_as_float(r[j]) + b.x, 0.f);
        v[j + 1] = fmaxf(__uint_as_float(r[j + 1]) + b.y, 0.f);
        v[j + 2] = fmaxf(__uint_as_float(r[j + 2]) + b.z, 0.f);
        v[j + 3] = fmaxf(__uint_as_float(r[j + 3]) + b.w, 0.f);
      }
      if (want_bits) {
        uint32_t bits = 0;
#pragma unroll
        for (int j = 0; j < 16; ++j) bits |= (v[j] > 0.f ? 1u : 0u) << j;
        relu_bits |= bits << (cl & 16);
      }
    } else {  // NFK_EPI_MASK_BF16: ReLU backward through the 1-bit activation mask of the forward pass
#pragma unroll
      for (int j = 0; j < 16; ++j) v[j] = (row_ok && ((bits16 >> j) & 1u)) ? __uint_as_float(r[j]) : 0.f;
    }
    const uint4 p0 = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]),
                                pack_bf16x2(v[6], v[7]));
    const uint4 p1 = make_uint4(pack_bf16x2(v[8], v[9]), pack_bf16x2(v[10], v[11]), pack_bf16x2(v[12], v[13]),
                                pack_bf16x2(v[14], v[15]));
    if (slab) {
      uint8_t* base = slab + lane * 128;
      const uint32_t cc = static_cast<uint32_t>(sc & 63) >> 3;
      *reinterpret_cast<uint4*>(base + ((cc ^ sw) << 4)) = p0;
      *reinterpret_cast<uint4*>(base + (((cc + 1) ^ sw) << 4)) = p1;
    } else if (row_ok) {
      uint4* o = reinterpret_cast<uint4*>(static_cast<__nv_bfloat16*>(g.out) + row * g.ldo + col);
      o[0] = p0;
      o[1] = p1;
    }
    if constexpr (EPI == NFK_EPI_MASK_BF16) {
      if (g.colsum && !slab) {
        // direct-store fallback: 32 lanes x 16 columns -> lane j (< 16) ends with the sum of column j
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] += __shfl_xor_sync(0xffffffffu, v[j], 16);
#pragma unroll
        for (int off = 8; off >= 1; off >>= 1) {
          const bool up = (lane & off) != 0;
#pragma unroll
          for (int j = 0; j < off; ++j) {
            const float send = up ? v[j] : v[j + off];
            const float keep = up ? v[j + off] : v[j];
            v[j] = keep + __shfl_xor_sync(0xffffffffu, send, off);
          }
        }
        if (lane < 16) atomicAdd(g.colsum + col + lane, v[0]);
      }
    }
  }
}

template <int EPI, bool PAIR>
__device__ __forceinline__ void gemm_nt_body(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmC,
                                             const GemmArgs& g) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  pdl_launch_dependents();
  uint8_t* smem = smem_raw;   // 1024-byte aligned (no static shared memory in this kernel): SWIZZLE_128B requirement
  if (smem_u32(smem) & 1023u) __trap();
  const int warp = static_cast<int>(uniform_u32(threadIdx.x >> 5)), lane = threadIdx.x & 31;
  const int a_bytes = BM * 128;
  const int b_bytes = (PAIR ? g.BN / 2 : g.BN) * 128;
  const int stage_bytes = a_bytes + b_bytes;
  uint8_t* cstage = smem + g.stages * stage_bytes;                 // 8 warp slabs (1024-byte aligned)
  uint64_t* full = reinterpret_cast<uint64_t*>(cstage + 8 * g.slab_bytes);
  uint64_t* empty = full + g.stages;
  uint64_t* tmem_full = empty + g.stages;   // [2]
  uint64_t* tmem_empty = tmem_full + 2;     // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);
  float* bias_s = reinterpret_cast<float*>(tmem_slot + 4);  // [2][256] (one per accumulator stage)

  const uint32_t rank = PAIR ? (blockIdx.x & 1u) : 0u;   // == %cluster_ctarank ((2,1,1) clusters along x), provably uniform
  const int worker = PAIR ? (blockIdx.x >> 1) : blockIdx.x;
  const int num_workers = PAIR ? (gridDim.x >> 1) : gridDim.x;
  constexpr int TM = PAIR ? 2 * BM : BM;    // tile rows
  const int num_kb = g.K / BK;
  const int m_tiles = (g.M + TM - 1) / TM;
  const int num_tiles = m_tiles * g.n_tiles;
  const uint32_t ncols = tmem_cols_pow2(2 * g.BN);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    if (g.slab_bytes) tma_prefetch_desc(&tmC);
    for (int s = 0; s < g.stages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tmem_full[a], 1);
      mbar_init(&tmem_empty[a], PAIR ? 16 : 8);  // one arrival per epilogue warp (of both CTAs; leader's copy is used)
    }
    fence_mbar_init();
  }
  if (warp == 1) {
    if constexpr (PAIR) { tmem_alloc_pair(tmem_slot, ncols); tmem_relinquish_pair(); }
    else { tmem_alloc(tmem_slot, ncols); tmem_relinquish(); }
  }
  tc_fence_before();
  if constexpr (PAIR) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = uniform_u32(*tmem_slot);
  pdl_wait();      // prologue overlapped the previous kernel's tail; global memory only from here on

  if (warp == 0) {
    {   // whole warp, uniform control flow: single-thread instructions are elected inside the asm (ptx.cuh)
      int s = 0;
      uint32_t ph = 0;
      for (int t = worker; t < num_tiles; t += num_workers) {
        const int n_tile = t % g.n_tiles, m_tile = t / g.n_tiles;
        const int kb0 = g.kb_begin[n_tile & 15], kb1 = g.kb_end[n_tile & 15] ? g.kb_end[n_tile & 15] : num_kb;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait_warp(&empty[s], ph ^ 1);
          uint8_t* sa = smem + s * stage_bytes;
          if constexpr (PAIR) {
            if (rank == 0) mbar_expect_tx_elect(&full[s], 2 * stage_bytes);  // both CTAs' bytes land on the leader's barrier
            tma_load_2d_pair_elect(sa, &tmA, &full[s], kb * BK, m_tile * TM + static_cast<int>(rank) * BM);
            tma_load_2d_pair_elect(sa + a_bytes, &tmB, &full[s], kb * BK,
                             n_tile * g.BN + static_cast<int>(rank) * (g.BN / 2));
          } else {
            mbar_expect_tx_elect(&full[s], stage_bytes);
            tma_load_2d_elect(sa, &tmA, &full[s], kb * BK, m_tile * BM);
            tma_load_2d_elect(sa + a_bytes, &tmB, &full[s], kb * BK, n_tile * g.BN);
          }
          if (++s == g.stages) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (rank == 0) {   // whole warp, uniform control flow (ptx.cuh: *_elect)
      const uint32_t idesc = umma_idesc_bf16(TM, g.BN, false, false);
      int s = 0;
      uint32_t ph = 0;
      int it = 0;
      long long pw_tmem = 0, pw_full = 0;
      const long long pt0 = g.prof ? clock64() : 0;
      for (int t = worker; t < num_tiles; t += num_workers, ++it) {
        const int acc = it & 1;
        const uint32_t acc_ph = (it >> 1) & 1;
        long long t0 = g.prof ? clock64() : 0;
        mbar_wait_warp(&tmem_empty[acc], acc_ph ^ 1);  // epilogue has drained this accumulator stage
        if (g.prof) { pw_tmem += clock64() - t0; }
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + acc * g.BN;
        const int n_tile = t % g.n_tiles;
        const int kb0 = g.kb_begin[n_tile & 15], kb1 = g.kb_end[n_tile & 15] ? g.kb_end[n_tile & 15] : num_kb;
        for (int kb = kb0; kb < kb1; ++kb) {
          t0 = g.prof ? clock64() : 0;
          mbar_wait_warp(&full[s], ph);
          if (g.prof) { pw_full += clock64() - t0; }
          tc_fence_after();
          const uint32_t a_addr = smem_u32(smem + s * stage_bytes);
          const uint32_t b_addr = a_addr + a_bytes;
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k) {
            const uint64_t ad = umma_desc_sw128(a_addr + k * (UMMA_K * 2), 16, 1024);
            const uint64_t bd = umma_desc_sw128(b_addr + k * (UMMA_K * 2), 16, 1024);
            if constexpr (PAIR) umma_f16_pair_elect(tmem_d, ad, bd, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
            else umma_f16_elect(tmem_d, ad, bd, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
          }
          // free the smem stage (in both CTAs of a pair) when these MMAs retire
          if constexpr (PAIR) umma_commit_pair_elect(&empty[s], 3); else umma_commit_elect(&empty[s]);
          if (++s == g.stages) { s = 0; ph ^= 1; }
        }
        if constexpr (PAIR) umma_commit_pair_elect(&tmem_full[acc], 3); else umma_commit_elect(&tmem_full[acc]);
      }
      if (g.prof && lane == 0) {
        g.prof[blockIdx.x * 8 + 0] = clock64() - pt0;
        g.prof[blockIdx.x * 8 + 1] = pw_tmem;
        g.prof[blockIdx.x * 8 + 2] = pw_full;
        g.prof[blockIdx.x * 8 + 3] = it;
      }
    }
  } else {
    // 8 epilogue warps: warp w reads TMEM lanes (w % 4) * 32.., and of the tile's BN columns the half (w - 2) / 4
    const int q = warp & 3;
    const int half = (warp - 2) >> 2;
    const int et = threadIdx.x - 64;  // 0..255
    constexpr int panel_w = (EPI == NFK_EPI_F32) ? 32 : 64;   // columns per 128-byte staging panel
    const bool split = (g.BN % (2 * panel_w)) == 0;            // both halves get whole panels (and whole mask words)
    const int c_begin = split ? half * (g.BN / 2) : 0;
    const int c_end = split ? c_begin + g.BN / 2 : (half == 0 ? g.BN : 0);
    uint8_t* slab = g.slab_bytes ? cstage + (warp - 2) * g.slab_bytes : nullptr;   // ONE panel: 32 rows x 128 B
    const bool want_bits = g.mask_out != nullptr;
    // bias-gradient column sums (EPI_MASK): lane owns the column pair (lane>>2)*8 + (lane&3)*2 of each 64-col panel;
    // accumulated over this CTA's tiles while they share one n-tile, flushed with one atomic per column at the end
    float cs[4][2] = {};
    int cs_ntile = -1;
    auto flush_colsum = [&]() {
      if (cs_ntile < 0) return;
#pragma unroll
      for (int p = 0; p < 4; ++p) {
        const int col = cs_ntile * g.BN + c_begin + p * 64 + (lane >> 2) * 8 + (lane & 3) * 2;
        if (c_begin + p * 64 < c_end && col < g.N) {
          atomicAdd(g.colsum + col, cs[p][0]);
          atomicAdd(g.colsum + col + 1, cs[p][1]);
        }
        cs[p][0] = cs[p][1] = 0.f;
      }
    };
    // 1-bit ReLU mask words of a tile (EPI_MASK), fetched one tile ahead so their HBM latency is never exposed
    auto load_mask = [&](int t, uint32_t (&mb)[8]) {
      const int n_tile = t % g.n_tiles, m_tile = t / g.n_tiles;
      const long long row = static_cast<long long>(m_tile) * TM + rank * BM + q * 32 + lane;
#pragma unroll
      for (int j = 0; j < 8; ++j) {   // up to 8 words: a warp that is not sharing its tile owns all BN <= 256 columns
        const int c = c_begin + 32 * j;
        const int col = n_tile * g.BN + c;
        mb[j] = (t < num_tiles && row < g.M && c < c_end && col < g.N)
                    ? __ldg(g.mask_in + static_cast<long long>(col >> 5) * g.ldmask + row) : 0u;
      }
    };
    uint32_t mbits[8] = {}, mnext[8] = {};
    if constexpr (EPI == NFK_EPI_MASK_BF16) load_mask(worker, mnext);
    int it = 0;
    long long ew_full = 0, ew_work = 0;
    for (int t = worker; t < num_tiles; t += num_workers, ++it) {
      const int n_tile = t % g.n_tiles, m_tile = t / g.n_tiles;
      const int acc = it & 1;
      const uint32_t acc_ph = (it >> 1) & 1;
      float* bs = bias_s + acc * 256;
      if (EPI != NFK_EPI_MASK_BF16 && g.bias) {
        // stage this tile's bias slice; the named barrier also orders it against the previous use of this stage
        for (int c = et; c < g.BN; c += 256) {
          const int col = n_tile * g.BN + c;
          bs[c] = col < g.N ? __ldg(g.bias + col) : 0.f;
        }
        asm volatile("bar.sync 1, 256;" ::: "memory");
      }
      const long long row0 = static_cast<long long>(m_tile) * TM + rank * BM + q * 32;
      const long long row = row0 + lane;
      const bool row_ok = row < g.M;
      if constexpr (EPI == NFK_EPI_MASK_BF16) {
#pragma unroll
        for (int j = 0; j < 8; ++j) mbits[j] = mnext[j];
        load_mask(t + num_workers, mnext);
        if (g.colsum && slab && cs_ntile != n_tile) { flush_colsum(); cs_ntile = n_tile; }
      }
      long long e0 = g.prof ? clock64() : 0;
      mbar_wait(&tmem_full[acc], acc_ph);
      if (g.prof) { ew_full += clock64() - e0; e0 = clock64(); }
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * g.BN;
      // one staging panel per pass: drain -> (column sums) -> fence -> TMA store; the slab is reused by the next pass
      // once the previous bulk store has finished reading it
      const int pass_w = slab ? panel_w : (c_end - c_begin);
#pragma unroll 1
      for (int pc = c_begin; pc < c_end; pc += pass_w) {
        if (slab) {
          if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
          __syncwarp();
        }
        const int pe = min(pc + pass_w, c_end);
#pragma unroll 1
        for (int c = pc; c < pe; c += 32) {
          uint32_t r0[16], r1[16];
          const bool two = c + 16 < pe;
          tmem_ld16(taddr + c, r0);
          if (two) tmem_ld16(taddr + c + 16, r1);
          tmem_ld_wait();
          const int col = n_tile * g.BN + c;
          uint32_t bits = 0, relu_bits = 0;
          if constexpr (EPI == NFK_EPI_MASK_BF16) {   // consume word 0, rotate (no dynamic register indexing)
            bits = mbits[0];
#pragma unroll
            for (int j = 0; j < 7; ++j) mbits[j] = mbits[j + 1];
          }
          if (col < g.N)
            nt_epilogue_16<EPI>(g, r0, row, row_ok, col, c, c - pc, bs, lane, bits & 0xFFFFu, slab, want_bits,
                                relu_bits);
          if (two && col + 16 < g.N)
            nt_epilogue_16<EPI>(g, r1, row, row_ok, col + 16, c + 16, c + 16 - pc, bs, lane, bits >> 16, slab,
                                want_bits, relu_bits);
          if constexpr (EPI == NFK_EPI_BIAS_RELU_BF16) {
            if (want_bits && row_ok && col < g.N)
              g.mask_out[static_cast<long long>(col >> 5) * g.ldmask + row] = relu_bits;   // word-major: coalesced
          }
        }
        if (pe == c_end) {   // last TMEM read of this tile is done: hand the accumulator stage back to the MMA warp
          tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            if constexpr (PAIR) mbar_arrive_cluster(&tmem_empty[acc], 0); else mbar_arrive(&tmem_empty[acc]);
          }
        }
        if (slab) {
          __syncwarp();
          if constexpr (EPI == NFK_EPI_MASK_BF16) {
            if (g.colsum) {
              // column sums straight from the staged bf16 panel: at row r the 32 lanes read the whole 128-byte row
              // (conflict-free); rows outside the matrix were staged as zeros
              const uint8_t* pb = slab + (lane & 3) * 4;
              const uint32_t chunk = static_cast<uint32_t>(lane >> 2);
              float a0 = 0.f, a1 = 0.f, b0 = 0.f, b1 = 0.f;
#pragma unroll 8
              for (int r = 0; r < 32; r += 2) {
                const uint32_t w0 = *reinterpret_cast<const uint32_t*>(pb + r * 128 + ((chunk ^ (r & 7)) << 4));
                const uint32_t w1 =
                    *reinterpret_cast<const uint32_t*>(pb + (r + 1) * 128 + ((chunk ^ ((r + 1) & 7)) << 4));
                a0 += __uint_as_float(w0 << 16);
                a1 += __uint_as_float(w0 & 0xFFFF0000u);
                b0 += __uint_as_float(w1 << 16);
                b1 += __uint_as_float(w1 & 0xFFFF0000u);
              }
              const int p = (pc - c_begin) / 64;
#pragma unroll
              for (int k = 0; k < 4; ++k)
                if (k == p) { cs[k][0] += a0 + b0; cs[k][1] += a1 + b1; }
            }
          }
          fence_proxy_async();   // generic-proxy smem writes -> visible to the TMA (async proxy)
          __syncwarp();
          const int col = n_tile * g.BN + pc;
          if (lane == 0 && row0 < g.M && col < g.N) {
            tma_store_2d(slab, &tmC, col, static_cast<int>(row0));
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          }
        }
      }
      if (c_begin >= c_end) {   // idle half (tile too narrow to split): still part of the accumulator hand-back
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if constexpr (PAIR) mbar_arrive_cluster(&tmem_empty[acc], 0); else mbar_arrive(&tmem_empty[acc]);
        }
      }
      if (g.prof) ew_work += clock64() - e0;
    }
    if constexpr (EPI == NFK_EPI_MASK_BF16) {
      if (g.colsum && slab) flush_colsum();
    }
    if (slab && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    if (g.prof && warp == 2 && lane == 0) {
      g.prof[blockIdx.x * 8 + 4] = ew_full;
      g.prof[blockIdx.x * 8 + 5] = ew_work;
    }
  }
  tc_fence_before();
  if constexpr (PAIR) cluster_sync_all(); else __syncthreads();
  if (warp == 1) {
    if constexpr (PAIR) tmem_dealloc_pair(tmem_base, ncols); else tmem_dealloc(tmem_base, ncols);
  }
}

template <int EPI>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_nt_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmC, const GemmArgs g) {
  gemm_nt_body<EPI, false>(tmA, tmB, tmC, g);
}

template <int EPI>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(GEMM_THREADS, 1)
gemm_nt_pair_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                    const __grid_constant__ CUtensorMap tmC, const GemmArgs g) {
  gemm_nt_body<EPI, true>(tmA, tmB, tmC, g);
}

// ------------------------------------------------------------------------------------------------ TN kernel
// out[Mo, No] (fp32, pre-zeroed) += sum over this CTA's pixel range of A[k, m] * B[k, n].
__global__ void __launch_bounds__(TN_THREADS, 1)
gemm_tn_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const GemmArgs g) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  pdl_launch_dependents();
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int warp = static_cast<int>(uniform_u32(threadIdx.x >> 5)), lane = threadIdx.x & 31;
  constexpr int BOX = 64 * 128;  // one TMA box: 64 pixel rows x 64 channels (128 B)
  const int a_bytes = 2 * BOX;
  const int nb_boxes = g.BN / 64;
  const int stage_bytes = a_bytes + nb_boxes * BOX;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + g.stages * stage_bytes);
  uint64_t* empty = full + g.stages;
  uint64_t* tmem_full = empty + g.stages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full + 1);

  const int n_tile = blockIdx.x % g.n_tiles;
  const int m_tile = blockIdx.x / g.n_tiles;
  const int total_kb = (g.K + BK - 1) / BK;
  const int kb0 = blockIdx.y * g.kb_per_split;
  const int kb1 = min(kb0 + g.kb_per_split, total_kb);
  const int num_kb = kb1 - kb0;
  if (num_kb <= 0) return;
  const uint32_t ncols = tmem_cols_pow2(g.BN);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int s = 0; s < g.stages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    mbar_init(tmem_full, 1);
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, ncols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = uniform_u32(*tmem_slot);
  pdl_wait();

  if (warp == 0) {
    {   // whole warp, uniform control flow: single-thread instructions are elected inside the asm (ptx.cuh)
      int s = 0;
      uint32_t ph = 0;
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait_warp(&empty[s], ph ^ 1);
        uint8_t* sa = smem + s * stage_bytes;
        mbar_expect_tx_elect(&full[s], stage_bytes);
        tma_load_2d_elect(sa, &tmA, &full[s], m_tile * BM, kb * BK);
        tma_load_2d_elect(sa + BOX, &tmA, &full[s], m_tile * BM + 64, kb * BK);
        for (int j = 0; j < nb_boxes; ++j)
          tma_load_2d_elect(sa + a_bytes + j * BOX, &tmB, &full[s], n_tile * g.BN + j * 64, kb * BK);
        if (++s == g.stages) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp == 1) {
    {   // whole warp, uniform control flow: single-thread instructions are elected inside the asm (ptx.cuh)
      const uint32_t idesc = umma_idesc_bf16(BM, g.BN, true, true);
      int s = 0;
      uint32_t ph = 0;
      for (int i = 0; i < num_kb; ++i) {
        mbar_wait_warp(&full[s], ph);
        tc_fence_after();
        const uint32_t a_addr = smem_u32(smem + s * stage_bytes);
        const uint32_t b_addr = a_addr + a_bytes;
#pragma unroll
        for (int k = 0; k < BK / UMMA_K; ++k) {
          // 16 pixel rows per MMA = two 8-row swizzle groups (SBO = 1024 B); 64-channel blocks are BOX apart (LBO).
          const uint64_t ad = umma_desc_sw128(a_addr + k * (UMMA_K * 128), BOX, 1024);
          const uint64_t bd = umma_desc_sw128(b_addr + k * (UMMA_K * 128), BOX, 1024);
          umma_f16_elect(tmem_base, ad, bd, idesc, (i | k) != 0 ? 1u : 0u);
        }
        umma_commit_elect(&empty[s]);
        if (++s == g.stages) { s = 0; ph ^= 1; }
      }
      umma_commit_elect(tmem_full);
    }
  } else {
    mbar_wait(tmem_full, 0);
    tc_fence_after();
    const int q = warp & 3;
    const long long row = static_cast<long long>(m_tile) * BM + q * 32 + lane;
    const bool row_ok = row < g.M;
    for (int c = 0; c < g.BN; c += 16) {
      uint32_t r[16];
      tmem_ld16(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + c, r);
      tmem_ld_wait();
      const int col = n_tile * g.BN + c;
      if (col >= g.N) break;
      if (row_ok) {
        float* o = static_cast<float*>(g.out) + row * g.ldo + col;
#pragma unroll
        for (int j = 0; j < 16; j += 4) {
          asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(o + j), "f"(__uint_as_float(r[j])),
                       "f"(__uint_as_float(r[j + 1])), "f"(__uint_as_float(r[j + 2])), "f"(__uint_as_float(r[j + 3]))
                       : "memory");
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, ncols);
}

// ------------------------------------------------------------------------------------------------ TN kernel, CTA pairs
// Same contraction on cta_group::2: one 256 x BN output tile per PAIR of SMs (M = 256 rows = channels of A, 128 per
// CTA; the BN columns of B are split, BN/2 per CTA). Per k-block of 64 pixels a CTA now stages 16 KB of A and
// BN/2 * 128 B of B for a 128 x BN x 64 share of the MMAs: half the shared-memory fill and half the B-operand reads per
// FLOP of the single-CTA 128 x BN tile, which is shared-memory-bandwidth bound (94 B/clk of fills + 94 B/clk of operand
// reads against 128 B/clk: 0.68 of the tensor peak, measured 0.64-0.68). Used when Mo % 256 == 0-ish and BN >= 128.
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(TN_THREADS, 1)
gemm_tn_pair_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                    const GemmArgs g) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  pdl_launch_dependents();
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int warp = static_cast<int>(uniform_u32(threadIdx.x >> 5)), lane = threadIdx.x & 31;
  const uint32_t rank = blockIdx.x & 1u;   // == %cluster_ctarank ((2,1,1) clusters along x), provably uniform
  constexpr int BOX = 64 * 128;          // one TMA box: 64 pixel rows x 64 channels (128 B)
  const int a_bytes = 2 * BOX;           // this CTA's 128 rows of the tile
  const int nb_boxes = g.BN / 128;       // this CTA's BN/2 columns of B, 64 per box
  const int stage_bytes = a_bytes + nb_boxes * BOX;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + g.stages * stage_bytes);   // (leader's copy collects both CTAs' bytes)
  uint64_t* empty = full + g.stages;
  uint64_t* tmem_full = empty + g.stages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full + 1);

  const int pair = blockIdx.x >> 1;
  const int n_tile = pair % g.n_tiles;
  const int m_tile = pair / g.n_tiles;
  const int total_kb = (g.K + BK - 1) / BK;
  const int kb0 = blockIdx.y * g.kb_per_split;
  const int kb1 = min(kb0 + g.kb_per_split, total_kb);
  const int num_kb = kb1 - kb0;           // (the host sizes the splits so that no pair is empty)
  const uint32_t ncols = tmem_cols_pow2(g.BN);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int s = 0; s < g.stages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(tmem_full, 1);
    fence_mbar_init();
  }
  if (warp == 1) { tmem_alloc_pair(tmem_slot, ncols); tmem_relinquish_pair(); }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = uniform_u32(*tmem_slot);
  pdl_wait();

  if (warp == 0) {
    {   // whole warp, uniform control flow: single-thread instructions are elected inside the asm (ptx.cuh)
      int s = 0;
      uint32_t ph = 0;
      const int m0 = m_tile * 2 * BM + static_cast<int>(rank) * BM;
      const int n0 = n_tile * g.BN + static_cast<int>(rank) * (g.BN / 2);
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait_warp(&empty[s], ph ^ 1);
        uint8_t* sa = smem + s * stage_bytes;
        if (rank == 0) mbar_expect_tx_elect(&full[s], 2 * stage_bytes);
        tma_load_2d_pair_elect(sa, &tmA, &full[s], m0, kb * BK);
        tma_load_2d_pair_elect(sa + BOX, &tmA, &full[s], m0 + 64, kb * BK);
        for (int j = 0; j < nb_boxes; ++j)
          tma_load_2d_pair_elect(sa + a_bytes + j * BOX, &tmB, &full[s], n0 + j * 64, kb * BK);
        if (++s == g.stages) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp == 1) {
    if (rank == 0) {   // whole warp, uniform control flow (ptx.cuh: *_elect)
      const uint32_t idesc = umma_idesc_bf16(2 * BM, g.BN, true, true);
      int s = 0;
      uint32_t ph = 0;
      for (int i = 0; i < num_kb; ++i) {
        mbar_wait_warp(&full[s], ph);
        tc_fence_after();
        const uint32_t a_addr = smem_u32(smem + s * stage_bytes);
        const uint32_t b_addr = a_addr + a_bytes;
#pragma unroll
        for (int k = 0; k < BK / UMMA_K; ++k) {
          const uint64_t ad = umma_desc_sw128(a_addr + k * (UMMA_K * 128), BOX, 1024);
          const uint64_t bd = umma_desc_sw128(b_addr + k * (UMMA_K * 128), BOX, 1024);
          umma_f16_pair_elect(tmem_base, ad, bd, idesc, (i | k) != 0 ? 1u : 0u);
        }
        umma_commit_pair_elect(&empty[s], 3);
        if (++s == g.stages) { s = 0; ph ^= 1; }
      }
      umma_commit_pair_elect(tmem_full, 3);
    }
  } else {
    mbar_wait(tmem_full, 0);
    tc_fence_after();
    const int q = warp & 3;
    const long long row = static_cast<long long>(m_tile) * 2 * BM + rank * BM + q * 32 + lane;
    const bool row_ok = row < g.M;
    for (int c = 0; c < g.BN; c += 16) {
      uint32_t r[16];
      tmem_ld16(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + c, r);
      tmem_ld_wait();
      const int col = n_tile * g.BN + c;
      if (col >= g.N) break;
      if (row_ok) {
        float* o = static_cast<float*>(g.out) + row * g.ldo + col;
#pragma unroll
        for (int j = 0; j < 16; j += 4) {
          asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(o + j), "f"(__uint_as_float(r[j])),
                       "f"(__uint_as_float(r[j + 1])), "f"(__uint_as_float(r[j + 2])), "f"(__uint_as_float(r[j + 3]))
                       : "memory");
        }
      }
    }
  }
  tc_fence_before();
  cluster_sync_all();
  if (warp == 1) tmem_dealloc_pair(tmem_base, ncols);
}

// ------------------------------------------------------------------------------------------------ host side
static long long* g_prof_buffer = nullptr;   // set by nfk_gemm_set_prof (diagnostics only)

static bool use_pairs() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("NFK_GEMM_PAIRS");
    v = (e && e[0] == '0') ? 0 : 1;
  }
  return v == 1;
}

static int pick_bn(int N, int cap) {
  // Widest tile (multiple of 16, <= cap) that wastes the fewest padded columns.
  const int n16 = (N + 15) / 16 * 16;
  if (n16 <= cap) return n16;
  int best = cap, best_waste = 1 << 30;
  for (int bn = cap; bn >= 128; bn -= 16) {
    const int tiles = (n16 + bn - 1) / bn;
    const int waste = tiles * bn - n16;
    if (waste < best_waste) { best = bn; best_waste = waste; }
  }
  return best;
}

template <typename K>
static int set_smem(K kernel, int bytes) {
  return ensure_dyn_smem(reinterpret_cast<const void*>(kernel), bytes);
}

}  // namespace nfk

using namespace nfk;

static int gemm_nt_launch(const void* A, long long lda, const void* B, long long ldb, int M, int N, int K, int epi,
                          void* out, long long ldo, const float* bias, const void* aux, long long ldaux,
                          float* colsum, int bn_force, const int* kb_begin, const int* kb_end, void* stream);

extern "C" int nfk_gemm_nt_bf16(const void* A, long long lda, const void* B, long long ldb, int M, int N, int K,
                                int epi, void* out, long long ldo, const float* bias, const void* aux,
                                long long ldaux, float* colsum, void* stream) {
  return gemm_nt_launch(A, lda, B, ldb, M, N, K, epi, out, ldo, bias, aux, ldaux, colsum, 0, nullptr, nullptr,
                        stream);
}

extern "C" int nfk_gemm_set_prof(void* buf) {
  g_prof_buffer = static_cast<long long*>(buf);
  return NFK_OK;
}

extern "C" int nfk_gemm_nt_bf16_ranged(const void* A, long long lda, const void* B, long long ldb, int M, int N,
                                       int K, int epi, void* out, long long ldo, const float* bias, const void* aux,
                                       long long ldaux, float* colsum, int bn, const int* kb_begin,
                                       const int* kb_end, void* stream) {
  if (bn <= 0 || bn % 16 || bn > 256 || (N + bn - 1) / bn > 16 || !kb_begin || !kb_end) return NFK_ERR_ARG;
  return gemm_nt_launch(A, lda, B, ldb, M, N, K, epi, out, ldo, bias, aux, ldaux, colsum, bn, kb_begin, kb_end,
                        stream);
}

static int gemm_nt_launch(const void* A, long long lda, const void* B, long long ldb, int M, int N, int K, int epi,
                          void* out, long long ldo, const float* bias, const void* aux, long long ldaux,
                          float* colsum, int bn_force, const int* kb_begin, const int* kb_end, void* stream) {
  if (M <= 0 || N <= 0 || K <= 0) return NFK_ERR_SHAPE;
  if (K % BK || N % 16 || ldo % 8) return NFK_ERR_SHAPE;
  if (epi == NFK_EPI_BIAS_RELU_BF16 && !bias) return NFK_ERR_ARG;
  if (epi == NFK_EPI_MASK_BF16 && (!aux || ldaux < M)) return NFK_ERR_ARG;
  if (epi == NFK_EPI_BIAS_RELU_BF16 && aux && ldaux < M) return NFK_ERR_ARG;
  const bool f32 = epi == NFK_EPI_F32;
  // TMA-store epilogue needs whole 128-byte panels per tile: 64 bf16 / 32 fp32 columns
  const int panel = f32 ? 32 : 64;
  const bool staged = N % panel == 0 && (!bn_force || bn_force % panel == 0);
  GemmArgs g{};
  g.M = M; g.N = N; g.K = K;
  const int cap = f32 ? 128 : 256;   // fp32 tiles are twice as wide in bytes: keep the staging slabs at <= 64 KB
  if (staged) {
    g.BN = N <= cap ? N : cap;
    if (N > cap && N % cap) {        // e.g. N = 448: 256 + 192, prefer an even split when it wastes nothing
      for (int bn = cap; bn >= 64; bn -= panel)
        if (N % bn == 0) { g.BN = bn; break; }
    }
  } else {
    g.BN = pick_bn(N, cap);
  }
  // few row tiles (small images x small batch): narrower accumulator tiles so the grid still covers the SMs
  const int m_tiles = (M + BM - 1) / BM;
  while (m_tiles * ((N + g.BN - 1) / g.BN) < 148 && g.BN >= 128 && g.BN % (2 * panel) == 0) g.BN /= 2;
  if (bn_force) g.BN = bn_force;
  g.n_tiles = (N + g.BN - 1) / g.BN;
  if (g.n_tiles > 16 && kb_begin) return NFK_ERR_ARG;
  if (kb_begin)
    for (int i = 0; i < g.n_tiles && i < 16; ++i) {
      if (kb_begin[i] < 0 || kb_end[i] > K / BK || kb_begin[i] >= kb_end[i]) return NFK_ERR_ARG;
      g.kb_begin[i] = static_cast<short>(kb_begin[i]);
      g.kb_end[i] = static_cast<short>(kb_end[i]);
    }
  const int m_tiles2 = (M + 2 * BM - 1) / (2 * BM);
  // CTA pairs once there are enough 256-row tiles to give every pair of SMs work (and B halves stay swizzle-aligned)
  const bool pair = use_pairs() && g.BN % 32 == 0 && m_tiles2 * g.n_tiles >= num_sms() / 2;
  const int stage_bytes = BM * 128 + (pair ? g.BN / 2 : g.BN) * 128;
  // 8 epilogue warps, each with ONE 32-row x 128-byte staging panel that it refills once per 128 bytes of columns
  g.slab_bytes = staged ? 4096 : 0;
  const int fixed = 8 * g.slab_bytes + 256 + 2 * 256 * 4;
  g.stages = min(8, (227 * 1024 - fixed) / stage_bytes);
  if (g.stages < 2) return NFK_ERR_SHAPE;
  g.out = out; g.ldo = ldo; g.bias = bias;
  g.mask_out = epi == NFK_EPI_BIAS_RELU_BF16 ? static_cast<uint32_t*>(const_cast<void*>(aux)) : nullptr;
  g.mask_in = epi == NFK_EPI_MASK_BF16 ? static_cast<const uint32_t*>(aux) : nullptr;
  g.ldmask = ldaux; g.colsum = colsum;
  g.prof = g_prof_buffer;
  CUtensorMap tmA, tmB, tmC;
  int rc;
  if ((rc = make_tmap_2d(&tmA, A, K, M, lda, BM)) != NFK_OK) return rc;
  if ((rc = make_tmap_2d(&tmB, B, K, N, ldb, pair ? g.BN / 2 : g.BN)) != NFK_OK) return rc;
  if (staged) {
    if ((rc = make_tmap_2d(&tmC, out, N, M, ldo, 32, f32)) != NFK_OK) return rc;
  } else {
    tmC = tmA;
  }
  const int smem = g.stages * stage_bytes + fixed;
  const int tiles = (pair ? m_tiles2 : m_tiles) * g.n_tiles;
  const int sms = num_sms();
  const dim3 grid(pair ? 2 * (tiles < sms / 2 ? tiles : sms / 2) : (tiles < sms ? tiles : sms));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
#define NFK_LAUNCH_NT(E)                                                                     \
  if (pair) {                                                                                \
    if ((rc = set_smem(gemm_nt_pair_kernel<E>, smem))) return rc;                            \
    if (launch_pdl(gemm_nt_pair_kernel<E>, grid, dim3(GEMM_THREADS), smem, st, tmA, tmB, tmC, g) != cudaSuccess) \
      return NFK_ERR_LAUNCH;                                                                  \
  } else {                                                                                   \
    if ((rc = set_smem(gemm_nt_kernel<E>, smem))) return rc;                                 \
    if (launch_pdl(gemm_nt_kernel<E>, grid, dim3(GEMM_THREADS), smem, st, tmA, tmB, tmC, g) != cudaSuccess) \
      return NFK_ERR_LAUNCH;                                                                  \
  }
  switch (epi) {
    case NFK_EPI_F32: NFK_LAUNCH_NT(NFK_EPI_F32); break;
    case NFK_EPI_BIAS_RELU_BF16: NFK_LAUNCH_NT(NFK_EPI_BIAS_RELU_BF16); break;
    case NFK_EPI_MASK_BF16: NFK_LAUNCH_NT(NFK_EPI_MASK_BF16); break;
    default: return NFK_ERR_ARG;
  }
#undef NFK_LAUNCH_NT
  return cudaGetLastError() == cudaSuccess ? NFK_OK : NFK_ERR_LAUNCH;
}

extern "C" int nfk_gemm_tn_bf16(const void* A, long long lda, const void* B, long long ldb, int Mo, int No, int Kpix,
                                float* out, long long ldo, int sm_count, void* stream) {
  if (Mo <= 0 || No <= 0 || Kpix <= 0) return NFK_ERR_SHAPE;
  if (No % 64 || ldo % 4 || Mo % 8) return NFK_ERR_SHAPE;
  GemmArgs g{};
  g.M = Mo; g.N = No; g.K = Kpix;
  g.BN = No <= 256 ? No : (No % 256 == 0 ? 256 : (No % 192 == 0 ? 192 : (No % 128 == 0 ? 128 : 64)));
  g.n_tiles = (No + g.BN - 1) / g.BN;
  if (sm_count <= 0) sm_count = 148;
  // CTA pairs (256-row tiles) when the output is tall and wide enough to fill them: conv#2 weight gradients (512 x 512)
  // and the deeper levels' Conv2dZeros ones; the narrow ones (64 / 128 wide) are HBM-bound and stay on single CTAs
  static const bool tn_pairs = [] { const char* e = getenv("NFK_TN_PAIRS"); return !(e && e[0] == '0'); }();
  if (tn_pairs && Mo > BM && g.BN % 128 == 0 && Kpix >= 4096) {
    const int m_tiles2 = (Mo + 2 * BM - 1) / (2 * BM);
    const int ptiles = m_tiles2 * g.n_tiles;
    const int total_kb2 = (Kpix + BK - 1) / BK;
    int psplits = max(1, min(total_kb2, (sm_count / 2) / ptiles));
    g.kb_per_split = (total_kb2 + psplits - 1) / psplits;
    psplits = (total_kb2 + g.kb_per_split - 1) / g.kb_per_split;
    const int pstage = 2 * 64 * 128 + (g.BN / 128) * 64 * 128;
    g.stages = min(8, (196 * 1024) / pstage);
    g.out = out; g.ldo = ldo;
    CUtensorMap ptmA, ptmB;
    int prc;
    if ((prc = make_tmap_2d(&ptmA, A, Mo, Kpix, lda, 64)) != NFK_OK) return prc;
    if ((prc = make_tmap_2d(&ptmB, B, No, Kpix, ldb, 64)) != NFK_OK) return prc;
    const int psmem = g.stages * pstage + 1024 + 256;
    if ((prc = set_smem(gemm_tn_pair_kernel, psmem))) return prc;
    const cudaError_t ple = launch_pdl(gemm_tn_pair_kernel, dim3(2 * ptiles, psplits), dim3(TN_THREADS), psmem,
                                       static_cast<cudaStream_t>(stream), ptmA, ptmB, g);
    return (ple == cudaSuccess && cudaGetLastError() == cudaSuccess) ? NFK_OK : NFK_ERR_LAUNCH;
  }
  const int stage_bytes = 2 * 64 * 128 + (g.BN / 64) * 64 * 128;
  g.stages = min(8, (196 * 1024) / stage_bytes);
  g.out = out; g.ldo = ldo;
  const int tiles = ((Mo + BM - 1) / BM) * g.n_tiles;
  const int total_kb = (Kpix + BK - 1) / BK;
  // one wave: tiles * splits <= SMs (one CTA per SM; 152 CTAs on 148 SMs would run as two waves at half the speed)
  int splits = max(1, min(total_kb, sm_count / tiles));
  g.kb_per_split = (total_kb + splits - 1) / splits;
  splits = (total_kb + g.kb_per_split - 1) / g.kb_per_split;
  CUtensorMap tmA, tmB;
  int rc;
  if ((rc = make_tmap_2d(&tmA, A, Mo, Kpix, lda, 64)) != NFK_OK) return rc;
  if ((rc = make_tmap_2d(&tmB, B, No, Kpix, ldb, 64)) != NFK_OK) return rc;
  const int smem = g.stages * stage_bytes + 1024 + 256;
  if ((rc = set_smem(gemm_tn_kernel, smem))) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const cudaError_t le = launch_pdl(gemm_tn_kernel, dim3(tiles, splits), dim3(TN_THREADS), smem, st, tmA, tmB, g);
  return (le == cudaSuccess && cudaGetLastError() == cudaSuccess) ? NFK_OK : NFK_ERR_LAUNCH;
}
