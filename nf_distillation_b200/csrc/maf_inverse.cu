// MADE autoregressive inverse with the activations resident in shared memory (north_star kernel (4)).
//
// The reference repository ships no MAF/MADE code (SURVEY.md §0.2), so this follows Papamakarios et al. 2017 eq. 3:
//   x_i = u_i * exp(alpha_i(x_<i)) + mu_i(x_<i),  i = 0 .. D-1,   log|det| += sum_i alpha_i.
// Instead of D full passes of the three masked linears (D x one forward's FLOPs, activations through HBM / L2), the
// pre-activation of every hidden unit is finalised exactly ONCE: hidden units are sorted by degree, so after x_{d-1}
// is known the layer-1 units of degree d are final, then the layer-2 units of degree d (they read layer-1 units of
// degree <= d only), then (mu_d, alpha_d) (layer-2 units of degree <= d). Total work ~ one forward pass.
//
// Two kernels share the machinery below. A CTA owns warps x 16 samples for the whole D-step recursion; each WARP keeps
// the bf16 activations of its own samples (the roundings the forward GEMM epilogues apply) in its slice of shared
// memory; every product is a warp-level mma.sync.m16n8k16 (bf16 operands, fp32 accumulation), activations as the A
// operand and the masked bf16 weights as the B operand, both through ldmatrix. tcgen05 does not fit this recursion: a
// step touches 16 output columns of a 16-row tile, far below its tile shapes, with a TMEM round trip per step on the
// dependent chain.
//   made_inverse_resident_kernel (PULL): x, h1 and h2 resident; (mu_d, alpha_d) recomputed from h2 at every step.
//     Any sorted degrees: units go in aligned 8-column tiles, a tile that straddles two degrees is evaluated at both
//     steps (its not-yet-final columns hold finite scratch values that only meet masked-zero weights).
//   made_inverse_push_kernel (PUSH, further down): degrees change on whole tiles; finished layer-2 tiles go straight
//     from their accumulators into running (mu | alpha) sums in registers, h2 never exists in memory.
// The recursion is a fixed stream of JOBS (step d: layer-1 tile pairs of degree d, layer-2 tile pairs, the
// (mu_d, alpha_d) row pair), the same for every sample tile, so the host plans it once (nfk_made_inverse_jobs): per job
// its byte range in a shared-memory weight ring, the distance back to the job whose bytes it overwrites, and its
// offset in a packed weight stream that holds every job's weights already in shared-memory layout
// (nfk_made_inverse_pack, redone when the weights change). A producer warp copies each job's block into its range
// with ONE cp.async.bulk (completion on the job's "full" mbarrier); consumer warps wait on it, multiply, and release
// the job through its "empty" mbarrier — no block-wide barrier in the recursion, warps drift apart freely.
// What bounds it (profiles/r01_prof_maf_inverse.txt): a warp advances about one instruction per 6 cycles whatever the
// other warps do (a dependent scalar + MMA chain), so a tile costs (instructions per step) x D steps; the measured
// time followed the instruction count per step and nothing else — not the copy engine (one bulk copy per weight row,
// 51 per step, ran as fast as one per job), not the ring depth, not the warp count.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <cstdint>

#include "../../include/nfk.h"
#include "launch_util.h"
#include "ptx.cuh"

namespace nfk {

constexpr int MI_SLOTS = 16;   // jobs in flight at most (mbarrier pairs); the byte ring usually binds first

struct MiArgs {
  const float* u_in;            // [B, D] layer output order (flipped if flip)
  const unsigned char* wstream; // every job's weight bytes in shared-memory layout, job after job (nfk_made_inverse_pack)
  const float *b1, *b2, *b3;    // [H], [H], [>= 2D]
  const int4* jobs;             // [njobs][2]: {phase | second tile << 2 | k-chunks << 3, row0 (phase 2: d), ring offset,
                                //              back}, {stream offset / 16, bytes / 16, push: output tiles fed (bit mask),
                                //              push: d + 1 when the job also finishes x_d}
  int njobs, ring_bytes;
  float* x;                     // [B, D]
  const float* ld_in;           // [B] or null
  float* ld_out;                // [B] or null
  int B, D, H, Dp, flip;
};

template <int OFF = 0>
__device__ __forceinline__ void mi_ldsm_x4(uint32_t addr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4+%5];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(addr), "n"(OFF)
               : "memory");
}

template <int OFF = 0>
__device__ __forceinline__ void mi_ldsm_x2(uint32_t addr, uint32_t (&r)[2]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.shared.b16 {%0,%1}, [%2+%3];"
               : "=r"(r[0]), "=r"(r[1])
               : "r"(addr), "n"(OFF)
               : "memory");
}

__device__ __forceinline__ void mi_mma(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// one contiguous block, global -> shared, completion counted in bytes on `bar`
__device__ __forceinline__ void mi_bulk_copy(uint32_t dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

__device__ __forceinline__ uint32_t mi_pack_relu(float a, float b) {
  const __nv_bfloat162 v = __floats2bfloat162_rn(fmaxf(a, 0.f), fmaxf(b, 0.f));
  return *reinterpret_cast<const uint32_t*>(&v);
}

// job descriptor in 4 x 32 bits: x = phase [0,2) | second tile [2] | k-chunks [3,11) | first row (phase 2: d) [11,23)
//                                   | push kernel: step d finished by this job [23,31), flag [31]
//                               y = ring offset / 16 [0,16) | jobs back to the latest job whose ring bytes it overwrites [16,32)
//                               z = offset / 16 in the packed weight stream
//                               w = bytes / 16 [0,16) (0: the job carries nothing) | push kernel: output tiles fed [16,32)
__device__ __forceinline__ uint4 mi_pack_job(int4 a, int4 b) {
  const uint32_t back = a.w > 65535 ? 65535u : static_cast<uint32_t>(a.w);
  // (push kernel) b.w = d + 1 on the last layer-2 job of step d: x_d is finished right after it, no job of its own
  const uint32_t fin = b.w ? ((static_cast<uint32_t>(b.w - 1) << 23) | (1u << 31)) : 0u;
  return make_uint4(static_cast<uint32_t>(a.x) | (static_cast<uint32_t>(a.y) << 11) | fin,
                    (static_cast<uint32_t>(a.z) >> 4) | (back << 16), static_cast<uint32_t>(b.x),
                    static_cast<uint32_t>(b.y) | (static_cast<uint32_t>(b.z) << 16));
}

// blockDim = (consumer warps + 1) * 32; the last warp is the weight producer
template <int MT>
__global__ void __launch_bounds__(288) made_inverse_resident_kernel(const MiArgs p) {
  extern __shared__ __align__(128) unsigned char mi_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, cwarps = (blockDim.x >> 5) - 1;
  const int D = p.D, H = p.H, Dp = p.Dp;
  const int ldx = Dp + 8, ldh = H + 8;                       // bf16 elements; +8 keeps ldmatrix rows on distinct banks
  constexpr int R = MT * 16;
  const int per_warp = R * (ldx + 2 * ldh) * 2;              // bytes
  unsigned char* ring = mi_smem;
  uint64_t* full = reinterpret_cast<uint64_t*>(mi_smem + p.ring_bytes);
  uint64_t* empty = full + MI_SLOTS;
  uint4* jobs_s = reinterpret_cast<uint4*>(mi_smem + p.ring_bytes + 256);   // packed, see mi_pack_job
  unsigned char* act = mi_smem + p.ring_bytes + 256 + p.njobs * 16;
  const uint32_t ring_s = smem_u32(ring);
  for (int i = threadIdx.x; i < p.njobs; i += blockDim.x) jobs_s[i] = mi_pack_job(__ldg(p.jobs + 2 * i), __ldg(p.jobs + 2 * i + 1));

  if (threadIdx.x == 0) {
    for (int s = 0; s < MI_SLOTS; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], cwarps);
    }
    fence_mbar_init();
  }
  __syncthreads();

  const int ctiles = (p.B + R * cwarps - 1) / (R * cwarps);   // CTA tiles of cwarps * R samples
  const int my_tiles = (ctiles - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);
  const int njobs = p.njobs;

  if (warp == cwarps) {
    // ---------------- producer: the same job stream once per CTA tile. A job's weights are ONE contiguous block of
    // the packed stream (already in shared-memory layout: row stride = row bytes + 16 keeps ldmatrix rows on distinct
    // banks) -> one bulk copy per job into its byte range of the ring. (One copy per weight ROW, 16-17 per job, made
    // the copy engine the bottleneck: ~100 cycles per bulk operation, 51 per step.) Before overwriting, wait until
    // the latest job that used any of those bytes — or this job's slot — has been released by every consumer warp.
    int slot = 0, par = 0, q = 0;
    for (int tile = 0; tile < my_tiles; ++tile) {
      for (int j = 0; j < njobs; ++j, ++q) {
        const uint4 cur = jobs_s[j];
        int back = cur.y >> 16;
        if (back > MI_SLOTS) back = MI_SLOTS;
        if (q >= back) {
          const int ws = slot >= back ? slot - back : slot - back + MI_SLOTS;
          mbar_wait(&empty[ws], slot >= back ? par : par ^ 1);
        }
        if (lane == 0) {
          const uint32_t bytes = (cur.w & 0xffff) * 16;
          if (bytes == 0) {
            mbar_arrive(&full[slot]);
          } else {
            mbar_expect_tx(&full[slot], bytes);
            mi_bulk_copy(ring_s + (cur.y & 0xffff) * 16, p.wstream + static_cast<size_t>(cur.z) * 16, bytes, &full[slot]);
          }
        }
        if (++slot == MI_SLOTS) { slot = 0; par ^= 1; }
      }
    }
    return;
  }

  // ---------------- consumers: warp w owns samples [base, base + R) of the CTA tile
  const int g = lane >> 2, t = lane & 3;
  __nv_bfloat16* xb = reinterpret_cast<__nv_bfloat16*>(act + static_cast<size_t>(warp) * per_warp);
  __nv_bfloat16* h1 = xb + R * ldx;
  __nv_bfloat16* h2 = h1 + R * ldh;
  const int lrow = lane & 15, lcol = (lane >> 4) * 8;
  const uint32_t xb_lane = smem_u32(xb + lrow * ldx + lcol);
  const uint32_t h1_lane = smem_u32(h1 + lrow * ldh + lcol);
  const uint32_t h2_lane = smem_u32(h2 + lrow * ldh + lcol);
  // B-operand ldmatrix row / column of this lane inside a job: matrices = (tile 0, k 0-7), (tile 0, k 8-15), (tile 1, ..)
  const uint32_t b_row = (lane & 7) + ((lane >> 4) << 3), b_col = ((lane >> 3) & 1) * 16;

  // biases of a job (phase < 2: the two column pairs this lane finishes; phase 2: b3[d], b3[D + d]); requested one
  // job ahead of their use so the L2 round trip hides behind the previous job's products
  auto fetch_bias = [&](uint32_t jd) -> float4 {   // jd = descriptor word x
    const int phase = jd & 3, row0 = jd >> 11;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (phase < 2) {
      const float* bias = (phase == 0 ? p.b1 : p.b2) + row0 + 2 * t;
      v.x = __ldg(bias);
      v.y = __ldg(bias + 1);
      if (jd & 4) {
        v.z = __ldg(bias + 8);
        v.w = __ldg(bias + 9);
      }
    } else {
      v.x = __ldg(p.b3 + row0);
      v.y = __ldg(p.b3 + D + row0);
    }
    return v;
  };

  int slot = 0, par = 0;
  for (int tile = 0; tile < my_tiles; ++tile) {
    const long long base = ((static_cast<long long>(tile) * gridDim.x + blockIdx.x) * cwarps + warp) * R;
    float ldacc[MT][2], unext[MT][2];
    const float* urow[MT][2];     // lanes t == 0: this lane's samples' rows of u (null past the batch end)
    {
      // clear this warp's slice: scratch columns must be finite (they meet masked-zero weights)
      uint4* z = reinterpret_cast<uint4*>(xb);
      const uint4 zero = make_uint4(0u, 0u, 0u, 0u);
      for (int i = lane; i < per_warp / 16; i += 32) z[i] = zero;
#pragma unroll
      for (int mt = 0; mt < MT; ++mt)
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          const long long b = base + mt * 16 + g + 8 * hh;
          ldacc[mt][hh] = 0.f;
          urow[mt][hh] = (t == 0 && b < p.B) ? p.u_in + b * D : nullptr;
          unext[mt][hh] = urow[mt][hh] ? __ldg(urow[mt][hh] + (p.flip ? D - 1 : 0)) : 0.f;
        }
      __syncwarp();
    }
    uint4 jd = jobs_s[0];
    float4 bnext = fetch_bias(jd.x);
    for (int j = 0; j < njobs; ++j) {
      const uint32_t cur = jd.x;
      const float4 bv = bnext;
      const int phase = cur & 3, kch = (cur >> 3) & 255, row0 = cur >> 11;
      uint32_t b_addr = ring_s + (jd.y & 0xffff) * 16 + b_row * (kch * 32 + 16) + b_col;
      if (j + 1 < njobs) {
        jd = jobs_s[j + 1];
        bnext = fetch_bias(jd.x);
      }

      if (phase < 2) {
        // out[:, row0 .. row0 + 16) = bf16(relu(in[:, 0 .. 16*kch) . W^T + bias))
        const bool l1 = phase == 0, two = (cur & 4) != 0;
        uint32_t a_addr = l1 ? xb_lane : h1_lane;
        const int lda_bytes = (l1 ? ldx : ldh) * 2;
        float acc[MT][2][2][4];   // [m-tile][n-tile][even / odd k-chunk chain]
#pragma unroll
        for (int mt = 0; mt < MT; ++mt)
#pragma unroll
          for (int n = 0; n < 2; ++n)
#pragma unroll
            for (int c = 0; c < 2; ++c)
#pragma unroll
              for (int e = 0; e < 4; ++e) acc[mt][n][c][e] = 0.f;
        mbar_wait(&full[slot], par);
        // fragments are requested one k-chunk ahead of the products that use them (ping-pong register sets)
        uint32_t a0[MT][4], a1[MT][4], b0[4], b1[4];
        if (kch > 0) {
          mi_ldsm_x4<0>(b_addr, b0);
#pragma unroll
          for (int mt = 0; mt < MT; ++mt) mi_ldsm_x4<0>(a_addr + mt * 16 * lda_bytes, a0[mt]);
        }
        int kc = kch;
        for (; kc >= 2; kc -= 2, a_addr += 64, b_addr += 64) {
          mi_ldsm_x4<32>(b_addr, b1);
#pragma unroll
          for (int mt = 0; mt < MT; ++mt) mi_ldsm_x4<32>(a_addr + mt * 16 * lda_bytes, a1[mt]);
#pragma unroll
          for (int mt = 0; mt < MT; ++mt) {
            mi_mma(acc[mt][0][0], a0[mt], b0[0], b0[1]);
            mi_mma(acc[mt][1][0], a0[mt], b0[2], b0[3]);
          }
          if (kc > 2) {
            mi_ldsm_x4<64>(b_addr, b0);
#pragma unroll
            for (int mt = 0; mt < MT; ++mt) mi_ldsm_x4<64>(a_addr + mt * 16 * lda_bytes, a0[mt]);
          }
#pragma unroll
          for (int mt = 0; mt < MT; ++mt) {
            mi_mma(acc[mt][0][1], a1[mt], b1[0], b1[1]);
            mi_mma(acc[mt][1][1], a1[mt], b1[2], b1[3]);
          }
        }
        if (kc) {
#pragma unroll
          for (int mt = 0; mt < MT; ++mt) {
            mi_mma(acc[mt][0][0], a0[mt], b0[0], b0[1]);
            mi_mma(acc[mt][1][0], a0[mt], b0[2], b0[3]);
          }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[slot]);             // weights consumed: the bytes may be refilled
        __nv_bfloat16* out = (l1 ? h1 : h2) + row0 + 2 * t;
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) {
          *reinterpret_cast<uint32_t*>(out + (mt * 16 + g) * ldh) = mi_pack_relu(
              acc[mt][0][0][0] + acc[mt][0][1][0] + bv.x, acc[mt][0][0][1] + acc[mt][0][1][1] + bv.y);
          *reinterpret_cast<uint32_t*>(out + (mt * 16 + g + 8) * ldh) = mi_pack_relu(
              acc[mt][0][0][2] + acc[mt][0][1][2] + bv.x, acc[mt][0][0][3] + acc[mt][0][1][3] + bv.y);
          if (two) {
            *reinterpret_cast<uint32_t*>(out + (mt * 16 + g) * ldh + 8) = mi_pack_relu(
                acc[mt][1][0][0] + acc[mt][1][1][0] + bv.z, acc[mt][1][0][1] + acc[mt][1][1][1] + bv.w);
            *reinterpret_cast<uint32_t*>(out + (mt * 16 + g + 8) * ldh + 8) = mi_pack_relu(
                acc[mt][1][0][2] + acc[mt][1][1][2] + bv.z, acc[mt][1][0][3] + acc[mt][1][1][3] + bv.w);
          }
        }
        __syncwarp();
      } else {
        // (mu_d, alpha_d) from the layer-2 units of degree <= d; job row 0 = mu weights, row 1 = alpha weights
        const int d = row0;
        float uv[MT][2];
#pragma unroll
        for (int mt = 0; mt < MT; ++mt)
#pragma unroll
          for (int hh = 0; hh < 2; ++hh) {
            uv[mt][hh] = unext[mt][hh];                          // next step's u, requested a whole step ahead
            unext[mt][hh] = (urow[mt][hh] && d + 1 < D) ? __ldg(urow[mt][hh] + (p.flip ? D - 2 - d : d + 1)) : 0.f;
          }
        float acc[MT][4][4];      // four independent k-chunk chains
#pragma unroll
        for (int mt = 0; mt < MT; ++mt)
#pragma unroll
          for (int c = 0; c < 4; ++c)
#pragma unroll
            for (int e = 0; e < 4; ++e) acc[mt][c][e] = 0.f;
        uint32_t a_addr = h2_lane;
        mbar_wait(&full[slot], par);
        // chunk c of a group of four feeds chain c; the next group's fragments are requested before this group's
        // products (only matrices 0/1 of the B operand are needed: rows 0 (mu) and 1 (alpha) of the job)
        uint32_t a[2][MT][4][4], b[2][4][2];
        auto load_group = [&](int buf, int n) {   // n = live chunks of the group (1..4)
#pragma unroll
          for (int c = 0; c < 4; ++c)
            if (c < n) {
              if (c == 0) mi_ldsm_x2<0>(b_addr, b[buf][0]);
              if (c == 1) mi_ldsm_x2<32>(b_addr, b[buf][1]);
              if (c == 2) mi_ldsm_x2<64>(b_addr, b[buf][2]);
              if (c == 3) mi_ldsm_x2<96>(b_addr, b[buf][3]);
#pragma unroll
              for (int mt = 0; mt < MT; ++mt) {
                if (c == 0) mi_ldsm_x4<0>(a_addr + mt * 16 * ldh * 2, a[buf][mt][0]);
                if (c == 1) mi_ldsm_x4<32>(a_addr + mt * 16 * ldh * 2, a[buf][mt][1]);
                if (c == 2) mi_ldsm_x4<64>(a_addr + mt * 16 * ldh * 2, a[buf][mt][2]);
                if (c == 3) mi_ldsm_x4<96>(a_addr + mt * 16 * ldh * 2, a[buf][mt][3]);
              }
            }
          a_addr += 128;
          b_addr += 128;
        };
        auto mma_group = [&](int buf, int n) {
#pragma unroll
          for (int c = 0; c < 4; ++c)
            if (c < n) {
#pragma unroll
              for (int mt = 0; mt < MT; ++mt) mi_mma(acc[mt][c], a[buf][mt][c], b[buf][c][0], b[buf][c][1]);
            }
        };
        int kc = kch;                                  // chunks not yet multiplied
        if (kc > 0) load_group(0, kc < 4 ? kc : 4);
        while (kc > 0) {
          const int n0 = kc < 4 ? kc : 4, r1 = kc - n0;
          if (r1 > 0) load_group(1, r1 < 4 ? r1 : 4);
          mma_group(0, n0);
          if (r1 <= 0) break;
          const int n1 = r1 < 4 ? r1 : 4, r2 = r1 - n1;
          if (r2 > 0) load_group(0, r2 < 4 ? r2 : 4);
          mma_group(1, n1);
          kc = r2;
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[slot]);
        if (t == 0) {   // lanes t == 0 hold columns 0 (mu) and 1 (alpha) of samples g and g + 8
#pragma unroll
          for (int mt = 0; mt < MT; ++mt)
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
              const float mu = (acc[mt][0][2 * hh] + acc[mt][1][2 * hh]) + (acc[mt][2][2 * hh] + acc[mt][3][2 * hh]) + bv.x;
              const float al = (acc[mt][0][2 * hh + 1] + acc[mt][1][2 * hh + 1]) +
                               (acc[mt][2][2 * hh + 1] + acc[mt][3][2 * hh + 1]) + bv.y;
              const float xv = uv[mt][hh] * expf(al) + mu;
              const int s = mt * 16 + g + 8 * hh;
              if (urow[mt][hh]) p.x[(urow[mt][hh] - p.u_in) + d] = xv;
              xb[s * ldx + d] = __float2bfloat16_rn(xv);
              ldacc[mt][hh] += al;
            }
        }
        __syncwarp();
      }
      if (++slot == MI_SLOTS) { slot = 0; par ^= 1; }
    }
    if (t == 0 && p.ld_out) {
#pragma unroll
      for (int mt = 0; mt < MT; ++mt)
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          const long long b = base + mt * 16 + g + 8 * hh;
          if (b < p.B) p.ld_out[b] = (p.ld_in ? p.ld_in[b] : 0.f) + ldacc[mt][hh];
        }
    }
  }
}

// ------------------------------------------------------------------------------------------------------------------
// PUSH variant (degree boundaries on multiples of 8 units, 2D <= 128): the layer-2 activations never reach shared
// memory. When the layer-2 tile pair of degree d comes out of its accumulators it is packed (bias, ReLU, bf16) straight
// into an A fragment and multiplied into the running (mu | alpha) sums of ALL outputs, kept in NO x 4 registers per
// thread for the whole recursion: out[:, r] += h2[:, 16 units] . B3[r, 16 units]^T. Step d then only extracts columns d
// and D + d. Against the pull kernel above: no h2 slice (19 KB instead of 35 KB per warp -> 9 consumer warps instead
// of 5), no K = (units of degree <= d) product per step for two useful columns out of eight.
template <int NO>
__global__ void __launch_bounds__(384) made_inverse_push_kernel(const MiArgs p) {
  extern __shared__ __align__(128) unsigned char mi_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, cwarps = (blockDim.x >> 5) - 1;
  const int D = p.D, H = p.H, Dp = p.Dp;
  const int ldx = Dp + 8, ldh = H + 8;
  constexpr int R = 16, N3p = NO * 8;
  const int per_warp = R * (ldx + ldh) * 2;                  // bytes: x and h1 only
  uint64_t* full = reinterpret_cast<uint64_t*>(mi_smem + p.ring_bytes);
  uint64_t* empty = full + MI_SLOTS;
  uint4* jobs_s = reinterpret_cast<uint4*>(mi_smem + p.ring_bytes + 256);
  float* bias_s = reinterpret_cast<float*>(mi_smem + p.ring_bytes + 256 + p.njobs * 16);   // [b1 | b2 | b3 (N3p)]
  unsigned char* act = mi_smem + p.ring_bytes + 256 + p.njobs * 16 + (2 * H + N3p) * 4;
  const uint32_t ring_s = smem_u32(mi_smem);
  for (int i = threadIdx.x; i < p.njobs; i += blockDim.x) jobs_s[i] = mi_pack_job(__ldg(p.jobs + 2 * i), __ldg(p.jobs + 2 * i + 1));
  // the biases live in shared memory: an L2 round trip per job sat on every warp's dependent chain
  for (int i = threadIdx.x; i < 2 * H + N3p; i += blockDim.x)
    bias_s[i] = i < H ? __ldg(p.b1 + i) : i < 2 * H ? __ldg(p.b2 + i - H) : (i - 2 * H < 2 * D ? __ldg(p.b3 + i - 2 * H) : 0.f);
  if (threadIdx.x == 0) {
    for (int s = 0; s < MI_SLOTS; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], cwarps);
    }
    fence_mbar_init();
  }
  __syncthreads();

  const int ctiles = (p.B + R * cwarps - 1) / (R * cwarps);
  const int my_tiles = (ctiles - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);
  const int njobs = p.njobs;

  if (warp == cwarps) {
    // ---------------- producer (see the pull kernel); a layer-2 job's block also holds its two push-table tiles,
    // after the B2 rows; a (mu_d, alpha_d) job carries nothing
    int slot = 0, par = 0, q = 0;
    for (int tile = 0; tile < my_tiles; ++tile) {
      for (int j = 0; j < njobs; ++j, ++q) {
        const uint4 cur = jobs_s[j];
        int back = cur.y >> 16;
        if (back > MI_SLOTS) back = MI_SLOTS;
        if (q >= back) {
          const int ws = slot >= back ? slot - back : slot - back + MI_SLOTS;
          mbar_wait(&empty[ws], slot >= back ? par : par ^ 1);
        }
        if (lane == 0) {
          const uint32_t bytes = (cur.w & 0xffff) * 16;
          if (bytes == 0) {
            mbar_arrive(&full[slot]);
          } else {
            mbar_expect_tx(&full[slot], bytes);
            mi_bulk_copy(ring_s + (cur.y & 0xffff) * 16, p.wstream + static_cast<size_t>(cur.z) * 16, bytes, &full[slot]);
          }
        }
        if (++slot == MI_SLOTS) { slot = 0; par ^= 1; }
      }
    }
    return;
  }

  // ---------------- consumers
  const int g = lane >> 2, t = lane & 3;
  __nv_bfloat16* xb = reinterpret_cast<__nv_bfloat16*>(act + static_cast<size_t>(warp) * per_warp);
  __nv_bfloat16* h1 = xb + R * ldx;
  const int lrow = lane & 15, lcol = (lane >> 4) * 8;
  const uint32_t xb_lane = smem_u32(xb + lrow * ldx + lcol);
  const uint32_t h1_lane = smem_u32(h1 + lrow * ldh + lcol);
  const uint32_t b_row = (lane & 7) + ((lane >> 4) << 3), b_col = ((lane >> 3) & 1) * 16;
  // push-table ldmatrix.x4: matrices = (n-tile n, tile block 0), (n, block 1), (n + 1, block 0), (n + 1, block 1);
  // a tile block is [N3p outputs][8 units] dense: 8 rows x 16 bytes = all 32 banks once
  const uint32_t pb_lane = ((lane >> 3) & 1) * (N3p * 16) + (((lane >> 4) << 3) + (lane & 7)) * 16;

  int slot = 0, par = 0;
  for (int tile = 0; tile < my_tiles; ++tile) {
    const long long base = ((static_cast<long long>(tile) * gridDim.x + blockIdx.x) * cwarps + warp) * R;
    float ldacc[2], unext[2];
    const float* urow[2];        // lanes t == 0: rows of u and x of this lane's two samples (null past the batch end)
    float* xrow[2];
    float out[NO][4];            // running (mu | alpha) sums: C fragments of the [16 samples x N3p] output
#pragma unroll
    for (int n = 0; n < NO; ++n)
#pragma unroll
      for (int e = 0; e < 4; ++e) out[n][e] = 0.f;
    {
      uint4* z = reinterpret_cast<uint4*>(xb);
      const uint4 zero = make_uint4(0u, 0u, 0u, 0u);
      for (int i = lane; i < per_warp / 16; i += 32) z[i] = zero;
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        const long long b = base + g + 8 * hh;
        ldacc[hh] = 0.f;
        urow[hh] = (t == 0 && b < p.B) ? p.u_in + b * D : nullptr;
        xrow[hh] = p.x + b * D;
        unext[hh] = urow[hh] ? __ldg(urow[hh] + (p.flip ? D - 1 : 0)) : 0.f;
      }
      __syncwarp();
    }
    // (mu_d, alpha_d) = columns d and D + d of the running sums -> x_d, its bf16 copy for the next layer-1 tile, log-det
    auto finalize = [&](const int d) {
        float uv[2];
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          uv[hh] = unext[hh];
          unext[hh] = (urow[hh] && d + 1 < D) ? __ldg(urow[hh] + (p.flip ? D - 2 - d : d + 1)) : 0.f;
        }
        const int nm = d >> 3, cm = d & 7, na = (D + d) >> 3, ca = (D + d) & 7;
        float m0 = 0.f, m1 = 0.f, l0 = 0.f, l1v = 0.f;
        // (a real switch = one indexed branch; an unrolled chain of n == nm tests costs 4 instructions per tile)
#define MI_PICK(N, ODD, V0, V1)                \
  case N:                                      \
    if (N < NO) {                              \
      V0 = (ODD) ? out[N < NO ? N : 0][1] : out[N < NO ? N : 0][0]; \
      V1 = (ODD) ? out[N < NO ? N : 0][3] : out[N < NO ? N : 0][2]; \
    }                                          \
    break;
#define MI_PICK_ALL(SEL, ODD, V0, V1)                                                                      \
  switch (SEL) {                                                                                           \
    MI_PICK(0, ODD, V0, V1) MI_PICK(1, ODD, V0, V1) MI_PICK(2, ODD, V0, V1) MI_PICK(3, ODD, V0, V1)        \
    MI_PICK(4, ODD, V0, V1) MI_PICK(5, ODD, V0, V1) MI_PICK(6, ODD, V0, V1) MI_PICK(7, ODD, V0, V1)        \
    MI_PICK(8, ODD, V0, V1) MI_PICK(9, ODD, V0, V1) MI_PICK(10, ODD, V0, V1) MI_PICK(11, ODD, V0, V1)      \
    MI_PICK(12, ODD, V0, V1) MI_PICK(13, ODD, V0, V1) MI_PICK(14, ODD, V0, V1) MI_PICK(15, ODD, V0, V1)    \
    default: break;                                                                                        \
  }
        MI_PICK_ALL(nm, cm & 1, m0, m1)
        MI_PICK_ALL(na, ca & 1, l0, l1v)
#undef MI_PICK_ALL
#undef MI_PICK
        const int srcm = (lane & ~3) | (cm >> 1), srca = (lane & ~3) | (ca >> 1);
        m0 = __shfl_sync(0xffffffffu, m0, srcm);
        m1 = __shfl_sync(0xffffffffu, m1, srcm);
        l0 = __shfl_sync(0xffffffffu, l0, srca);
        l1v = __shfl_sync(0xffffffffu, l1v, srca);
        if (t == 0) {
#pragma unroll
          for (int hh = 0; hh < 2; ++hh) {
            const float mu = (hh ? m1 : m0) + bias_s[2 * H + d], al = (hh ? l1v : l0) + bias_s[2 * H + D + d];
            const float xv = uv[hh] * expf(al) + mu;
            if (urow[hh]) xrow[hh][d] = xv;
            xb[(g + 8 * hh) * ldx + d] = __float2bfloat16_rn(xv);
            ldacc[hh] += al;
          }
        }
        __syncwarp();
    };
    uint4 jd = jobs_s[0];
    for (int j = 0; j < njobs; ++j) {
      const uint32_t cur = jd.x;
      const int phase = cur & 3, kch = (cur >> 3) & 255, row0 = (cur >> 11) & 0xfff;
      const uint32_t job_s = ring_s + (jd.y & 0xffff) * 16, live = jd.w >> 16;
      if (j + 1 < njobs) jd = jobs_s[j + 1];

      if (phase < 2) {
        const bool l1 = phase == 0, two = (cur & 4) != 0;
        uint32_t a_addr = l1 ? xb_lane : h1_lane;
        uint32_t b_addr = job_s + b_row * (kch * 32 + 16) + b_col;
        float acc[2][2][4];      // [n-tile][even / odd k-chunk chain]
#pragma unroll
        for (int n = 0; n < 2; ++n)
#pragma unroll
          for (int c = 0; c < 2; ++c)
#pragma unroll
            for (int e = 0; e < 4; ++e) acc[n][c][e] = 0.f;
        const float* bsrc = bias_s + (l1 ? 0 : H) + row0 + 2 * t;   // columns row0 + 2t, + 1 (tile 0) and + 8 (tile 1)
        const float2 bv01 = *reinterpret_cast<const float2*>(bsrc), bv23 = *reinterpret_cast<const float2*>(bsrc + 8);
        mbar_wait(&full[slot], par);
        // k-chunk counts are even (the host rounds up: the extra chunk meets masked-zero weights); fragments are
        // requested one chunk ahead, the last request of a job reads past its last chunk and is never used
        uint32_t a0[4], a1[4], b0[4], b1[4];
        mi_ldsm_x4<0>(b_addr, b0);
        mi_ldsm_x4<0>(a_addr, a0);
        for (int kc = kch; kc > 0; kc -= 2, a_addr += 64, b_addr += 64) {
          mi_ldsm_x4<32>(b_addr, b1);
          mi_ldsm_x4<32>(a_addr, a1);
          mi_mma(acc[0][0], a0, b0[0], b0[1]);
          mi_mma(acc[1][0], a0, b0[2], b0[3]);
          mi_ldsm_x4<64>(b_addr, b0);
          mi_ldsm_x4<64>(a_addr, a0);
          mi_mma(acc[0][1], a1, b1[0], b1[1]);
          mi_mma(acc[1][1], a1, b1[2], b1[3]);
        }
        // bias + ReLU + bf16: rows g / g + 8, columns row0 + 2t, + 1 (tile 0) and row0 + 8 + 2t, + 1 (tile 1)
        uint32_t hA[4];
        hA[0] = mi_pack_relu(acc[0][0][0] + acc[0][1][0] + bv01.x, acc[0][0][1] + acc[0][1][1] + bv01.y);
        hA[1] = mi_pack_relu(acc[0][0][2] + acc[0][1][2] + bv01.x, acc[0][0][3] + acc[0][1][3] + bv01.y);
        hA[2] = two ? mi_pack_relu(acc[1][0][0] + acc[1][1][0] + bv23.x, acc[1][0][1] + acc[1][1][1] + bv23.y) : 0u;
        hA[3] = two ? mi_pack_relu(acc[1][0][2] + acc[1][1][2] + bv23.x, acc[1][0][3] + acc[1][1][3] + bv23.y) : 0u;
        if (l1) {
          __syncwarp();
          if (lane == 0) mbar_arrive(&empty[slot]);
          __nv_bfloat16* o = h1 + row0 + 2 * t;
          *reinterpret_cast<uint32_t*>(o + g * ldh) = hA[0];
          *reinterpret_cast<uint32_t*>(o + (g + 8) * ldh) = hA[1];
          if (two) {
            *reinterpret_cast<uint32_t*>(o + g * ldh + 8) = hA[2];
            *reinterpret_cast<uint32_t*>(o + (g + 8) * ldh + 8) = hA[3];
          }
        } else {
          // push: these 16 layer-2 units (degree d) feed outputs mu_i, alpha_i for i >= d only
          // (hA is exactly the A fragment of a 16 x 16 tile: C fragments of two adjacent 8-column tiles)
          const uint32_t pb = job_s + ((16 * (kch * 32 + 16) + 127) & ~127) + pb_lane;
#pragma unroll
          for (int n = 0; n < NO; n += 2) {
            if (live & (3u << n)) {      // the host marked the output tiles these units reach (i >= their degree)
              uint32_t w[4];
              mi_ldsm_x4<0>(pb + n * 128, w);
              if (live & (1u << n)) mi_mma(out[n], hA, w[0], w[1]);
              if (live & (2u << n)) mi_mma(out[n + 1], hA, w[2], w[3]);
            }
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(&empty[slot]);
          if (cur >> 31) finalize((cur >> 23) & 0xff);         // last layer-2 job of its step: x_d is complete
        }
        __syncwarp();
      } else {
        // a step without layer-2 units of its own degree (step 0; sparse degrees): x_d gets a job of its own
        mbar_wait(&full[slot], par);                           // (empty job: keeps the slot sequence in step)
        __syncwarp();                                          // every lane has seen the phase before the slot is released
        if (lane == 0) mbar_arrive(&empty[slot]);
        finalize(row0);
      }
      if (++slot == MI_SLOTS) { slot = 0; par ^= 1; }
    }
    if (t == 0 && p.ld_out) {
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        const long long b = base + g + 8 * hh;
        if (b < p.B) p.ld_out[b] = (p.ld_in ? p.ld_in[b] : 0.f) + ldacc[hh];
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------------------------
// REVERSE SOLVE (gradients of the inverse): the mirror of the pull kernel. With upstream g_x [B, D] and g_ld [B], one
// sweep d = D-1 .. 0 over the outputs gives every gradient of the inverse:
//   c_d = sum_{k > d} (dmu_k/dx_d . mubar_k + dalpha_k/dx_d . alphabar_k)    (VJP of the rows already final)
//   v_d = e^{alpha_d} (g_x,d + c_d),  mubar_d = g_x,d + c_d,  alphabar_d = v_d u_d + g_ld,   g_u = v (output order)
// c_d is a masked VJP whose order the degrees fix, the exact transpose of the order in which the pull kernel finalises
// units: layer-2 units of degree d + 1 get g2 = m2 . (dout[:, outputs > d] B3), then layer-1 units of degree d + 1 get
// g1 = m1 . (g2[:, degree >= d + 1] B2), then c_d = g1[:, degree >= d + 1] B1[:, d]. Every pre-activation gradient
// is final once (~ one backward pass of work). A warp keeps, for its samples, the bf16 dout rows finished so far and
// g2 / g1 in shared memory (the roundings the dgrad GEMM epilogues apply); the weights are the transposed operands of
// nfk_made_prep (B3T, B2T, B1T rows), streamed job by job through the same byte ring as the forward. A job's k range
// starts at its first k-chunk that can be non-zero (descriptor word w, bits [16,32)). Tiles that straddle two degrees
// are evaluated at both steps: their not-yet-final columns meet masked-zero weights only.
struct MibArgs {
  const float* g_x;             // [B, D] input order
  const float* g_ld;            // [B] or null
  const float* out;             // [B, N3p] (mu | alpha) at x, fp32
  const uint32_t *m1, *m2;      // ReLU masks at x, word-major [H / 32][B]
  const float* u_in;            // [B, D] layer output order (the inverse's input)
  const unsigned char* wstream; // nfk_made_inverse_bwd_pack
  const int4* jobs;
  int njobs, ring_bytes;
  float* g_u;                   // [B, D] output order
  __nv_bfloat16* dout;          // [B, N3p] = [mubar | alphabar | 0]
  float* db3;                   // [>= 2D] += column sums of dout (fp32 values before rounding)
  int B, D, H, N3p, flip;
};

template <int MT>
__global__ void __launch_bounds__(288) made_inverse_bwd_resident_kernel(const MibArgs p) {
  extern __shared__ __align__(128) unsigned char mi_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, cwarps = (blockDim.x >> 5) - 1;
  const int D = p.D, H = p.H, N3p = p.N3p, HW = H >> 5;
  const int ldo = N3p + 8, ldh = H + 8;
  constexpr int R = MT * 16;
  const int act_bytes = R * (ldo + 2 * ldh) * 2;
  const int per_warp = act_bytes + 2 * HW * R * 4 + N3p * 4;   // + masks [2][HW][R] + column sums [N3p]
  uint64_t* full = reinterpret_cast<uint64_t*>(mi_smem + p.ring_bytes);
  uint64_t* empty = full + MI_SLOTS;
  uint4* jobs_s = reinterpret_cast<uint4*>(mi_smem + p.ring_bytes + 256);
  unsigned char* act = mi_smem + p.ring_bytes + 256 + p.njobs * 16;
  const uint32_t ring_s = smem_u32(mi_smem);
  for (int i = threadIdx.x; i < p.njobs; i += blockDim.x) jobs_s[i] = mi_pack_job(__ldg(p.jobs + 2 * i), __ldg(p.jobs + 2 * i + 1));
  if (threadIdx.x == 0) {
    for (int s = 0; s < MI_SLOTS; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], cwarps);
    }
    fence_mbar_init();
  }
  __syncthreads();

  const int ctiles = (p.B + R * cwarps - 1) / (R * cwarps);
  const int my_tiles = (ctiles - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);
  const int njobs = p.njobs;

  if (warp == cwarps) {
    // ---------------- producer: identical to the pull kernel's
    int slot = 0, par = 0, q = 0;
    for (int tile = 0; tile < my_tiles; ++tile) {
      for (int j = 0; j < njobs; ++j, ++q) {
        const uint4 cur = jobs_s[j];
        int back = cur.y >> 16;
        if (back > MI_SLOTS) back = MI_SLOTS;
        if (q >= back) {
          const int ws = slot >= back ? slot - back : slot - back + MI_SLOTS;
          mbar_wait(&empty[ws], slot >= back ? par : par ^ 1);
        }
        if (lane == 0) {
          const uint32_t bytes = (cur.w & 0xffff) * 16;
          if (bytes == 0) {
            mbar_arrive(&full[slot]);
          } else {
            mbar_expect_tx(&full[slot], bytes);
            mi_bulk_copy(ring_s + (cur.y & 0xffff) * 16, p.wstream + static_cast<size_t>(cur.z) * 16, bytes, &full[slot]);
          }
        }
        if (++slot == MI_SLOTS) { slot = 0; par ^= 1; }
      }
    }
    return;
  }

  // ---------------- consumers: warp w owns samples [base, base + R) of the CTA tile
  const int g = lane >> 2, t = lane & 3;
  unsigned char* mine = act + static_cast<size_t>(warp) * per_warp;
  __nv_bfloat16* ds = reinterpret_cast<__nv_bfloat16*>(mine);     // dout rows [R][ldo]
  __nv_bfloat16* g2 = ds + R * ldo;                               // [R][ldh]
  __nv_bfloat16* g1 = g2 + R * ldh;                               // [R][ldh]
  uint32_t* mk = reinterpret_cast<uint32_t*>(mine + act_bytes);   // m1 words [HW][R], then m2 words [HW][R]
  float* csum = reinterpret_cast<float*>(mk + 2 * HW * R);        // this warp's column sums, every tile
  for (int i = lane; i < N3p; i += 32) csum[i] = 0.f;
  const int lrow = lane & 15, lcol = (lane >> 4) * 8;
  const uint32_t ds_lane = smem_u32(ds + lrow * ldo + lcol);
  const uint32_t g2_lane = smem_u32(g2 + lrow * ldh + lcol);
  const uint32_t g1_lane = smem_u32(g1 + lrow * ldh + lcol);
  const uint32_t b_row = (lane & 7) + ((lane >> 4) << 3), b_col = ((lane >> 3) & 1) * 16;

  int slot = 0, par = 0;
  for (int tile = 0; tile < my_tiles; ++tile) {
    const long long base = ((static_cast<long long>(tile) * gridDim.x + blockIdx.x) * cwarps + warp) * R;
    long long brow[MT][2];       // lanes t == 0: this lane's samples (-1 past the batch end)
    float gl[MT][2], nx[MT][2][3];   // g_ld; next step's (g_x, alpha, u), requested a whole step ahead
    {
      uint4* z = reinterpret_cast<uint4*>(ds);
      const uint4 zero = make_uint4(0u, 0u, 0u, 0u);
      for (int i = lane; i < act_bytes / 16; i += 32) z[i] = zero;   // scratch columns must be finite
      for (int i = lane; i < HW * R; i += 32) {
        const int w = i / R, s = i - w * R;
        const long long b = base + s;
        mk[i] = b < p.B ? __ldg(p.m1 + static_cast<long long>(w) * p.B + b) : 0u;
        mk[HW * R + i] = b < p.B ? __ldg(p.m2 + static_cast<long long>(w) * p.B + b) : 0u;
      }
#pragma unroll
      for (int mt = 0; mt < MT; ++mt)
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          const long long b = base + mt * 16 + g + 8 * hh;
          brow[mt][hh] = (t == 0 && b < p.B) ? b : -1;
          const bool ok = brow[mt][hh] >= 0;
          gl[mt][hh] = (ok && p.g_ld) ? __ldg(p.g_ld + b) : 0.f;
          nx[mt][hh][0] = ok ? __ldg(p.g_x + b * D + D - 1) : 0.f;
          nx[mt][hh][1] = ok ? __ldg(p.out + b * N3p + 2 * D - 1) : 0.f;
          nx[mt][hh][2] = ok ? __ldg(p.u_in + b * D + (p.flip ? 0 : D - 1)) : 0.f;
        }
      __syncwarp();
    }
    for (int j = 0; j < njobs; ++j) {
      const uint4 jd = jobs_s[j];
      const uint32_t cur = jd.x;
      const int phase = cur & 3, kch = (cur >> 3) & 255, row0 = cur >> 11, k0 = jd.w >> 16;
      uint32_t b_addr = ring_s + (jd.y & 0xffff) * 16 + b_row * (kch * 32 + 16) + b_col;

      if (phase < 2) {
        // phase 1: g2[:, row0 .. row0 + 16) = m2 . (dout . B3T rows); phase 0: g1 = m1 . (g2 . B2T rows)
        const bool two = (cur & 4) != 0;
        uint32_t a_addr = (phase == 1 ? ds_lane : g2_lane) + k0 * 32;
        const int lda_bytes = (phase == 1 ? ldo : ldh) * 2;
        float acc[MT][2][2][4];
#pragma unroll
        for (int mt = 0; mt < MT; ++mt)
#pragma unroll
          for (int n = 0; n < 2; ++n)
#pragma unroll
            for (int c = 0; c < 2; ++c)
#pragma unroll
              for (int e = 0; e < 4; ++e) acc[mt][n][c][e] = 0.f;
        mbar_wait(&full[slot], par);
        uint32_t a0[MT][4], a1[MT][4], b0[4], b1[4];
        if (kch > 0) {
          mi_ldsm_x4<0>(b_addr, b0);
#pragma unroll
          for (int mt = 0; mt < MT; ++mt) mi_ldsm_x4<0>(a_addr + mt * 16 * lda_bytes, a0[mt]);
        }
        int kc = kch;
        for (; kc >= 2; kc -= 2, a_addr += 64, b_addr += 64) {
          mi_ldsm_x4<32>(b_addr, b1);
#pragma unroll
          for (int mt = 0; mt < MT; ++mt) mi_ldsm_x4<32>(a_addr + mt * 16 * lda_bytes, a1[mt]);
#pragma unroll
          for (int mt = 0; mt < MT; ++mt) {
            mi_mma(acc[mt][0][0], a0[mt], b0[0], b0[1]);
            mi_mma(acc[mt][1][0], a0[mt], b0[2], b0[3]);
          }
          if (kc > 2) {
            mi_ldsm_x4<64>(b_addr, b0);
#pragma unroll
            for (int mt = 0; mt < MT; ++mt) mi_ldsm_x4<64>(a_addr + mt * 16 * lda_bytes, a0[mt]);
          }
#pragma unroll
          for (int mt = 0; mt < MT; ++mt) {
            mi_mma(acc[mt][0][1], a1[mt], b1[0], b1[1]);
            mi_mma(acc[mt][1][1], a1[mt], b1[2], b1[3]);
          }
        }
        if (kc) {
#pragma unroll
          for (int mt = 0; mt < MT; ++mt) {
            mi_mma(acc[mt][0][0], a0[mt], b0[0], b0[1]);
            mi_mma(acc[mt][1][0], a0[mt], b0[2], b0[3]);
          }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[slot]);
        __nv_bfloat16* o = (phase == 1 ? g2 : g1) + row0 + 2 * t;
        const uint32_t* mw = mk + (phase == 1 ? HW * R : 0);
        const int c0 = row0 + 2 * t, c1 = c0 + 8;
#pragma unroll
        for (int mt = 0; mt < MT; ++mt)
#pragma unroll
          for (int hh = 0; hh < 2; ++hh) {
            const int s = mt * 16 + g + 8 * hh;
            const uint32_t w0 = mw[(c0 >> 5) * R + s] >> (c0 & 31);
            __nv_bfloat162 v = __floats2bfloat162_rn((w0 & 1u) ? acc[mt][0][0][2 * hh] + acc[mt][0][1][2 * hh] : 0.f,
                                                     (w0 & 2u) ? acc[mt][0][0][2 * hh + 1] + acc[mt][0][1][2 * hh + 1] : 0.f);
            *reinterpret_cast<__nv_bfloat162*>(o + s * ldh) = v;
            if (two) {
              const uint32_t w1 = mw[(c1 >> 5) * R + s] >> (c1 & 31);
              v = __floats2bfloat162_rn((w1 & 1u) ? acc[mt][1][0][2 * hh] + acc[mt][1][1][2 * hh] : 0.f,
                                        (w1 & 2u) ? acc[mt][1][0][2 * hh + 1] + acc[mt][1][1][2 * hh + 1] : 0.f);
              *reinterpret_cast<__nv_bfloat162*>(o + s * ldh + 8) = v;
            }
          }
        __syncwarp();
      } else {
        // step d: c_d = g1[:, k0 .. H) . B1T[d, k0 .. H) (job row 0), then row d of every gradient
        const int d = row0;
        float cur_v[MT][2][3];
#pragma unroll
        for (int mt = 0; mt < MT; ++mt)
#pragma unroll
          for (int hh = 0; hh < 2; ++hh) {
            const long long b = brow[mt][hh];
#pragma unroll
            for (int e = 0; e < 3; ++e) cur_v[mt][hh][e] = nx[mt][hh][e];
            const bool ok = b >= 0 && d > 0;
            nx[mt][hh][0] = ok ? __ldg(p.g_x + b * D + d - 1) : 0.f;
            nx[mt][hh][1] = ok ? __ldg(p.out + b * N3p + D + d - 1) : 0.f;
            nx[mt][hh][2] = ok ? __ldg(p.u_in + b * D + (p.flip ? D - d : d - 1)) : 0.f;
          }
        float acc[MT][4][4];
#pragma unroll
        for (int mt = 0; mt < MT; ++mt)
#pragma unroll
          for (int c = 0; c < 4; ++c)
#pragma unroll
            for (int e = 0; e < 4; ++e) acc[mt][c][e] = 0.f;
        uint32_t a_addr = g1_lane + k0 * 32;
        mbar_wait(&full[slot], par);
        uint32_t a[2][MT][4][4], b[2][4][2];
        auto load_group = [&](int buf, int n) {
#pragma unroll
          for (int c = 0; c < 4; ++c)
            if (c < n) {
              if (c == 0) mi_ldsm_x2<0>(b_addr, b[buf][0]);
              if (c == 1) mi_ldsm_x2<32>(b_addr, b[buf][1]);
              if (c == 2) mi_ldsm_x2<64>(b_addr, b[buf][2]);
              if (c == 3) mi_ldsm_x2<96>(b_addr, b[buf][3]);
#pragma unroll
              for (int mt = 0; mt < MT; ++mt) {
                if (c == 0) mi_ldsm_x4<0>(a_addr + mt * 16 * ldh * 2, a[buf][mt][0]);
                if (c == 1) mi_ldsm_x4<32>(a_addr + mt * 16 * ldh * 2, a[buf][mt][1]);
                if (c == 2) mi_ldsm_x4<64>(a_addr + mt * 16 * ldh * 2, a[buf][mt][2]);
                if (c == 3) mi_ldsm_x4<96>(a_addr + mt * 16 * ldh * 2, a[buf][mt][3]);
              }
            }
          a_addr += 128;
          b_addr += 128;
        };
        auto mma_group = [&](int buf, int n) {
#pragma unroll
          for (int c = 0; c < 4; ++c)
            if (c < n) {
#pragma unroll
              for (int mt = 0; mt < MT; ++mt) mi_mma(acc[mt][c], a[buf][mt][c], b[buf][c][0], b[buf][c][1]);
            }
        };
        int kc = kch;
        if (kc > 0) load_group(0, kc < 4 ? kc : 4);
        while (kc > 0) {
          const int n0 = kc < 4 ? kc : 4, r1 = kc - n0;
          if (r1 > 0) load_group(1, r1 < 4 ? r1 : 4);
          mma_group(0, n0);
          if (r1 <= 0) break;
          const int n1 = r1 < 4 ? r1 : 4, r2 = r1 - n1;
          if (r2 > 0) load_group(0, r2 < 4 ? r2 : 4);
          mma_group(1, n1);
          kc = r2;
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[slot]);
        float smu = 0.f, sal = 0.f;
        if (t == 0) {   // lanes t == 0 hold column 0 (c_d) of samples g and g + 8
#pragma unroll
          for (int mt = 0; mt < MT; ++mt)
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
              const float c = (acc[mt][0][2 * hh] + acc[mt][1][2 * hh]) + (acc[mt][2][2 * hh] + acc[mt][3][2 * hh]);
              const float mub = cur_v[mt][hh][0] + c;
              const float v = expf(cur_v[mt][hh][1]) * mub;
              const float alb = v * cur_v[mt][hh][2] + gl[mt][hh];
              const __nv_bfloat16 bm = __float2bfloat16_rn(mub), ba = __float2bfloat16_rn(alb);
              const int s = mt * 16 + g + 8 * hh;
              ds[s * ldo + d] = bm;
              ds[s * ldo + D + d] = ba;
              const long long b = brow[mt][hh];
              if (b >= 0) {
                p.g_u[b * D + (p.flip ? D - 1 - d : d)] = v;
                p.dout[b * N3p + d] = bm;
                p.dout[b * N3p + D + d] = ba;
                smu += mub;
                sal += alb;
              }
            }
        }
        // column sums: a fixed order over the warp's samples, then over its tiles
#pragma unroll
        for (int o = 4; o < 32; o <<= 1) {
          smu += __shfl_xor_sync(0xffffffffu, smu, o);
          sal += __shfl_xor_sync(0xffffffffu, sal, o);
        }
        if (lane == 0) {
          csum[d] += smu;
          csum[D + d] += sal;
        }
        __syncwarp();
      }
      if (++slot == MI_SLOTS) { slot = 0; par ^= 1; }
    }
    const int pad = N3p - 2 * D;   // dout's padding columns are zero
    for (int i = lane; i < R * pad; i += 32) {
      const int s = i / pad;
      const long long b = base + s;
      if (b < p.B) p.dout[b * N3p + 2 * D + (i - s * pad)] = __float2bfloat16_rn(0.f);
    }
  }
  // db3: the consumer warps' sums in warp order, one atomic per column per CTA
  asm volatile("bar.sync 1, %0;" ::"r"(cwarps * 32) : "memory");
  for (int i = threadIdx.x; i < 2 * D; i += cwarps * 32) {
    float s = 0.f;
    for (int w = 0; w < cwarps; ++w) s += reinterpret_cast<const float*>(act + static_cast<size_t>(w) * per_warp + act_bytes + 2 * HW * R * 4)[i];
    atomicAdd(p.db3 + i, s);
  }
}

// Packed weight stream: every job's bytes exactly as the inverse kernels want them in shared memory — rows of
// (kch * 32) weight bytes + 16 bytes of padding (zero), rows the job does not own zeroed, for a push-mode layer-2 job
// followed (128-byte aligned) by its two push-table tiles B3[r][row0 .. row0 + 16) regrouped as [tile][r][8].
// One CTA per job; rebuilt when the weights change (the job table itself depends on the degrees only).
__global__ void made_inverse_pack_kernel(const int4* __restrict__ jobs, const __nv_bfloat16* __restrict__ B1,
                                         const __nv_bfloat16* __restrict__ B2, const __nv_bfloat16* __restrict__ B3,
                                         int N3p, int D, int H, int Dp, int push, unsigned char* __restrict__ wstream) {
  const int4 a = jobs[2 * blockIdx.x], b = jobs[2 * blockIdx.x + 1];
  if (b.y == 0) return;
  const int phase = a.x & 3, two = (a.x >> 2) & 1, kch = a.x >> 3, row0 = a.y;
  uint4* dst = reinterpret_cast<uint4*>(wstream + static_cast<size_t>(b.x) * 16);
  const int per_row = kch * 2 + 1;                                      // 16-byte pieces per row, the last one padding
  const int rows_valid = phase == 2 ? 2 : (two ? 16 : 8);
  const int rows_block = (push && phase == 1) ? 16 : rows_valid;
  for (int i = threadIdx.x; i < rows_block * per_row; i += blockDim.x) {
    const int r = i / per_row, c = i - r * per_row;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (r < rows_valid && c < kch * 2) {
      const __nv_bfloat16* src = phase == 0   ? B1 + static_cast<size_t>(row0 + r) * Dp
                                 : phase == 1 ? B2 + static_cast<size_t>(row0 + r) * H
                                              : B3 + static_cast<size_t>(row0 + r * D) * H;   // rows d (mu), D + d (alpha)
      v = *reinterpret_cast<const uint4*>(src + c * 8);
    }
    dst[i] = v;
  }
  if (push && phase == 1) {
    // push tiles: [2 tiles][N3p rows][8 units]; units past H (a last, single tile) are zero
    __nv_bfloat16* pt = reinterpret_cast<__nv_bfloat16*>(dst + ((rows_block * per_row * 16 + 127) & ~127) / 16);
    for (int i = threadIdx.x; i < 2 * N3p; i += blockDim.x) {
      const int tb = i / N3p, r = i - tb * N3p, u0 = row0 + 8 * tb;
      uint4 v = make_uint4(0u, 0u, 0u, 0u);
      if (u0 < H) v = *reinterpret_cast<const uint4*>(B3 + static_cast<size_t>(r) * H + u0);
      reinterpret_cast<uint4*>(pt)[i] = v;
    }
  }
}

// Packed weight stream of the reverse solve: rows of the transposed operands from the job's first k-chunk on (phase
// 1: B3T [H, N3p], phase 0: B2T [H, H], phase 2: row d of B1T [Dp, H]), same row layout as above.
__global__ void made_inverse_bwd_pack_kernel(const int4* __restrict__ jobs, const __nv_bfloat16* __restrict__ B1T,
                                             const __nv_bfloat16* __restrict__ B2T,
                                             const __nv_bfloat16* __restrict__ B3T, int H, int N3p,
                                             unsigned char* __restrict__ wstream) {
  const int4 a = jobs[2 * blockIdx.x], b = jobs[2 * blockIdx.x + 1];
  if (b.y == 0) return;
  const int phase = a.x & 3, two = (a.x >> 2) & 1, kch = a.x >> 3, row0 = a.y, k0 = b.z;
  uint4* dst = reinterpret_cast<uint4*>(wstream + static_cast<size_t>(b.x) * 16);
  const int per_row = kch * 2 + 1;
  const int rows = phase == 2 ? 1 : (two ? 16 : 8);
  const __nv_bfloat16* src = phase == 0 ? B2T + static_cast<size_t>(row0) * H
                             : phase == 1 ? B3T + static_cast<size_t>(row0) * N3p
                                          : B1T + static_cast<size_t>(row0) * H;
  const int ld = phase == 1 ? N3p : H;
  for (int i = threadIdx.x; i < rows * per_row; i += blockDim.x) {
    const int r = i / per_row, c = i - r * per_row;
    dst[i] = c < kch * 2 ? *reinterpret_cast<const uint4*>(src + static_cast<size_t>(r) * ld + k0 * 16 + c * 8)
                         : make_uint4(0u, 0u, 0u, 0u);
  }
}

static inline int mi_per_warp_bytes(int mt, int H, int Dp) { return mt * 16 * ((Dp + 8) + 2 * (H + 8)) * 2; }
// reverse solve: dout rows, g2, g1 (bf16), the two ReLU masks of the warp's samples, its column sums of dout
static inline int mib_per_warp_bytes(int mt, int H, int N3p) {
  return mt * 16 * ((N3p + 8) + 2 * (H + 8)) * 2 + 2 * (H / 32) * mt * 16 * 4 + N3p * 4;
}
static inline int mi_per_warp_bytes_push(int H, int Dp) { return 16 * ((Dp + 8) + (H + 8)) * 2; }
static inline int mi_rows_bytes(int rows, int kch) { return (rows * (kch * 32 + 16) + 127) & ~127; }
// bytes of a job in the weight ring. pull: its rows (nothing for kch == 0). push: layer-1 job = its rows, layer-2 job =
// a 16-row block + two push-table tiles, (mu, alpha) job = nothing.
static inline int mi_job_bytes(int desc, int push, int N3p) {
  const int phase = desc & 3, kch = desc >> 3, rows = phase == 2 ? 2 : ((desc & 4) ? 16 : 8);
  if (!push) return kch ? mi_rows_bytes(rows, kch) : 0;
  if (phase == 2) return 0;
  if (phase == 0) return mi_rows_bytes(rows, kch);
  return mi_rows_bytes(16, kch) + 2 * N3p * 16;
}
// barriers + packed job table + 128 spare bytes at the very end of the allocation (the product loops request one
// fragment past a row's last k-chunk; for the last row of the last warp that is past the activations)
static inline int mi_side_bytes(int njobs, int bias_floats = 0) { return 256 + njobs * 16 + bias_floats * 4 + 128; }   // barriers + packed job table

}  // namespace nfk

using namespace nfk;

static constexpr int MI_SMEM_MAX = 227 * 1024;

// Weight ring size for a layer shape: what is left after the barriers, the job table (the biases) and as many one-tile
// warps as fit next to a ring of two or three largest jobs.
static int mi_ring_fit(int biggest, int avail, int per_warp, int max_warps) {
  // room for four (else three) of the largest jobs when that still leaves 8 warps — with two, the copy of job j + 2
  // cannot start before job j is released and its latency shows when jobs are few and large (D = 6); a ring of exactly
  // three wastes its tail on jobs of unequal size — else for two
  int warps = 0;
  for (int k = 4; k >= 2 && warps < 8; --k) warps = (avail - k * biggest) / per_warp;
  if (warps > 8 && (avail - 4 * biggest) / per_warp < 8) warps = 8;   // (k = 3 or 2 chosen for the 8 warps: keep 8)
  if (warps < 1) return -1;
  if (warps > max_warps) warps = max_warps;
  int ring = (avail - warps * per_warp) & ~127;
  if (ring > (1 << 20) - 128) ring = (1 << 20) - 128;   // offsets are stored in 16 bits of 16-byte units
  return ring;
}

static int mi_ring_bytes(int H, int Dp, int njobs, int push, int N3p) {
  const int kmax = (H > Dp ? H : Dp) / 16;
  const int biggest = push ? mi_rows_bytes(16, kmax) + 2 * N3p * 16 : mi_rows_bytes(16, kmax);
  const int avail = MI_SMEM_MAX - mi_side_bytes(njobs, push ? 2 * H + N3p : 0);
  const int per_warp = push ? mi_per_warp_bytes_push(H, Dp) : mi_per_warp_bytes(1, H, Dp);
  return mi_ring_fit(biggest, avail, per_warp, push ? 11 : 8);
}

// reverse solve: the largest job multiplies 16 rows over max(H, N3p) columns
static int mib_ring_bytes(int H, int N3p, int njobs) {
  const int kmax = (H > N3p ? H : N3p) / 16;
  return mi_ring_fit(mi_rows_bytes(16, kmax), MI_SMEM_MAX - mi_side_bytes(njobs), mib_per_warp_bytes(1, H, N3p), 8);
}

// Ring placement of a planned job table (8 int32 per job; [0] descriptor, [2] ring offset, [3] back, [4] stream
// offset / 16, [5] bytes / 16): consecutive byte ranges, wrapping to 0 when a job does not fit before the end; every
// tile replays the same offsets, so `back` looks through the cyclic job order (a job of the previous tile counts).
// Stream placement: job after job.
template <class Size>
static int mi_place_jobs(int* jobs, int n, int ring, Size size_of) {
  int cur = 0;
  long long soff = 0;
  for (int j = 0; j < n; ++j) {
    const int size = size_of(jobs[8 * j]);
    if (size > ring) return NFK_ERR_SHAPE;
    if (cur + size > ring) cur = 0;
    jobs[8 * j + 2] = cur;
    cur += size;
    if (soff / 16 > 0x7fffffff) return NFK_ERR_SHAPE;
    jobs[8 * j + 4] = static_cast<int>(soff / 16);
    jobs[8 * j + 5] = size / 16;
    soff += size;
  }
  for (int j = 0; j < n; ++j) {
    const int lo = jobs[8 * j + 2], hi = lo + jobs[8 * j + 5] * 16;
    int back = n;                                  // nothing overlaps within a whole period: only the slot binds
    for (int b = 1; b < n && hi > lo; ++b) {
      const int i = ((j - b) % n + n) % n;
      const int lo2 = jobs[8 * i + 2], hi2 = lo2 + jobs[8 * i + 5] * 16;
      if (lo < hi2 && lo2 < hi) { back = b; break; }
    }
    jobs[8 * j + 3] = back;
  }
  return n;
}

extern "C" int nfk_made_inverse_resident_supported(int D, int H, int Dp) {
  if (D <= 0 || H <= 0 || H % 64 || Dp % 64 || Dp < D || H > 255 * 16 || Dp > 255 * 16) return 0;
  // (the packed job table also lives in shared memory: at most 4 D + H / 8 jobs of 16 bytes)
  return mi_ring_bytes(H, Dp, 4 * D + H / 8, 0, 0) > 0 ? 1 : 0;
}

extern "C" int nfk_made_inverse_push_supported(int D, int H, int Dp, int N3p) {
  if (!nfk_made_inverse_resident_supported(D, H, Dp)) return 0;
  if ((N3p != 64 && N3p != 128) || 2 * D > N3p) return 0;
  return mi_ring_bytes(H, Dp, 4 * D + H / 8, 1, N3p) > 0 ? 1 : 0;
}

// Host-side: the job stream of one sample tile from the degree counts (cnt[d] = units with degree <= d, d = 0..D),
// each job with its byte range in the weight ring and the distance back to the latest job that used those bytes.
extern "C" int nfk_made_inverse_jobs(const int* cnt1, const int* cnt2, int D, int H, int Dp, int N3p, int push,
                                     int* jobs, int cap) {
  if (!cnt1 || !cnt2 || D <= 0 || cap < 0 || (cap > 0 && !jobs)) return NFK_ERR_ARG;
  if (!(push ? nfk_made_inverse_push_supported(D, H, Dp, N3p) : nfk_made_inverse_resident_supported(D, H, Dp)))
    return NFK_ERR_SHAPE;
  int n = 0;
  // k-chunk counts of the hidden layers are rounded up to even (H / 16 and Dp / 16 are even): the kernels' product
  // loops take two chunks per trip; the extra chunk multiplies masked-zero weights
  auto even = [](int k) { return (k + 1) & ~1; };
  auto put = [&](int phase, int row0, int kch, int two) {
    if (n < cap) {
      int* q = jobs + 8 * n;
      q[0] = phase | (two << 2) | (kch << 3); q[1] = row0;
      for (int e = 2; e < 8; ++e) q[e] = 0;
    }
    ++n;
  };
  for (int d = 0; d < D; ++d) {
    const int c1p = d ? cnt1[d - 1] : 0, c1 = cnt1[d], c2p = d ? cnt2[d - 1] : 0, c2 = cnt2[d];
    if (c1 < c1p || c2 < c2p || c1p < 0 || c2p < 0 || c1 > H || c2 > H) return NFK_ERR_ARG;
    if (push && ((c1 | c2) & 7)) return NFK_ERR_SHAPE;   // the push kernel needs degree boundaries on whole 8-unit tiles
    if (d > 0) {
      if (c1 > c1p)   // layer-1 units of degree d: inputs x_0 .. x_{d-1}
        for (int nt = c1p >> 3, hi = (c1 + 7) >> 3; nt < hi; nt += 2) put(0, nt * 8, even((d + 15) >> 4), nt + 1 < hi);
      if (c2 > c2p)   // layer-2 units of degree d: layer-1 units of degree <= d
        for (int nt = c2p >> 3, hi = (c2 + 7) >> 3; nt < hi; nt += 2) {
          put(1, nt * 8, even((c1 + 15) >> 4), nt + 1 < hi);
          if (push && n <= cap) {   // output tiles (8 rows of [mu | alpha]) holding an output i >= d
            int mask = 0;
            for (int t = 0; t < N3p / 8; ++t)
              if ((8 * t + 7 >= d && 8 * t < D) || (8 * t + 7 >= D + d && 8 * t < 2 * D)) mask |= 1 << t;
            jobs[8 * (n - 1) + 6] = mask;
          }
        }
    }
    if (push && d > 0 && c2 > c2p) {
      if (n <= cap) jobs[8 * (n - 1) + 7] = d + 1;   // push: the step's last layer-2 job also finishes x_d
    } else {
      put(2, d, push ? 0 : (c2 + 15) >> 4, 0);       // (mu_d, alpha_d): layer-2 units of degree <= d (push: already summed)
    }
  }
  if (n > cap) return n;            // sizing call (or a short buffer): offsets need the whole table
  const int ring = mi_ring_bytes(H, Dp, n, push, N3p);
  if (ring <= 0) return NFK_ERR_SHAPE;
  return mi_place_jobs(jobs, n, ring, [&](int desc) { return mi_job_bytes(desc, push, N3p); });
}

extern "C" int nfk_made_inverse_bwd_supported(int D, int H, int N3p) {
  if (D <= 0 || D > 4095 || H <= 0 || H % 64 || N3p % 64 || N3p < 2 * D || H > 255 * 16 || N3p > 255 * 16) return 0;
  return mib_ring_bytes(H, N3p, 4 * D + H / 8) > 0 ? 1 : 0;
}

// Host-side: the job stream of the reverse solve, steps d = D-1 .. 0, from the same degree counts as the forward's
// planner. Per step: layer-2 tile pairs of degree d + 1 (k: dout columns of outputs > d), layer-1 tile pairs of
// degree d + 1 (k: layer-2 units of degree >= d + 1), then the row job of step d (k: layer-1 units of degree >= d + 1).
// jobs[6] = the job's first 16-wide k-chunk.
extern "C" int nfk_made_inverse_bwd_jobs(const int* cnt1, const int* cnt2, int D, int H, int N3p, int* jobs, int cap) {
  if (!cnt1 || !cnt2 || D <= 0 || cap < 0 || (cap > 0 && !jobs)) return NFK_ERR_ARG;
  if (!nfk_made_inverse_bwd_supported(D, H, N3p)) return NFK_ERR_SHAPE;
  for (int d = 0; d <= D; ++d)
    if (cnt1[d] < (d ? cnt1[d - 1] : 0) || cnt2[d] < (d ? cnt2[d - 1] : 0) || cnt1[d] > H || cnt2[d] > H)
      return NFK_ERR_ARG;
  int n = 0;
  auto put = [&](int phase, int row0, int k0, int k1, int two) {
    if (n < cap) {
      int* q = jobs + 8 * n;
      q[0] = phase | (two << 2) | ((k1 > k0 ? k1 - k0 : 0) << 3); q[1] = row0; q[6] = k1 > k0 ? k0 : 0;
      q[2] = q[3] = q[4] = q[5] = q[7] = 0;
    }
    ++n;
  };
  const int kh = H / 16, ko = (2 * D + 15) / 16;
  for (int d = D - 1; d >= 0; --d) {
    if (d + 1 < D) {
      const int c2p = cnt2[d], c2 = cnt2[d + 1], c1p = cnt1[d], c1 = cnt1[d + 1];
      for (int nt = c2p >> 3, hi = (c2 + 7) >> 3; c2 > c2p && nt < hi; nt += 2) put(1, nt * 8, (d + 1) >> 4, ko, nt + 1 < hi);
      for (int nt = c1p >> 3, hi = (c1 + 7) >> 3; c1 > c1p && nt < hi; nt += 2) put(0, nt * 8, c2p >> 4, kh, nt + 1 < hi);
    }
    put(2, d, cnt1[d] >> 4, kh, 0);
  }
  if (n > cap) return n;
  const int ring = mib_ring_bytes(H, N3p, n);
  if (ring <= 0) return NFK_ERR_SHAPE;
  return mi_place_jobs(jobs, n, ring, [](int desc) {
    const int kch = desc >> 3, rows = (desc & 3) == 2 ? 1 : ((desc & 4) ? 16 : 8);
    return kch ? mi_rows_bytes(rows, kch) : 0;
  });
}

extern "C" int nfk_made_inverse_bwd_pack(const int* jobs, int njobs, const void* B1T, const void* B2T, const void* B3T,
                                         int D, int H, int N3p, void* wstream, void* stream) {
  if (njobs <= 0 || !nfk_made_inverse_bwd_supported(D, H, N3p)) return NFK_ERR_SHAPE;
  if (!jobs || !B1T || !B2T || !B3T || !wstream || (reinterpret_cast<uintptr_t>(jobs) & 15) ||
      (reinterpret_cast<uintptr_t>(wstream) & 127))
    return NFK_ERR_ARG;
  made_inverse_bwd_pack_kernel<<<njobs, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const int4*>(jobs), static_cast<const __nv_bfloat16*>(B1T),
      static_cast<const __nv_bfloat16*>(B2T), static_cast<const __nv_bfloat16*>(B3T), H, N3p,
      static_cast<unsigned char*>(wstream));
  return cudaGetLastError() == cudaSuccess ? NFK_OK : NFK_ERR_LAUNCH;
}

extern "C" int nfk_made_inverse_pack(const int* jobs, int njobs, const void* B1, const void* B2, const void* B3,
                                     int N3p, int D, int H, int Dp, int push, void* wstream, void* stream) {
  if (njobs <= 0 || !nfk_made_inverse_resident_supported(D, H, Dp) || N3p < 2 * D || N3p % 8) return NFK_ERR_SHAPE;
  if (!jobs || !B1 || !B2 || !B3 || !wstream || (reinterpret_cast<uintptr_t>(jobs) & 15) ||
      (reinterpret_cast<uintptr_t>(wstream) & 127))
    return NFK_ERR_ARG;
  made_inverse_pack_kernel<<<njobs, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const int4*>(jobs), static_cast<const __nv_bfloat16*>(B1),
      static_cast<const __nv_bfloat16*>(B2), static_cast<const __nv_bfloat16*>(B3), N3p, D, H, Dp, push,
      static_cast<unsigned char*>(wstream));
  return cudaGetLastError() == cudaSuccess ? NFK_OK : NFK_ERR_LAUNCH;
}

template <int MT>
static int mi_launch(MiArgs p, cudaStream_t st) {
  const int per_warp = mi_per_warp_bytes(MT, p.H, p.Dp);
  p.ring_bytes = mi_ring_bytes(p.H, p.Dp, p.njobs, 0, 0);
  if (p.ring_bytes <= 0) return NFK_ERR_SHAPE;
  const int fixed = p.ring_bytes + mi_side_bytes(p.njobs);
  int warps = (MI_SMEM_MAX - fixed) / per_warp;
  if (warps > 8) warps = 8;
  if (warps < 1) return NFK_ERR_SHAPE;
  const int wtiles = (p.B + MT * 16 - 1) / (MT * 16);
  if (warps > wtiles) warps = wtiles;
  const int sms = num_sms();
  const int smem = fixed + warps * per_warp;
  if (cudaFuncSetAttribute(made_inverse_resident_kernel<MT>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) !=
      cudaSuccess)
    return NFK_ERR_LAUNCH;
  int grid = (wtiles + warps - 1) / warps;
  if (grid > sms) grid = sms;
  made_inverse_resident_kernel<MT><<<grid, (warps + 1) * 32, smem, st>>>(p);
  return cudaGetLastError() == cudaSuccess ? NFK_OK : NFK_ERR_LAUNCH;
}

template <int NO>
static int mi_launch_push(MiArgs p, cudaStream_t st) {
  const int per_warp = mi_per_warp_bytes_push(p.H, p.Dp);
  p.ring_bytes = mi_ring_bytes(p.H, p.Dp, p.njobs, 1, NO * 8);
  if (p.ring_bytes <= 0) return NFK_ERR_SHAPE;
  const int fixed = p.ring_bytes + mi_side_bytes(p.njobs, 2 * p.H + NO * 8);
  int warps = (MI_SMEM_MAX - fixed) / per_warp;
  if (warps > 11) warps = 11;
  if (warps < 1) return NFK_ERR_SHAPE;
  const int wtiles = (p.B + 15) / 16;
  if (warps > wtiles) warps = wtiles;
  const int sms = num_sms();
  const int smem = fixed + warps * per_warp;
  if (cudaFuncSetAttribute(made_inverse_push_kernel<NO>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) !=
      cudaSuccess)
    return NFK_ERR_LAUNCH;
  int grid = (wtiles + warps - 1) / warps;
  if (grid > sms) grid = sms;
  made_inverse_push_kernel<NO><<<grid, (warps + 1) * 32, smem, st>>>(p);
  return cudaGetLastError() == cudaSuccess ? NFK_OK : NFK_ERR_LAUNCH;
}

extern "C" int nfk_made_inverse_resident(const float* u_in, const void* wstream, const float* b1, const float* b2,
                                         const float* b3, const int* jobs, int njobs, int push, int N3p, float* x,
                                         const float* ld_in, float* ld_out, int B, int D, int H, int Dp, int flip,
                                         int mtiles, void* stream) {
  if (B <= 0 || njobs <= 0 || njobs > (1 << 20) || !nfk_made_inverse_resident_supported(D, H, Dp) || mtiles < 0 ||
      mtiles > 2)
    return NFK_ERR_SHAPE;
  if (push && !nfk_made_inverse_push_supported(D, H, Dp, N3p)) return NFK_ERR_SHAPE;
  if (!u_in || !wstream || !b1 || !b2 || !b3 || !jobs || !x) return NFK_ERR_ARG;
  if ((reinterpret_cast<uintptr_t>(jobs) & 15) || (reinterpret_cast<uintptr_t>(wstream) & 15)) return NFK_ERR_ARG;
  MiArgs p;
  p.u_in = u_in;
  p.wstream = static_cast<const unsigned char*>(wstream);
  p.b1 = b1; p.b2 = b2; p.b3 = b3;
  p.jobs = reinterpret_cast<const int4*>(jobs); p.njobs = njobs; p.ring_bytes = 0;
  p.x = x; p.ld_in = ld_in; p.ld_out = ld_out;
  p.B = B; p.D = D; p.H = H; p.Dp = Dp; p.flip = flip;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (push) return N3p == 128 ? mi_launch_push<16>(p, st) : mi_launch_push<8>(p, st);
  // pull kernel: one 16-sample tile per warp leaves room for the most warps; two halve the B-operand reads
  const int ring = mi_ring_bytes(H, Dp, njobs, 0, 0);
  if (ring <= 0) return NFK_ERR_SHAPE;
  int mt = mtiles == 0 ? 1 : mtiles;
  if (mt == 2 && ring + mi_side_bytes(njobs) + mi_per_warp_bytes(2, H, Dp) > MI_SMEM_MAX) mt = 1;
  return mt == 2 ? mi_launch<2>(p, st) : mi_launch<1>(p, st);
}

template <int MT>
static int mib_launch(MibArgs p, cudaStream_t st) {
  const int per_warp = mib_per_warp_bytes(MT, p.H, p.N3p);
  p.ring_bytes = mib_ring_bytes(p.H, p.N3p, p.njobs);
  if (p.ring_bytes <= 0) return NFK_ERR_SHAPE;
  const int fixed = p.ring_bytes + mi_side_bytes(p.njobs);
  int warps = (MI_SMEM_MAX - fixed) / per_warp;
  if (warps > 8) warps = 8;
  if (warps < 1) return NFK_ERR_SHAPE;
  const int wtiles = (p.B + MT * 16 - 1) / (MT * 16);
  if (warps > wtiles) warps = wtiles;
  const int sms = num_sms();
  const int smem = fixed + warps * per_warp;
  if (cudaFuncSetAttribute(made_inverse_bwd_resident_kernel<MT>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) !=
      cudaSuccess)
    return NFK_ERR_LAUNCH;
  int grid = (wtiles + warps - 1) / warps;
  if (grid > sms) grid = sms;
  made_inverse_bwd_resident_kernel<MT><<<grid, (warps + 1) * 32, smem, st>>>(p);
  return cudaGetLastError() == cudaSuccess ? NFK_OK : NFK_ERR_LAUNCH;
}

extern "C" int nfk_made_inverse_bwd_resident(const float* g_x, const float* g_ld, const float* out, const void* m1,
                                             const void* m2, const float* u_in, const void* wstream, const int* jobs,
                                             int njobs, float* g_u, void* dout, float* db3, int B, int D, int H,
                                             int N3p, int flip, int mtiles, void* stream) {
  if (B <= 0 || njobs <= 0 || njobs > (1 << 20) || !nfk_made_inverse_bwd_supported(D, H, N3p) || mtiles < 0 ||
      mtiles > 2)
    return NFK_ERR_SHAPE;
  if (!g_x || !out || !m1 || !m2 || !u_in || !wstream || !jobs || !g_u || !dout || !db3) return NFK_ERR_ARG;
  if ((reinterpret_cast<uintptr_t>(jobs) & 15) || (reinterpret_cast<uintptr_t>(wstream) & 15)) return NFK_ERR_ARG;
  MibArgs p;
  p.g_x = g_x; p.g_ld = g_ld; p.out = out;
  p.m1 = static_cast<const uint32_t*>(m1); p.m2 = static_cast<const uint32_t*>(m2);
  p.u_in = u_in;
  p.wstream = static_cast<const unsigned char*>(wstream);
  p.jobs = reinterpret_cast<const int4*>(jobs); p.njobs = njobs; p.ring_bytes = 0;
  p.g_u = g_u; p.dout = static_cast<__nv_bfloat16*>(dout); p.db3 = db3;
  p.B = B; p.D = D; p.H = H; p.N3p = N3p; p.flip = flip;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int ring = mib_ring_bytes(H, N3p, njobs);
  if (ring <= 0) return NFK_ERR_SHAPE;
  int mt = mtiles == 0 ? 1 : mtiles;
  if (mt == 2 && ring + mi_side_bytes(njobs) + mib_per_warp_bytes(2, H, N3p) > MI_SMEM_MAX) mt = 1;
  return mt == 2 ? mib_launch<2>(p, st) : mib_launch<1>(p, st);
}
