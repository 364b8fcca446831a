// Attention, ping-pong variant: TWO 128-row query tiles per CTA, each owned by its own softmax warpgroup,
// sharing every K/V tile.  Profiling of the one-tile kernel (attention.cu) showed its period is the serial
// chain  S-tile TMEM read -> max/exp -> P write  of a single warpgroup (~2.5x the MMA time, tensor pipe 41 %);
// with two tiles in flight the tensor pipe works on tile B (P.V and the next Q.K^T) while warpgroup A drains
// S_A from tensor memory, and vice versa.
//
//   warp 0      TMA producer (Q_A, Q_B once; K_j, V_j rings)          warp 2   TMEM allocator
//   warp 1      tcgen05.mma issuer                                     warps 4-7 / 8-11  softmax of tile A / B
//   TMEM        S_A @0, S_B @128 (fp32, 128 cols), O_A @256, O_B @384; P_X (bf16) overwrites the first 64
//               columns of S_X once S_X sits in registers and feeds the P.V MMA as a TMEM A operand.
//   registers   setmaxnreg: 56 for the producer/MMA warpgroup, 208 for the softmax warpgroups.
//
// KV2 (D = 128, NS = 1): two key/value sources, out = softmax(q K1^T) V1 + softmax(q K2^T) V2 in one launch (WAN2.1
// I2V / FLF2V cross-attention: text tokens and CLIP image tokens).  The producer streams the n1 tiles of source 1 and
// then the n2 tiles of source 2 through the same rings (only the tensor map and the key row change); at tile n1 the
// softmax warpgroups store the normalised segment-1 rows as bf16, restart the running max / sum and release the first
// segment-2 P.V (accumulate = 0) through `o_drain`; the final store adds the segment-1 row back in fp32 and rounds once.
#include <cuda_bf16.h>
#include <cuda_fp8.h>
#include <cuda_runtime.h>

#include "../common/host.h"
#include "../common/ptx.cuh"
#include "softmax_math.cuh"

namespace pa {
namespace a2 {

using namespace smx;

// timeline capture for DBG & 64: [role 0..4][kv tile 0..63][slot 0..7] clock64 stamps of CTA (1, 1)
__device__ long long g_trace[5 * 64 * 8];
#define PA_TR(role, j, slot)                                                          \
  do {                                                                                \
    if ((DBG & 64) && blockIdx.x == 1 && blockIdx.y == 1 && (j) < 64)                 \
      g_trace[((role) * 64 + (j)) * 8 + (slot)] = clock64();                          \
  } while (0)

#ifndef PA_POLY_MASK
#define PA_POLY_MASK 0x22
#endif

// Optional MXFP8 output (the next GEMM's A operand): e4m3 bytes [B, rows8, ld8] + UE8M0 scale chunks in the layout
// of gemm_mxfp8.cu.  q == nullptr -> bf16 output as usual.
struct Fp8Out {
  uint8_t* q;
  uint8_t* sf;
  long long ld8, bstride;
  int mtiles, kchunks;
};

template <int D>
struct Cfg {
  static constexpr int BN = 128;
  static constexpr uint32_t SLICE = 128 * 64 * 2;
  static constexpr uint32_t TILE = 128 * D * 2;
  static constexpr uint32_t OFF_Q = 0;                      // Q_A, Q_B
  static constexpr uint32_t OFF_K = 2 * TILE;               // 2 stages
  static constexpr uint32_t OFF_V = 4 * TILE;               // 2 stages
  static constexpr uint32_t OFF_BAR = 6 * TILE;
  static constexpr uint32_t OFF_XCHG = OFF_BAR + 256;       // float[2 tiles][2 parities][2 halves][128 rows]
  static constexpr uint32_t SMEM = OFF_XCHG + 4096 + 1024;
};

// DBG (timing experiments only, results are garbage for DBG != 0), bit mask: 1 = skip the softmax math, 2 = skip the
// TMEM read of S, 4 = Q.K^T issues one MMA instead of D/16, 8 = P.V issues one MMA instead of 8, 16 = P.V reads its
// A operand from shared memory (SS form) instead of tensor memory.
// NS: softmax warpgroups per query tile.  NS = 2 splits every S row between two threads (key columns 0..63 / 64..127,
// row maxima exchanged through shared memory): two warps per scheduler work on the same tile, so one warp's MUFU.EX2
// stalls are filled with the other's FMA-pipe work and the  S -> P  latency (the period-setting chain once the MMAs
// issue back to back) roughly halves.  640 threads, setmaxnreg 56 / 104 (640 x 96 registers at launch).
// KV2: this thread's normalised 128-column O row (tensor memory) -> bf16 at `dst`; `add`: sum with the bf16 row that is
// already there (segment 1) in fp32 and round once
__device__ __forceinline__ void store_o_row(uint32_t o_addr, __nv_bfloat16* dst, float inv, bool add, bool row_ok) {
#pragma unroll 1
  for (int c = 0; c < 4; ++c) {
    uint32_t t[32];
    ptx::tmem_ld_32x32b_x32(o_addr + c * 32, t);
    ptx::tmem_ld_wait();
    if (row_ok) {
#pragma unroll
      for (int i = 0; i < 32; i += 8) {
        float f[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) f[e] = __uint_as_float(t[i + e]) * inv;
        uint4* d = reinterpret_cast<uint4*>(dst + c * 32 + i);
        if (add) {
          const uint4 prev = *d;
          const __nv_bfloat162* pv = reinterpret_cast<const __nv_bfloat162*>(&prev);
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float2 pf = __bfloat1622float2(pv[e]);
            f[2 * e] += pf.x;
            f[2 * e + 1] += pf.y;
          }
        }
        uint4 u;
        __nv_bfloat162* hv = reinterpret_cast<__nv_bfloat162*>(&u);
#pragma unroll
        for (int e = 0; e < 4; ++e) hv[e] = __floats2bfloat162_rn(f[2 * e], f[2 * e + 1]);
        *d = u;
      }
    }
  }
}

template <int D, int DBG, int NS, bool KV2 = false>
__global__ void __launch_bounds__(128 + 256 * NS, 1)
attention2_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                  const __grid_constant__ CUtensorMap tmV, __nv_bfloat16* __restrict__ out, long long ldo,
                  long long o_bstride, int H, int Lq, int Lk, float scale_log2, const Fp8Out f8,
                  const __grid_constant__ CUtensorMap tmK2, const __grid_constant__ CUtensorMap tmV2, int Lk2) {
  static_assert(!KV2 || (D == 128 && NS == 1 && DBG == 0), "two K/V sources: D = 128, NS = 1 only");
  using C = Cfg<D>;
  constexpr int BN = C::BN;
  constexpr uint32_t SLICE = C::SLICE, TILE = C::TILE;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C::OFF_BAR);
  uint64_t* q_full = bars;          // 1
  uint64_t* k_full = bars + 1;      // 2
  uint64_t* k_empty = bars + 3;     // 2
  uint64_t* v_full = bars + 5;      // 2
  uint64_t* v_empty = bars + 7;     // 2
  uint64_t* s_full = bars + 9;      // 2 (tile A, B)
  uint64_t* p_full = bars + 11;     // 2: P_X keys 0..63 stored (the first four P.V MMAs may start)
  uint64_t* o_full = bars + 13;     // 2
  uint64_t* p_hi = bars + 15;       // 2: P_X keys 64..127 stored
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 17);
  uint64_t* o_drain = bars + 18;    // 2 (KV2): segment-1 O of tile X stored, its TMEM columns may be overwritten

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int warp_u = __shfl_sync(0xffffffffu, warp, 0);      // provably warp-uniform role index
  const int q0 = blockIdx.x * 256;
  const int bh = blockIdx.y;
  const int n1 = (Lk + BN - 1) / BN;                  // key tiles of source 1
  const int n_kv = KV2 ? n1 + (Lk2 + BN - 1) / BN : n1;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmQ);
    ptx::prefetch_tmap(&tmK);
    ptx::prefetch_tmap(&tmV);
    if constexpr (KV2) {
      ptx::prefetch_tmap(&tmK2);
      ptx::prefetch_tmap(&tmV2);
    }
  }
  if (warp == 1 && lane == 0) {
    ptx::mbar_init(q_full, 1);
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&k_full[i], 1);
      ptx::mbar_init(&k_empty[i], 1);
      ptx::mbar_init(&v_full[i], 1);
      ptx::mbar_init(&v_empty[i], 1);
      ptx::mbar_init(&s_full[i], 1);
      ptx::mbar_init(&p_full[i], 4);
      ptx::mbar_init(&p_hi[i], 4);
      ptx::mbar_init(&o_full[i], 1);
      if constexpr (KV2) ptx::mbar_init(&o_drain[i], 4);
    }
    ptx::fence_barrier_init();
    ptx::fence_proxy_async_smem();
  }
  if (warp == 2) ptx::tmem_alloc<512>(tmem_slot);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp < 4) {
    ptx::setmaxnreg_dec<56>();
    if (warp_u == 0) {
      // ===================== TMA producer (whole warp, one elected lane issues) =====================
      const bool leader = ptx::elect_one();
      const uint32_t smem_base = __shfl_sync(0xffffffffu, ptx::smem_u32(smem), 0);
      const int hb = bh / H, hh = bh - hb * H;
      if (leader) {
        ptx::mbar_arrive_expect_tx(q_full, 2 * TILE);
#pragma unroll
        for (int t = 0; t < 2; ++t)
#pragma unroll
          for (int sl = 0; sl < D / 64; ++sl)
            ptx::tma_load_4d_s(smem_base + C::OFF_Q + t * TILE + sl * SLICE, &tmQ, q_full, sl * 64, q0 + t * 128, hh, hb);
      }
      for (int j = 0; j < n_kv; ++j) {
        const int s = j & 1;
        const uint32_t ph = (j >> 1) & 1;
        ptx::mbar_wait(&k_empty[s], ph ^ 1);
        if (leader) {
          PA_TR(4, j, 0);
          ptx::mbar_arrive_expect_tx(&k_full[s], TILE);
          if (KV2 && j >= n1) {                            // ring and phase run over both sources; map and row switch
#pragma unroll
            for (int sl = 0; sl < D / 64; ++sl)
              ptx::tma_load_4d_s(smem_base + C::OFF_K + s * TILE + sl * SLICE, &tmK2, &k_full[s], sl * 64, (j - n1) * BN,
                                 hh, hb);
          } else {
#pragma unroll
            for (int sl = 0; sl < D / 64; ++sl)
              ptx::tma_load_4d_s(smem_base + C::OFF_K + s * TILE + sl * SLICE, &tmK, &k_full[s], sl * 64, j * BN, hh, hb);
          }
        }
        ptx::mbar_wait(&v_empty[s], ph ^ 1);
        if (leader) {
          PA_TR(4, j, 1);
          ptx::mbar_arrive_expect_tx(&v_full[s], TILE);
          if (KV2 && j >= n1) {
#pragma unroll
            for (int sl = 0; sl < D / 64; ++sl)
              ptx::tma_load_4d_s(smem_base + C::OFF_V + s * TILE + sl * SLICE, &tmV2, &v_full[s], sl * 64, (j - n1) * BN,
                                 hh, hb);
          } else {
#pragma unroll
            for (int sl = 0; sl < D / 64; ++sl)
              ptx::tma_load_4d_s(smem_base + C::OFF_V + s * TILE + sl * SLICE, &tmV, &v_full[s], sl * 64, j * BN, hh, hb);
          }
        }
      }
      __syncwarp();
    } else if (warp_u == 1) {
      // ===================== MMA issuer =====================
      // The whole warp runs this role with warp-uniform values and one elected lane issues the tcgen05 ops: inside a
      // `lane == 0` branch ptxas cannot prove the descriptors uniform and wraps EVERY UTCHMMA in an
      // ELECT / R2UR.BROADCAST / BRA.U.ANY waterfall loop (~90 cycles per MMA, more than the 64 cycles a 128x128x16
      // MMA executes) - measured with the PA_TR timeline: the issue thread, not the tensor pipe, set the period.
      constexpr uint32_t IDESC_QK = ptx::make_idesc_f16(128, 128, 1, 0, 0);
      constexpr uint32_t IDESC_PV = ptx::make_idesc_f16(128, D, 1, 0, 1);
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem, 0);
      const uint32_t smem_base = __shfl_sync(0xffffffffu, ptx::smem_u32(smem), 0);
      const bool leader = ptx::elect_one();
      auto qk = [&](int x, int i) {            // S_X = Q_X K_i^T
        if (leader) {
          const uint64_t qd = ptx::make_desc_kmajor_sw128(smem_base + C::OFF_Q + x * TILE);
          const uint64_t kd = ptx::make_desc_kmajor_sw128(smem_base + C::OFF_K + (i & 1) * TILE);
#pragma unroll
          for (int kk = 0; kk < ((DBG & 4) ? 1 : D / 16); ++kk) {
            const uint32_t off = ((kk >> 2) * SLICE + (kk & 3) * 32) >> 4;     // descriptor address field: bytes / 16
            ptx::mma_f16_ss(tmem_u + x * 128, qd + off, kd + off, IDESC_QK, kk != 0);
          }
          ptx::tc_commit(&s_full[x]);
        }
      };
      ptx::mbar_wait(q_full, 0);
      ptx::mbar_wait(&k_full[0], 0);
      ptx::tc_fence_after();
      qk(0, 0);
      qk(1, 0);
      if (leader) ptx::tc_commit(&k_empty[0]);
      for (int j = 0; j < n_kv; ++j) {
        const int st = j & 1;
        ptx::mbar_wait(&v_full[st], (j >> 1) & 1);
        if (leader) PA_TR(0, j, 4);
        const uint64_t vd = ptx::make_desc_mnmajor_sw128(smem_base + C::OFF_V + st * TILE, SLICE, 1024);
#pragma unroll 1
        for (int x = 0; x < 2; ++x) {
          ptx::mbar_wait(&p_full[x], j & 1);
          if (KV2 && j == n1) ptx::mbar_wait(&o_drain[x], 0);   // segment-1 O of tile x has left tensor memory
          ptx::tc_fence_after();
          if (leader) {
            PA_TR(x, j, 0);
#pragma unroll
            for (int kk = 0; kk < ((DBG & 8) ? 1 : 4); ++kk) {
              if (DBG & 16) {
                const uint32_t off = ((kk >> 2) * SLICE + (kk & 3) * 32) >> 4;
                ptx::mma_f16_ss(tmem_u + 256 + x * 128,
                                ptx::make_desc_kmajor_sw128(smem_base + C::OFF_Q + x * TILE) + off, vd + kk * 128, IDESC_PV,
                                (j | kk) != 0);
              } else {
                ptx::mma_f16_ts(tmem_u + 256 + x * 128, tmem_u + x * 128 + kk * 8, vd + kk * 128, IDESC_PV,
                                ((KV2 && j >= n1 ? j - n1 : j) | kk) != 0);
              }
            }
          }
          // second half of P_X (keys 64..127) is released separately: the first four MMAs overlap the rest of the exps
          ptx::mbar_wait(&p_hi[x], j & 1);
          ptx::tc_fence_after();
          if (leader) {
            if (!(DBG & 8)) {
#pragma unroll
              for (int kk = 4; kk < 8; ++kk)
                ptx::mma_f16_ts(tmem_u + 256 + x * 128, tmem_u + x * 128 + kk * 8, vd + kk * 128, IDESC_PV, 1u);
            }
            ptx::tc_commit(&o_full[x]);
            if (x == 1) ptx::tc_commit(&v_empty[st]);
            PA_TR(x, j, 1);
          }
          if (j + 1 < n_kv) {
            if (x == 0) {
              ptx::mbar_wait(&k_full[(j + 1) & 1], ((j + 1) >> 1) & 1);
              ptx::tc_fence_after();
            }
            if (leader) PA_TR(x, j, 2);
            qk(x, j + 1);                      // overwrites S_X / P_X: ordered after P_X.V in the tensor pipe
            if (leader) {
              if (x == 1) ptx::tc_commit(&k_empty[(j + 1) & 1]);
              PA_TR(x, j, 3);
            }
          }
        }
      }
      __syncwarp();
    }
  } else {
    ptx::setmaxnreg_inc<(NS == 2 ? 104 : 208)>();
    // ===================== softmax warpgroups =====================
    constexpr int CW = 128 / NS;                        // key columns of every S row owned by this thread
    constexpr int OW = D / NS;                          // output columns owned by this thread
    const int wg = (warp - 4) >> 2;
    const int x = wg / NS;                              // query tile of this warpgroup
    const int half = wg - x * NS;
    const int q4 = warp & 3;
    const int r = q4 * 32 + lane;
    const bool tracer = (q4 == 0 && lane == 0 && half == 0);
    const uint32_t lane_addr = tmem + (static_cast<uint32_t>(q4 * 32) << 16);
    const uint32_t s_addr = lane_addr + x * 128 + half * CW;
    const uint32_t p_addr = lane_addr + x * 128 + half * (CW / 2);     // bf16x2-packed P columns of this thread
    const uint32_t o_addr = lane_addr + 256 + x * 128 + half * OW;
    float* xchg = reinterpret_cast<float*>(smem + C::OFF_XCHG) + x * 512;
    float m_used = -INFINITY, l = 0.f;
    const unsigned long long sl2 = pack2(scale_log2, scale_log2);

    for (int j = 0; j < n_kv; ++j) {
      if (KV2 && j == n1) {
        // segment 1 done: store it normalised, restart the running max / sum, hand O's columns back to the MMA warp
        ptx::mbar_wait(&o_full[x], (n1 - 1) & 1);
        ptx::tc_fence_after();
        const int q_row = q0 + x * 128 + r;
        const int b = bh / H, h = bh - b * H;
        store_o_row(o_addr, out + b * o_bstride + static_cast<long long>(q_row) * ldo + h * D, 1.0f / l, false,
                    q_row < Lq);
        m_used = -INFINITY;
        l = 0.f;
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&o_drain[x]);
      }
      const bool seg2 = KV2 && j >= n1;
      const int jj = seg2 ? j - n1 : j;                  // tile index inside its own source
      ptx::mbar_wait(&s_full[x], j & 1);
      if (tracer) PA_TR(2 + x, j, 0);
      ptx::tc_fence_after();
      uint32_t sv[CW];
      if (DBG & 2) {
#pragma unroll
        for (int i = 0; i < CW; ++i) sv[i] = 0x3c000000u + i + j;
      } else {
#pragma unroll
        for (int c = 0; c < CW / 32; ++c)
          ptx::tmem_ld_32x32b_x32(s_addr + c * 32, *reinterpret_cast<uint32_t(*)[32]>(&sv[c * 32]));
        ptx::tmem_ld_wait();
      }
      if (tracer) PA_TR(2 + x, j, 1);
      if (DBG & 1) {
        if (NS == 2) ptx::named_bar_sync(1 + x, 256);    // S of both halves is in registers before P overwrites it
#pragma unroll
        for (int c = 0; c < CW / 32; ++c) {
          uint32_t pk[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) pk[i] = (sv[c * 32 + 2 * i] >> 16) | (sv[c * 32 + 2 * i + 1] & 0xffff0000u);
          ptx::tmem_st_32x32b_x16(p_addr + c * 16, pk);
        }
        ptx::tmem_st_wait();
        l = 1.f;
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (NS == 1 || half == 0) ptx::mbar_arrive(&p_full[x]);
          if (NS == 1 || half == 1) ptx::mbar_arrive(&p_hi[x]);
        }
        if (tracer) PA_TR(2 + x, j, 4);
        continue;
      }
      const int kv_left = (seg2 ? Lk2 : Lk) - jj * BN - half * CW;
      if (kv_left < CW) {
#pragma unroll
        for (int i = 0; i < CW; ++i)
          if (i >= kv_left) sv[i] = 0xff800000u;
      }
      float mx0 = -INFINITY, mx1 = -INFINITY, mx2 = -INFINITY, mx3 = -INFINITY;
#pragma unroll
      for (int i = 0; i < CW; i += 8) {
        mx0 = fmax3(mx0, __uint_as_float(sv[i]), __uint_as_float(sv[i + 1]));
        mx1 = fmax3(mx1, __uint_as_float(sv[i + 2]), __uint_as_float(sv[i + 3]));
        mx2 = fmax3(mx2, __uint_as_float(sv[i + 4]), __uint_as_float(sv[i + 5]));
        mx3 = fmax3(mx3, __uint_as_float(sv[i + 6]), __uint_as_float(sv[i + 7]));
      }
      float m_new = fmaxf(fmaxf(mx0, mx1), fmaxf(mx2, mx3));
      if (NS == 2) {
        // the two column halves of every row exchange maxima; the barrier also orders "S in registers (both halves)"
        // before the P stores below, which overwrite columns of S that belong to the other half
        float* xb = xchg + (j & 1) * 256;
        xb[half * 128 + r] = m_new;
        ptx::named_bar_sync(1 + x, 256);
        m_new = fmaxf(m_new, xb[(half ^ 1) * 128 + r]);
      }
      m_new = fmaxf(m_new, m_used);
      const bool need = (m_new - m_used) * scale_log2 > 8.0f;
      if (__any_sync(0xffffffffu, need)) {
        const float alpha = need ? ex2f((m_used - m_new) * scale_log2) : 1.0f;
        if (need) m_used = m_new;
        l *= alpha;
        if (jj > 0) {
          ptx::mbar_wait(&o_full[x], (j - 1) & 1);
          ptx::tc_fence_after();
#pragma unroll 1
          for (int c = 0; c < OW / 32; ++c) {
            uint32_t t[32];
            ptx::tmem_ld_32x32b_x32(o_addr + c * 32, t);
            ptx::tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 32; ++i) t[i] = __float_as_uint(__uint_as_float(t[i]) * alpha);
            ptx::tmem_st_32x32b_x32(o_addr + c * 32, t);
          }
          ptx::tmem_st_wait();
        }
      }
      if (tracer) PA_TR(2 + x, j, 2);
      const float mneg_f = -m_used * scale_log2;
      const unsigned long long mneg = pack2(mneg_f, mneg_f);
      unsigned long long sum2 = pack2(0.f, 0.f);
#pragma unroll
      for (int c = 0; c < CW / 32; ++c) {
        uint32_t pk[16];
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
          float a0, a1;
          const unsigned long long x2 =
              fma2(pack2(__uint_as_float(sv[c * 32 + i]), __uint_as_float(sv[c * 32 + i + 1])), sl2, mneg);
          // PA_POLY_MASK: which of every 8 pairs take the FMA-pipe polynomial instead of MUFU.EX2 (16 lanes/clk/SM);
          // tools/microbench/softmax_phase.cu: 2/8 is the fastest mix for one or two warps per scheduler
          if ((PA_POLY_MASK >> ((i >> 1) & 7)) & 1) {
            exp2_poly2(x2, a0, a1);
          } else {
            unpack2(x2, a0, a1);
            a0 = ex2f(a0);
            a1 = ex2f(a1);
          }
          sum2 = add2(sum2, pack2(a0, a1));
          __nv_bfloat162 hv = __floats2bfloat162_rn(a0, a1);
          pk[i >> 1] = *reinterpret_cast<uint32_t*>(&hv);
        }
        ptx::tmem_st_32x32b_x16(p_addr + c * 16, pk);    // keys 32c..32c+31 of this half -> packed columns 16c..16c+15
        if (NS == 1 && c == 1) {                         // keys 0..63 of P_X are complete: release the first four MMAs
          ptx::tmem_st_wait();
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(&p_full[x]);
        }
      }
      if (tracer) PA_TR(2 + x, j, 3);
      ptx::tmem_st_wait();
      float s0, s1;
      unpack2(sum2, s0, s1);
      l += s0 + s1;
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive((NS == 1 || half == 1) ? &p_hi[x] : &p_full[x]);
      if (tracer) PA_TR(2 + x, j, 4);
    }

    if (NS == 2) {                                        // combine the two partial row sums
      float* xl = xchg + (n_kv & 1) * 256;
      xl[half * 128 + r] = l;
      ptx::named_bar_sync(1 + x, 256);
      l += xl[(half ^ 1) * 128 + r];
    }
    ptx::mbar_wait(&o_full[x], (n_kv - 1) & 1);
    ptx::tc_fence_after();
    const int q_row = q0 + x * 128 + r;
    const float inv = 1.0f / l;
    const int b = bh / H, h = bh - b * H;
    __nv_bfloat16* dst = out + b * o_bstride + static_cast<long long>(q_row) * ldo + h * D + half * OW;
    if (KV2) {
      store_o_row(o_addr, dst, inv, true, q_row < Lq);
    } else if (f8.q != nullptr && NS == 1 && D == 128) {
      // MX-quantised output: each 32-column TMEM chunk of this thread's row is one MX block (amax -> UE8M0 scale ->
      // e4m3); half the bytes of the bf16 store and no separate quantise kernel before the projection GEMM
      uint8_t* qrow = f8.q + b * f8.bstride + static_cast<long long>(q_row) * f8.ld8 + h * D;
      uint32_t sfw = 0;
#pragma unroll 1
      for (int c = 0; c < 4; ++c) {
        uint32_t t[32];
        ptx::tmem_ld_32x32b_x32(o_addr + c * 32, t);
        ptx::tmem_ld_wait();
        float amax = 0.f;
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          t[i] = __float_as_uint(__uint_as_float(t[i]) * inv);
          amax = fmaxf(amax, fabsf(__uint_as_float(t[i])));
        }
        int e = -127;
        if (amax > 0.f) {
          e = static_cast<int>(ceilf(log2f(amax * (1.0f / 448.0f))));
          e = max(-127, min(127, e));
        }
        const float sc = exp2f(static_cast<float>(-e));
        uint32_t pk[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const __nv_fp8x2_storage_t lo = __nv_cvt_float2_to_fp8x2(
              make_float2(__uint_as_float(t[4 * j]) * sc, __uint_as_float(t[4 * j + 1]) * sc), __NV_SATFINITE, __NV_E4M3);
          const __nv_fp8x2_storage_t hi = __nv_cvt_float2_to_fp8x2(
              make_float2(__uint_as_float(t[4 * j + 2]) * sc, __uint_as_float(t[4 * j + 3]) * sc), __NV_SATFINITE, __NV_E4M3);
          pk[j] = static_cast<uint32_t>(lo) | (static_cast<uint32_t>(hi) << 16);
        }
        if (q_row < Lq) {
          uint4* d = reinterpret_cast<uint4*>(qrow + c * 32);
          d[0] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
          d[1] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
        }
        sfw |= static_cast<uint32_t>(e + 127) << (8 * c);
      }
      if (q_row < Lq) {
        const long long chunk = (static_cast<long long>(b) * f8.mtiles + (q_row >> 7)) * f8.kchunks + h;   // D == 128
        *reinterpret_cast<uint32_t*>(f8.sf + chunk * 512 + (q_row & 31) * 16 + ((q_row >> 5) & 3) * 4) = sfw;
      }
    } else
#pragma unroll 1
    for (int c = 0; c < OW / 32; ++c) {
      uint32_t t[32];
      ptx::tmem_ld_32x32b_x32(o_addr + c * 32, t);
      ptx::tmem_ld_wait();
      if (q_row < Lq) {
#pragma unroll
        for (int i = 0; i < 32; i += 8) {
          uint4 u;
          __nv_bfloat162 a0 = __floats2bfloat162_rn(__uint_as_float(t[i]) * inv, __uint_as_float(t[i + 1]) * inv);
          __nv_bfloat162 a1 = __floats2bfloat162_rn(__uint_as_float(t[i + 2]) * inv, __uint_as_float(t[i + 3]) * inv);
          __nv_bfloat162 a2 = __floats2bfloat162_rn(__uint_as_float(t[i + 4]) * inv, __uint_as_float(t[i + 5]) * inv);
          __nv_bfloat162 a3 = __floats2bfloat162_rn(__uint_as_float(t[i + 6]) * inv, __uint_as_float(t[i + 7]) * inv);
          u.x = *reinterpret_cast<uint32_t*>(&a0);
          u.y = *reinterpret_cast<uint32_t*>(&a1);
          u.z = *reinterpret_cast<uint32_t*>(&a2);
          u.w = *reinterpret_cast<uint32_t*>(&a3);
          *reinterpret_cast<uint4*>(dst + c * 32 + i) = u;
        }
      }
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc<512>(tmem);
  }
}

// second K/V source of a KV2 launch
struct Kv2 {
  const void *k, *v;
  int Lk;
  const long long *ks, *vs;
};

template <int D, int DBG, int NS = 1, bool KV2 = false>
static int launch(const void* q, const void* k, const void* v, void* out, long long ldo, long long o_bstride, int B,
                  int H, int Lq, int Lk, const long long* qs, const long long* ks, const long long* vs, float scale,
                  cudaStream_t st, Fp8Out f8 = Fp8Out{nullptr, nullptr, 0, 0, 0, 0},
                  Kv2 kv2 = Kv2{nullptr, nullptr, 0, nullptr, nullptr}) {
  using C = Cfg<D>;
  CUtensorMap tq, tk, tv, tk2, tv2;
  const uint32_t box[4] = {64, 128, 1, 1};
  auto mk = [&](CUtensorMap* m, const void* p, int L, const long long* s3) {
    uint64_t dims[4] = {(uint64_t)D, (uint64_t)L, (uint64_t)H, (uint64_t)B};
    uint64_t str[4] = {2, (uint64_t)s3[2] * 2, (uint64_t)s3[1] * 2, (uint64_t)s3[0] * 2};
    return make_tmap(m, p, 4, dims, str, box, 2, nullptr);
  };
  if (mk(&tq, q, Lq, qs)) return -20;
  if (mk(&tk, k, Lk, ks)) return -21;
  if (mk(&tv, v, Lk, vs)) return -22;
  if (KV2) {
    if (mk(&tk2, kv2.k, kv2.Lk, kv2.ks)) return -23;
    if (mk(&tv2, kv2.v, kv2.Lk, kv2.vs)) return -24;
  } else {
    tk2 = tk;                                            // unused by the one-source kernel
    tv2 = tv;
  }
  static bool attr_set[64] = {false};
  int dev = 0;
  cudaGetDevice(&dev);
  if (!attr_set[dev]) {
    cudaError_t e = cudaFuncSetAttribute(attention2_kernel<D, DBG, NS, KV2>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)C::SMEM);
    if (e != cudaSuccess) return (int)e;
    attr_set[dev] = true;
  }
  dim3 grid((Lq + 255) / 256, B * H);
  attention2_kernel<D, DBG, NS, KV2><<<grid, 128 + 256 * NS, C::SMEM, st>>>(
      tq, tk, tv, static_cast<__nv_bfloat16*>(out), ldo, o_bstride, H, Lq, Lk, scale * 1.4426950408889634f, f8, tk2, tv2,
      kv2.Lk);
  return (int)cudaGetLastError();
}
}  // namespace a2

int attention2_bf16(const void* q, const void* k, const void* v, void* out, long long ldo, long long o_bstride, int B,
                    int H, int Lq, int Lk, int D, const long long* qs, const long long* ks, const long long* vs,
                    float scale, cudaStream_t st) {
  for (int i = 0; i < 3; ++i)
    if (qs[i] % 8 || ks[i] % 8 || vs[i] % 8) return -10;
  if (D == 128) return a2::launch<128, 0>(q, k, v, out, ldo, o_bstride, B, H, Lq, Lk, qs, ks, vs, scale, st);
  if (D == 64) return a2::launch<64, 0>(q, k, v, out, ldo, o_bstride, B, H, Lq, Lk, qs, ks, vs, scale, st);
  return -11;
}

// head_dim 128 only: out = softmax(q k^T) v + softmax(q k2^T) v2 in one launch (the query tiles are loaded once)
int attention2_kv2_bf16(const void* q, const void* k, const void* v, const void* k2, const void* v2, void* out,
                        long long ldo, long long o_bstride, int B, int H, int Lq, int Lk, int Lk2, const long long* qs,
                        const long long* ks, const long long* vs, const long long* ks2, const long long* vs2, float scale,
                        cudaStream_t st) {
  for (int i = 0; i < 3; ++i)
    if (qs[i] % 8 || ks[i] % 8 || vs[i] % 8 || ks2[i] % 8 || vs2[i] % 8) return -10;
  if (Lk < 1 || Lk2 < 1) return -13;
  return a2::launch<128, 0, 1, true>(q, k, v, out, ldo, o_bstride, B, H, Lq, Lk, qs, ks, vs, scale, st,
                                     a2::Fp8Out{nullptr, nullptr, 0, 0, 0, 0}, a2::Kv2{k2, v2, Lk2, ks2, vs2});
}

// head_dim 128 only: the output goes out MX-quantised (e4m3 [B, rows8, ld8] + scale chunks) for a following fp8 GEMM
int attention2_fp8out(const void* q, const void* k, const void* v, void* out8, void* sf8, long long ld8, long long rows8,
                      int B, int H, int Lq, int Lk, const long long* qs, const long long* ks, const long long* vs,
                      float scale, cudaStream_t st) {
  for (int i = 0; i < 3; ++i)
    if (qs[i] % 8 || ks[i] % 8 || vs[i] % 8) return -10;
  if (ld8 % 128 || H * 128 > ld8) return -12;
  a2::Fp8Out f8{static_cast<uint8_t*>(out8), static_cast<uint8_t*>(sf8), ld8, rows8 * ld8,
                static_cast<int>((rows8 + 127) / 128), static_cast<int>(ld8 / 128)};
  return a2::launch<128, 0>(q, k, v, nullptr, 0, 0, B, H, Lq, Lk, qs, ks, vs, scale, st, f8);
}

// timing experiments (D = 128 only): dbg = DBG mask (see attention2_kernel) + 128 for one softmax warpgroup per tile
int attention2_debug(const void* q, const void* k, const void* v, void* out, long long ldo, long long o_bstride, int B,
                     int H, int Lq, int Lk, int dbg, const long long* qs, const long long* ks, const long long* vs,
                     float scale, cudaStream_t st) {
#define PA_A2_DBG(N) \
  if (dbg == N) return a2::launch<128, N, 2>(q, k, v, out, ldo, o_bstride, B, H, Lq, Lk, qs, ks, vs, scale, st); \
  if (dbg == N + 128) return a2::launch<128, N, 1>(q, k, v, out, ldo, o_bstride, B, H, Lq, Lk, qs, ks, vs, scale, st);
  PA_A2_DBG(0) PA_A2_DBG(1) PA_A2_DBG(3) PA_A2_DBG(15) PA_A2_DBG(64) PA_A2_DBG(67)
#undef PA_A2_DBG
  return -11;
}

// copies the DBG & 64 timeline (5 x 64 x 8 clock64 stamps) of the last traced launch to `host`
int attention2_trace_read(long long* host) {
  return (int)cudaMemcpyFromSymbol(host, a2::g_trace, sizeof(long long) * 5 * 64 * 8);
}

}  // namespace pa
