// Fused SCATTER + patch-embed GEMM + timestep embedding (SURVEY K1/K2, north-star fused path #1).
//
// Each CTA owns one 128-token tile of this rank's shard.  Its four producer/epilogue warps pull the
// latent pixels of those tokens straight out of the LEAD GPU's buffer (plain ld.global on an
// NVLink peer mapping; 4-byte loads, coalesced along W), applying the 2x2 patchify permutation on
// the fly, and write them as the 128B-swizzled K-major A operand of a tcgen05 GEMM:
//
//     X[b, Lt + token, :] = patchify(x_peer[off + b])[token, :] @ W_img_in^T + bias      (K = 4*C)
//
// Up to 16 latent channels the patch is one 64-column K block (FLUX, Z-Image, WAN T2V).  Wider latents (WAN2.2 I2V:
// 36 channels = noise | mask | image latent) take NKB = ceil(C / 16) K blocks: the producers write one swizzled slab
// per block, the weight ring streams (n-tile, k-block) slabs (columns past 4*C come from the tensor map's zero fill,
// so the weight stays the plain [N, 4*C] reshape) and the MMA warp accumulates over the blocks.
//
// W tiles stream through a TMA ring, accumulators are double buffered in TMEM, the epilogue adds the
// bias and stores bf16 rows of the residual stream.  A spare warp of CTA 0 reads the shard's
// timesteps / guidance values from the peer and emits their sinusoidal embeddings, so after this one
// launch the replica holds everything of the step's per-sample inputs that changes between steps.
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include "../common/host.h"
#include "../common/ptx.cuh"
#include "scatter_params.h"

namespace pa {

namespace se {
constexpr int BM = 128, BN = 256, BK = 64, WSTAGES = 3, MAX_KB = 4;
constexpr uint32_t A_BYTES = BM * BK * 2, W_BYTES = BN * BK * 2;   // A_BYTES: one K block (slab) of the token tile
constexpr uint32_t STAGE_BYTES = BM * BN * 2;                      // 4 slabs of [128 rows x 64 cols] bf16, 128B-swizzled

// shared-memory layout for NKB K blocks: [A slabs | W ring | store staging | barriers]
template <int NKB>
struct Smem {
  static constexpr uint32_t OFF_W = NKB * A_BYTES;
  static constexpr uint32_t OFF_STAGE = OFF_W + WSTAGES * W_BYTES;
  static constexpr uint32_t OFF_BAR = OFF_STAGE + STAGE_BYTES;
  static constexpr uint32_t BYTES = OFF_BAR + 256 + 1024;
  static_assert(BYTES <= 227 * 1024, "scatter_patch_embed: shared memory over the 227 KB per-block limit");
};
}  // namespace se

template <int NKB>
__global__ void __launch_bounds__(256, 1)
scatter_patch_embed_kernel(const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmO,
                           const ScatterEmbedParams p) {
  using namespace se;
  constexpr uint32_t OFF_W = Smem<NKB>::OFF_W, OFF_STAGE = Smem<NKB>::OFF_STAGE, OFF_BAR = Smem<NKB>::OFF_BAR;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + OFF_BAR);
  uint64_t* a_full = bars;              // 1 (128 arrivals)
  uint64_t* w_full = bars + 1;          // WSTAGES
  uint64_t* w_empty = w_full + WSTAGES; // WSTAGES
  uint64_t* tfull = w_empty + WSTAGES;  // 2
  uint64_t* tempty = tfull + 2;         // 2
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int warp_u = __shfl_sync(0xffffffffu, warp, 0);      // provably warp-uniform role index
  // grid = samples x token tiles x N-splits: with one sample per rank (8-GPU runs) 32 token tiles alone would leave
  // 3/4 of the SMs idle and serialise 12 weight tiles per CTA, so the output columns are split over `nsplit` CTAs
  // (each re-gathers the same 128 tokens: 16 KB of peer loads, L1-cached per SM)
  const int m_per = (p.Li + BM - 1) / BM;
  const int nsplit = p.nsplit;
  const int mb = blockIdx.x / nsplit, ns_i = blockIdx.x - mb * nsplit;
  const int b = mb / m_per;
  const int tok0 = (mb - b * m_per) * BM;
  const int num_n_all = (p.N + BN - 1) / BN;
  const int n_per = (num_n_all + nsplit - 1) / nsplit;
  const int nt0 = ns_i * n_per;
  const int num_n = max(0, min(num_n_all, nt0 + n_per) - nt0);      // this CTA's weight tiles: nt0 .. nt0 + num_n

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmW);
    ptx::prefetch_tmap(&tmO);
  }
  if (warp == 1 && lane == 0) {
    ptx::mbar_init(a_full, 128);
    for (int s = 0; s < WSTAGES; ++s) {
      ptx::mbar_init(&w_full[s], 1);
      ptx::mbar_init(&w_empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      ptx::mbar_init(&tfull[a], 1);
      ptx::mbar_init(&tempty[a], 4);
    }
    ptx::fence_barrier_init();
    ptx::fence_proxy_async_smem();
  }
  if (warp == 2) ptx::tmem_alloc<512>(tmem_slot);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp_u == 0) {
    // weight-tile producer (whole warp on uniform values, one elected lane issues; see gemm_tcgen05.cuh)
    const bool leader = ptx::elect_one();
    const uint32_t smem_u = __shfl_sync(0xffffffffu, ptx::smem_u32(smem), 0);
    for (int nt = 0; nt < num_n; ++nt) {
#pragma unroll
      for (int kb = 0; kb < NKB; ++kb) {
        const int it = nt * NKB + kb;
        const int s = it % WSTAGES;
        const uint32_t ph = (it / WSTAGES) & 1;
        ptx::mbar_wait(&w_empty[s], ph ^ 1);
        if (leader) {
          ptx::mbar_arrive_expect_tx(&w_full[s], W_BYTES);
          ptx::tma_load_2d_s(smem_u + OFF_W + s * W_BYTES, &tmW, &w_full[s], kb * BK, (nt0 + nt) * BN);
        }
      }
    }
    __syncwarp();
  } else if (warp_u == 1) {
    constexpr uint32_t IDESC = ptx::make_idesc_f16(BM, BN);
    const bool leader = ptx::elect_one();
    const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem, 0);
    const uint32_t smem_u = __shfl_sync(0xffffffffu, ptx::smem_u32(smem), 0);
    ptx::mbar_wait(a_full, 0);
    ptx::tc_fence_after();
    const uint64_t adesc = ptx::make_desc_kmajor_sw128(smem_u);
    for (int nt = 0; nt < num_n; ++nt) {
      const int acc = nt & 1;
#pragma unroll
      for (int kb = 0; kb < NKB; ++kb) {
        const int it = nt * NKB + kb;
        const int s = it % WSTAGES;
        ptx::mbar_wait(&w_full[s], (it / WSTAGES) & 1);
        if (kb == 0) ptx::mbar_wait(&tempty[acc], ((nt >> 1) & 1) ^ 1);
        ptx::tc_fence_after();
        if (leader) {
          const uint64_t bdesc = ptx::make_desc_kmajor_sw128(smem_u + OFF_W + s * W_BYTES);
          const uint64_t ad = adesc + kb * (A_BYTES >> 4);                 // descriptor address field is in 16 B units
#pragma unroll
          for (int k = 0; k < 4; ++k)
            ptx::mma_f16_ss(tmem_u + acc * BN, ad + 2 * k, bdesc + 2 * k, IDESC, (kb | k) != 0);
          ptx::tc_commit(&w_empty[s]);
          if (kb == NKB - 1) ptx::tc_commit(&tfull[acc]);
        }
      }
    }
    __syncwarp();
  } else if (warp == 3) {
    // timestep / guidance sinusoidal embeddings of the shard (values read from the lead GPU): n_t timesteps (n, or
    // one per video frame), guidance values only with n_t == n
    if (blockIdx.x == 0) {
      for (int i = lane; i < p.n_t * 128; i += 32) {
        const int s = i >> 7, f = i & 127;
        const float freq = __expf(-9.210340371976184f * static_cast<float>(f) * (1.0f / 128.0f));   // ln(1e4)
        float sn, cs;
        const float tv = __bfloat162float(p.t_src[s]) * p.time_factor;
        sincosf(tv * freq, &sn, &cs);
        p.t_emb[s * 256 + f] = __float2bfloat16(cs);
        p.t_emb[s * 256 + 128 + f] = __float2bfloat16(sn);
        if (p.g_src != nullptr) {
          const float gv = __bfloat162float(p.g_src[s]) * p.time_factor;
          sincosf(gv * freq, &sn, &cs);
          p.g_emb[s * 256 + f] = __float2bfloat16(cs);
          p.g_emb[s * 256 + 128 + f] = __float2bfloat16(sn);
        }
      }
    }
  } else if (warp >= 4) {
    // ---- A-operand producer: peer loads + patchify + swizzled smem stores
    const int q4 = warp & 3;
    const int r = q4 * 32 + lane;
    const int tok = tok0 + r;
    const int Wp = p.Wl >> 1;
    uint8_t* arow = smem + r * 128;
    const int sw = r & 7;
    if (tok < p.Li) {
      const int hh = tok / Wp, ww = tok - hh * Wp;
      const long long sample = static_cast<long long>(b) * p.C * p.Hl * p.Wl;
      const __nv_bfloat16* xs = p.x_src + sample;
      // every peer load of the row is issued before the first use: one NVLink round trip (~2-3 us) instead of one per
      // channel pair (NKB * 32 four-byte loads; with four K blocks 128 registers, still without spills)
      uint32_t v[NKB * 32];
#pragma unroll
      for (int c = 0; c < NKB * 16; ++c) {
#pragma unroll
        for (int ph = 0; ph < 2; ++ph) {
          const long long pix = (static_cast<long long>(c) * p.Hl + (hh * 2 + ph)) * p.Wl + ww * 2;
          v[c * 2 + ph] = c < p.C ? *reinterpret_cast<const uint32_t*>(xs + pix) : 0u;
        }
      }
#pragma unroll
      for (int c = 0; c < NKB * 16; ++c) {
#pragma unroll
        for (int ph = 0; ph < 2; ++ph) {
          if (p.x_copy && ns_i == 0 && c < p.C) {
            const long long pix = (static_cast<long long>(c) * p.Hl + (hh * 2 + ph)) * p.Wl + ww * 2;
            *reinterpret_cast<uint32_t*>(p.x_copy + sample + pix) = v[c * 2 + ph];
          }
          const int chunk = ((c & 15) >> 1) ^ sw;                          // K column 4*c + 2*ph + pw, slab c / 16
          *reinterpret_cast<uint32_t*>(arow + (c >> 4) * A_BYTES + chunk * 16 + (c & 1) * 8 + ph * 4) = v[c * 2 + ph];
        }
      }
    } else {
#pragma unroll
      for (int i = 0; i < NKB * 8; ++i) *reinterpret_cast<uint4*>(arow + (i >> 3) * A_BYTES + (i & 7) * 16) = make_uint4(0, 0, 0, 0);
    }
    ptx::fence_proxy_async_smem();
    ptx::mbar_arrive(a_full);
    // ---- epilogue: bias -> bf16 -> 128B-swizzled shared-memory staging -> TMA store.  A thread owns one accumulator
    // ROW, so storing straight to global memory makes every warp-level store touch 32 different 128-byte lines (16
    // useful bytes each); staged through shared memory the tile leaves the SM as whole 128-byte rows of a bulk tensor
    // store (UTMASTG), rows past the end of the sample are clipped by the tensor map.
    uint8_t* stage = smem + OFF_STAGE;
    const uint32_t stage_u = ptx::smem_u32(stage);
    const uint32_t lane_addr = tmem + (static_cast<uint32_t>(q4 * 32) << 16);
    for (int nt = 0; nt < num_n; ++nt) {
      const int acc = nt & 1;
      ptx::mbar_wait(&tfull[acc], (nt >> 1) & 1);
      ptx::tc_fence_after();
#pragma unroll 1
      for (int c = 0; c < BN / 32; ++c) {
        const int n = (nt0 + nt) * BN + c * 32;
        if (n >= p.N) break;
        uint32_t t[32];
        ptx::tmem_ld_32x32b_x32(lane_addr + acc * BN + c * 32, t);
        ptx::tmem_ld_wait();
        uint8_t* srow = stage + (c >> 1) * (BM * 128) + r * 128;          // slab of 64 columns, this thread's row
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          const uint4 bu = __ldg(reinterpret_cast<const uint4*>(p.bias + n + g * 8));
          const uint32_t bw[4] = {bu.x, bu.y, bu.z, bu.w};
          uint32_t o[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            __nv_bfloat162 bb = *reinterpret_cast<const __nv_bfloat162*>(&bw[e]);
            const float2 bf = __bfloat1622float2(bb);
            __nv_bfloat162 ov = __floats2bfloat162_rn(__uint_as_float(t[g * 8 + 2 * e]) + bf.x,
                                                      __uint_as_float(t[g * 8 + 2 * e + 1]) + bf.y);
            o[e] = *reinterpret_cast<uint32_t*>(&ov);
          }
          const int chunk = ((c & 1) * 4 + g) ^ sw;                        // 16-byte chunk inside the 128-byte row
          *reinterpret_cast<uint4*>(srow + chunk * 16) = make_uint4(o[0], o[1], o[2], o[3]);
        }
      }
      // accumulator drained: hand it back to the MMA warp before the (asynchronous) store
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&tempty[acc]);
      ptx::fence_proxy_async_smem();
      ptx::named_bar_sync(1, 128);                                         // all 128 rows of the tile are staged
      if (warp == 4 && ptx::elect_one()) {
#pragma unroll
        for (int sl = 0; sl < BN / 64; ++sl)
          if ((nt0 + nt) * BN + sl * 64 < p.N)
            ptx::tma_store_3d(&tmO, stage_u + sl * (BM * 128), (nt0 + nt) * BN + sl * 64, tok0, b);
        ptx::tma_store_commit();
        ptx::tma_store_wait_read<0>();                                     // staging may be overwritten afterwards
      }
      ptx::named_bar_sync(1, 128);
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc<512>(tmem);
  }
}

template <int NKB>
static int launch_scatter_patch_embed(const CUtensorMap& tw, const CUtensorMap& to, const ScatterEmbedParams& q,
                                      int blocks, cudaStream_t st) {
  constexpr int bytes = static_cast<int>(se::Smem<NKB>::BYTES);
  static bool attr_set[64] = {false};
  int dev = 0;
  cudaGetDevice(&dev);
  if (!attr_set[dev]) {
    cudaError_t e = cudaFuncSetAttribute(scatter_patch_embed_kernel<NKB>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         bytes);
    if (e != cudaSuccess) return (int)e;
    attr_set[dev] = true;
  }
  scatter_patch_embed_kernel<NKB><<<blocks, 256, bytes, st>>>(tw, to, q);
  return (int)cudaGetLastError();
}

// W: [N, 64] for C <= 16 (the one-block layout), else [N, 4*C] with C even (16-byte aligned rows)
int scatter_patch_embed(const void* W, long long ldw, const ScatterEmbedParams& p, cudaStream_t st) {
  using namespace se;
  if (p.C < 1 || p.C > MAX_KB * 16 || (p.C > 16 && (p.C & 1)) || p.N % 32 || (p.Wl & 1)) return -1;
  if (p.n_t < p.n || (p.g_src != nullptr && p.n_t != p.n)) return -3;
  const int nkb = p.C <= 16 ? 1 : (p.C + 15) / 16;
  CUtensorMap tw;
  uint64_t dims[2] = {nkb == 1 ? 64u : (uint64_t)(4 * p.C), (uint64_t)p.N};
  uint64_t str[2] = {2, (uint64_t)ldw * 2};
  uint32_t box[2] = {64, (uint32_t)BN};
  if (make_tmap(&tw, W, 2, dims, str, box, 2)) return -20;
  CUtensorMap to;                                   // output rows X[b, Lt + token, :] for the epilogue's TMA stores
  {
    uint64_t od[3] = {(uint64_t)p.N, (uint64_t)p.Li, (uint64_t)p.n};
    uint64_t os[3] = {2, (uint64_t)p.ldo * 2, (uint64_t)p.out_bstride * 2};
    uint32_t ob[3] = {64, (uint32_t)BM, 1};
    if ((p.ldo % 8) || (p.out_bstride % 8) || (reinterpret_cast<uintptr_t>(p.out) & 15)) return -2;
    if (make_tmap(&to, p.out, 3, od, os, ob, 2)) return -21;
  }
  ScatterEmbedParams q = p;
  const int mtiles = p.n * ((p.Li + BM - 1) / BM);
  const int num_n = (p.N + BN - 1) / BN;
  q.nsplit = 1;
  while (mtiles * q.nsplit * 2 <= 160 && q.nsplit * 2 <= num_n) q.nsplit *= 2;      // fill ~148 SMs, whole tiles per CTA
  switch (nkb) {
    case 1: return launch_scatter_patch_embed<1>(tw, to, q, mtiles * q.nsplit, st);
    case 2: return launch_scatter_patch_embed<2>(tw, to, q, mtiles * q.nsplit, st);
    case 3: return launch_scatter_patch_embed<3>(tw, to, q, mtiles * q.nsplit, st);
    default: return launch_scatter_patch_embed<4>(tw, to, q, mtiles * q.nsplit, st);
  }
}

}  // namespace pa
