// Persistent, warp-specialised bf16 GEMM for sm_100a:
//   TMA (128B-swizzled tiles) -> smem ring -> tcgen05.mma (one elected thread) -> fp32 accumulators in
//   TMEM (double buffered) -> tcgen05.ld -> fused epilogue -> global (or NVLink peer) stores.
//
//   C[b, m, n] = epilogue( sum_k A[b, m, k] * W[n, k] )       A, W: bf16, K contiguous ("K-major")
//
// A is addressed as a 3-D tensor (K, rows-per-batch, batch) so that strided row subsets of one
// activation buffer (e.g. the txt / img token ranges of every sample) are GEMM operands without
// a gather/cat.  W is the nn.Linear weight [N, K] as stored.
//
// Epilogues (runtime `mode`, warp-uniform branch): bias, bias+GELU(tanh), bias+SiLU,
// residual + gate[b,n]*(acc+bias)  (AdaLN gated residual), fused QKV split + per-head RMSNorm + RoPE
// (+ GELU'd MLP columns for FLUX single blocks), GEGLU, and the "gather" epilogue: unpatchify + CFG
// + Euler update stored straight into the lead GPU's buffer over NVLink.
#pragma once
#include "../common/ptx.cuh"
#include <cuda_fp8.h>

#include "gemm_params.h"

namespace pa {

__device__ __forceinline__ float gelu_tanh(float x) {
  const float k0 = 0.7978845608028654f, k1 = 0.044715f;
  float u = k0 * (x + k1 * x * x * x);
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(u));
  return 0.5f * x * (1.0f + t);
}

__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752f)); }

__device__ __forceinline__ float silu(float x) { return x / (1.0f + __expf(-x)); }

__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}

__device__ __forceinline__ float2 unpack_bf16(uint32_t u) {
  __nv_bfloat162 v = *reinterpret_cast<__nv_bfloat162*>(&u);
  return __bfloat1622float2(v);
}

template <int BN>
struct GemmCfg {
  static constexpr int BM = 128, BK = 64;
  static constexpr int STAGES = BN == 256 ? 4 : (BN == 160 ? 5 : (BN == 128 ? 6 : 8));
  static constexpr uint32_t A_BYTES = BM * BK * 2;
  static constexpr uint32_t B_BYTES = BN * BK * 2;
  static constexpr uint32_t STAGE_BYTES = A_BYTES + B_BYTES;
  // two accumulator stages; the allocation must be a power of two >= 32 columns
  static constexpr uint32_t TMEM_COLS = 2 * BN <= 128 ? 128 : (2 * BN <= 256 ? 256 : 512);
  static constexpr uint32_t SMEM_BYTES = STAGES * STAGE_BYTES + 256 /*barriers*/ + 1024 /*align slack*/;
  static constexpr int THREADS = 384;                // 4 control warps + 8 epilogue warps
  // accumulator columns drained by the first / second warp of every TMEM lane quadrant (GLU epilogues walk
  // 64-column groups, the QKV epilogue 128-column heads: both stay whole)
  static constexpr int EPI_H0 = BN == 256 ? 128 : (BN == 160 ? 96 : 64);
  static constexpr int EPI_H1 = BN - EPI_H0;       // 128 | 64 | 64 | 0
};

// 8 bf16 (16 B) <-> 8 floats
__device__ __forceinline__ void cvt8(const uint4& u, float (&o)[8]) {
  float2 a = unpack_bf16(u.x), b = unpack_bf16(u.y), c = unpack_bf16(u.z), d = unpack_bf16(u.w);
  o[0] = a.x; o[1] = a.y; o[2] = b.x; o[3] = b.y; o[4] = c.x; o[5] = c.y; o[6] = d.x; o[7] = d.y;
}

__device__ __forceinline__ void ldg8(const __nv_bfloat16* p, float (&o)[8]) {
  cvt8(__ldg(reinterpret_cast<const uint4*>(p)), o);
}

__device__ __forceinline__ void ld8(const __nv_bfloat16* p, float (&o)[8]) {
  cvt8(*reinterpret_cast<const uint4*>(p), o);
}

__device__ __forceinline__ void st8(__nv_bfloat16* p, const float (&v)[8]) {
  uint4 u;
  u.x = pack_bf16(v[0], v[1]);
  u.y = pack_bf16(v[2], v[3]);
  u.z = pack_bf16(v[4], v[5]);
  u.w = pack_bf16(v[6], v[7]);
  *reinterpret_cast<uint4*>(p) = u;
}

// acc (+ bias) for 8 consecutive columns starting at register index g*8 of a 32-column TMEM chunk
__device__ __forceinline__ void acc8(const uint32_t (&r)[32], int g, const __nv_bfloat16* bias_at, float (&x)[8]) {
#pragma unroll
  for (int e = 0; e < 8; ++e) x[e] = __uint_as_float(r[g * 8 + e]);
  if (bias_at) {
    float bv[8];
    ldg8(bias_at, bv);
#pragma unroll
    for (int e = 0; e < 8; ++e) x[e] += bv[e];
  }
}

// One MX block: 32 consecutive fp32 values of a row -> 32 e4m3 bytes at `dst` (32-byte aligned) and the UE8M0 scale
// byte (returned).  Same arithmetic as quantize_mxfp8_kernel: scale = 2^ceil(log2(amax / 448)).
__device__ __forceinline__ uint32_t mx_quant32_store(const float (&v)[32], uint8_t* dst, bool do_store) {
  float amax = 0.f;
#pragma unroll
  for (int i = 0; i < 32; ++i) amax = fmaxf(amax, fabsf(v[i]));
  int e = -127;
  if (amax > 0.f) {
    e = static_cast<int>(ceilf(log2f(amax * (1.0f / 448.0f))));
    e = max(-127, min(127, e));
  }
  const float inv = exp2f(static_cast<float>(-e));
  uint32_t pk[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const __nv_fp8x2_storage_t lo =
        __nv_cvt_float2_to_fp8x2(make_float2(v[4 * j] * inv, v[4 * j + 1] * inv), __NV_SATFINITE, __NV_E4M3);
    const __nv_fp8x2_storage_t hi =
        __nv_cvt_float2_to_fp8x2(make_float2(v[4 * j + 2] * inv, v[4 * j + 3] * inv), __NV_SATFINITE, __NV_E4M3);
    pk[j] = static_cast<uint32_t>(lo) | (static_cast<uint32_t>(hi) << 16);
  }
  if (do_store) {
    uint4* d = reinterpret_cast<uint4*>(dst);
    d[0] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
    d[1] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
  }
  return static_cast<uint32_t>(e + 127);
}

// scale byte of (batch b, row, destination column dcol) inside the chunk layout
__device__ __forceinline__ uint8_t* mx_sf_ptr(const GemmParams& p, int b, int row, long long dcol) {
  const long long chunk = (static_cast<long long>(b) * p.sf8_mtiles + (row >> 7)) * p.sf8_kchunks + (dcol >> 7);
  return p.sf8 + chunk * 512 + (row & 31) * 16 + ((row >> 5) & 3) * 4 + ((dcol >> 5) & 3);
}

// QKV + RoPE (+ GELU'd MLP columns) epilogue of ONE 128-column head group whose accumulator row already sits in
// registers.  Used by single-accumulator mainloops (block-scaled fp8, 256-wide tiles): the epilogue warps first drain
// their TMEM slice into registers and hand the accumulator back to the MMA warp, so the next tile's main loop runs
// under this (expensive) math instead of waiting for it - double buffering through the register file.
__device__ __forceinline__ void epilogue_qkv_from_regs(const GemmParams& p, const uint32_t (&acc)[128], int b, int row,
                                                       bool row_ok, int ng) {
  const int qkv_cols = 3 * p.heads * 128;
  if (ng < qkv_cols) {
    const int sec = ng / (p.heads * 128);
    const int head = (ng - sec * p.heads * 128) >> 7;
    float rrms = 1.0f;
    if (sec < 2) {
      float ss = 0.f;
#pragma unroll
      for (int g = 0; g < 16; ++g) {
        float x[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) x[e] = __uint_as_float(acc[g * 8 + e]);
        if (p.bias) {
          float bv[8];
          ldg8(p.bias + ng + g * 8, bv);
#pragma unroll
          for (int e = 0; e < 8; ++e) x[e] += bv[e];
        }
#pragma unroll
        for (int e = 0; e < 8; ++e) ss += x[e] * x[e];
      }
      rrms = rsqrtf(ss * (1.0f / 128.0f) + p.qk_eps);
    }
    __nv_bfloat16* dst_base = (sec == 0 ? p.q : (sec == 1 ? p.k : p.v));
    const long long pos = p.seq_off + row;
    __nv_bfloat16* dst = dst_base + ((static_cast<long long>(b) * p.heads + head) * p.seq_total + pos) * 128;
    const __nv_bfloat16* nw = sec == 0 ? p.q_scale : p.k_scale;
    const bool do_rope = sec < 2 && p.rope != nullptr && row_ok;
#pragma unroll
    for (int g = 0; g < 16; ++g) {
      float x[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) x[e] = __uint_as_float(acc[g * 8 + e]);
      if (p.bias) {
        float bv[8];
        ldg8(p.bias + ng + g * 8, bv);
#pragma unroll
        for (int e = 0; e < 8; ++e) x[e] += bv[e];
      }
      if (sec < 2) {
        float w[8];
        ldg8(nw + g * 8, w);
#pragma unroll
        for (int e = 0; e < 8; ++e) x[e] = x[e] * rrms * w[e];
        if (do_rope) {
          const float4* rp = reinterpret_cast<const float4*>(p.rope + (pos + (row < p.seg_rows ? p.rope_off : p.rope_off2)) * 64 + g * 4);
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            const float4 cs = __ldg(rp + j);     // (cos0, sin0, cos1, sin1)
            const float x0 = x[4 * j], x1 = x[4 * j + 1], x2 = x[4 * j + 2], x3 = x[4 * j + 3];
            x[4 * j] = cs.x * x0 - cs.y * x1;
            x[4 * j + 1] = cs.y * x0 + cs.x * x1;
            x[4 * j + 2] = cs.z * x2 - cs.w * x3;
            x[4 * j + 3] = cs.w * x2 + cs.z * x3;
          }
        }
      }
      if (row_ok) st8(dst + g * 8, x);
    }
  } else {
    // GELU'd MLP columns of a FLUX single block -> concat buffer
    if (p.out8 != nullptr) {
      // ... already quantised to MXFP8 for linear2 (its A operand): half the bytes of the bf16 store, no quantise pass
      const long long dcol = p.out8_col_off + (ng - qkv_cols);
      uint8_t* qrow = p.out8 + b * p.out8_bstride + static_cast<long long>(row) * p.ld8 + dcol;
      uint32_t sfw = 0;
#pragma unroll
      for (int kb = 0; kb < 4; ++kb) {
        float x[32];
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          float bv[8];
          if (p.bias) ldg8(p.bias + ng + kb * 32 + g * 8, bv);
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            float t = __uint_as_float(acc[kb * 32 + g * 8 + e]);
            if (p.bias) t += bv[e];
            x[g * 8 + e] = gelu_tanh(t);
          }
        }
        sfw |= mx_quant32_store(x, qrow + kb * 32, row_ok) << (8 * kb);
      }
      if (row_ok) *reinterpret_cast<uint32_t*>(mx_sf_ptr(p, b, row, dcol)) = sfw;      // 4 K-blocks of one chunk
      return;
    }
    const long long col = p.mlp_col_off + (ng - qkv_cols);
    __nv_bfloat16* orow = p.out + b * p.out_bstride + static_cast<long long>(row) * p.ldc + col;
#pragma unroll
    for (int g = 0; g < 16; ++g) {
      float x[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) x[e] = __uint_as_float(acc[g * 8 + e]);
      if (p.bias) {
        float bv[8];
        ldg8(p.bias + ng + g * 8, bv);
#pragma unroll
        for (int e = 0; e < 8; ++e) x[e] += bv[e];
      }
#pragma unroll
      for (int e = 0; e < 8; ++e) x[e] = gelu_tanh(x[e]);
      if (row_ok) st8(orow + g * 8, x);
    }
  }
}

// The same epilogue for the common case (bias and RoPE table present), written as straight-line code: no per-group
// `if (p.bias)` / `if (do_rope)` control flow, so ptxas can hoist the loads, and the per-lane RoPE rows (the only loads
// that miss L1: 512 B per accumulator row and head) run six column groups ahead of their use.  ncu of the branchy
// version: the eight epilogue warps were busy for the whole tile period, > 40 % of their samples `long_scoreboard` on the
// first use of a just-issued load, tensor pipe 65 % (profiles/r2/ncu_mxfp8_l1_ctapair_run31.txt).
__device__ __forceinline__ void epilogue_qkv_from_regs_fast(const GemmParams& p, uint32_t (&acc)[128], int b, int row,
                                                            bool row_ok, int ng) {
  const int qkv_cols = 3 * p.heads * 128;
  if (ng < qkv_cols) {
    const int sec = ng / (p.heads * 128);
    const int head = (ng - sec * p.heads * 128) >> 7;
    const long long pos = p.seq_off + row;
    __nv_bfloat16* dst_base = (sec == 0 ? p.q : (sec == 1 ? p.k : p.v));
    __nv_bfloat16* dst = dst_base + ((static_cast<long long>(b) * p.heads + head) * p.seq_total + pos) * 128;
    const __nv_bfloat16* bias = p.bias + ng;
    if (sec == 2) {
#pragma unroll
      for (int g = 0; g < 16; ++g) {
        float x[8], bv[8];
        ldg8(bias + g * 8, bv);
#pragma unroll
        for (int e = 0; e < 8; ++e) x[e] = __uint_as_float(acc[g * 8 + e]) + bv[e];
        if (row_ok) st8(dst + g * 8, x);
      }
      return;
    }
    // RoPE row of this accumulator row (rows past the end read row 0 and store nothing)
    const long long rrow = row_ok ? pos + (row < p.seg_rows ? p.rope_off : p.rope_off2) : 0;
    const float4* rp = reinterpret_cast<const float4*>(p.rope + rrow * 64);
    constexpr int RD = 6;                   // column groups of RoPE values in flight per thread
    float4 rb[RD][2];
#pragma unroll
    for (int g = 0; g < RD; ++g) {
      rb[g][0] = __ldg(rp + 2 * g);
      rb[g][1] = __ldg(rp + 2 * g + 1);
    }
    float ss = 0.f;
#pragma unroll
    for (int g = 0; g < 16; ++g) {          // bias folded into the register copy of the accumulator
      float bv[8];
      ldg8(bias + g * 8, bv);
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float x = __uint_as_float(acc[g * 8 + e]) + bv[e];
        acc[g * 8 + e] = __float_as_uint(x);
        ss += x * x;
      }
    }
    const float rrms = rsqrtf(ss * (1.0f / 128.0f) + p.qk_eps);
    const __nv_bfloat16* nw = sec == 0 ? p.q_scale : p.k_scale;
#pragma unroll
    for (int g = 0; g < 16; ++g) {
      const float4 c0 = rb[g % RD][0], c1 = rb[g % RD][1];     // (cos0, sin0, cos1, sin1) x 2
      if (g + RD < 16) {
        rb[g % RD][0] = __ldg(rp + 2 * (g + RD));
        rb[g % RD][1] = __ldg(rp + 2 * (g + RD) + 1);
      }
      float w[8], x[8];
      ldg8(nw + g * 8, w);
#pragma unroll
      for (int e = 0; e < 8; ++e) x[e] = __uint_as_float(acc[g * 8 + e]) * rrms * w[e];
      float y[8];
      y[0] = c0.x * x[0] - c0.y * x[1];
      y[1] = c0.y * x[0] + c0.x * x[1];
      y[2] = c0.z * x[2] - c0.w * x[3];
      y[3] = c0.w * x[2] + c0.z * x[3];
      y[4] = c1.x * x[4] - c1.y * x[5];
      y[5] = c1.y * x[4] + c1.x * x[5];
      y[6] = c1.z * x[6] - c1.w * x[7];
      y[7] = c1.w * x[6] + c1.z * x[7];
      if (row_ok) st8(dst + g * 8, y);
    }
    return;
  }
  if (p.out8 != nullptr) {
    const long long dcol = p.out8_col_off + (ng - qkv_cols);
    uint8_t* qrow = p.out8 + b * p.out8_bstride + static_cast<long long>(row) * p.ld8 + dcol;
    uint32_t sfw = 0;
#pragma unroll
    for (int kb = 0; kb < 4; ++kb) {
      float x[32];
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        float bv[8];
        ldg8(p.bias + ng + kb * 32 + g * 8, bv);
#pragma unroll
        for (int e = 0; e < 8; ++e) x[g * 8 + e] = gelu_tanh(__uint_as_float(acc[kb * 32 + g * 8 + e]) + bv[e]);
      }
      sfw |= mx_quant32_store(x, qrow + kb * 32, row_ok) << (8 * kb);
    }
    if (row_ok) *reinterpret_cast<uint32_t*>(mx_sf_ptr(p, b, row, dcol)) = sfw;
    return;
  }
  const long long col = p.mlp_col_off + (ng - qkv_cols);
  __nv_bfloat16* orow = p.out + b * p.out_bstride + static_cast<long long>(row) * p.ldc + col;
#pragma unroll
  for (int g = 0; g < 16; ++g) {
    float x[8], bv[8];
    ldg8(p.bias + ng + g * 8, bv);
#pragma unroll
    for (int e = 0; e < 8; ++e) x[e] = gelu_tanh(__uint_as_float(acc[g * 8 + e]) + bv[e]);
    if (row_ok) st8(orow + g * 8, x);
  }
}

// Fused epilogue of one accumulator tile (thread == accumulator row `row` of batch `b`; `taddr` = this warp's
// TMEM lane quadrant + accumulator column base; `n0` = first output column of the tile).  Shared by the bf16 and
// the block-scaled fp8 mainloops.
template <int BN>
__device__ __forceinline__ void epilogue_tile(const GemmParams& p, uint32_t taddr, int b, int row, bool row_ok,
                                              int n0) {
  if (p.mode == EPI_QKV_ROPE) {
    const int qkv_cols = 3 * p.heads * 128;
#pragma unroll 1
    for (int hg = 0; hg < BN / 128; ++hg) {
      const int ng = n0 + hg * 128;
      if (ng >= p.N) break;
      if (ng < qkv_cols) {
        const int sec = ng / (p.heads * 128);
        const int head = (ng - sec * p.heads * 128) >> 7;
        float rrms = 1.0f;
        if (sec < 2) {
          float ss = 0.f;
#pragma unroll 1
          for (int c = 0; c < 4; ++c) {
            uint32_t r[32];
            ptx::tmem_ld_32x32b_x32(taddr + hg * 128 + c * 32, r);
            ptx::tmem_ld_wait();
#pragma unroll
            for (int g = 0; g < 4; ++g) {
              float x[8];
              acc8(r, g, p.bias ? p.bias + ng + c * 32 + g * 8 : nullptr, x);
#pragma unroll
              for (int e = 0; e < 8; ++e) ss += x[e] * x[e];
            }
          }
          rrms = rsqrtf(ss * (1.0f / 128.0f) + p.qk_eps);
        }
        __nv_bfloat16* dst_base = (sec == 0 ? p.q : (sec == 1 ? p.k : p.v));
        const long long pos = p.seq_off + row;
        __nv_bfloat16* dst = dst_base + ((static_cast<long long>(b) * p.heads + head) * p.seq_total + pos) * 128;
        const __nv_bfloat16* nw = sec == 0 ? p.q_scale : p.k_scale;
        const bool do_rope = sec < 2 && p.rope != nullptr && row_ok;
#pragma unroll 1
        for (int c = 0; c < 4; ++c) {
          uint32_t r[32];
          ptx::tmem_ld_32x32b_x32(taddr + hg * 128 + c * 32, r);
          ptx::tmem_ld_wait();
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            float x[8];
            acc8(r, g, p.bias ? p.bias + ng + c * 32 + g * 8 : nullptr, x);
            if (sec < 2) {
              float w[8];
              ldg8(nw + c * 32 + g * 8, w);
#pragma unroll
              for (int e = 0; e < 8; ++e) x[e] = x[e] * rrms * w[e];
              if (do_rope) {
                const float4* rp = reinterpret_cast<const float4*>(p.rope + (pos + (row < p.seg_rows ? p.rope_off : p.rope_off2)) * 64 + c * 16 + g * 4);
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                  const float4 cs = __ldg(rp + j);     // (cos0, sin0, cos1, sin1)
                  const float x0 = x[4 * j], x1 = x[4 * j + 1], x2 = x[4 * j + 2], x3 = x[4 * j + 3];
                  x[4 * j] = cs.x * x0 - cs.y * x1;
                  x[4 * j + 1] = cs.y * x0 + cs.x * x1;
                  x[4 * j + 2] = cs.z * x2 - cs.w * x3;
                  x[4 * j + 3] = cs.w * x2 + cs.z * x3;
                }
              }
            }
            if (row_ok) st8(dst + c * 32 + g * 8, x);
          }
        }
      } else {
        // GELU'd MLP columns of a FLUX single block -> concat buffer
        const long long col = p.mlp_col_off + (ng - qkv_cols);
        __nv_bfloat16* orow = p.out + b * p.out_bstride + static_cast<long long>(row) * p.ldc + col;
#pragma unroll 1
        for (int c = 0; c < 4; ++c) {
          uint32_t r[32];
          ptx::tmem_ld_32x32b_x32(taddr + hg * 128 + c * 32, r);
          ptx::tmem_ld_wait();
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            float x[8];
            acc8(r, g, p.bias ? p.bias + ng + c * 32 + g * 8 : nullptr, x);
#pragma unroll
            for (int e = 0; e < 8; ++e) x[e] = gelu_tanh(x[e]);
            if (row_ok) st8(orow + c * 32 + g * 8, x);
          }
        }
      }
    }
  } else if (p.mode == EPI_EULER_UNPATCH) {
    // token `row` = (hh, ww) of the patch grid; column n = (c, ph, pw), ps == 2.
    const int Wp = p.Wl / p.ps;
    const int tokg = row + p.tok_off;
    const int hh = tokg / Wp, ww = tokg - hh * Wp;
    const bool euler = p.sigmas != nullptr;
    float dt = 0.f;
    if (euler) dt = p.sigmas[2 * b + 1] - p.sigmas[2 * b];
    const long long sample_elems = static_cast<long long>(p.C) * p.Hl * p.Wl;
    const long long xin_elems = p.xin_bstride ? p.xin_bstride : sample_elems;
#pragma unroll 1
    for (int c = 0; c < BN / 32; ++c) {
      if (n0 + c * 32 >= p.N) break;
      uint32_t r[32];
      ptx::tmem_ld_32x32b_x32(taddr + c * 32, r);
      ptx::tmem_ld_wait();
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        float x[8];
        acc8(r, g, p.bias ? p.bias + n0 + c * 32 + g * 8 : nullptr, x);
        if (row_ok) {
#pragma unroll
          for (int j = 0; j < 8; j += 2) {     // (pw = 0, 1) are adjacent pixels -> one 4-byte store
            const int n = n0 + c * 32 + g * 8 + j;
            const int ch = n >> 2, ph = (n >> 1) & 1;
            const long long pix = (static_cast<long long>(ch) * p.Hl + (hh * 2 + ph)) * p.Wl + ww * 2;
            float v0 = x[j], v1 = x[j + 1];
            if (euler) {
              const float2 xi = unpack_bf16(*reinterpret_cast<const uint32_t*>(p.x_in + b * xin_elems + pix));
              v0 = xi.x + dt * v0;
              v1 = xi.y + dt * v1;
            }
            *reinterpret_cast<uint32_t*>(p.x_out + (p.xout_sample_off + b) * sample_elems + pix) =
                pack_bf16(v0, v1);
          }
        }
      }
    }
  } else if (p.mode == EPI_GEGLU || p.mode == EPI_SWIGLU) {
    // columns come in groups of 64 = [a(32) | g(32)]; output column = n/2
    __nv_bfloat16* orow = p.out + b * p.out_bstride + static_cast<long long>(row) * p.ldc;
#pragma unroll 1
    for (int c = 0; c < BN / 64; ++c) {
      const int n = n0 + c * 64;
      if (n >= p.N) break;
      uint32_t ra[32], rg[32];
      ptx::tmem_ld_32x32b_x32(taddr + c * 64, ra);
      ptx::tmem_ld_32x32b_x32(taddr + c * 64 + 32, rg);
      ptx::tmem_ld_wait();
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        float a[8], gt[8];
        acc8(ra, g, p.bias ? p.bias + n + g * 8 : nullptr, a);
        acc8(rg, g, p.bias ? p.bias + n + 32 + g * 8 : nullptr, gt);
#pragma unroll
        for (int e = 0; e < 8; ++e) a[e] = a[e] * (p.mode == EPI_GEGLU ? gelu_erf(gt[e]) : gt[e] / (1.0f + __expf(-gt[e])));
        if (row_ok) st8(orow + n / 2 + g * 8, a);
      }
    }
  } else if (p.mode == EPI_BIAS_GELU && p.out8 != nullptr) {
    // GELU + MX quantisation: the 32 columns of one TMEM chunk are exactly one MX block of this thread's row
    uint8_t* qrow = p.out8 + b * p.out8_bstride + static_cast<long long>(row) * p.ld8 + p.out8_col_off;
#pragma unroll 1
    for (int c = 0; c < BN / 32; ++c) {
      const int n = n0 + c * 32;
      if (n >= p.N) break;
      uint32_t r[32];
      ptx::tmem_ld_32x32b_x32(taddr + c * 32, r);
      ptx::tmem_ld_wait();
      float x[32];
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        float t8[8];
        acc8(r, g, p.bias ? p.bias + n + g * 8 : nullptr, t8);
#pragma unroll
        for (int e = 0; e < 8; ++e) x[g * 8 + e] = gelu_tanh(t8[e]);
      }
      const uint32_t sb = mx_quant32_store(x, qrow + n, row_ok);
      if (row_ok) *mx_sf_ptr(p, b, row, p.out8_col_off + n) = static_cast<uint8_t>(sb);
    }
  } else {
    __nv_bfloat16* orow = p.out + b * p.out_bstride + static_cast<long long>(row) * p.ldc;
    const __nv_bfloat16* rrow =
        p.residual ? p.residual + b * p.res_bstride + static_cast<long long>(row) * p.ldr : nullptr;
    // per-frame gates: the group of THIS thread's row (a 128-row tile spans several frames)
    const int gb = p.gate_rows ? (b * p.rows + row + p.gate_row_off) / p.gate_rows : b;
    const __nv_bfloat16* grow = p.gate ? p.gate + gb * p.gate_bstride : nullptr;
#pragma unroll 1
    for (int c = 0; c < BN / 32; ++c) {
      const int n = n0 + c * 32;
      if (n >= p.N) break;
      uint32_t r[32];
      ptx::tmem_ld_32x32b_x32(taddr + c * 32, r);
      ptx::tmem_ld_wait();
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        float x[8];
        acc8(r, g, p.bias ? p.bias + n + g * 8 : nullptr, x);
        if (p.mode == EPI_BIAS_GELU) {
#pragma unroll
          for (int e = 0; e < 8; ++e) x[e] = gelu_tanh(x[e]);
        } else if (p.mode == EPI_BIAS_GELU_ERF) {
#pragma unroll
          for (int e = 0; e < 8; ++e) x[e] = gelu_erf(x[e]);
        } else if (p.mode == EPI_BIAS_SILU) {
#pragma unroll
          for (int e = 0; e < 8; ++e) x[e] = silu(x[e]);
        } else if (p.mode == EPI_BIAS_BCAST) {
          float gv[8];
          ldg8(grow + n + g * 8, gv);
#pragma unroll
          for (int e = 0; e < 8; ++e) x[e] += gv[e];
        } else if ((p.mode == EPI_GATE_RES || p.mode == EPI_RES) && row_ok) {
          float res[8];
          ld8(rrow + n + g * 8, res);
          if (p.mode == EPI_GATE_RES) {
            float gv[8];
            ldg8(grow + n + g * 8, gv);
#pragma unroll
            for (int e = 0; e < 8; ++e) x[e] = res[e] + gv[e] * x[e];
          } else {
#pragma unroll
            for (int e = 0; e < 8; ++e) x[e] = res[e] + x[e];
          }
        }
        if (row_ok) st8(orow + n + g * 8, x);
      }
    }
  }
}

template <int BN>
__global__ void __launch_bounds__(384, 1)
gemm_bf16_tcgen05_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                         const GemmParams p) {
  using Cfg = GemmCfg<BN>;
  constexpr int BM = Cfg::BM, BK = Cfg::BK, STAGES = Cfg::STAGES;
  constexpr uint32_t IDESC = ptx::make_idesc_f16(BM, BN);

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + STAGES * Cfg::STAGE_BYTES);
  uint64_t* empty = full + STAGES;
  uint64_t* tfull = empty + STAGES;
  uint64_t* tempty = tfull + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

  const int warp = threadIdx.x >> 5;
  const int warp_u = __shfl_sync(0xffffffffu, warp, 0);      // provably warp-uniform role index
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmA);
    ptx::prefetch_tmap(&tmB);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      ptx::mbar_init(&full[s], 1);
      ptx::mbar_init(&empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      ptx::mbar_init(&tfull[a], 1);
      ptx::mbar_init(&tempty[a], 8);          // one arrive per epilogue warp
    }
    ptx::fence_barrier_init();
    ptx::fence_proxy_async_smem();
  }
  if (warp == 2) ptx::tmem_alloc<Cfg::TMEM_COLS>(tmem_slot);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const bool conv = p.conv_taps > 0;
  const int m_per_batch = conv ? p.conv_tiles_w * p.conv_tiles_h : (p.rows + BM - 1) / BM;
  const int num_m = m_per_batch * p.batch;
  const int num_n = (p.N + BN - 1) / BN;
  const int num_tiles = num_m * num_n;
  const int num_k = conv ? p.conv_taps * p.conv_cblocks : (p.K + BK - 1) / BK;
  constexpr int GROUP_M = 8;

  auto decode = [&](int t, int& mt, int& nt) {
    const int per_group = GROUP_M * num_n;
    const int g = t / per_group;
    const int first = g * GROUP_M;
    const int gsz = min(num_m - first, GROUP_M);
    const int r = t - g * per_group;
    mt = first + r % gsz;
    nt = r / gsz;
  };

  if (warp_u == 0) {
    // ===================== TMA producer (whole warp, one elected lane issues; see the MMA role) =====================
    const bool leader = ptx::elect_one();
    const uint32_t smem_u = __shfl_sync(0xffffffffu, ptx::smem_u32(smem), 0);
    int stage = 0;
    uint32_t phase = 0;
    for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
      int mt, nt;
      decode(t, mt, nt);
      const int b = mt / m_per_batch, mrow = (mt - b * m_per_batch) * BM;
      int h0 = 0, w0 = 0;
      if (conv) {
        const int t_in = mt - b * m_per_batch;
        const int ti_h = t_in / p.conv_tiles_w;
        h0 = ti_h * p.conv_th * p.conv_stride - p.conv_pad;
        w0 = (t_in - ti_h * p.conv_tiles_w) * p.conv_tw * p.conv_stride - p.conv_pad;
      }
      for (int kb = 0; kb < num_k; ++kb) {
        ptx::mbar_wait(&empty[stage], phase ^ 1);
        if (leader) {
          ptx::mbar_arrive_expect_tx(&full[stage], Cfg::STAGE_BYTES);
          const uint32_t sa = smem_u + stage * Cfg::STAGE_BYTES;
          if (conv) {
            const int tap = kb / p.conv_cblocks, cb = kb - tap * p.conv_cblocks;
            const int kh = p.conv_taps == 9 ? tap / 3 : 0, kw = p.conv_taps == 9 ? tap - kh * 3 : 0;
            ptx::tma_load_4d_s(sa, &tmA, &full[stage], cb * BK, w0 + kw, h0 + kh, b);
          } else {
            ptx::tma_load_3d_s(sa, &tmA, &full[stage], kb * BK, mrow, b);
          }
          ptx::tma_load_2d_s(sa + Cfg::A_BYTES, &tmB, &full[stage], kb * BK, nt * BN);
        }
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
    }
    __syncwarp();
  } else if (warp_u == 1) {
    // ===================== MMA issuer =====================
    // Whole warp, warp-uniform values, one elected lane issues: inside a `lane == 0` branch ptxas wraps every
    // UTCHMMA in an ELECT / R2UR.BROADCAST / BRA.U.ANY waterfall (~90 cycles per MMA - slower than a 128x128x16 MMA
    // executes); with uniform descriptors the MMAs issue back to back from uniform registers.
    const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
    const uint32_t smem_u = __shfl_sync(0xffffffffu, ptx::smem_u32(smem), 0);
    const bool leader = ptx::elect_one();
    int stage = 0;
    uint32_t phase = 0;
    int it = 0;
    for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++it) {
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      ptx::mbar_wait(&tempty[acc], acc_phase ^ 1);
      ptx::tc_fence_after();
      const uint32_t d_tmem = tmem_u + acc * BN;
      for (int kb = 0; kb < num_k; ++kb) {
        ptx::mbar_wait(&full[stage], phase);
        ptx::tc_fence_after();
        if (leader) {
          const uint32_t sa = smem_u + stage * Cfg::STAGE_BYTES;
          const uint64_t adesc = ptx::make_desc_kmajor_sw128(sa);
          const uint64_t bdesc = ptx::make_desc_kmajor_sw128(sa + Cfg::A_BYTES);
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            // +32 bytes per K=16 slice inside the 128-byte swizzle row (descriptor address unit = 16 B)
            ptx::mma_f16_ss(d_tmem, adesc + 2 * k, bdesc + 2 * k, IDESC, (kb | k) != 0 ? 1u : 0u);
          }
          ptx::tc_commit(&empty[stage]);
          if (kb == num_k - 1) ptx::tc_commit(&tfull[acc]);
        }
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
    }
    __syncwarp();
  } else if (warp >= 4) {
    // ===================== epilogue (8 warps, thread == accumulator row x column half) =====================
    const int q4 = warp & 3;                       // TMEM lane quadrant this warp may read
    const int half = (warp - 4) >> 2;              // which part of the accumulator columns (see GemmCfg::EPI_H0/H1)
    const int r_in_tile = q4 * 32 + lane;
    int it = 0;
    for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++it) {
      int mt, nt;
      decode(t, mt, nt);
      const int b = mt / m_per_batch;
      int row = (mt - b * m_per_batch) * BM + r_in_tile;
      bool row_ok = row < p.rows;
      if (conv) {
        const int t_in = mt - b * m_per_batch;
        const int ti_h = t_in / p.conv_tiles_w;
        const int rh = r_in_tile / p.conv_tw;
        const int oh = ti_h * p.conv_th + rh;
        const int ow = (t_in - ti_h * p.conv_tiles_w) * p.conv_tw + (r_in_tile - rh * p.conv_tw);
        row_ok = oh < p.conv_ho && ow < p.conv_wo;
        row = oh * p.conv_wo + ow;
      }
      const int n0 = nt * BN;
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      ptx::mbar_wait(&tfull[acc], acc_phase);
      ptx::tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q4 * 32) << 16) + acc * BN;

      if (half == 0) {
        epilogue_tile<Cfg::EPI_H0>(p, taddr, b, row, row_ok, n0);
      } else if (Cfg::EPI_H1 > 0 && n0 + Cfg::EPI_H0 < p.N) {
        epilogue_tile<(Cfg::EPI_H1 > 0 ? Cfg::EPI_H1 : 32)>(p, taddr + Cfg::EPI_H0, b, row, row_ok, n0 + Cfg::EPI_H0);
      }
      // accumulator drained: hand it back to the MMA warp
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&tempty[acc]);
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc<Cfg::TMEM_COLS>(tmem_base);
  }
}

}  // namespace pa
