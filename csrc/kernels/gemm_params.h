// GEMM epilogue modes + parameter block shared by device code and the host binding.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>

namespace pa {

enum EpiMode : int {
  EPI_BIAS = 0,
  EPI_BIAS_GELU = 1,
  EPI_BIAS_SILU = 2,
  EPI_GATE_RES = 3,     // out = residual + gate[b, n] * (acc + bias)
  EPI_QKV_ROPE = 4,     // N = 3*H*128 (+ mlp columns when mlp_cols > 0)
  EPI_EULER_UNPATCH = 5,// N = C*ps*ps : velocity -> x_next written in NCHW, possibly to a peer
  EPI_GEGLU = 6,        // W rows interleaved [a(32) | g(32)]...: out[:, n/2] = a * gelu(g)
  EPI_RES = 7,          // out = residual + acc + bias
  EPI_BIAS_BCAST = 8,   // out = acc + bias + gate[b, n]   (per-sample channel bias, e.g. time embedding)
  EPI_SWIGLU = 9,       // same interleaving as EPI_GEGLU: out[:, n/2] = a * silu(g)
  EPI_BIAS_GELU_ERF = 10,  // out = gelu(acc + bias), exact erf form (nn.GELU()); EPI_BIAS_GELU is the tanh form
};

struct GemmParams {
  int rows;          // rows per batch
  int batch;
  int N, K;
  int mode;
  // generic output
  __nv_bfloat16* out;
  long long ldc, out_bstride;
  const __nv_bfloat16* bias;        // [N] or nullptr
  const __nv_bfloat16* residual;    // EPI_GATE_RES / EPI_RES
  long long ldr, res_bstride;
  const __nv_bfloat16* gate;        // [batch, N] with stride gate_bstride
  long long gate_bstride;
  // EPI_GATE_RES with gate_rows > 0: the gate row of (sample b, row r) is (b * rows + r + gate_row_off) / gate_rows
  // instead of b (one gate vector per video frame; gate_row_off = global token index of row 0 of a token slice)
  int gate_rows, gate_row_off;
  // Fused MXFP8 output (the NEXT GEMM's A operand, written by this epilogue instead of bf16 + a quantise kernel):
  // EPI_BIAS_GELU: every column; EPI_QKV_ROPE: the GELU'd MLP columns.  e4m3 bytes row-major [batch, rows8, ld8]
  // plus UE8M0 scale chunks in the layout of gemm_mxfp8.cu (128-row x 128-column chunks of 512 bytes).
  uint8_t* out8;                    // nullptr = bf16 output as usual
  uint8_t* sf8;
  long long ld8, out8_bstride;      // row length / batch stride in bytes
  long long out8_col_off;           // destination column of the first fp8 column (multiple of 32)
  int sf8_mtiles, sf8_kchunks;      // 128-row tiles per batch, ld8 / 128
  // QKV
  __nv_bfloat16 *q, *k, *v;         // [batch, H, seq_total, 128]
  const __nv_bfloat16 *q_scale, *k_scale;   // [128] RMSNorm weights
  const float2* rope;               // [seq_total, 64] (cos, sin); nullptr = no rope
  int heads, seq_off, seq_total;
  // RoPE row = destination row + rope_off (rows < seg_rows) or + rope_off2 (rows >= seg_rows): sequence-parallel replicas
  // keep a LOCAL [txt slice | img slice] token layout whose global positions are two separate ranges
  int rope_off, rope_off2, seg_rows;
  int mlp_cols;                     // columns after the 3*H*128 qkv columns (FLUX single blocks)
  long long mlp_col_off;            // where they start inside `out`
  float qk_eps;
  // Euler / unpatchify epilogue (the fused "gather")
  const __nv_bfloat16* x_in;        // local latent shard  [batch, C, Hl, Wl]
  __nv_bfloat16* x_out;             // destination (lead GPU buffer, possibly a peer mapping)
  long long xout_sample_off;        // first sample of this rank inside x_out
  long long xin_bstride;            // elements per sample of x_in (0: C*Hl*Wl); a wider input (WAN I2V: noise | mask |
                                    // image latent) is updated from its first C channels
  const float* sigmas;              // [batch, 2] (sigma, sigma_next) per sample, or nullptr => out = v
  int C, Hl, Wl, ps;
  int sfa_mtiles;                   // block-scaled fp8: 128-row scale chunks per batch entry of the A operand's buffer (0: ceil(rows/128));
                                    // lets a row range of a larger [B, L, K] buffer (txt / img rows of the joint attention output) be an operand
  int tok_off;                      // EULER_UNPATCH: global token index of row 0 (sequence-parallel replicas own a token range)
  // implicit-GEMM convolution: A is an NHWC activation addressed through a 4-D TMA tensor
  // (C, W, H, N); the K loop walks taps x Cin-blocks with shifted spatial coordinates, padding
  // comes from TMA out-of-bounds zero fill.  rows = Ho*Wo, batch = N.
  int conv_taps;             // 0 = plain GEMM, 1 (1x1) or 9 (3x3)
  int conv_cblocks;          // ceil(Cin / 64)
  int conv_tw, conv_th;      // spatial tile, tw * th == 128
  int conv_wo, conv_ho;      // output size
  int conv_stride, conv_pad;
  int conv_tiles_w, conv_tiles_h;
};

}  // namespace pa
