// Parameter block of the fused scatter + patch-embed kernel (shared with the host binding).
#pragma once
#include <cuda_bf16.h>

namespace pa {

struct ScatterEmbedParams {
  const __nv_bfloat16* x_src;     // [n, C, Hl, Wl] at the lead (peer mapping or local)
  const __nv_bfloat16* t_src;     // [n_t]
  const __nv_bfloat16* g_src;     // [n] or nullptr
  __nv_bfloat16* t_emb;           // [n_t, 256]
  __nv_bfloat16* g_emb;           // [n, 256]
  __nv_bfloat16* x_copy;          // optional local copy of the latent shard (for the Euler epilogue)
  __nv_bfloat16* out;             // X[:, Lt:, :]
  long long ldo, out_bstride;
  const __nv_bfloat16* bias;      // [N]
  int n, C, Hl, Wl, N, Li;
  int n_t;                        // timesteps to embed: n, or n * T with one per video frame (WAN2.2 TI2V)
  float time_factor;
  int nsplit;                     // CTAs sharing one token tile, each owning a slice of the N weight tiles (set by the launcher)
};

}  // namespace pa

namespace pa {

// Fused scatter + first 3x3 convolution (UNet ``conv_in``) + timestep sinusoid.
struct ScatterConvParams {
  const __nv_bfloat16* x_src;     // [n, C, H, W] at the lead (peer mapping or local), NCHW
  const __nv_bfloat16* t_src;     // [n] timesteps at the lead (or local)
  __nv_bfloat16* t_emb;           // [n, temb_dim]  (cos | sin)
  __nv_bfloat16* x_copy;          // optional local NCHW copy of the shard (x_in of the Euler gather)
  __nv_bfloat16* out;             // [n, H*W, N] NHWC rows
  const __nv_bfloat16* bias;      // [N]
  int n, C, H, W, N, temb_dim;
  float time_factor, max_period;
};

}  // namespace pa
