// Host-callable entry points of the native library (plain C++ signatures, no torch headers, so the
// .cu files compile in seconds; csrc/bind.cpp adapts them to torch tensors).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace pa {

struct GemmParams;
struct ScatterEmbedParams;
struct ScatterConvParams;
int scatter_conv_in(const void* W, long long ldw, const ScatterConvParams& p, cudaStream_t st);
int scatter_patch_embed(const void* W, long long ldw, const ScatterEmbedParams& p, cudaStream_t st);

int multimem_bcast(const void* src, void* mc_dst, long long bytes, cudaStream_t st);
struct SpPullDesc;
int sp_signal(uint32_t* const* peer_flags, int n_peers, int slot, int me, const uint32_t* epoch, cudaStream_t st);
int sp_pull(const SpPullDesc* descs, int n_desc, int blocks_per_desc, const uint32_t* flags, int slot, int n_peers,
            const uint32_t* epoch, long long timeout, uint32_t* err, cudaStream_t st);
int sp_epoch_inc(uint32_t* epoch, cudaStream_t st);
int num_sms();
void set_sm_limit(int n);   // per-thread SM budget for persistent-kernel grids (0 = all)
int make_tmap(CUtensorMap* out, const void* ptr, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
              const uint32_t* box, int elem_bytes, const uint32_t* elem_strides = nullptr, bool swizzle128 = true);
int conv_bf16(const void* x, int N, int H, int W, int Cin, const void* w, int taps, int stride, GemmParams p,
              cudaStream_t st);

int gemm_bf16(const void* A, long long lda, long long a_bstride, const void* W, long long ldw, GemmParams p,
              int force_bn, cudaStream_t st);

// block-scaled FP8 (MXFP8) GEMM + quantiser (csrc/kernels/gemm_mxfp8.cu)
int quantize_mxfp8_rows(const void* x, long long ldx, long long x_bs, void* q, void* sf, int batch, int rows, int K,
                        int tile_rows, cudaStream_t st);
int gemm_mxfp8(const void* A, const void* sfa, const void* W, const void* sfb, GemmParams p, int w_tile,
               cudaStream_t st, int pair = -1, long long a_bstride = 0);   // a_bstride: bytes between batch entries of A (0: rows*K)   // pair: -1 auto, 0 one CTA per tile, 1 CTA pairs (single accumulator for 256-wide tiles), 2 CTA pairs + split-N accumulators

// out = LN(x) * (1 + scale[b]) + shift[b]   (scale/shift optional; gamma/beta optional affine)
int rmsnorm_mod(const void* x, long long ldx, long long x_bs, void* out, long long ldo, long long o_bs,
                const void* weight, const void* scale, const void* gate, long long mod_bs, const void* residual,
                long long ldr, long long r_bs, int batch, int rows, int D, float eps, int tanh_gate, cudaStream_t st);
int layernorm_modulate_fp8(const void* x, long long ldx, long long x_bs, void* q8, void* sf8, const void* scale,
                           const void* shift, long long mod_bs, int batch, int rows, int D, float eps, cudaStream_t st);
int layernorm_modulate(const void* x, long long ldx, long long x_bstride, void* out, long long ldo,
                       long long o_bstride, const void* scale, const void* shift, long long mod_bstride,
                       const void* gamma, const void* beta, int batch, int rows, int D, float eps, int mod_rows,
                       int mod_row_off, cudaStream_t st);   // scale/shift row = b, or (b*rows + r + mod_row_off) / mod_rows

// sinusoidal embedding: out[b, :] = [cos(t*f_i) | sin(t*f_i)], f_i = exp(-ln(max_period) * i / half)
int timestep_embedding(const void* t, void* out, long long ldo, int B, int dim, float time_factor,
                       float max_period, int t_is_bf16, cudaStream_t st);

// x[b, c, H, W] (NCHW latent, possibly on a peer GPU) -> tokens[b, (h w), (c ph pw)]
int patchify(const void* x, void* out, long long ldo, long long o_bstride, int B, int C, int H, int W, int ps,
             cudaStream_t st);

// layout / glue for the convolutional executors (csrc/kernels/layout.cu)
int nchw_to_nhwc_pad(const void* x, void* out, int B, int C, int HW, int Cpad, cudaStream_t st);
int upsample_nearest2x_nhwc(const void* x, void* out, int B, int H, int W, int C, cudaStream_t st);
int concat_channels(const void* a, const void* b, void* out, long long rows, int C1, int C2, cudaStream_t st);
int unet_out_gather(const void* eps, const void* x, void* x_out, const void* sigmas, int n, int C, int HW, int Cpad,
                    int cfg_pairs, float cfg, int mode, long long out_sample_off, cudaStream_t st);

int rms_rope_inplace(void* x, long long ldx, long long x_bs, const void* w, const void* rope, int batch, int rows,
                     int D, float eps, cudaStream_t st);
int bcast_add(const void* a, const void* m, void* out, int B, int nblk, int n, cudaStream_t st);

int softmax_rows(void* x, long long ld, int rows, int n, float scale, cudaStream_t st);

// elementwise helpers
int silu_bf16(const void* x, void* out, long long n, cudaStream_t st);
int add_bf16(const void* a, const void* b, void* out, long long n, cudaStream_t st);

// fused attention (head_dim 64 / 128, bf16): q,k,v [B, H, L, D] strided views -> out[b, l, h*D + d]
int attention_bf16(const void* q, const void* k, const void* v, void* out, long long ldo, long long o_bstride, int B,
                   int H, int Lq, int Lk, int D, const long long* q_strides, const long long* k_strides,
                   const long long* v_strides, float scale, cudaStream_t st);

int attention2_trace_read(long long* host);
int attention3_trace_read(long long* host);
// CTA-pair ping-pong variant (csrc/kernels/attention3.cu, head dim 128 only); same contract
int attention3_bf16(const void* q, const void* k, const void* v, void* out, long long ldo, long long o_bstride, int B,
                    int H, int Lq, int Lk, int D, const long long* q_strides, const long long* k_strides,
                    const long long* v_strides, float scale, cudaStream_t st);
// ping-pong variant (two query tiles per CTA, csrc/kernels/attention2.cu); same contract
int attention2_bf16(const void* q, const void* k, const void* v, void* out, long long ldo, long long o_bstride, int B,
                    int H, int Lq, int Lk, int D, const long long* q_strides, const long long* k_strides,
                    const long long* v_strides, float scale, cudaStream_t st);
// two key/value sources (head dim 128): out = softmax(q k^T) v + softmax(q k2^T) v2, one launch
int attention2_kv2_bf16(const void* q, const void* k, const void* v, const void* k2, const void* v2, void* out,
                        long long ldo, long long o_bstride, int B, int H, int Lq, int Lk, int Lk2,
                        const long long* q_strides, const long long* k_strides, const long long* v_strides,
                        const long long* k2_strides, const long long* v2_strides, float scale, cudaStream_t st);

// small-KV cross-attention (Lk <= 128, head_dim 64): a CTA pair shares one multicast K/V tile (csrc/kernels/xattn_cluster.cu)
int xattn_cluster_bf16(const void* q, const void* k, const void* v, void* out, long long ldo, long long o_bstride, int B,
                       int H, int Lq, int Lk, int D, const long long* q_strides, const long long* k_strides,
                       const long long* v_strides, float scale, cudaStream_t st);
int attention2_fp8out(const void* q, const void* k, const void* v, void* out8, void* sf8, long long ld8, long long rows8,
                      int B, int H, int Lq, int Lk, const long long* qs, const long long* ks, const long long* vs,
                      float scale, cudaStream_t st);
int attention2_debug(const void* q, const void* k, const void* v, void* out, long long ldo, long long o_bstride, int B,
                     int H, int Lq, int Lk, int dbg, const long long* q_strides, const long long* k_strides,
                     const long long* v_strides, float scale, cudaStream_t st);

// GroupNorm (+ optional SiLU) on NHWC bf16
int groupnorm_silu_nhwc_cluster(const void* x, void* out, const void* gamma, const void* beta, int B, int HW, int C,
                                int groups, float eps, int apply_silu, cudaStream_t st);
int groupnorm_silu_nhwc_ws(const void* x, void* out, const void* gamma, const void* beta, float* workspace, int B,
                           int HW, int C, int groups, float eps, int apply_silu, cudaStream_t st);

// CFG + Euler update + peer store (elementwise "gather" for models whose last op is not a GEMM)
int cfg_euler_store(const void* x, const void* eps_cond, const void* eps_uncond, void* x_out, const void* sigmas,
                    float cfg_scale, long long n_per_sample, int batch, long long out_sample_off, int mode,
                    cudaStream_t st);

// flag words (release/acquire at .sys scope) for the cross-GPU step protocol
int signal_flags(uint32_t* const* peer_flag_ptrs, int n_peers, int slot, uint32_t value, cudaStream_t st);
int wait_flags(const uint32_t* flags, int first_slot, int n_slots, uint32_t value, long long timeout_cycles,
               uint32_t* error_word, cudaStream_t st);

}  // namespace pa
