// torch <-> native library glue.  Everything below adapts at::Tensor arguments (pointers, strides, the
// current CUDA stream) to the plain C++ entry points in common/host.h.
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>
#include <torch/extension.h>

#include <cstdlib>

#include "common/host.h"
#include "comm/scatter_params.h"
#include "comm/sp_params.h"
#include "kernels/gemm_params.h"
#include "runtime/runtime.h"

namespace py = pybind11;
using at::Tensor;

static cudaStream_t cur_stream() { return at::cuda::getCurrentCUDAStream().stream(); }

static void check(int rc, const char* what) {
  TORCH_CHECK(rc == 0, "[pa] ", what, " failed with code ", rc, " (", rc > 0 ? cudaGetErrorString((cudaError_t)rc) : "argument error", ")");
}

static bool has(const py::kwargs& kw, const char* k) { return kw.contains(k) && !kw[k].is_none(); }
static Tensor ten(const py::kwargs& kw, const char* k) { return kw[k].cast<Tensor>(); }
static const __nv_bfloat16* bfp(const py::kwargs& kw, const char* k) {
  if (!has(kw, k)) return nullptr;
  Tensor t = ten(kw, k);
  TORCH_CHECK(t.is_cuda() && t.scalar_type() == at::kBFloat16, k, " must be a CUDA bf16 tensor");
  return reinterpret_cast<const __nv_bfloat16*>(t.data_ptr());
}

// views: 2-D [M, K] or 3-D [B, rows, K], innermost stride 1
static void view3(const Tensor& t, int& batch, int& rows, long long& ld, long long& bs) {
  TORCH_CHECK(t.dim() == 2 || t.dim() == 3, "expected a 2-D or 3-D tensor");
  TORCH_CHECK(t.stride(-1) == 1, "innermost dimension must be contiguous");
  if (t.dim() == 2) {
    batch = 1; rows = (int)t.size(0); ld = t.stride(0); bs = (long long)t.size(0) * t.stride(0);
  } else {
    batch = (int)t.size(0); rows = (int)t.size(1); ld = t.stride(1); bs = t.stride(0);
  }
}

// out= / bias= / residual= / gate= (shared by gemm and conv)
static void parse_epilogue(const py::kwargs& kw, pa::GemmParams& p, bool check_shape) {
  if (has(kw, "out")) {
    Tensor o = ten(kw, "out");
    int ob, orows;
    view3(o, ob, orows, p.ldc, p.out_bstride);
    TORCH_CHECK(!check_shape || (ob == p.batch && orows == p.rows), "out shape mismatch");
    p.out = reinterpret_cast<__nv_bfloat16*>(o.data_ptr());
  }
  p.bias = bfp(kw, "bias");
  if (has(kw, "residual")) {
    Tensor r = ten(kw, "residual");
    int rb, rr;
    view3(r, rb, rr, p.ldr, p.res_bstride);
    p.residual = reinterpret_cast<const __nv_bfloat16*>(r.data_ptr());
  }
  if (has(kw, "gate")) {
    Tensor g = ten(kw, "gate");
    TORCH_CHECK(g.stride(-1) == 1, "gate must be contiguous in its last dim");
    p.gate = reinterpret_cast<const __nv_bfloat16*>(g.data_ptr());
    p.gate_bstride = g.dim() >= 2 ? g.stride(0) : 0;
    if (has(kw, "gate_rows")) {
      // one gate vector per group of gate_rows rows (video frames): the last row's group must be a row of `gate`
      p.gate_rows = kw["gate_rows"].cast<int>();
      p.gate_row_off = has(kw, "gate_row_off") ? kw["gate_row_off"].cast<int>() : 0;
      TORCH_CHECK(p.mode == pa::EPI_GATE_RES, "gate_rows needs the gate_res epilogue");
      TORCH_CHECK(p.gate_rows > 0 && p.gate_row_off >= 0, "gate_rows must be > 0, gate_row_off >= 0");
      TORCH_CHECK(g.dim() == 2, "gate_rows needs a 2-D [groups, N] gate view");
      TORCH_CHECK(((long long)p.batch * p.rows - 1 + p.gate_row_off) / p.gate_rows < g.size(0),
                  "gate_rows: the last row's group is outside the gate's ", g.size(0), " rows");
    }
  }
  if (has(kw, "out8")) {
    // fused MXFP8 output: e4m3 bytes [batch, rows8, ld8] contiguous + scale chunks; written at column out8_col_off
    Tensor o8 = ten(kw, "out8");
    Tensor s8 = ten(kw, "sf8");
    TORCH_CHECK(o8.element_size() == 1 && s8.element_size() == 1 && o8.is_contiguous() && s8.is_contiguous() &&
                    o8.dim() == 3, "out8 must be contiguous uint8 [batch, rows, K], sf8 contiguous uint8");
    TORCH_CHECK(o8.size(0) == p.batch && o8.size(1) >= p.rows && o8.size(2) % 128 == 0, "out8 shape mismatch");
    p.out8 = reinterpret_cast<uint8_t*>(o8.data_ptr());
    p.sf8 = reinterpret_cast<uint8_t*>(s8.data_ptr());
    p.ld8 = o8.size(2);
    p.out8_bstride = o8.size(1) * o8.size(2);
    p.sf8_mtiles = (int)((o8.size(1) + 127) / 128);
    p.sf8_kchunks = (int)(o8.size(2) / 128);
    p.out8_col_off = has(kw, "out8_col_off") ? kw["out8_col_off"].cast<long long>() : 0;
    TORCH_CHECK(p.out8_col_off % 32 == 0, "out8_col_off must be a multiple of 32");
    TORCH_CHECK(s8.numel() >= (int64_t)p.batch * p.sf8_mtiles * p.sf8_kchunks * 512, "sf8 too small");
  }
}

// gemm(A, W, mode, out=..., bias=..., residual=..., gate=..., q=,k=,v=,q_scale=,k_scale=,rope=,heads=,seq_off=,
//      mlp_col_off=, qk_eps=, x_in=, xin_bstride=, x_out= | x_out_ptr=, xout_sample_off=, sigmas=, C=,Hl=,Wl=, force_bn=)
static void parse_modes(int mode, const py::kwargs& kw, pa::GemmParams& p);

static void gemm(Tensor A, Tensor W, int mode, py::kwargs kw) {
  TORCH_CHECK(A.is_cuda() && W.is_cuda(), "gemm: CUDA tensors required");
  TORCH_CHECK(A.scalar_type() == at::kBFloat16 && W.scalar_type() == at::kBFloat16, "gemm: bf16 required");
  TORCH_CHECK(W.dim() == 2 && W.stride(1) == 1, "gemm: W must be [N, K] with contiguous K");
  c10::cuda::CUDAGuard guard(A.device());
  pa::GemmParams p{};
  long long lda, abs_;
  view3(A, p.batch, p.rows, lda, abs_);
  p.N = (int)W.size(0);
  p.K = (int)W.size(1);
  TORCH_CHECK(A.size(-1) == p.K, "gemm: K mismatch");
  p.mode = mode;
  parse_epilogue(kw, p, /*check_shape=*/true);
  parse_modes(mode, kw, p);
  int force_bn = has(kw, "force_bn") ? kw["force_bn"].cast<int>() : 0;
  check(pa::gemm_bf16(A.data_ptr(), lda, abs_, W.data_ptr(), W.stride(0), p, force_bn, cur_stream()), "gemm_bf16");
}

// MXFP8: A_q / W_q are uint8 (e4m3 bit patterns) contiguous, sfa / sfb uint8 scale chunks (see gemm_mxfp8.cu)
static void gemm_fp8(Tensor A, Tensor sfa, Tensor W, Tensor sfb, int mode, int w_tile, py::kwargs kw) {
  TORCH_CHECK(A.is_cuda() && W.is_contiguous() && A.element_size() == 1 && W.element_size() == 1 && A.stride(-1) == 1,
              "gemm_fp8: 1-byte operands, contiguous rows required");
  c10::cuda::CUDAGuard guard(A.device());
  pa::GemmParams p{};
  long long lda, abs_;
  view3(A, p.batch, p.rows, lda, abs_);
  p.N = (int)W.size(0);
  p.K = (int)W.size(1);
  TORCH_CHECK(A.size(-1) == p.K, "gemm_fp8: K mismatch");
  // A may be a row range of a larger [B, L, K] buffer (rows contiguous, batch stride L*K): pass `sfa_mtiles` = L/128 and a
  // scale tensor that starts at the range's first 128-row chunk
  TORCH_CHECK(lda == p.K, "gemm_fp8: rows of A must be contiguous (lda == K)");
  p.sfa_mtiles = has(kw, "sfa_mtiles") ? kw["sfa_mtiles"].cast<int>() : 0;
  TORCH_CHECK(p.batch == 1 || abs_ == (long long)p.rows * p.K || p.sfa_mtiles > 0,
              "gemm_fp8: a strided batch needs sfa_mtiles");
  p.mode = mode;
  parse_epilogue(kw, p, /*check_shape=*/true);
  parse_modes(mode, kw, p);
  const int pair = has(kw, "pair") ? kw["pair"].cast<int>() : -1;      // -1 auto | 0 one-CTA kernel | 1 CTA pairs
  check(pa::gemm_mxfp8(A.data_ptr(), sfa.data_ptr(), W.data_ptr(), sfb.data_ptr(), p, w_tile, cur_stream(), pair,
                       p.batch > 1 ? abs_ : 0),
        "gemm_mxfp8");
}

// bf16 [B, rows, K] / [rows, K] view -> (e4m3 bytes [B, rows, K], scale chunks)
static std::vector<Tensor> quantize_mxfp8(Tensor x, int tile_rows) {
  c10::cuda::CUDAGuard guard(x.device());
  TORCH_CHECK(x.scalar_type() == at::kBFloat16, "quantize_mxfp8: bf16 input");
  int b, rows;
  long long ld, bs;
  view3(x, b, rows, ld, bs);
  const int K = (int)x.size(-1);
  TORCH_CHECK(K % 128 == 0, "quantize_mxfp8: K must be a multiple of 128");
  auto o8 = x.options().dtype(at::kByte);
  Tensor q = x.dim() == 2 ? at::empty({rows, K}, o8) : at::empty({b, rows, K}, o8);
  const int64_t chunks = (int64_t)((rows + tile_rows - 1) / tile_rows) * ((tile_rows + 127) / 128);
  Tensor sf = at::zeros({(int64_t)b * chunks * (K / 128) * 512}, o8);
  check(pa::quantize_mxfp8_rows(x.data_ptr(), ld, bs, q.data_ptr(), sf.data_ptr(), b, rows, K, tile_rows,
                                cur_stream()),
        "quantize_mxfp8_rows");
  return {q, sf};
}

static void parse_modes(int mode, const py::kwargs& kw, pa::GemmParams& p) {
  if (mode == pa::EPI_QKV_ROPE) {
    Tensor q = ten(kw, "q");
    TORCH_CHECK(q.dim() == 4 && q.size(3) == 128 && q.is_contiguous(), "q must be [B, H, L, 128] contiguous");
    p.q = reinterpret_cast<__nv_bfloat16*>(q.data_ptr());
    p.k = reinterpret_cast<__nv_bfloat16*>(ten(kw, "k").data_ptr());
    p.v = reinterpret_cast<__nv_bfloat16*>(ten(kw, "v").data_ptr());
    p.q_scale = bfp(kw, "q_scale");
    p.k_scale = bfp(kw, "k_scale");
    TORCH_CHECK(p.q_scale && p.k_scale, "q_scale/k_scale required");
    p.heads = (int)q.size(1);
    p.seq_total = (int)q.size(2);
    p.seq_off = has(kw, "seq_off") ? kw["seq_off"].cast<int>() : 0;
    p.qk_eps = has(kw, "qk_eps") ? kw["qk_eps"].cast<float>() : 1e-6f;
    if (has(kw, "rope")) {
      Tensor r = ten(kw, "rope");
      TORCH_CHECK(r.scalar_type() == at::kFloat && r.is_contiguous() && r.size(-1) == 2 && r.size(-2) == 64,
                  "rope must be float32 [L, 64, 2]");
      p.rope = reinterpret_cast<const float2*>(r.data_ptr());
    }
    p.rope_off = has(kw, "rope_off") ? kw["rope_off"].cast<int>() : 0;
    p.rope_off2 = has(kw, "rope_off2") ? kw["rope_off2"].cast<int>() : p.rope_off;
    p.seg_rows = has(kw, "seg_rows") ? kw["seg_rows"].cast<int>() : 0;
    if (!has(kw, "seg_rows")) p.rope_off2 = p.rope_off;         // one segment: every row uses rope_off
    p.mlp_cols = p.N - 3 * p.heads * 128;
    p.mlp_col_off = has(kw, "mlp_col_off") ? kw["mlp_col_off"].cast<long long>() : 0;
    TORCH_CHECK(p.mlp_cols == 0 || p.out != nullptr || p.out8 != nullptr, "single-block QKV+MLP needs out= or out8=");
  }
  if (mode == pa::EPI_EULER_UNPATCH) {
    p.tok_off = has(kw, "tok_off") ? kw["tok_off"].cast<int>() : 0;
    p.C = kw["C"].cast<int>();
    p.Hl = kw["Hl"].cast<int>();
    p.Wl = kw["Wl"].cast<int>();
    p.ps = 2;
    TORCH_CHECK(p.N == p.C * 4, "EULER_UNPATCH expects N == C*4 (2x2 patches)");
    if (has(kw, "x_in")) p.x_in = bfp(kw, "x_in");
    if (has(kw, "x_out_ptr")) p.x_out = reinterpret_cast<__nv_bfloat16*>(kw["x_out_ptr"].cast<uintptr_t>());
    else p.x_out = reinterpret_cast<__nv_bfloat16*>(ten(kw, "x_out").data_ptr());
    p.xout_sample_off = has(kw, "xout_sample_off") ? kw["xout_sample_off"].cast<long long>() : 0;
    p.xin_bstride = has(kw, "xin_bstride") ? kw["xin_bstride"].cast<long long>() : 0;
    TORCH_CHECK(p.xin_bstride == 0 || p.xin_bstride >= (long long)p.C * p.Hl * p.Wl,
                "xin_bstride must cover the C*Hl*Wl elements the update reads");
    if (has(kw, "sigmas")) {
      Tensor s = ten(kw, "sigmas");
      TORCH_CHECK(s.scalar_type() == at::kFloat && s.is_contiguous(), "sigmas must be float32 [B, 2]");
      p.sigmas = reinterpret_cast<const float*>(s.data_ptr());
      TORCH_CHECK(p.x_in != nullptr, "Euler update needs x_in");
    }
  } else {
    TORCH_CHECK(p.out != nullptr || p.out8 != nullptr || mode == pa::EPI_QKV_ROPE, "gemm: out= (or out8=) required");
  }
}

// conv(x[N,H,W,Cin], w[Cout, taps*Cin_pad], taps, stride, mode, out=[N, Ho*Wo, Cout], bias=, residual=, gate=)
static void conv(Tensor x, Tensor w, int taps, int stride, int mode, py::kwargs kw) {
  TORCH_CHECK(x.is_cuda() && x.dim() == 4 && x.is_contiguous() && x.scalar_type() == at::kBFloat16,
              "conv: x must be a contiguous NHWC bf16 tensor [N, H, W, C]");
  TORCH_CHECK(w.dim() == 2 && w.is_contiguous() && w.scalar_type() == at::kBFloat16, "conv: w must be [Cout, taps*Cin_pad]");
  c10::cuda::CUDAGuard guard(x.device());
  pa::GemmParams p{};
  p.mode = mode;
  p.N = (int)w.size(0);
  const int Cin = (int)x.size(3);
  const int cpad = (Cin + 63) / 64 * 64;
  TORCH_CHECK(w.size(1) == (int64_t)taps * cpad, "conv: weight K must be taps * 64*ceil(Cin/64)");
  parse_epilogue(kw, p, /*check_shape=*/false);
  TORCH_CHECK(p.out != nullptr, "conv: out= required");
  check(pa::conv_bf16(x.data_ptr(), (int)x.size(0), (int)x.size(1), (int)x.size(2), Cin, w.data_ptr(), taps, stride, p,
                      cur_stream()),
        "conv_bf16");
}

// scale / shift: [B, D] views (one vector per sample), or with mod_rows > 0 [G, D] views with one vector per group of
// mod_rows rows: row r of sample b reads vector (b * rows + r + mod_row_off) / mod_rows (video frames)
static void layernorm_modulate(Tensor x, Tensor out, c10::optional<Tensor> scale, c10::optional<Tensor> shift,
                               c10::optional<Tensor> gamma, c10::optional<Tensor> beta, double eps, int mod_rows,
                               int mod_row_off) {
  c10::cuda::CUDAGuard guard(x.device());
  int b, rows, ob, orows;
  long long ldx, xbs, ldo, obs;
  view3(x, b, rows, ldx, xbs);
  view3(out, ob, orows, ldo, obs);
  TORCH_CHECK(b == ob && rows == orows, "layernorm_modulate: shape mismatch");
  long long mod_bs = 0;
  const void *sc = nullptr, *sh = nullptr;
  if (scale) { sc = scale->data_ptr(); mod_bs = scale->dim() >= 2 ? scale->stride(0) : 0; TORCH_CHECK(scale->stride(-1) == 1); }
  if (shift) { sh = shift->data_ptr(); long long s2 = shift->dim() >= 2 ? shift->stride(0) : 0; TORCH_CHECK(!scale || s2 == mod_bs, "scale/shift batch strides differ"); mod_bs = s2; }
  if (mod_rows > 0) {
    TORCH_CHECK(mod_row_off >= 0, "mod_row_off must be >= 0");
    const long long last = ((long long)b * rows - 1 + mod_row_off) / mod_rows;
    for (const c10::optional<Tensor>* m : {&scale, &shift})
      if (*m) TORCH_CHECK((*m)->dim() == 2 && last < (*m)->size(0), "mod_rows: the last row's group ", last,
                          " is outside the [", (*m)->size(0), ", D] scale / shift view");
  } else {
    TORCH_CHECK(mod_rows == 0 && mod_row_off == 0, "mod_row_off needs mod_rows > 0");      // one vector per sample
  }
  check(pa::layernorm_modulate(x.data_ptr(), ldx, xbs, out.data_ptr(), ldo, obs, sc, sh, mod_bs,
                               gamma ? gamma->data_ptr() : nullptr, beta ? beta->data_ptr() : nullptr, b, rows,
                               (int)x.size(-1), (float)eps, mod_rows, mod_row_off, cur_stream()),
        "layernorm_modulate");
}

// LayerNorm + (1 + scale) * . + shift with MXFP8 output: q8 uint8 [B, rows, D] contiguous, sf8 scale chunks
static void layernorm_modulate_fp8(Tensor x, Tensor q8, Tensor sf8, Tensor scale, Tensor shift, double eps) {
  c10::cuda::CUDAGuard guard(x.device());
  int b, rows;
  long long ldx, xbs;
  view3(x, b, rows, ldx, xbs);
  const int D = (int)x.size(-1);
  TORCH_CHECK(q8.is_contiguous() && q8.element_size() == 1 && q8.numel() == (int64_t)b * rows * D, "q8 must be [B, rows, D] uint8");
  TORCH_CHECK(sf8.is_contiguous() && sf8.numel() >= (int64_t)b * ((rows + 127) / 128) * (D / 128) * 512, "sf8 too small");
  TORCH_CHECK(scale.stride(-1) == 1 && shift.stride(-1) == 1);
  const long long mod_bs = scale.dim() >= 2 ? scale.stride(0) : 0;
  TORCH_CHECK((shift.dim() >= 2 ? shift.stride(0) : 0) == mod_bs, "scale/shift batch strides differ");
  check(pa::layernorm_modulate_fp8(x.data_ptr(), ldx, xbs, q8.data_ptr(), sf8.data_ptr(), scale.data_ptr(),
                                   shift.data_ptr(), mod_bs, b, rows, D, (float)eps, cur_stream()),
        "layernorm_modulate_fp8");
}

// out = [residual +] [tanh](gate) * rms(x) * weight * (1 + scale); scale / gate: [B, D] views (or [D]), any may be None
static void rmsnorm_mod(Tensor x, Tensor out, c10::optional<Tensor> weight, c10::optional<Tensor> scale,
                        c10::optional<Tensor> gate, c10::optional<Tensor> residual, double eps, bool tanh_gate) {
  c10::cuda::CUDAGuard guard(x.device());
  int b, rows, ob, orows;
  long long ldx, xbs, ldo, obs, ldr = 0, rbs = 0;
  view3(x, b, rows, ldx, xbs);
  view3(out, ob, orows, ldo, obs);
  TORCH_CHECK(b == ob && rows == orows, "rmsnorm_mod: shape mismatch");
  long long mod_bs = 0;
  const void *sc = nullptr, *gt = nullptr, *rs = nullptr;
  if (scale) { sc = scale->data_ptr(); mod_bs = scale->dim() >= 2 ? scale->stride(0) : 0; TORCH_CHECK(scale->stride(-1) == 1); }
  if (gate) { gt = gate->data_ptr(); long long s2 = gate->dim() >= 2 ? gate->stride(0) : 0; TORCH_CHECK(!scale || s2 == mod_bs, "scale/gate batch strides differ"); mod_bs = s2; TORCH_CHECK(gate->stride(-1) == 1); }
  if (residual) {
    int rb, rr;
    view3(*residual, rb, rr, ldr, rbs);
    TORCH_CHECK(rb == b && rr == rows, "rmsnorm_mod: residual shape mismatch");
    rs = residual->data_ptr();
  }
  check(pa::rmsnorm_mod(x.data_ptr(), ldx, xbs, out.data_ptr(), ldo, obs, weight ? weight->data_ptr() : nullptr, sc, gt,
                        mod_bs, rs, ldr, rbs, b, rows, (int)x.size(-1), (float)eps, tanh_gate ? 1 : 0, cur_stream()),
        "rmsnorm_mod");
}

static void timestep_embedding(Tensor t, Tensor out, double time_factor, double max_period) {
  c10::cuda::CUDAGuard guard(t.device());
  TORCH_CHECK(out.dim() == 2 && out.stride(1) == 1 && out.scalar_type() == at::kBFloat16);
  TORCH_CHECK(t.scalar_type() == at::kBFloat16 || t.scalar_type() == at::kFloat);
  check(pa::timestep_embedding(t.data_ptr(), out.data_ptr(), out.stride(0), (int)out.size(0), (int)out.size(1),
                               (float)time_factor, (float)max_period, t.scalar_type() == at::kBFloat16, cur_stream()),
        "timestep_embedding");
}

static void patchify(uintptr_t x_ptr, Tensor out, int B, int C, int H, int W, int ps) {
  c10::cuda::CUDAGuard guard(out.device());
  int ob, orows;
  long long ldo, obs;
  view3(out, ob, orows, ldo, obs);
  check(pa::patchify(reinterpret_cast<const void*>(x_ptr), out.data_ptr(), ldo, obs, B, C, H, W, ps, cur_stream()),
        "patchify");
}

// Fused scatter: peer latent shard -> patchify -> img_in GEMM (+ bias) -> X[:, Lt:], plus the
// sinusoidal embeddings of the shard's timesteps / guidance values (read from the peer).
// n_t: timesteps to embed into t_emb (0: one per sample; samples x frames with per-frame timesteps)
static void scatter_patch_embed(Tensor W, Tensor bias, uintptr_t x_src, uintptr_t t_src, uintptr_t g_src, Tensor t_emb,
                                c10::optional<Tensor> g_emb, c10::optional<Tensor> x_copy, Tensor out, int C, int Hl,
                                int Wl, double time_factor, int n_t) {
  c10::cuda::CUDAGuard guard(out.device());
  // up to 16 channels the patch is one 64-column K block; wider latents use the plain [N, 4*C] patch reshape
  const int64_t K = C <= 16 ? 64 : 4 * (int64_t)C;
  TORCH_CHECK(W.dim() == 2 && W.size(1) == K && W.stride(1) == 1, "img_in weight must be [N, ", K, "]");
  TORCH_CHECK(C <= 16 || (C <= 64 && C % 2 == 0), "scatter_patch_embed: wide latents need an even C <= 64, got ", C);
  pa::ScatterEmbedParams p{};
  int ob, orows;
  view3(out, ob, orows, p.ldo, p.out_bstride);
  p.x_src = reinterpret_cast<const __nv_bfloat16*>(x_src);
  p.t_src = reinterpret_cast<const __nv_bfloat16*>(t_src);
  p.g_src = reinterpret_cast<const __nv_bfloat16*>(g_src);
  p.t_emb = reinterpret_cast<__nv_bfloat16*>(t_emb.data_ptr());
  p.g_emb = g_emb ? reinterpret_cast<__nv_bfloat16*>(g_emb->data_ptr()) : nullptr;
  TORCH_CHECK(p.g_src == nullptr || p.g_emb != nullptr, "g_emb required with g_src");
  p.x_copy = x_copy ? reinterpret_cast<__nv_bfloat16*>(x_copy->data_ptr()) : nullptr;
  p.out = reinterpret_cast<__nv_bfloat16*>(out.data_ptr());
  p.bias = reinterpret_cast<const __nv_bfloat16*>(bias.data_ptr());
  p.n = ob; p.C = C; p.Hl = Hl; p.Wl = Wl; p.N = (int)W.size(0); p.Li = orows;
  p.n_t = n_t > 0 ? n_t : ob;
  TORCH_CHECK(p.n_t % ob == 0 && (p.g_src == nullptr || p.n_t == ob), "n_t must be a multiple of the ", ob,
              " samples (and equal to it with guidance)");
  TORCH_CHECK(t_emb.numel() >= (int64_t)p.n_t * 256, "t_emb must hold n_t = ", p.n_t, " rows of 256");
  TORCH_CHECK(p.Li == (Hl / 2) * (Wl / 2), "out rows must equal the number of 2x2 patches");
  p.time_factor = (float)time_factor;
  check(pa::scatter_patch_embed(W.data_ptr(), W.stride(0), p, cur_stream()), "scatter_patch_embed");
}

static void scatter_conv_in(Tensor W, Tensor bias, uintptr_t x_src, uintptr_t t_src, Tensor t_emb,
                            c10::optional<Tensor> x_copy, Tensor out, int C, int H, int Wd, double time_factor,
                            double max_period) {
  // fused scatter: (peer) NCHW latent shard -> 3x3 im2col -> conv_in GEMM -> NHWC rows, + timestep sinusoid
  c10::cuda::CUDAGuard guard(out.device());
  TORCH_CHECK(W.dim() == 2 && W.size(1) == 64 && W.stride(1) == 1, "packed conv_in weight must be [N, 64]");
  TORCH_CHECK(out.dim() == 3 && out.is_contiguous() && out.size(1) == (int64_t)H * Wd && out.size(2) == W.size(0),
              "out must be contiguous [n, H*W, N]");
  TORCH_CHECK(t_emb.dim() == 2 && t_emb.is_contiguous() && t_emb.size(0) == out.size(0), "t_emb must be [n, dim]");
  pa::ScatterConvParams p{};
  p.x_src = reinterpret_cast<const __nv_bfloat16*>(x_src);
  p.t_src = reinterpret_cast<const __nv_bfloat16*>(t_src);
  p.t_emb = reinterpret_cast<__nv_bfloat16*>(t_emb.data_ptr());
  p.x_copy = x_copy ? reinterpret_cast<__nv_bfloat16*>(x_copy->data_ptr()) : nullptr;
  p.out = reinterpret_cast<__nv_bfloat16*>(out.data_ptr());
  p.bias = reinterpret_cast<const __nv_bfloat16*>(bias.data_ptr());
  p.n = (int)out.size(0); p.C = C; p.H = H; p.W = Wd; p.N = (int)W.size(0); p.temb_dim = (int)t_emb.size(1);
  p.time_factor = (float)time_factor;
  p.max_period = (float)max_period;
  check(pa::scatter_conv_in(W.data_ptr(), W.stride(0), p, cur_stream()), "scatter_conv_in");
}

static void nchw_to_nhwc_pad(uintptr_t x_ptr, Tensor out, int B, int C, int HW) {
  c10::cuda::CUDAGuard guard(out.device());
  TORCH_CHECK(out.is_contiguous() && out.size(-1) % 8 == 0);
  check(pa::nchw_to_nhwc_pad(reinterpret_cast<const void*>(x_ptr), out.data_ptr(), B, C, HW, (int)out.size(-1),
                             cur_stream()), "nchw_to_nhwc_pad");
}

static void upsample2x(Tensor x, Tensor out) {
  c10::cuda::CUDAGuard guard(x.device());
  TORCH_CHECK(x.dim() == 4 && x.is_contiguous() && out.is_contiguous(), "x must be NHWC [B, H, W, C]");
  check(pa::upsample_nearest2x_nhwc(x.data_ptr(), out.data_ptr(), (int)x.size(0), (int)x.size(1), (int)x.size(2),
                                    (int)x.size(3), cur_stream()), "upsample2x");
}

static void concat_channels(Tensor a, Tensor b, Tensor out) {
  c10::cuda::CUDAGuard guard(a.device());
  TORCH_CHECK(a.is_contiguous() && b.is_contiguous() && out.is_contiguous());
  const long long rows = a.numel() / a.size(-1);
  TORCH_CHECK(b.numel() / b.size(-1) == rows, "concat: row mismatch");
  check(pa::concat_channels(a.data_ptr(), b.data_ptr(), out.data_ptr(), rows, (int)a.size(-1), (int)b.size(-1),
                            cur_stream()), "concat_channels");
}

static void unet_out_gather(Tensor eps, c10::optional<Tensor> x, uintptr_t x_out_ptr, c10::optional<Tensor> sigmas,
                            int n, int C, bool cfg_pairs, double cfg, int mode, long long out_sample_off) {
  c10::cuda::CUDAGuard guard(eps.device());
  TORCH_CHECK(eps.dim() == 3 && eps.is_contiguous(), "eps must be [B, HW, Cpad]");
  TORCH_CHECK(mode == 0 || (x && sigmas), "Euler update needs x and sigmas");
  check(pa::unet_out_gather(eps.data_ptr(), x ? x->data_ptr() : nullptr, reinterpret_cast<void*>(x_out_ptr),
                            sigmas ? sigmas->data_ptr() : nullptr, n, C, (int)eps.size(1), (int)eps.size(2),
                            cfg_pairs ? 1 : 0, (float)cfg, mode, out_sample_off, cur_stream()),
        "unet_out_gather");
}

static void rms_rope(Tensor x, Tensor w, c10::optional<Tensor> rope, double eps) {
  c10::cuda::CUDAGuard guard(x.device());
  int b, rows;
  long long ld, bs;
  view3(x, b, rows, ld, bs);
  if (rope) TORCH_CHECK(rope->scalar_type() == at::kFloat && rope->is_contiguous() && rope->size(-1) == 2 &&
                        rope->size(-2) == 64 && rope->size(0) >= rows, "rope must be float32 [L, 64, 2]");
  check(pa::rms_rope_inplace(x.data_ptr(), ld, bs, w.data_ptr(), rope ? rope->data_ptr() : nullptr, b, rows,
                             (int)x.size(-1), (float)eps, cur_stream()), "rms_rope");
}

static void bcast_add(Tensor a, Tensor m, Tensor out) {
  c10::cuda::CUDAGuard guard(a.device());
  TORCH_CHECK(a.dim() == 2 && m.dim() == 2 && a.size(1) == m.size(1) && a.is_contiguous() && m.is_contiguous() &&
              out.is_contiguous());
  check(pa::bcast_add(a.data_ptr(), m.data_ptr(), out.data_ptr(), (int)a.size(0), (int)m.size(0), (int)a.size(1),
                      cur_stream()), "bcast_add");
}

// [B, R, D] -> [B, R, D] where each sample's [R, D] block is contiguous on both sides (e.g. the cached caption tokens
// into the token buffer): one strided DMA copy (cudaMemcpy2DAsync), no kernel.
static void copy_rows(Tensor src, Tensor dst) {
  c10::cuda::CUDAGuard guard(src.device());
  TORCH_CHECK(src.dim() == 3 && dst.dim() == 3 && src.sizes() == dst.sizes() && src.element_size() == dst.element_size());
  TORCH_CHECK(src.stride(2) == 1 && dst.stride(2) == 1 && src.stride(1) == src.size(2) && dst.stride(1) == dst.size(2),
              "copy_rows: per-sample blocks must be contiguous");
  const size_t es = src.element_size();
  const size_t width = (size_t)src.size(1) * src.size(2) * es;
  cudaError_t e = cudaMemcpy2DAsync(dst.data_ptr(), (size_t)dst.stride(0) * es, src.data_ptr(), (size_t)src.stride(0) * es,
                                    width, (size_t)src.size(0), cudaMemcpyDeviceToDevice, cur_stream());
  check((int)e, "copy_rows");
}

static void softmax_rows(Tensor x, double scale) {
  c10::cuda::CUDAGuard guard(x.device());
  TORCH_CHECK(x.dim() == 2 && x.stride(1) == 1 && x.scalar_type() == at::kBFloat16);
  check(pa::softmax_rows(x.data_ptr(), x.stride(0), (int)x.size(0), (int)x.size(1), (float)scale, cur_stream()),
        "softmax_rows");
}

static void silu_(Tensor x, Tensor out) {
  c10::cuda::CUDAGuard guard(x.device());
  TORCH_CHECK(x.is_contiguous() && out.is_contiguous());
  check(pa::silu_bf16(x.data_ptr(), out.data_ptr(), x.numel(), cur_stream()), "silu");
}

static void add_(Tensor a, Tensor b, Tensor out) {
  c10::cuda::CUDAGuard guard(a.device());
  TORCH_CHECK(a.is_contiguous() && b.is_contiguous() && out.is_contiguous());
  check(pa::add_bf16(a.data_ptr(), b.data_ptr(), out.data_ptr(), a.numel(), cur_stream()), "add");
}

static void attention(Tensor q, Tensor k, Tensor v, Tensor out, double scale, int variant, c10::optional<Tensor> k2,
                      c10::optional<Tensor> v2) {
  c10::cuda::CUDAGuard guard(q.device());
  TORCH_CHECK(q.dim() == 4 && k.dim() == 4 && v.dim() == 4, "q/k/v must be [B, H, L, D] views");
  const int D = (int)q.size(3);
  TORCH_CHECK((D == 64 || D == 128) && k.size(3) == D && v.size(3) == D, "head_dim must be 64 or 128");
  TORCH_CHECK(q.stride(3) == 1 && k.stride(3) == 1 && v.stride(3) == 1, "innermost dim must be contiguous");
  TORCH_CHECK(q.scalar_type() == at::kBFloat16, "bf16 required");
  TORCH_CHECK(out.dim() == 3 && out.stride(2) == 1, "out must be [B, L, H*D] (row stride free)");
  long long qs[3] = {q.stride(0), q.stride(1), q.stride(2)};
  long long ks[3] = {k.stride(0), k.stride(1), k.stride(2)};
  long long vs[3] = {v.stride(0), v.stride(1), v.stride(2)};
  if (k2.has_value() || v2.has_value()) {
    // two key/value sources: always the two-source ping-pong kernel, whatever `variant` says
    TORCH_CHECK(k2.has_value() && v2.has_value(), "attention: k2 and v2 go together");
    const Tensor& K2 = *k2;
    const Tensor& V2 = *v2;
    TORCH_CHECK(D == 128, "attention: a second K/V source needs head_dim 128");
    TORCH_CHECK(K2.dim() == 4 && V2.dim() == 4 && K2.size(3) == D && V2.size(3) == D && K2.stride(3) == 1 &&
                    V2.stride(3) == 1 && K2.scalar_type() == at::kBFloat16 && V2.scalar_type() == at::kBFloat16,
                "attention: k2/v2 must be bf16 [B, H, L2, 128] views with a contiguous innermost dim");
    TORCH_CHECK(K2.size(0) == q.size(0) && K2.size(1) == q.size(1) && V2.sizes() == K2.sizes() &&
                    k.size(0) == q.size(0) && k.size(1) == q.size(1) && v.sizes() == k.sizes(),
                "attention: batch / heads / lengths of the key and value sources do not match");
    long long ks2[3] = {K2.stride(0), K2.stride(1), K2.stride(2)};
    long long vs2[3] = {V2.stride(0), V2.stride(1), V2.stride(2)};
    check(pa::attention2_kv2_bf16(q.data_ptr(), k.data_ptr(), v.data_ptr(), K2.data_ptr(), V2.data_ptr(), out.data_ptr(),
                                  out.stride(1), out.stride(0), (int)q.size(0), (int)q.size(1), (int)q.size(2),
                                  (int)k.size(2), (int)K2.size(2), qs, ks, vs, ks2, vs2, (float)scale, cur_stream()),
          "attention2_kv2");
    return;
  }
  if (variant >= 20 && variant <= 250) {      // timing experiments of the ping-pong kernel (garbage results)
    check(pa::attention2_debug(q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr(), out.stride(1), out.stride(0),
                               (int)q.size(0), (int)q.size(1), (int)q.size(2), (int)k.size(2), variant - 20, qs, ks, vs,
                               (float)scale, cur_stream()),
          "attention2_debug");
    return;
  }
  static const bool xattn_cluster = []() { const char* e = std::getenv("PA_XATTN_CLUSTER"); return !(e && e[0] == '0'); }();
  if ((xattn_cluster || variant == 5) && D == 64 && k.size(2) <= 128 && (variant == 2 || variant == 5)) {
    // cross-attention over a short conditioning sequence: CTA pairs share one multicast K/V tile
    check(pa::xattn_cluster_bf16(q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr(), out.stride(1), out.stride(0),
                                 (int)q.size(0), (int)q.size(1), (int)q.size(2), (int)k.size(2), D, qs, ks, vs, (float)scale,
                                 cur_stream()),
          "xattn_cluster");
    return;
  }
  auto fn = (variant == 3 && D == 128) ? pa::attention3_bf16 : (variant >= 2 ? pa::attention2_bf16 : pa::attention_bf16);
  check(fn(q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr(), out.stride(1), out.stride(0), (int)q.size(0),
           (int)q.size(1), (int)q.size(2), (int)k.size(2), D, qs, ks, vs, (float)scale, cur_stream()),
        "attention");
}

// attention with MX-quantised output: out8 uint8 [B, rows8 >= Lq, ld8 >= H*128] contiguous (e4m3), sf8 scale chunks
static void attention_fp8out(Tensor q, Tensor k, Tensor v, Tensor out8, Tensor sf8, double scale) {
  c10::cuda::CUDAGuard guard(q.device());
  TORCH_CHECK(q.dim() == 4 && q.size(3) == 128 && k.size(3) == 128 && v.size(3) == 128, "head_dim 128 required");
  TORCH_CHECK(q.stride(3) == 1 && k.stride(3) == 1 && v.stride(3) == 1 && q.scalar_type() == at::kBFloat16);
  TORCH_CHECK(out8.dim() == 3 && out8.is_contiguous() && out8.element_size() == 1 && sf8.is_contiguous() &&
                  out8.size(0) == q.size(0) && out8.size(1) >= q.size(2), "out8 must be uint8 [B, rows, K] contiguous");
  TORCH_CHECK(sf8.numel() >= out8.size(0) * ((out8.size(1) + 127) / 128) * (out8.size(2) / 128) * 512, "sf8 too small");
  long long qs[3] = {q.stride(0), q.stride(1), q.stride(2)};
  long long ks[3] = {k.stride(0), k.stride(1), k.stride(2)};
  long long vs[3] = {v.stride(0), v.stride(1), v.stride(2)};
  check(pa::attention2_fp8out(q.data_ptr(), k.data_ptr(), v.data_ptr(), out8.data_ptr(), sf8.data_ptr(), out8.size(2),
                              out8.size(1), (int)q.size(0), (int)q.size(1), (int)q.size(2), (int)k.size(2), qs, ks, vs,
                              (float)scale, cur_stream()),
        "attention_fp8out");
}

static Tensor attention3_trace() {
  Tensor t = at::zeros({7, 64, 8}, at::TensorOptions().dtype(at::kLong));
  check(pa::attention3_trace_read(reinterpret_cast<long long*>(t.data_ptr<int64_t>())), "attention3_trace_read");
  return t;
}

static Tensor attention2_trace() {
  Tensor t = at::zeros({5, 64, 8}, at::TensorOptions().dtype(at::kLong));
  check(pa::attention2_trace_read(reinterpret_cast<long long*>(t.data_ptr<int64_t>())), "attention2_trace_read");
  return t;
}

static void groupnorm_silu(Tensor x, Tensor out, Tensor gamma, Tensor beta, int groups, double eps, bool silu) {
  c10::cuda::CUDAGuard guard(x.device());
  TORCH_CHECK(x.dim() == 3 && x.is_contiguous() && out.is_contiguous(), "x must be NHWC flattened: [B, HW, C]");
  static const bool use_cluster = []() { const char* e = std::getenv("PA_GROUPNORM_CLUSTER"); return !(e && e[0] == '0'); }();
  if (use_cluster) {
    // one launch: a thread-block cluster per (sample, channel slab), statistics exchanged through distributed shared memory
    const int rc = pa::groupnorm_silu_nhwc_cluster(x.data_ptr(), out.data_ptr(), gamma.data_ptr(), beta.data_ptr(),
                                                   (int)x.size(0), (int)x.size(1), (int)x.size(2), groups, (float)eps,
                                                   silu ? 1 : 0, cur_stream());
    if (rc != -100) {
      check(rc, "groupnorm_silu(cluster)");
      return;
    }
  }
  Tensor ws = at::zeros({x.size(0) * groups * 2}, x.options().dtype(at::kFloat));
  check(pa::groupnorm_silu_nhwc_ws(x.data_ptr(), out.data_ptr(), gamma.data_ptr(), beta.data_ptr(),
                                   ws.data_ptr<float>(), (int)x.size(0), (int)x.size(1), (int)x.size(2), groups,
                                   (float)eps, silu ? 1 : 0, cur_stream()),
        "groupnorm_silu");
}

static void cfg_euler_store(Tensor x, Tensor eps_c, c10::optional<Tensor> eps_u, uintptr_t x_out_ptr,
                            c10::optional<Tensor> sigmas, double cfg, long long out_sample_off, int mode) {
  c10::cuda::CUDAGuard guard(eps_c.device());
  TORCH_CHECK(eps_c.is_contiguous());
  const int batch = (int)eps_c.size(0);
  const long long per = eps_c.numel() / batch;
  check(pa::cfg_euler_store(x.data_ptr(), eps_c.data_ptr(), eps_u ? eps_u->data_ptr() : nullptr,
                            reinterpret_cast<void*>(x_out_ptr), sigmas ? sigmas->data_ptr() : nullptr, (float)cfg, per,
                            batch, out_sample_off, mode, cur_stream()),
        "cfg_euler_store");
}

// ---- sequence-parallel (Ulysses) exchange: flags with device-resident epochs + table-driven peer pull
static void sp_signal(Tensor peer_flag_table, int n_peers, int slot, int me, Tensor epoch) {
  c10::cuda::CUDAGuard guard(peer_flag_table.device());
  check(pa::sp_signal(reinterpret_cast<uint32_t* const*>(peer_flag_table.data_ptr()), n_peers, slot, me,
                      reinterpret_cast<const uint32_t*>(epoch.data_ptr()), cur_stream()),
        "sp_signal");
}

static void sp_pull(Tensor descs, int n_desc, int blocks_per_desc, Tensor flags, int slot, int n_peers, Tensor epoch,
                    long long timeout_cycles, Tensor err) {
  c10::cuda::CUDAGuard guard(descs.device());
  TORCH_CHECK(descs.is_contiguous() && descs.numel() * descs.element_size() >= (int64_t)n_desc * (int64_t)sizeof(pa::SpPullDesc),
              "descriptor table too small");
  check(pa::sp_pull(reinterpret_cast<const pa::SpPullDesc*>(descs.data_ptr()), n_desc, blocks_per_desc,
                    reinterpret_cast<const uint32_t*>(flags.data_ptr()), slot, n_peers,
                    reinterpret_cast<const uint32_t*>(epoch.data_ptr()), timeout_cycles,
                    reinterpret_cast<uint32_t*>(err.data_ptr()), cur_stream()),
        "sp_pull");
}

static void sp_epoch_inc(Tensor epoch) {
  c10::cuda::CUDAGuard guard(epoch.device());
  check(pa::sp_epoch_inc(reinterpret_cast<uint32_t*>(epoch.data_ptr()), cur_stream()), "sp_epoch_inc");
}

static void signal_flags(Tensor peer_ptr_table, int n_peers, int slot, uint32_t value) {
  c10::cuda::CUDAGuard guard(peer_ptr_table.device());
  check(pa::signal_flags(reinterpret_cast<uint32_t* const*>(peer_ptr_table.data_ptr()), n_peers, slot, value,
                         cur_stream()),
        "signal_flags");
}

static void wait_flags(Tensor flags, int first, int n, uint32_t value, long long timeout_cycles, Tensor err) {
  c10::cuda::CUDAGuard guard(flags.device());
  check(pa::wait_flags(reinterpret_cast<const uint32_t*>(flags.data_ptr()), first, n, value, timeout_cycles,
                       reinterpret_cast<uint32_t*>(err.data_ptr()), cur_stream()),
        "wait_flags");
}

PYBIND11_MODULE(_C, m) {
  m.doc() = "comfyui-parallelanything_b200 native library (sm_100a kernels + runtime)";
  m.def("gemm", &gemm, py::arg("A"), py::arg("W"), py::arg("mode"));
  m.def("gemm_fp8", &gemm_fp8, py::arg("A"), py::arg("sfa"), py::arg("W"), py::arg("sfb"), py::arg("mode"),
        py::arg("w_tile"));
  m.def("quantize_mxfp8", &quantize_mxfp8, py::arg("x"), py::arg("tile_rows") = 128);
  m.def("conv", &conv, py::arg("x"), py::arg("w"), py::arg("taps"), py::arg("stride"), py::arg("mode"));
  m.def("layernorm_modulate_fp8", &layernorm_modulate_fp8);
  m.def("layernorm_modulate", &layernorm_modulate, py::arg("x"), py::arg("out"), py::arg("scale") = py::none(),
        py::arg("shift") = py::none(), py::arg("gamma") = py::none(), py::arg("beta") = py::none(),
        py::arg("eps") = 1e-6, py::arg("mod_rows") = 0, py::arg("mod_row_off") = 0);
  m.def("timestep_embedding", &timestep_embedding);
  m.def("patchify", &patchify);
  m.def("scatter_patch_embed", &scatter_patch_embed, py::arg("W"), py::arg("bias"), py::arg("x_src"), py::arg("t_src"),
        py::arg("g_src"), py::arg("t_emb"), py::arg("g_emb"), py::arg("x_copy"), py::arg("out"), py::arg("C"),
        py::arg("Hl"), py::arg("Wl"), py::arg("time_factor"), py::arg("n_t") = 0);
  m.def("scatter_conv_in", &scatter_conv_in);
  m.def("nchw_to_nhwc_pad", &nchw_to_nhwc_pad);
  m.def("upsample2x", &upsample2x);
  m.def("concat_channels", &concat_channels);
  m.def("unet_out_gather", &unet_out_gather);
  m.def("rms_rope", &rms_rope);
  m.def("bcast_add", &bcast_add);
  m.def("softmax_rows", &softmax_rows);
  m.def("silu", &silu_);
  m.def("add", &add_);
  m.def("attention", &attention, py::arg("q"), py::arg("k"), py::arg("v"), py::arg("out"), py::arg("scale"),
        py::arg("variant") = 1, py::arg("k2") = py::none(), py::arg("v2") = py::none());
  m.def("attention2_trace", &attention2_trace);
  m.def("attention_fp8out", &attention_fp8out);
  m.def("attention3_trace", &attention3_trace);
  m.def("copy_rows", &copy_rows);
  m.def("rmsnorm_mod", &rmsnorm_mod, py::arg("x"), py::arg("out"), py::arg("weight") = py::none(),
        py::arg("scale") = py::none(), py::arg("gate") = py::none(), py::arg("residual") = py::none(),
        py::arg("eps") = 1e-5, py::arg("tanh_gate") = true);
  m.def("groupnorm_silu", &groupnorm_silu);
  m.def("cfg_euler_store", &cfg_euler_store);
  m.def("sp_signal", &sp_signal);
  m.def("sp_pull", &sp_pull);
  m.def("sp_epoch_inc", &sp_epoch_inc);
  m.attr("SP_MAX_RANKS") = (int)pa::SP_MAX_RANKS;
  m.attr("SP_MAX_SLOTS") = (int)pa::SP_MAX_SLOTS;
  m.attr("SP_DESC_BYTES") = (int)sizeof(pa::SpPullDesc);
  m.def("signal_flags", &signal_flags);
  m.def("wait_flags", &wait_flags);
  m.def("num_sms", &pa::num_sms);
  m.def("set_sm_limit", &pa::set_sm_limit);
  pa::rt::bind(m);
  m.attr("EPI_BIAS") = (int)pa::EPI_BIAS;
  m.attr("EPI_BIAS_GELU") = (int)pa::EPI_BIAS_GELU;
  m.attr("EPI_BIAS_SILU") = (int)pa::EPI_BIAS_SILU;
  m.attr("EPI_GATE_RES") = (int)pa::EPI_GATE_RES;
  m.attr("EPI_QKV_ROPE") = (int)pa::EPI_QKV_ROPE;
  m.attr("EPI_EULER_UNPATCH") = (int)pa::EPI_EULER_UNPATCH;
  m.attr("EPI_GEGLU") = (int)pa::EPI_GEGLU;
  m.attr("EPI_RES") = (int)pa::EPI_RES;
  m.attr("EPI_BIAS_BCAST") = (int)pa::EPI_BIAS_BCAST;
}
