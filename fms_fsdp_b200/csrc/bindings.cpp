// Python bindings (torch tensors -> raw launchers).  Compiled by g++ only; every kernel lives in a
// torch-free .cu so nvcc never parses the torch headers.
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>
#include <torch/extension.h>

#include <cmath>
#include <cstdint>

#define DECL extern "C"
DECL int b200_gemm_bf16(const void*, const void*, void*, const void*, int, int, int, int, int, int, int, int, int, int,
                        int, cudaStream_t);
DECL int b200_gemm2_bf16(const void*, const void*, void*, const void*, int, int, int, int, int, int, int, int, int, int,
                         int, cudaStream_t);
DECL int b200_gemm2_ag_bf16(const void*, const void*, void*, const void*, int, int, int, int, int, int, int, int, int, int,
                            const void* const*, void*, unsigned long long, unsigned long long, unsigned long long, int, int,
                            uint32_t*, uint32_t, int, cudaStream_t);
DECL int b200_bgemm_bf16(const void*, const void*, void*, int, int, int, int, int, int, int, int, long long, long long,
                         long long, long long, long long, long long, int, int, int, int, cudaStream_t);
DECL int b200_ssd_prep(const void*, const float*, const float*, float*, float*, float*, int, int, int, cudaStream_t);
DECL int b200_ssd_mask(const void*, const float*, const float*, void*, int, int, int, cudaStream_t);
DECL int b200_ssd_xs(const void*, const float*, const float*, const float*, void*, long long, int, int, cudaStream_t);
DECL int b200_ssd_state_pass(const float*, const float*, void*, int, int, int, int, int, cudaStream_t);
DECL int b200_ssd_combine(const void*, const void*, const void*, const float*, const float*, void*, long long, int, int,
                          cudaStream_t);
DECL int b200_ssd_dyoff(const void*, const void*, const void*, const float*, void*, float*, float*, long long, int,
                        cudaStream_t);
DECL int b200_ssd_mask_bwd(const void*, const void*, const float*, const float*, void*, float*, float*, int, int, int,
                           cudaStream_t);
DECL int b200_ssd_state_pass_bwd(const float*, const void*, const float*, void*, float*, int, int, int, int, int,
                                 cudaStream_t);
DECL int b200_ssd_dx(const void*, const void*, const void*, const void*, const float*, const float*, const float*,
                     const float*, void*, float*, float*, float*, long long, int, int, cudaStream_t);
DECL int b200_ssd_dt_bwd(const void*, const float*, const float*, const float*, const float*, const float*, const float*,
                         void*, float*, float*, int, int, int, cudaStream_t);
DECL int b200_selscan_fwd(const void*, const void*, const float*, const void*, const void*, const float*, const void*,
                          const float*, float*, void*, int, int, int, int, int, cudaStream_t);
DECL int b200_selscan_bwd(const void*, const void*, const void*, const float*, const void*, const void*, const float*,
                          const void*, const float*, float*, void*, void*, void*, float*, float*, float*, float*, float*, int,
                          int, int, int, int, cudaStream_t);
DECL void b200_comm_set_reduce_ctas(int);
DECL int b200_p2p_gather_range(const void* const*, void*, long long, long long, long long, cudaStream_t);
DECL int b200_ts_mma_probe(const void*, const void*, float*, cudaStream_t);
DECL int b200_rmsnorm_fwd(const void*, const void*, void*, float*, int, int, float, cudaStream_t);
DECL int b200_rmsnorm_bwd_grid(int);
DECL int b200_rmsnorm_bwd(const void*, const void*, const void*, const float*, const void*, void*, float*, float*, int, int,
                          cudaStream_t);
DECL int b200_add_rmsnorm_fwd(const void*, const float*, const void*, void*, float*, float*, int, int, float, cudaStream_t);
DECL int b200_rmsnorm_bwd_f32(const void*, const float*, const void*, const float*, float*, float*, float*, int, int, cudaStream_t);
DECL int b200_rmsnorm_gated_fwd(const void*, const void*, const void*, void*, float*, int, int, float, cudaStream_t);
DECL int b200_rmsnorm_gated_bwd(const void*, const void*, const void*, const void*, const float*, void*, void*, float*, float*, int, int, cudaStream_t);
DECL int b200_rope(void*, const float*, int, int, int, int, int, int, int, int, int, cudaStream_t);
DECL int b200_swiglu_fwd(const void*, void*, long long, int, int, cudaStream_t);
DECL int b200_swiglu_bwd(const void*, const void*, void*, long long, int, int, cudaStream_t);
DECL int b200_embedding_fwd(const void*, int, const void*, void*, long long, int, cudaStream_t);
DECL int b200_embedding_bwd(const void*, int, const void*, void*, int, long long, int, cudaStream_t);
DECL int b200_count_valid(const long long*, int, long long, float*, cudaStream_t);
DECL int b200_ce_grad_inplace(void*, const long long*, const float*, float*, int, int, int, long long, cudaStream_t);
DECL int b200_adamw(float*, const void*, int, float*, float*, void*, long long, float, float, float, float, float,
                    float, float, const float*, cudaStream_t);
DECL int b200_sumsq(const void*, int, long long, float*, cudaStream_t);
DECL void b200_attn_set_fwd_version(int);
DECL void b200_attn_set_bwd_version(int);
DECL void b200_attn_set_poly(int, int);
DECL int b200_attn_fwd(const void*, void*, float*, int, int, int, int, int, float, cudaStream_t);
DECL int b200_attn_bwd(const void*, const void*, const void*, const float*, void*, float*, int, int, int, int, int,
                       float, const float*, cudaStream_t);
DECL void b200_gemm2_set_rope(const float*, int, int, int);
DECL void b200_gemm2_set_swiglu(void*, int, int, int);
DECL int b200_gemm2_fp8(const void*, const void*, void*, const float*, const float*, int, int, int, int, int, int, cudaStream_t);
DECL int b200_bias_grad_partials(int, int);
DECL int b200_bias_grad(const void*, float*, void*, int, int, int, int, cudaStream_t);
DECL int b200_quant_rowwise_e4m3(const void*, void*, float*, int, int, int, int, cudaStream_t);
DECL void b200_gemm2_set_push(void* const*, long long, long long, int, int, int);
DECL int b200_p2p_push_range(const void*, void* const*, long long, long long, long long, int, cudaStream_t);
DECL int b200_p2p_allgather(const void* const*, void*, long long, int, int, cudaStream_t);
DECL int b200_reduce_scatter(const void* const*, float*, long long, long long, int, int, int, float, float*,
                             cudaStream_t);
DECL int b200_allreduce_inplace(void* const*, long long, int, int, int, float, float*, cudaStream_t);
DECL int b200_signal_barrier(uint32_t* const*, int, int, uint32_t, int, int, cudaStream_t);
DECL int b200_scalar_allreduce_bytes();
DECL int b200_scalar_allreduce(uint8_t* const*, int, int, uint32_t, float*, int, cudaStream_t);
DECL int b200_causal_conv1d_fwd(const void*, const void*, const void*, void*, int, int, int, int, int, cudaStream_t);
DECL int b200_causal_conv1d_bwd(const void*, const void*, const void*, const void*, void*, float*, float*, int, int,
                                int, int, int, cudaStream_t);

namespace {

static int64_t g_launches = 0;
static int g_reduce_ctas_default = 296;
static bool g_gemm_2cta = true;

inline cudaStream_t cur_stream() { return at::cuda::getCurrentCUDAStream().stream(); }

inline void check(int rc, const char* what, int n_kernels = 1) {
  TORCH_CHECK(rc == 0, "fms_fsdp_b200 kernel '", what, "' failed with code ", rc, " (",
              rc > 0 && rc < 1000 ? cudaGetErrorString((cudaError_t)rc) : "argument/descriptor error", ")");
  g_launches += n_kernels;
}
inline void need(const at::Tensor& t, const char* name, at::ScalarType dt) {
  TORCH_CHECK(t.is_cuda(), name, " must be a CUDA tensor");
  TORCH_CHECK(t.scalar_type() == dt, name, " has dtype ", t.scalar_type(), ", expected ", dt);
}
inline void need_rowmajor2d(const at::Tensor& t, const char* name) {
  TORCH_CHECK(t.dim() == 2 && t.stride(1) == 1, name, " must be 2-D with unit inner stride");
  TORCH_CHECK((reinterpret_cast<uintptr_t>(t.data_ptr()) & 15) == 0 && (t.stride(0) * t.element_size()) % 16 == 0,
              name, " must be 16-byte aligned (ptr and row stride)");
}

// epilogue flag (csrc/gemm2_sm100.cu P_EPI_BIAS): + bias[col] before the store / RoPE; the bias travels in the R slot
constexpr int kEpiBias = 16;
// bias [N] bf16, contiguous, 16-byte aligned: returns its pointer (the R operand of the launch)
inline const void* bias_operand(const c10::optional<at::Tensor>& bias, int64_t N) {
  need(*bias, "bias", at::kBFloat16);
  TORCH_CHECK(bias->is_contiguous() && bias->numel() == N && (reinterpret_cast<uintptr_t>(bias->data_ptr()) & 15) == 0,
              "bias must be a contiguous, 16-byte aligned [N] tensor");
  return bias->data_ptr();
}

// layout: 0 = nt, 1 = nn, 2 = tn ; epi: 0 store, 1 +residual, 2 accumulate into c
// bias (nt, epi 0 / 3, CTA-pair kernel, bf16 output): c = a b^T + bias[col] (then RoPE for epi 3)
void gemm(const at::Tensor& a, const at::Tensor& b, at::Tensor& c, int64_t layout, int64_t epi,
          const c10::optional<at::Tensor>& residual, const c10::optional<at::Tensor>& bias) {
  c10::cuda::CUDAGuard guard(a.device());
  need(a, "a", at::kBFloat16);
  need(b, "b", at::kBFloat16);
  need_rowmajor2d(a, "a");
  need_rowmajor2d(b, "b");
  need_rowmajor2d(c, "c");
  TORCH_CHECK(c.scalar_type() == at::kBFloat16 || c.scalar_type() == at::kFloat, "c must be bf16 or fp32");
  int M, N, K, a_mn = 0, b_mn = 0;
  if (layout == 0) {
    M = a.size(0); K = a.size(1); N = b.size(0);
    TORCH_CHECK(b.size(1) == K, "nt: K mismatch");
  } else if (layout == 1) {
    M = a.size(0); K = a.size(1); N = b.size(1); b_mn = 1;
    TORCH_CHECK(b.size(0) == K, "nn: K mismatch");
  } else {
    K = a.size(0); M = a.size(1); N = b.size(1); a_mn = b_mn = 1;
    TORCH_CHECK(b.size(0) == K, "tn: K mismatch");
  }
  TORCH_CHECK(c.size(0) == M && c.size(1) == (epi == 6 ? 2 * N : N), "c shape mismatch");
  TORCH_CHECK(K % 8 == 0 && N % 8 == 0 && M % 8 == 0, "M, N, K must be multiples of 8");
  TORCH_CHECK((epi != 5 && epi != 6) || (g_gemm_2cta && M >= 256 && c.scalar_type() == at::kBFloat16),
              "SwiGLU epilogues: CTA-pair kernel, bf16 output (call set_gemm_swiglu first)");
  const void* r = nullptr;
  int ldr = 0;
  if (epi == 1) {
    TORCH_CHECK(residual.has_value(), "residual epilogue needs a residual");
    need(*residual, "residual", at::kBFloat16);
    need_rowmajor2d(*residual, "residual");
    r = residual->data_ptr();
    ldr = residual->stride(0);
  }
  TORCH_CHECK(epi != 3 || (g_gemm_2cta && M >= 256 && layout == 0 && c.scalar_type() == at::kBFloat16),
              "RoPE epilogue: CTA-pair kernel, nt layout, bf16 output only (call set_gemm_rope first)");
  TORCH_CHECK(epi != 4, "push epilogue: use gemm_push (no output tensor)");
  if (bias.has_value() && bias->defined()) {
    TORCH_CHECK((epi == 0 || epi == 3) && layout == 0 && g_gemm_2cta && M >= 256 && c.scalar_type() == at::kBFloat16,
                "bias epilogue: CTA-pair kernel, nt layout, store or RoPE epilogue, bf16 output only");
    r = bias_operand(bias, N);
    ldr = 0;
    epi |= kEpiBias;
  }
  // CTA-pair kernel (cta_group::2, 256x256 tiles) for anything with at least one full pair tile of rows
  if (g_gemm_2cta && M >= 256) {
    check(b200_gemm2_bf16(a.data_ptr(), b.data_ptr(), c.data_ptr(), r, M, N, K, a.stride(0), b.stride(0), c.stride(0),
                          ldr, a_mn, b_mn, (int)epi, c.scalar_type() == at::kFloat ? 1 : 0, cur_stream()),
          "gemm2_bf16_tcgen05");
    return;
  }
  check(b200_gemm_bf16(a.data_ptr(), b.data_ptr(), c.data_ptr(), r, M, N, K, a.stride(0), b.stride(0), c.stride(0),
                       ldr, a_mn, b_mn, (int)epi, c.scalar_type() == at::kFloat ? 1 : 0, cur_stream()),
        "gemm_bf16_tcgen05");
}

std::vector<at::Tensor> rmsnorm_fwd(const at::Tensor& x, const at::Tensor& w, double eps) {
  c10::cuda::CUDAGuard guard(x.device());
  need(x, "x", at::kBFloat16);
  need(w, "w", at::kBFloat16);
  TORCH_CHECK(x.is_contiguous() && w.is_contiguous());
  const int D = x.size(-1), M = x.numel() / D;
  auto y = at::empty_like(x);
  auto rstd = at::empty({M}, x.options().dtype(at::kFloat));
  check(b200_rmsnorm_fwd(x.data_ptr(), w.data_ptr(), y.data_ptr(), rstd.data_ptr<float>(), M, D, (float)eps,
                         cur_stream()), "rmsnorm_fwd");
  return {y, rstd};
}
std::vector<at::Tensor> rmsnorm_bwd(const at::Tensor& dy, const at::Tensor& x, const at::Tensor& w,
                                    const at::Tensor& rstd, const c10::optional<at::Tensor>& dres) {
  c10::cuda::CUDAGuard guard(x.device());
  need(dy, "dy", at::kBFloat16);
  need(x, "x", at::kBFloat16);
  need(w, "w", at::kBFloat16);
  need(rstd, "rstd", at::kFloat);
  TORCH_CHECK(dy.is_contiguous() && x.is_contiguous());
  const int D = x.size(-1), M = x.numel() / D;
  auto dx = at::empty_like(x);
  auto part = at::empty({b200_rmsnorm_bwd_grid(M), D}, x.options().dtype(at::kFloat));
  auto dw = at::empty({D}, x.options().dtype(at::kFloat));
  const void* dres_p = nullptr;
  if (dres.has_value() && dres->defined()) {
    need(*dres, "dres", at::kBFloat16);
    TORCH_CHECK(dres->is_contiguous() && dres->numel() == x.numel(), "rmsnorm_bwd: dres shape");
    dres_p = dres->data_ptr();
  }
  check(b200_rmsnorm_bwd(dy.data_ptr(), x.data_ptr(), w.data_ptr(), rstd.data_ptr<float>(), dres_p, dx.data_ptr(),
                         part.data_ptr<float>(), dw.data_ptr<float>(), M, D, cur_stream()), "rmsnorm_bwd", 2);
  return {dx, dw};
}
std::vector<at::Tensor> add_rmsnorm_fwd(const at::Tensor& x, const at::Tensor& res, const at::Tensor& w, double eps) {
  c10::cuda::CUDAGuard guard(x.device());
  need(x, "x", at::kBFloat16);
  need(res, "res", at::kFloat);
  need(w, "w", at::kBFloat16);
  TORCH_CHECK(x.is_contiguous() && res.is_contiguous() && w.is_contiguous());
  const int D = x.size(-1), M = x.numel() / D;
  auto y = at::empty_like(x);
  auto res_out = at::empty_like(res);
  auto rstd = at::empty({M}, x.options().dtype(at::kFloat));
  check(b200_add_rmsnorm_fwd(x.data_ptr(), res.data_ptr<float>(), w.data_ptr(), y.data_ptr(), res_out.data_ptr<float>(),
                             rstd.data_ptr<float>(), M, D, (float)eps, cur_stream()), "add_rmsnorm_fwd");
  return {y, res_out, rstd};
}
std::vector<at::Tensor> rmsnorm_bwd_f32(const at::Tensor& dy, const at::Tensor& x, const at::Tensor& w,
                                        const at::Tensor& rstd) {
  c10::cuda::CUDAGuard guard(x.device());
  need(dy, "dy", at::kBFloat16);
  need(x, "x", at::kFloat);
  need(w, "w", at::kBFloat16);
  TORCH_CHECK(dy.is_contiguous() && x.is_contiguous());
  const int D = x.size(-1), M = x.numel() / D;
  auto dx = at::empty_like(x);
  auto part = at::empty({b200_rmsnorm_bwd_grid(M), D}, x.options());
  auto dw = at::empty({D}, x.options());
  check(b200_rmsnorm_bwd_f32(dy.data_ptr(), x.data_ptr<float>(), w.data_ptr(), rstd.data_ptr<float>(), dx.data_ptr<float>(),
                             part.data_ptr<float>(), dw.data_ptr<float>(), M, D, cur_stream()), "rmsnorm_bwd_f32", 2);
  return {dx, dw};
}
std::vector<at::Tensor> rmsnorm_gated_fwd(const at::Tensor& x, const at::Tensor& z, const at::Tensor& w, double eps) {
  c10::cuda::CUDAGuard guard(x.device());
  need(x, "x", at::kBFloat16);
  need(z, "z", at::kBFloat16);
  need(w, "w", at::kBFloat16);
  TORCH_CHECK(x.is_contiguous() && z.is_contiguous());
  const int D = x.size(-1), M = x.numel() / D;
  auto y = at::empty_like(x);
  auto rstd = at::empty({M}, x.options().dtype(at::kFloat));
  check(b200_rmsnorm_gated_fwd(x.data_ptr(), z.data_ptr(), w.data_ptr(), y.data_ptr(), rstd.data_ptr<float>(), M, D,
                               (float)eps, cur_stream()), "rmsnorm_gated_fwd");
  return {y, rstd};
}
std::vector<at::Tensor> rmsnorm_gated_bwd(const at::Tensor& dy, const at::Tensor& x, const at::Tensor& z,
                                          const at::Tensor& w, const at::Tensor& rstd) {
  c10::cuda::CUDAGuard guard(x.device());
  need(dy, "dy", at::kBFloat16);
  need(x, "x", at::kBFloat16);
  need(z, "z", at::kBFloat16);
  TORCH_CHECK(dy.is_contiguous() && x.is_contiguous() && z.is_contiguous());
  const int D = x.size(-1), M = x.numel() / D;
  auto dx = at::empty_like(x);
  auto dz = at::empty_like(z);
  auto part = at::empty({b200_rmsnorm_bwd_grid(M), D}, x.options().dtype(at::kFloat));
  auto dw = at::empty({D}, x.options().dtype(at::kFloat));
  check(b200_rmsnorm_gated_bwd(dy.data_ptr(), x.data_ptr(), z.data_ptr(), w.data_ptr(), rstd.data_ptr<float>(),
                               dx.data_ptr(), dz.data_ptr(), part.data_ptr<float>(), dw.data_ptr<float>(), M, D, cur_stream()),
        "rmsnorm_gated_bwd", 2);
  return {dx, dz, dw};
}
void rope(at::Tensor& qkv, const at::Tensor& table, int64_t seq_len, int64_t nrot_heads, int64_t hd, int64_t rot,
          bool inverse, int64_t pos_offset, bool interleaved) {
  c10::cuda::CUDAGuard guard(qkv.device());
  need(qkv, "qkv", at::kBFloat16);
  need(table, "table", at::kFloat);
  TORCH_CHECK(qkv.dim() == 2 && qkv.stride(1) == 1 && table.is_contiguous());
  TORCH_CHECK(table.size(0) >= seq_len + pos_offset && table.size(1) == rot / 2, "rope table too small");
  check(b200_rope(qkv.data_ptr(), table.data_ptr<float>(), qkv.size(0), seq_len, qkv.stride(0), nrot_heads, hd, rot,
                  inverse, pos_offset, interleaved, cur_stream()), "rope");
}
at::Tensor swiglu_fwd(const at::Tensor& gu, bool gate_first) {
  c10::cuda::CUDAGuard guard(gu.device());
  need(gu, "gu", at::kBFloat16);
  TORCH_CHECK(gu.is_contiguous());
  const int F = gu.size(-1) / 2;
  const int64_t M = gu.numel() / (2 * F);
  auto sizes = gu.sizes().vec();
  sizes.back() = F;
  auto out = at::empty(sizes, gu.options());
  check(b200_swiglu_fwd(gu.data_ptr(), out.data_ptr(), M, F, gate_first, cur_stream()), "swiglu_fwd");
  return out;
}
at::Tensor swiglu_bwd(const at::Tensor& ds, const at::Tensor& gu, bool gate_first) {
  c10::cuda::CUDAGuard guard(gu.device());
  need(gu, "gu", at::kBFloat16);
  need(ds, "ds", at::kBFloat16);
  TORCH_CHECK(gu.is_contiguous() && ds.is_contiguous());
  const int F = gu.size(-1) / 2;
  const int64_t M = gu.numel() / (2 * F);
  auto dgu = at::empty_like(gu);
  check(b200_swiglu_bwd(ds.data_ptr(), gu.data_ptr(), dgu.data_ptr(), M, F, gate_first, cur_stream()), "swiglu_bwd");
  return dgu;
}
at::Tensor embedding_fwd(const at::Tensor& tok, const at::Tensor& w) {
  c10::cuda::CUDAGuard guard(w.device());
  need(w, "w", at::kBFloat16);
  TORCH_CHECK(tok.is_cuda() && tok.is_contiguous() &&
              (tok.scalar_type() == at::kLong || tok.scalar_type() == at::kInt));
  const int D = w.size(1);
  const int64_t M = tok.numel();
  auto out = at::empty({M, D}, w.options());
  check(b200_embedding_fwd(tok.data_ptr(), tok.scalar_type() == at::kLong, w.data_ptr(), out.data_ptr(), M, D,
                           cur_stream()), "embedding_fwd");
  return out;
}
void embedding_bwd(const at::Tensor& dx, const at::Tensor& tok, at::Tensor& dw) {
  c10::cuda::CUDAGuard guard(dx.device());
  need(dx, "dx", at::kBFloat16);
  TORCH_CHECK(dx.is_contiguous() && tok.is_contiguous() && dw.is_contiguous());
  TORCH_CHECK(dw.scalar_type() == at::kBFloat16 || dw.scalar_type() == at::kFloat);
  const int D = dx.size(-1);
  const int64_t M = tok.numel();
  check(b200_embedding_bwd(tok.data_ptr(), tok.scalar_type() == at::kLong, dx.data_ptr(), dw.data_ptr(),
                           dw.scalar_type() == at::kFloat, M, D, cur_stream()), "embedding_bwd");
}
void count_valid(const at::Tensor& labels, int64_t ignore, at::Tensor& n_valid) {
  c10::cuda::CUDAGuard guard(labels.device());
  need(labels, "labels", at::kLong);
  need(n_valid, "n_valid", at::kFloat);
  check(b200_count_valid((const long long*)labels.data_ptr(), labels.numel(), ignore, n_valid.data_ptr<float>(),
                         cur_stream()), "count_valid");
}
void ce_grad_inplace(at::Tensor& logits, const at::Tensor& labels, const at::Tensor& n_valid, at::Tensor& loss_sum,
                     int64_t ignore) {
  c10::cuda::CUDAGuard guard(logits.device());
  need(logits, "logits", at::kBFloat16);
  need(labels, "labels", at::kLong);
  TORCH_CHECK(logits.dim() == 2 && logits.stride(1) == 1 && labels.is_contiguous());
  check(b200_ce_grad_inplace(logits.data_ptr(), (const long long*)labels.data_ptr(), n_valid.data_ptr<float>(),
                             loss_sum.data_ptr<float>(), logits.size(0), logits.size(1), logits.stride(0), ignore,
                             cur_stream()), "ce_grad_inplace");
}
void adamw(at::Tensor& master, const at::Tensor& grad, at::Tensor& m, at::Tensor& v,
           const c10::optional<at::Tensor>& lowp, double lr, double b1, double b2, double eps, double wd, int64_t step,
           const c10::optional<at::Tensor>& grad_scale) {
  c10::cuda::CUDAGuard guard(master.device());
  need(master, "master", at::kFloat);
  need(m, "m", at::kFloat);
  need(v, "v", at::kFloat);
  TORCH_CHECK(grad.scalar_type() == at::kBFloat16 || grad.scalar_type() == at::kFloat);
  TORCH_CHECK(grad.numel() == master.numel());
  void* lp = nullptr;
  if (lowp.has_value()) {
    need(*lowp, "lowp", at::kBFloat16);
    lp = lowp->data_ptr();
  }
  const float* gs = grad_scale.has_value() ? grad_scale->data_ptr<float>() : nullptr;
  const double bc1 = 1.0 - std::pow(b1, (double)step), bc2 = 1.0 - std::pow(b2, (double)step);
  check(b200_adamw(master.data_ptr<float>(), grad.data_ptr(), grad.scalar_type() == at::kBFloat16,
                   m.data_ptr<float>(), v.data_ptr<float>(), lp, master.numel(), (float)lr, (float)b1, (float)b2,
                   (float)eps, (float)wd, (float)bc1, (float)std::sqrt(bc2), gs, cur_stream()), "adamw");
}
void sumsq(const at::Tensor& x, at::Tensor& out) {
  c10::cuda::CUDAGuard guard(x.device());
  TORCH_CHECK(x.is_contiguous() && (x.scalar_type() == at::kBFloat16 || x.scalar_type() == at::kFloat));
  need(out, "out", at::kFloat);
  check(b200_sumsq(x.data_ptr(), x.scalar_type() == at::kBFloat16, x.numel(), out.data_ptr<float>(), cur_stream()),
        "sumsq");
}

std::vector<at::Tensor> attn_fwd(const at::Tensor& qkv, int64_t B, int64_t S, int64_t H, int64_t KVH, int64_t hd,
                                 double scale) {
  c10::cuda::CUDAGuard guard(qkv.device());
  need(qkv, "qkv", at::kBFloat16);
  TORCH_CHECK(qkv.is_contiguous());
  auto o = at::empty({B * S, H * hd}, qkv.options());
  auto lse = at::empty({B, H, S}, qkv.options().dtype(at::kFloat));
  check(b200_attn_fwd(qkv.data_ptr(), o.data_ptr(), lse.data_ptr<float>(), B, S, H, KVH, hd, (float)scale,
                      cur_stream()), "attn_fwd");
  return {o, lse};
}
at::Tensor attn_bwd(const at::Tensor& dout, const at::Tensor& qkv, const at::Tensor& o, const at::Tensor& lse,
                    int64_t B, int64_t S, int64_t H, int64_t KVH, int64_t hd, double scale,
                    const c10::optional<at::Tensor>& rope) {
  c10::cuda::CUDAGuard guard(qkv.device());
  need(qkv, "qkv", at::kBFloat16);
  need(dout, "do", at::kBFloat16);
  need(o, "o", at::kBFloat16);
  need(lse, "lse", at::kFloat);
  TORCH_CHECK(qkv.is_contiguous() && dout.is_contiguous() && o.is_contiguous() && lse.is_contiguous());
  auto dqkv = at::empty_like(qkv);
  // [2 planes: delta | lse*log2e][B][H][S padded to 128]
  auto delta = at::empty({2, B, H, ((S + 127) / 128) * 128}, qkv.options().dtype(at::kFloat));
  const float* rope_p = nullptr;
  if (rope.has_value() && rope->defined()) {   // inverse RoPE of dq, dk fused into the epilogue
    need(*rope, "rope", at::kFloat);
    TORCH_CHECK(rope->is_contiguous() && rope->numel() >= S * hd, "attn_bwd: rope table must be [S, hd/2, 2] fp32");
    rope_p = rope->data_ptr<float>();
  }
  check(b200_attn_bwd(dout.data_ptr(), qkv.data_ptr(), o.data_ptr(), lse.data_ptr<float>(), dqkv.data_ptr(),
                      delta.data_ptr<float>(), B, S, H, KVH, hd, (float)scale, rope_p, cur_stream()), "attn_bwd", 3);
  return dqkv;
}

// ---- peer-memory collectives: pointer tables live on the device (int64 tensors of peer addresses)
void p2p_allgather(const at::Tensor& peer_ptrs, at::Tensor& full, int64_t shard_bytes, int64_t world, int64_t rank) {
  c10::cuda::CUDAGuard guard(full.device());
  check(b200_p2p_allgather((const void* const*)peer_ptrs.data_ptr(), full.data_ptr(), shard_bytes, world, rank,
                           cur_stream()), "p2p_allgather");
}
void reduce_scatter(const at::Tensor& peer_ptrs, at::Tensor& out32, int64_t elem_offset, int64_t world, int64_t rank,
                    bool src_bf16, double scale, const c10::optional<at::Tensor>& sumsq_out, int64_t max_ctas) {
  c10::cuda::CUDAGuard guard(out32.device());
  need(out32, "out", at::kFloat);
  b200_comm_set_reduce_ctas(max_ctas > 0 ? (int)max_ctas : g_reduce_ctas_default);
  check(b200_reduce_scatter((const void* const*)peer_ptrs.data_ptr(), out32.data_ptr<float>(), out32.numel(),
                            elem_offset, world, rank, src_bf16, (float)scale,
                            sumsq_out.has_value() ? sumsq_out->data_ptr<float>() : nullptr, cur_stream()),
        "reduce_scatter");
}
void allreduce_inplace(const at::Tensor& peer_ptrs, int64_t numel, int64_t world, int64_t rank, bool is_bf16,
                       double scale, const c10::optional<at::Tensor>& sumsq_out, const at::Tensor& anchor) {
  c10::cuda::CUDAGuard guard(anchor.device());
  check(b200_allreduce_inplace((void* const*)peer_ptrs.data_ptr(), numel, world, rank, is_bf16, (float)scale,
                               sumsq_out.has_value() ? sumsq_out->data_ptr<float>() : nullptr, cur_stream()),
        "allreduce_inplace");
}
// mode 0 = barrier, 1 = post only, 2 = wait only; slot_base selects the 32-slot channel of the signal pad
void signal_barrier(const at::Tensor& pad_ptrs, int64_t world, int64_t rank, int64_t epoch, const at::Tensor& anchor,
                    int64_t slot_base, int64_t mode) {
  c10::cuda::CUDAGuard guard(anchor.device());
  check(b200_signal_barrier((uint32_t* const*)pad_ptrs.data_ptr(), world, rank, (uint32_t)epoch, (int)slot_base, (int)mode,
                            cur_stream()), "signal_barrier");
}
// one-shot sum of a few fp32 scalars across the group (in place), every rank gets the identical result
void scalar_allreduce(const at::Tensor& buf_ptrs, int64_t world, int64_t rank, int64_t epoch, at::Tensor& inout) {
  c10::cuda::CUDAGuard guard(inout.device());
  need(inout, "inout", at::kFloat);
  TORCH_CHECK(inout.is_contiguous());
  check(b200_scalar_allreduce((uint8_t* const*)buf_ptrs.data_ptr(), (int)world, (int)rank, (uint32_t)epoch,
                              inout.data_ptr<float>(), (int)inout.numel(), cur_stream()), "scalar_allreduce");
}

at::Tensor causal_conv1d_fwd(const at::Tensor& x, const at::Tensor& w, const c10::optional<at::Tensor>& b,
                             int64_t seq_len, bool act) {
  c10::cuda::CUDAGuard guard(x.device());
  need(x, "x", at::kBFloat16);
  need(w, "w", at::kBFloat16);
  TORCH_CHECK(x.is_contiguous() && w.is_contiguous());
  auto y = at::empty_like(x);
  check(b200_causal_conv1d_fwd(x.data_ptr(), w.data_ptr(), b.has_value() ? b->data_ptr() : nullptr, y.data_ptr(),
                               x.size(0), x.size(1), w.size(1), seq_len, act, cur_stream()), "causal_conv1d_fwd");
  return y;
}
std::vector<at::Tensor> causal_conv1d_bwd(const at::Tensor& dy, const at::Tensor& x, const at::Tensor& w,
                                          const c10::optional<at::Tensor>& b, int64_t seq_len, bool act) {
  c10::cuda::CUDAGuard guard(x.device());
  need(x, "x", at::kBFloat16);
  need(dy, "dy", at::kBFloat16);
  TORCH_CHECK(x.is_contiguous() && dy.is_contiguous());
  auto dx = at::empty_like(x);
  auto dw = at::zeros({w.size(0), w.size(1)}, x.options().dtype(at::kFloat));
  auto db = at::zeros({w.size(0)}, x.options().dtype(at::kFloat));
  check(b200_causal_conv1d_bwd(dy.data_ptr(), x.data_ptr(), w.data_ptr(), b.has_value() ? b->data_ptr() : nullptr,
                               dx.data_ptr(), dw.data_ptr<float>(), db.data_ptr<float>(), x.size(0), x.size(1),
                               w.size(1), seq_len, act, cur_stream()), "causal_conv1d_bwd");
  return {dx, dw, db};
}

void set_attn_fwd_version(int64_t v) { b200_attn_set_fwd_version((int)v); }
void set_attn_bwd_version(int64_t v) { b200_attn_set_bwd_version((int)v); }
void set_gemm_2cta(bool on) { g_gemm_2cta = on; }
bool get_gemm_2cta() { return g_gemm_2cta; }
// GEMM with the all-gather of a unit's parameters fused in (comm warps over NVLink peer memory)
void gemm_ag(const at::Tensor& a, const at::Tensor& b, const c10::optional<at::Tensor>& c_opt, int64_t layout, int64_t epi,
             const c10::optional<at::Tensor>& residual, const at::Tensor& peer_ptrs, at::Tensor& full,
             int64_t shard_bytes, int64_t begin, int64_t end, int64_t world, int64_t rank, at::Tensor& flags,
             int64_t epoch, bool dependent, const c10::optional<at::Tensor>& bias) {
  c10::cuda::CUDAGuard guard(a.device());
  need(a, "a", at::kBFloat16);
  need(b, "b", at::kBFloat16);
  need(flags, "flags", at::kInt);
  need_rowmajor2d(a, "a");
  need_rowmajor2d(b, "b");
  if (epi == 4) {   // push epilogue: the output goes to the owners' staging slots (set_gemm_push), there is no C
    TORCH_CHECK(layout == 2 && !c_opt.has_value(), "push epilogue: tn layout, no output tensor");
    const int K = a.size(0), M = a.size(1), N = b.size(1);
    TORCH_CHECK(b.size(0) == K && M >= 256 && K % 8 == 0 && N % 8 == 0 && M % 8 == 0);
    check(b200_gemm2_ag_bf16(a.data_ptr(), b.data_ptr(), nullptr, nullptr, M, N, K, a.stride(0), b.stride(0), N, 0, 1, 1, 4,
                             (const void* const*)peer_ptrs.data_ptr(), full.data_ptr(), (unsigned long long)shard_bytes,
                             (unsigned long long)begin, (unsigned long long)end, (int)world, (int)rank,
                             (uint32_t*)flags.data_ptr(), (uint32_t)epoch, dependent ? 1 : 0, cur_stream()),
          "gemm2_ag_push_bf16_tcgen05");
    return;
  }
  TORCH_CHECK(c_opt.has_value(), "gemm_ag: output tensor required");
  at::Tensor c = *c_opt;
  need(c, "c", at::kBFloat16);
  need_rowmajor2d(c, "c");
  int M, N, K, a_mn = 0, b_mn = 0;
  if (layout == 0) { M = a.size(0); K = a.size(1); N = b.size(0); TORCH_CHECK(b.size(1) == K); }
  else if (layout == 1) { M = a.size(0); K = a.size(1); N = b.size(1); b_mn = 1; TORCH_CHECK(b.size(0) == K); }
  else { K = a.size(0); M = a.size(1); N = b.size(1); a_mn = b_mn = 1; TORCH_CHECK(b.size(0) == K); }
  TORCH_CHECK(c.size(0) == M && c.size(1) == (epi == 6 ? 2 * N : N) && M >= 256 && K % 8 == 0 && N % 8 == 0 && M % 8 == 0);
  const void* r = nullptr;
  int ldr = 0;
  if (epi == 1) {
    TORCH_CHECK(residual.has_value());
    need(*residual, "residual", at::kBFloat16);
    r = residual->data_ptr();
    ldr = residual->stride(0);
  }
  if (bias.has_value() && bias->defined()) {
    TORCH_CHECK((epi == 0 || epi == 3) && layout == 0, "bias epilogue: nt layout, store or RoPE epilogue");
    r = bias_operand(bias, N);
    ldr = 0;
    epi |= kEpiBias;
  }
  check(b200_gemm2_ag_bf16(a.data_ptr(), b.data_ptr(), c.data_ptr(), r, M, N, K, a.stride(0), b.stride(0), c.stride(0), ldr,
                           a_mn, b_mn, (int)epi, (const void* const*)peer_ptrs.data_ptr(), full.data_ptr(),
                           (unsigned long long)shard_bytes, (unsigned long long)begin, (unsigned long long)end, (int)world,
                           (int)rank, (uint32_t*)flags.data_ptr(), (uint32_t)epoch, dependent ? 1 : 0, cur_stream()),
        "gemm2_ag_bf16_tcgen05");
}
// wgrad GEMM (tn: dW[M,N] = a[K,M]^T b[K,N]) whose epilogue pushes every tile to the owning rank's staging slot
void gemm_push(const at::Tensor& a, const at::Tensor& b) {
  c10::cuda::CUDAGuard guard(a.device());
  need(a, "a", at::kBFloat16);
  need(b, "b", at::kBFloat16);
  need_rowmajor2d(a, "a");
  need_rowmajor2d(b, "b");
  const int K = a.size(0), M = a.size(1), N = b.size(1);
  TORCH_CHECK(b.size(0) == K && g_gemm_2cta && M >= 256 && K % 8 == 0 && N % 8 == 0 && M % 8 == 0,
              "push epilogue: CTA-pair kernel (M >= 256), dims multiples of 8");
  check(b200_gemm2_bf16(a.data_ptr(), b.data_ptr(), nullptr, nullptr, M, N, K, a.stride(0), b.stride(0), N, 0, 1, 1, 4, 0,
                        cur_stream()), "gemm2_push_bf16_tcgen05");
}
// optional fp8 forward path: row-wise e4m3 quantisation and the e4m3 x e4m3 -> bf16 GEMM (kind::f8f6f4)
std::vector<at::Tensor> quant_rowwise_e4m3(const at::Tensor& x) {
  c10::cuda::CUDAGuard guard(x.device());
  need(x, "x", at::kBFloat16);
  need_rowmajor2d(x, "x");
  TORCH_CHECK(x.size(1) % 16 == 0, "quant_rowwise_e4m3: K must be a multiple of 16");
  auto q = at::empty({x.size(0), x.size(1)}, x.options().dtype(at::kByte));
  auto sc = at::empty({x.size(0)}, x.options().dtype(at::kFloat));
  check(b200_quant_rowwise_e4m3(x.data_ptr(), q.data_ptr(), sc.data_ptr<float>(), (int)x.size(0), (int)x.size(1),
                                (int)x.stride(0), (int)q.stride(0), cur_stream()), "quant_rowwise_e4m3");
  return {q, sc};
}
void gemm_fp8(const at::Tensor& aq, const at::Tensor& bq, const at::Tensor& sa, const at::Tensor& sb, at::Tensor& c) {
  c10::cuda::CUDAGuard guard(aq.device());
  need(aq, "a_q", at::kByte); need(bq, "b_q", at::kByte); need(sa, "scale_a", at::kFloat); need(sb, "scale_b", at::kFloat);
  need(c, "c", at::kBFloat16);
  need_rowmajor2d(aq, "a_q"); need_rowmajor2d(bq, "b_q"); need_rowmajor2d(c, "c");
  const int M = aq.size(0), K = aq.size(1), N = bq.size(0);
  TORCH_CHECK(bq.size(1) == K && c.size(0) == M && c.size(1) == N && sa.numel() == M && sb.numel() == N &&
              sa.is_contiguous() && sb.is_contiguous(), "gemm_fp8: shape mismatch");
  check(b200_gemm2_fp8(aq.data_ptr(), bq.data_ptr(), c.data_ptr(), sa.data_ptr<float>(), sb.data_ptr<float>(), M, N, K,
                       (int)aq.stride(0), (int)bq.stride(0), (int)c.stride(0), cur_stream()), "gemm2_fp8_tcgen05");
}
// db [N] (bf16 or fp32) = column sums of dy [M, N] bf16, or db += them (accumulate); deterministic (fixed split, no atomics)
void bias_grad(const at::Tensor& dy, at::Tensor& db, bool accumulate) {
  c10::cuda::CUDAGuard guard(dy.device());
  need(dy, "dy", at::kBFloat16);
  need_rowmajor2d(dy, "dy");
  const int M = dy.size(0), N = dy.size(1);
  TORCH_CHECK(dy.is_contiguous() && N % 8 == 0, "bias_grad: dy must be contiguous [M, N] with N % 8 == 0");
  TORCH_CHECK(db.is_cuda() && db.is_contiguous() && db.numel() == N &&
              (db.scalar_type() == at::kBFloat16 || db.scalar_type() == at::kFloat), "bias_grad: db must be [N] bf16 or fp32");
  auto part = at::empty({b200_bias_grad_partials(M, N), N}, dy.options().dtype(at::kFloat));
  check(b200_bias_grad(dy.data_ptr(), part.data_ptr<float>(), db.data_ptr(), db.scalar_type() == at::kFloat ? 1 : 0, M, N,
                       accumulate ? 1 : 0, cur_stream()), "bias_grad", 2);
}
void p2p_gather_range(const at::Tensor& peer_ptrs, at::Tensor& full, int64_t shard_bytes, int64_t begin, int64_t end) {
  c10::cuda::CUDAGuard guard(full.device());
  check(b200_p2p_gather_range((const void* const*)peer_ptrs.data_ptr(), full.data_ptr(), shard_bytes, begin, end, cur_stream()),
        "p2p_gather_range");
}

at::Tensor ts_mma_probe(const at::Tensor& a, const at::Tensor& b) {
  c10::cuda::CUDAGuard guard(a.device());
  need(a, "a", at::kBFloat16);
  need(b, "b", at::kBFloat16);
  TORCH_CHECK(a.is_contiguous() && b.is_contiguous() && a.size(0) == 128 && a.size(1) == 64 && b.size(0) == 64 && b.size(1) == 64);
  auto d = at::empty({128, 64}, a.options().dtype(at::kFloat));
  check(b200_ts_mma_probe(a.data_ptr(), b.data_ptr(), d.data_ptr<float>(), cur_stream()), "ts_mma_probe");
  return d;
}
int64_t launch_count() { return g_launches; }
void reset_launch_count() { g_launches = 0; }

}  // namespace


// ------------------------------------------------------------------------------ Mamba2 SSD chunk scan (csrc/ssd.cu)
// Orchestration of the batched tcgen05 GEMMs and the glue kernels.  Internal chunk length is 128 tokens whatever
// the model's chunk_size (the chunked form is exact for every chunking).
namespace {
constexpr int kL = 128;
struct SsdDims {
  long long M; int H, P, G, Nd, Hg, HP, GN, nbc, batch, nc;
};
struct SsdFwd {
  at::Tensor dtv, acs, aL, CB, Mh, xs, states, prev, yd, yoff;
};
SsdDims ssd_dims(const at::Tensor& x, const at::Tensor& Bm, int64_t seq_len) {
  SsdDims d;
  d.M = x.size(0); d.H = x.size(1); d.P = x.size(2); d.G = Bm.size(1); d.Nd = Bm.size(2);
  TORCH_CHECK(seq_len % kL == 0 && d.M % seq_len == 0, "ssd: seq_len must be a multiple of 128");
  TORCH_CHECK(d.H % d.G == 0 && d.P % 32 == 0 && d.Nd % 8 == 0, "ssd: unsupported head/state dims");
  d.Hg = d.H / d.G; d.HP = d.H * d.P; d.GN = d.G * d.Nd; d.nbc = (int)(d.M / kL);
  d.batch = (int)(d.M / seq_len); d.nc = (int)(seq_len / kL);
  return d;
}
void bg(const void* A, const void* B, void* C, int M, int N, int K, int lda, int ldb, int ldc, int nb0, int nb1,
        long long sa0, long long sa1, long long sb0, long long sb1, long long sc0, long long sc1, int a_mn, int b_mn, int epi,
        int f32, const char* what) {
  check(b200_bgemm_bf16(A, B, C, M, N, K, lda, ldb, ldc, nb0, nb1, sa0, sa1, sb0, sb1, sc0, sc1, a_mn, b_mn, epi, f32,
                        cur_stream()), what);
}
SsdFwd ssd_forward_internals(const SsdDims& d, const at::Tensor& x, const at::Tensor& dt, const at::Tensor& A,
                             const at::Tensor& Bm, const at::Tensor& Cm, const float* bias, bool softplus) {
  SsdFwd f;
  auto f32 = x.options().dtype(at::kFloat);
  auto bf = x.options();
  const long long LL = (long long)kL * kL;
  f.dtv = at::empty({d.M, d.H}, f32); f.acs = at::empty({d.M, d.H}, f32); f.aL = at::empty({d.nbc, d.H}, f32);
  check(b200_ssd_prep(dt.data_ptr(), A.data_ptr<float>(), bias, f.dtv.data_ptr<float>(), f.acs.data_ptr<float>(),
                      f.aL.data_ptr<float>(), d.nbc, d.H, softplus ? 1 : 0, cur_stream()), "ssd_prep");
  f.CB = at::empty({d.nbc, d.G, kL, kL}, bf);
  bg(Cm.data_ptr(), Bm.data_ptr(), f.CB.data_ptr(), kL, kL, d.Nd, d.GN, d.GN, kL, d.G, d.nbc, d.Nd, (long long)kL * d.GN,
     d.Nd, (long long)kL * d.GN, LL, d.G * LL, 0, 0, 0, 0, "ssd_bgemm_CB");
  f.Mh = at::empty({d.nbc, d.H, kL, kL}, bf);
  check(b200_ssd_mask(f.CB.data_ptr(), f.acs.data_ptr<float>(), f.dtv.data_ptr<float>(), f.Mh.data_ptr(), d.nbc, d.H, d.G,
                      cur_stream()), "ssd_mask");
  f.yd = at::empty({d.M, d.H, d.P}, bf);
  bg(f.Mh.data_ptr(), x.data_ptr(), f.yd.data_ptr(), kL, d.P, kL, kL, d.HP, d.HP, d.H, d.nbc, LL, d.H * LL, d.P,
     (long long)kL * d.HP, d.P, (long long)kL * d.HP, 0, 1, 0, 0, "ssd_bgemm_Ydiag");
  f.xs = at::empty({d.M, d.H, d.P}, bf);
  check(b200_ssd_xs(x.data_ptr(), f.dtv.data_ptr<float>(), f.acs.data_ptr<float>(), f.aL.data_ptr<float>(), f.xs.data_ptr(),
                    d.M, d.H, d.P, cur_stream()), "ssd_xs");
  f.states = at::empty({d.nbc, d.Nd, d.HP}, f32);
  bg(Bm.data_ptr(), f.xs.data_ptr(), f.states.data_ptr(), d.Nd, d.Hg * d.P, kL, d.GN, d.HP, d.HP, d.G, d.nbc, d.Nd,
     (long long)kL * d.GN, (long long)d.Hg * d.P, (long long)kL * d.HP, (long long)d.Hg * d.P, (long long)d.Nd * d.HP, 1, 1, 0, 1,
     "ssd_bgemm_states");
  f.prev = at::empty({d.nbc, d.Nd, d.HP}, bf);
  check(b200_ssd_state_pass(f.states.data_ptr<float>(), f.aL.data_ptr<float>(), f.prev.data_ptr(), d.batch, d.nc, d.Nd, d.H,
                            d.P, cur_stream()), "ssd_state_pass");
  f.yoff = at::empty({d.M, d.H, d.P}, bf);
  bg(Cm.data_ptr(), f.prev.data_ptr(), f.yoff.data_ptr(), kL, d.Hg * d.P, d.Nd, d.GN, d.HP, d.HP, d.G, d.nbc, d.Nd,
     (long long)kL * d.GN, (long long)d.Hg * d.P, (long long)d.Nd * d.HP, (long long)d.Hg * d.P, (long long)kL * d.HP, 0, 1, 0, 0,
     "ssd_bgemm_Yoff");
  return f;
}
void ssd_check_inputs(const at::Tensor& x, const at::Tensor& dt, const at::Tensor& A, const at::Tensor& Bm,
                      const at::Tensor& Cm) {
  need(x, "x", at::kBFloat16); need(dt, "dt", at::kBFloat16); need(Bm, "B", at::kBFloat16); need(Cm, "C", at::kBFloat16);
  need(A, "A", at::kFloat);
  TORCH_CHECK(x.dim() == 3 && dt.dim() == 2 && Bm.dim() == 3 && Cm.dim() == 3, "ssd: x [M,H,P], dt [M,H], B/C [M,G,N]");
  TORCH_CHECK(x.is_contiguous() && dt.is_contiguous() && Bm.is_contiguous() && Cm.is_contiguous() && A.is_contiguous(),
              "ssd: inputs must be contiguous");
}
}  // namespace

at::Tensor ssd_scan_fwd(const at::Tensor& x, const at::Tensor& dt, const at::Tensor& A, const at::Tensor& Bm,
                        const at::Tensor& Cm, const c10::optional<at::Tensor>& D, const c10::optional<at::Tensor>& dt_bias,
                        int64_t seq_len, bool softplus) {
  c10::cuda::CUDAGuard guard(x.device());
  ssd_check_inputs(x, dt, A, Bm, Cm);
  const SsdDims d = ssd_dims(x, Bm, seq_len);
  const float* bias = dt_bias.has_value() ? dt_bias->data_ptr<float>() : nullptr;
  SsdFwd f = ssd_forward_internals(d, x, dt, A, Bm, Cm, bias, softplus);
  auto y = at::empty_like(x);
  check(b200_ssd_combine(f.yd.data_ptr(), f.yoff.data_ptr(), x.data_ptr(), f.acs.data_ptr<float>(),
                         D.has_value() ? D->data_ptr<float>() : nullptr, y.data_ptr(), d.M, d.H, d.P, cur_stream()),
        "ssd_combine");
  return y;
}

// returns dx, ddt (bf16), dA, dB, dC (B/C dtype), dD, ddt_bias (fp32; undefined tensors when the input was absent)
std::vector<at::Tensor> ssd_scan_bwd(const at::Tensor& dy, const at::Tensor& x, const at::Tensor& dt, const at::Tensor& A,
                                     const at::Tensor& Bm, const at::Tensor& Cm, const c10::optional<at::Tensor>& D,
                                     const c10::optional<at::Tensor>& dt_bias, int64_t seq_len, bool softplus) {
  c10::cuda::CUDAGuard guard(x.device());
  ssd_check_inputs(x, dt, A, Bm, Cm);
  need(dy, "dy", at::kBFloat16);
  TORCH_CHECK(dy.is_contiguous() && dy.sizes() == x.sizes(), "ssd: dy must match x");
  const SsdDims d = ssd_dims(x, Bm, seq_len);
  const float* bias = dt_bias.has_value() ? dt_bias->data_ptr<float>() : nullptr;
  const float* Dp = D.has_value() ? D->data_ptr<float>() : nullptr;
  SsdFwd f = ssd_forward_internals(d, x, dt, A, Bm, Cm, bias, softplus);   // recompute (nothing but inputs is saved)
  auto f32 = x.options().dtype(at::kFloat);
  auto bf = x.options();
  const long long LL = (long long)kL * kL;
  const long long MH = d.M * d.H;
  // output branch: dYs = dy * exp(acs); dacs, dD partials
  auto dys = at::empty_like(x);
  auto dacs = at::empty({d.M, d.H}, f32), dDrow = at::empty({d.M, d.H}, f32);
  check(b200_ssd_dyoff(dy.data_ptr(), f.yoff.data_ptr(), x.data_ptr(), f.acs.data_ptr<float>(), dys.data_ptr(),
                       dacs.data_ptr<float>(), dDrow.data_ptr<float>(), MH, d.P, cur_stream()), "ssd_dyoff");
  // intra-chunk: dMh = dy x^T ; dx_diag = Mh^T dy
  auto dMh = at::empty({d.nbc, d.H, kL, kL}, bf);
  bg(dy.data_ptr(), x.data_ptr(), dMh.data_ptr(), kL, kL, d.P, d.HP, d.HP, kL, d.H, d.nbc, d.P, (long long)kL * d.HP, d.P,
     (long long)kL * d.HP, LL, d.H * LL, 0, 0, 0, 0, "ssd_bgemm_dMh");
  auto dxd = at::empty_like(x);
  bg(f.Mh.data_ptr(), dy.data_ptr(), dxd.data_ptr(), kL, d.P, kL, kL, d.HP, d.HP, d.H, d.nbc, LL, d.H * LL, d.P,
     (long long)kL * d.HP, d.P, (long long)kL * d.HP, 1, 1, 0, 0, "ssd_bgemm_dxdiag");
  f.Mh = at::Tensor();
  auto ddtv = at::zeros({d.M, d.H}, f32);
  auto dCB = at::empty({d.nbc, d.G, kL, kL}, bf);
  check(b200_ssd_mask_bwd(dMh.data_ptr(), f.CB.data_ptr(), f.acs.data_ptr<float>(), f.dtv.data_ptr<float>(), dCB.data_ptr(),
                          dacs.data_ptr<float>(), ddtv.data_ptr<float>(), d.nbc, d.H, d.G, cur_stream()), "ssd_mask_bwd");
  dMh = at::Tensor();
  auto dC32 = at::empty({d.M, d.G, d.Nd}, f32), dB32 = at::empty({d.M, d.G, d.Nd}, f32);
  bg(dCB.data_ptr(), Bm.data_ptr(), dC32.data_ptr(), kL, d.Nd, kL, kL, d.GN, d.GN, d.G, d.nbc, LL, d.G * LL, d.Nd,
     (long long)kL * d.GN, d.Nd, (long long)kL * d.GN, 0, 1, 0, 1, "ssd_bgemm_dC_diag");
  bg(dCB.data_ptr(), Cm.data_ptr(), dB32.data_ptr(), kL, d.Nd, kL, kL, d.GN, d.GN, d.G, d.nbc, LL, d.G * LL, d.Nd,
     (long long)kL * d.GN, d.Nd, (long long)kL * d.GN, 1, 1, 0, 1, "ssd_bgemm_dB_diag");
  // inter-chunk: dprev = C^T dYs ; dC += dYs prev^T
  auto dprev = at::empty({d.nbc, d.Nd, d.HP}, f32);
  bg(Cm.data_ptr(), dys.data_ptr(), dprev.data_ptr(), d.Nd, d.Hg * d.P, kL, d.GN, d.HP, d.HP, d.G, d.nbc, d.Nd,
     (long long)kL * d.GN, (long long)d.Hg * d.P, (long long)kL * d.HP, (long long)d.Hg * d.P, (long long)d.Nd * d.HP, 1, 1, 0, 1,
     "ssd_bgemm_dprev");
  bg(dys.data_ptr(), f.prev.data_ptr(), dC32.data_ptr(), kL, d.Nd, d.Hg * d.P, d.HP, d.HP, d.GN, d.G, d.nbc,
     (long long)d.Hg * d.P, (long long)kL * d.HP, (long long)d.Hg * d.P, (long long)d.Nd * d.HP, d.Nd, (long long)kL * d.GN, 0, 0, 2,
     1, "ssd_bgemm_dC_off");
  auto dstates = at::empty({d.nbc, d.Nd, d.HP}, bf);
  auto daL = at::zeros({d.nbc, d.H}, f32);
  check(b200_ssd_state_pass_bwd(dprev.data_ptr<float>(), f.prev.data_ptr(), f.aL.data_ptr<float>(), dstates.data_ptr(),
                                daL.data_ptr<float>(), d.batch, d.nc, d.Nd, d.H, d.P, cur_stream()), "ssd_state_pass_bwd");
  dprev = at::Tensor();
  // chunk states: dXs = B dS ; dB += Xs dS^T
  auto dxs = at::empty_like(x);
  bg(Bm.data_ptr(), dstates.data_ptr(), dxs.data_ptr(), kL, d.Hg * d.P, d.Nd, d.GN, d.HP, d.HP, d.G, d.nbc, d.Nd,
     (long long)kL * d.GN, (long long)d.Hg * d.P, (long long)d.Nd * d.HP, (long long)d.Hg * d.P, (long long)kL * d.HP, 0, 1, 0, 0,
     "ssd_bgemm_dXs");
  bg(f.xs.data_ptr(), dstates.data_ptr(), dB32.data_ptr(), kL, d.Nd, d.Hg * d.P, d.HP, d.HP, d.GN, d.G, d.nbc,
     (long long)d.Hg * d.P, (long long)kL * d.HP, (long long)d.Hg * d.P, (long long)d.Nd * d.HP, d.Nd, (long long)kL * d.GN, 0, 0, 2,
     1, "ssd_bgemm_dB_states");
  auto dx = at::empty_like(x);
  check(b200_ssd_dx(dxd.data_ptr(), dxs.data_ptr(), dy.data_ptr(), x.data_ptr(), f.dtv.data_ptr<float>(),
                    f.acs.data_ptr<float>(), f.aL.data_ptr<float>(), Dp, dx.data_ptr(), ddtv.data_ptr<float>(),
                    dacs.data_ptr<float>(), daL.data_ptr<float>(), MH, d.H, d.P, cur_stream()), "ssd_dx");
  auto ddt = at::empty_like(dt);
  auto dA = at::zeros({d.H}, f32);
  at::Tensor dbias;
  if (dt_bias.has_value()) dbias = at::zeros({d.H}, f32);
  check(b200_ssd_dt_bwd(dt.data_ptr(), A.data_ptr<float>(), bias, f.dtv.data_ptr<float>(), dacs.data_ptr<float>(),
                        ddtv.data_ptr<float>(), daL.data_ptr<float>(), ddt.data_ptr(), dA.data_ptr<float>(),
                        dbias.defined() ? dbias.data_ptr<float>() : nullptr, d.nbc, d.H, softplus ? 1 : 0, cur_stream()),
        "ssd_dt_bwd");
  at::Tensor dD;
  if (D.has_value()) dD = dDrow.sum(0);
  return {dx, ddt, dA, dB32.to(Bm.scalar_type()), dC32.to(Cm.scalar_type()), dD, dbias};
}


// ------------------------------------------------------------------------------ Mamba1 selective scan (csrc/selscan.cu)
// u, delta, z: [M, Dm] bf16; A: [Dm, 16] fp32; B, C: [M, 16] bf16; D, delta_bias: [Dm] fp32.
std::vector<at::Tensor> selective_scan_fwd(const at::Tensor& u, const at::Tensor& delta, const at::Tensor& A,
                                           const at::Tensor& Bm, const at::Tensor& Cm, const c10::optional<at::Tensor>& D,
                                           const c10::optional<at::Tensor>& z, const c10::optional<at::Tensor>& dbias,
                                           int64_t seq_len, bool softplus, bool save_carry) {
  c10::cuda::CUDAGuard guard(u.device());
  need(u, "u", at::kBFloat16); need(delta, "delta", at::kBFloat16); need(Bm, "B", at::kBFloat16); need(Cm, "C", at::kBFloat16);
  need(A, "A", at::kFloat);
  TORCH_CHECK(u.is_contiguous() && delta.is_contiguous() && Bm.is_contiguous() && Cm.is_contiguous() && A.is_contiguous());
  const int64_t M = u.size(0), Dm = u.size(1), N = A.size(1);
  TORCH_CHECK(M % seq_len == 0, "selective_scan: rows must be batch * seq_len");
  const int batch = (int)(M / seq_len);
  auto y = at::empty_like(u);
  at::Tensor hc;
  if (save_carry) hc = at::empty({batch, seq_len / 32, Dm, N}, u.options().dtype(at::kFloat));
  check(b200_selscan_fwd(u.data_ptr(), delta.data_ptr(), A.data_ptr<float>(), Bm.data_ptr(), Cm.data_ptr(),
                         D.has_value() ? D->data_ptr<float>() : nullptr, z.has_value() ? z->data_ptr() : nullptr,
                         dbias.has_value() ? dbias->data_ptr<float>() : nullptr, hc.defined() ? hc.data_ptr<float>() : nullptr,
                         y.data_ptr(), batch, (int)seq_len, (int)Dm, (int)N, softplus ? 1 : 0, cur_stream()), "selscan_fwd");
  return {y, hc};
}
std::vector<at::Tensor> selective_scan_bwd(const at::Tensor& dy, const at::Tensor& u, const at::Tensor& delta,
                                           const at::Tensor& A, const at::Tensor& Bm, const at::Tensor& Cm,
                                           const c10::optional<at::Tensor>& D, const c10::optional<at::Tensor>& z,
                                           const c10::optional<at::Tensor>& dbias, const at::Tensor& hcarry, int64_t seq_len,
                                           bool softplus) {
  c10::cuda::CUDAGuard guard(u.device());
  need(dy, "dy", at::kBFloat16);
  TORCH_CHECK(dy.is_contiguous() && dy.sizes() == u.sizes());
  const int64_t M = u.size(0), Dm = u.size(1), N = A.size(1);
  const int batch = (int)(M / seq_len);
  auto f32 = u.options().dtype(at::kFloat);
  auto du = at::empty_like(u), dd = at::empty_like(delta);
  at::Tensor dz, dD, ddb;
  if (z.has_value()) dz = at::empty_like(u);
  auto dA = at::zeros({Dm, N}, f32), dB = at::zeros({M, N}, f32), dC = at::zeros({M, N}, f32);
  if (D.has_value()) dD = at::zeros({Dm}, f32);
  if (dbias.has_value()) ddb = at::zeros({Dm}, f32);
  check(b200_selscan_bwd(dy.data_ptr(), u.data_ptr(), delta.data_ptr(), A.data_ptr<float>(), Bm.data_ptr(), Cm.data_ptr(),
                         D.has_value() ? D->data_ptr<float>() : nullptr, z.has_value() ? z->data_ptr() : nullptr,
                         dbias.has_value() ? dbias->data_ptr<float>() : nullptr, hcarry.data_ptr<float>(), du.data_ptr(),
                         dd.data_ptr(), dz.defined() ? dz.data_ptr() : nullptr, dA.data_ptr<float>(), dB.data_ptr<float>(),
                         dC.data_ptr<float>(), dD.defined() ? dD.data_ptr<float>() : nullptr,
                         ddb.defined() ? ddb.data_ptr<float>() : nullptr, batch, (int)seq_len, (int)Dm, (int)N,
                         softplus ? 1 : 0, cur_stream()), "selscan_bwd");
  return {du, dd, dA, dB, dC, dD, dz, ddb};
}

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m) {
  m.doc() = "fms_fsdp_b200 sm_100a kernels";
  m.def("gemm", &gemm, py::arg("a"), py::arg("b"), py::arg("c"), py::arg("layout"), py::arg("epi"), py::arg("residual"),
        py::arg("bias") = py::none());
  m.def("bias_grad", &bias_grad, py::arg("dy"), py::arg("db"), py::arg("accumulate") = false);
  m.def("bias_grad_partials", [](int64_t M, int64_t N) { return (int64_t)b200_bias_grad_partials((int)M, (int)N); });
  m.def("rmsnorm_fwd", &rmsnorm_fwd);
  m.def("rmsnorm_bwd", &rmsnorm_bwd, py::arg("dy"), py::arg("x"), py::arg("w"), py::arg("rstd"), py::arg("dres") = py::none());
  m.def("add_rmsnorm_fwd", &add_rmsnorm_fwd);
  m.def("rmsnorm_bwd_f32", &rmsnorm_bwd_f32);
  m.def("rmsnorm_gated_fwd", &rmsnorm_gated_fwd);
  m.def("rmsnorm_gated_bwd", &rmsnorm_gated_bwd);
  m.def("rope", &rope);
  m.def("swiglu_fwd", &swiglu_fwd);
  m.def("swiglu_bwd", &swiglu_bwd);
  m.def("embedding_fwd", &embedding_fwd);
  m.def("embedding_bwd", &embedding_bwd);
  m.def("count_valid", &count_valid);
  m.def("ce_grad_inplace", &ce_grad_inplace);
  m.def("adamw", &adamw);
  m.def("sumsq", &sumsq);
  m.def("attn_fwd", &attn_fwd);
  m.def("attn_bwd", &attn_bwd, py::arg("dout"), py::arg("qkv"), py::arg("o"), py::arg("lse"), py::arg("B"), py::arg("S"),
        py::arg("H"), py::arg("KVH"), py::arg("hd"), py::arg("scale"), py::arg("rope") = py::none());
  m.def("p2p_allgather", &p2p_allgather);
  m.def("reduce_scatter", &reduce_scatter, py::arg("peer_ptrs"), py::arg("out32"), py::arg("elem_offset"), py::arg("world"),
        py::arg("rank"), py::arg("src_bf16"), py::arg("scale"), py::arg("sumsq_out"), py::arg("max_ctas") = 0);
  m.def("allreduce_inplace", &allreduce_inplace);
  m.def("signal_barrier", &signal_barrier, py::arg("pad_ptrs"), py::arg("world"), py::arg("rank"), py::arg("epoch"),
        py::arg("anchor"), py::arg("slot_base") = 0, py::arg("mode") = 0);
  m.def("scalar_allreduce", &scalar_allreduce);
  m.def("scalar_allreduce_bytes", []() { return (int64_t)b200_scalar_allreduce_bytes(); });
  m.def("causal_conv1d_fwd", &causal_conv1d_fwd);
  m.def("causal_conv1d_bwd", &causal_conv1d_bwd);
  m.def("set_reduce_ctas", [](int64_t n) { g_reduce_ctas_default = n < 1 ? 1 : (int)n; b200_comm_set_reduce_ctas((int)n); });
  m.def("set_gemm_rope", [](const at::Tensor& table, int64_t S, int64_t hd, int64_t cols) {
    need(table, "rope table", at::kFloat);
    TORCH_CHECK(table.is_contiguous() && table.numel() >= S * hd, "rope table must be [S, hd/2, 2] fp32");
    b200_gemm2_set_rope(table.data_ptr<float>(), (int)S, (int)hd, (int)cols);
  });
  m.def("push_range", [](const at::Tensor& src, const at::Tensor& bases, int64_t n, int64_t off, int64_t rank) {
    // this rank's gradient elements [off, off + src.numel()) -> the owners' staging slots (norm gains / biases)
    c10::cuda::CUDAGuard guard(src.device());
    need(src, "src", at::kBFloat16);
    TORCH_CHECK(src.is_contiguous() && bases.scalar_type() == at::kLong && bases.is_cuda());
    check(b200_p2p_push_range(src.data_ptr(), (void* const*)bases.data_ptr(), n, off, src.numel(), (int)rank, cur_stream()),
          "p2p_push_range");
  });
  m.def("set_gemm_swiglu", [](const at::Tensor& aux, int64_t F, bool gate_first) {
    // aux: activation output [M, F] (epi 5, forward) or the saved bf16 projection [M, 2F] (epi 6, backward)
    need(aux, "aux", at::kBFloat16);
    TORCH_CHECK(aux.dim() == 2 && aux.stride(1) == 1 && (aux.size(1) == F || aux.size(1) == 2 * F));
    b200_gemm2_set_swiglu(aux.data_ptr(), (int)aux.stride(0), (int)F, gate_first ? 1 : 0);
  });
  m.def("set_gemm_push", [](const at::Tensor& bases, int64_t n, int64_t off, int64_t rank, bool bulk, int64_t rot_world) {
    // int64 device table of every rank's staging-buffer base address (fused wgrad GEMM -> reduce-scatter);
    // rot_world > 1 rotates the tile raster by rank / rot_world of a sweep (spreads the pushes over all owners)
    TORCH_CHECK(bases.is_cuda() && bases.scalar_type() == at::kLong && bases.is_contiguous(), "push table: int64 CUDA tensor");
    b200_gemm2_set_push((void* const*)bases.data_ptr(), n, off, (int)rank, bulk ? 1 : 0, (int)rot_world);
  }, py::arg("bases"), py::arg("n"), py::arg("off"), py::arg("rank"), py::arg("bulk") = true, py::arg("rot_world") = 1);
  m.def("ssd_scan_fwd", &ssd_scan_fwd);
  m.def("selective_scan_fwd", &selective_scan_fwd);
  m.def("selective_scan_bwd", &selective_scan_bwd);
  m.def("ssd_scan_bwd", &ssd_scan_bwd);
  m.def("set_attn_poly", [](int64_t f, int64_t b) { b200_attn_set_poly((int)f, (int)b); });
  m.def("set_attn_fwd_version", &set_attn_fwd_version);
  m.def("set_attn_bwd_version", &set_attn_bwd_version);
  m.def("set_gemm_2cta", &set_gemm_2cta);
  m.def("get_gemm_2cta", &get_gemm_2cta);
  m.def("gemm_ag", &gemm_ag, py::arg("a"), py::arg("b"), py::arg("c"), py::arg("layout"), py::arg("epi"), py::arg("residual"),
        py::arg("peer_ptrs"), py::arg("full"), py::arg("shard_bytes"), py::arg("begin"), py::arg("end"), py::arg("world"),
        py::arg("rank"), py::arg("flags"), py::arg("epoch"), py::arg("dependent"), py::arg("bias") = py::none());
  m.def("gemm_push", &gemm_push);
  m.def("quant_rowwise_e4m3", &quant_rowwise_e4m3);
  m.def("gemm_fp8", &gemm_fp8);
  m.def("p2p_gather_range", &p2p_gather_range);
  m.def("ts_mma_probe", &ts_mma_probe);
  m.def("launch_count", &launch_count);
  m.def("reset_launch_count", &reset_launch_count);
}
