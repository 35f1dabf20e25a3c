// Per-kernel C entry points of libdtxtune (raw device pointers) — used by the parity tests and ncu captures.
#include "kernels.h"
#include "../../include/dtxtune.h"

#include <math.h>
#include <string.h>
#include <vector>

using namespace dtx;

namespace {
inline cudaStream_t S(void* s) { return static_cast<cudaStream_t>(s); }
inline int32_t rc(cudaError_t e) { return e == cudaSuccess ? DTX_OK : (e == cudaErrorInvalidValue ? DTX_ERR_INVALID : DTX_ERR_CUDA); }
}  // namespace

extern "C" {

int32_t dtx_gemm_bf16(const void* A, int64_t lda, int32_t a_mn, const void* B, int64_t ldb, int32_t b_mn, const void* A2,
                      int64_t lda2, const void* B2, int64_t ldb2, int32_t K2, void* C, int64_t ldc, const void* R, int64_t ldr,
                      int32_t M, int32_t N, int32_t K, int32_t epilogue, int32_t split_k, int32_t block_n, void* stream) {
  GemmArgs g;
  g.A = static_cast<const bf16*>(A); g.lda = lda; g.a_mn_major = a_mn;
  g.B = static_cast<const bf16*>(B); g.ldb = ldb; g.b_mn_major = b_mn;
  g.A2 = static_cast<const bf16*>(A2); g.lda2 = lda2; g.B2 = static_cast<const bf16*>(B2); g.ldb2 = ldb2; g.K2 = K2;
  g.C = C; g.ldc = ldc; g.R = static_cast<const bf16*>(R); g.ldr = ldr;
  g.M = M; g.N = N; g.K = K; g.epilogue = epilogue; g.split_k = split_k; g.block_n = block_n;
  return rc(gemm_bf16(g, S(stream)));
}

int32_t dtx_gemm_fused(const void* A, int64_t lda, const void* B, int64_t ldb, int32_t b_mn, const void* A2, int64_t lda2,
                       const void* B2, int64_t ldb2, int32_t K2, void* C, int64_t ldc, void* aux, int64_t ld_aux, const void* rope_cs,
                       int32_t rope_S, int32_t rope_cols, int32_t M, int32_t N, int32_t K, int32_t epilogue, void* stream) {
  if (epilogue < EPI_ROPE || epilogue > EPI_SWIGLU_BWD) return DTX_ERR_INVALID;
  GemmArgs g;
  g.A = static_cast<const bf16*>(A); g.lda = lda;
  g.B = static_cast<const bf16*>(B); g.ldb = ldb; g.b_mn_major = b_mn;
  g.A2 = static_cast<const bf16*>(A2); g.lda2 = lda2; g.B2 = static_cast<const bf16*>(B2); g.ldb2 = ldb2; g.K2 = K2;
  g.C = C; g.ldc = ldc; g.aux = aux; g.ld_aux = ld_aux;
  g.rope_cs = static_cast<const float2*>(rope_cs); g.rope_S = rope_S; g.rope_cols = rope_cols;
  g.M = M; g.N = N; g.K = K; g.epilogue = epilogue;
  return rc(gemm_bf16(g, S(stream)));
}

int32_t dtx_set_option(const char* name, int32_t value) {
  if (!name) return DTX_ERR_INVALID;
  if (strcmp(name, "gemm_pair_kernel") == 0) {
    gemm_set_pair_kernel(value);
    return DTX_OK;
  }
  if (strcmp(name, "gemm_group_m") == 0) {
    gemm_set_pair_group_m(value);
    return DTX_OK;
  }
  if (strcmp(name, "attn_fwd_exp_fma_every") == 0) {
    attn_set_fwd_exp_fma_every(value);
    return DTX_OK;
  }
  if (strcmp(name, "attn_dq_exp_fma_every") == 0) {
    attn_set_dq_exp_fma_every(value);
    return DTX_OK;
  }
  if (strcmp(name, "varlen_split") == 0) {
    trainer_set_varlen_split(value);
    return DTX_OK;
  }
  if (strcmp(name, "varlen_pack") == 0) {
    trainer_set_varlen_pack(value);
    return DTX_OK;
  }
  if (strcmp(name, "varlen_group_cost") == 0) {
    trainer_set_varlen_group_cost(value);
    return DTX_OK;
  }
  if (strcmp(name, "nf4_prefetch") == 0) {
    trainer_set_nf4_prefetch(value);
    return DTX_OK;
  }
  if (strcmp(name, "fused_epilogues") == 0) {
    trainer_set_fused_epilogues(value);
    return DTX_OK;
  }
  return DTX_ERR_INVALID;
}

int32_t dtx_embedding_fwd(const void* ids, const void* table, void* out, int32_t M, int32_t d, int32_t vocab, void* stream) {
  return rc(embedding_fwd(static_cast<const int32_t*>(ids), static_cast<const bf16*>(table), static_cast<bf16*>(out), M, d, vocab,
                          S(stream)));
}
int32_t dtx_rmsnorm_fwd(const void* x, const void* w, void* y, void* rstd, int32_t M, int32_t d, float eps, void* stream) {
  return rc(rmsnorm_fwd(static_cast<const bf16*>(x), static_cast<const bf16*>(w), static_cast<bf16*>(y), static_cast<float*>(rstd), M,
                        d, eps, S(stream)));
}
int32_t dtx_rmsnorm_bwd(const void* dy, const void* x, const void* w, const void* rstd, const void* dres, void* dx, int32_t M,
                        int32_t d, void* stream) {
  return rc(rmsnorm_bwd(static_cast<const bf16*>(dy), static_cast<const bf16*>(x), static_cast<const bf16*>(w),
                        static_cast<const float*>(rstd), static_cast<const bf16*>(dres), static_cast<bf16*>(dx), M, d, S(stream)));
}
int32_t dtx_rope_table(void* cs_out_device, int32_t Sq, int32_t D, float theta, void* stream) {
  const int half = D / 2;
  std::vector<float2> cs(static_cast<size_t>(Sq) * half);
  for (int pos = 0; pos < Sq; ++pos)
    for (int i = 0; i < half; ++i) {
      const float inv_freq = 1.0f / powf(theta, static_cast<float>(2 * i) / static_cast<float>(D));
      const float ang = static_cast<float>(pos) * inv_freq;
      cs[static_cast<size_t>(pos) * half + i] =
          make_float2(static_cast<float>(cos(static_cast<double>(ang))), static_cast<float>(sin(static_cast<double>(ang))));
    }
  cudaError_t e = cudaMemcpyAsync(cs_out_device, cs.data(), cs.size() * sizeof(float2), cudaMemcpyHostToDevice, S(stream));
  if (e == cudaSuccess) e = cudaStreamSynchronize(S(stream));
  return rc(e);
}
int32_t dtx_rope_qk(void* qkv, const void* cs, int32_t B, int32_t Sq, int32_t H, int32_t Hkv, int32_t D, int32_t inverse,
                    void* stream) {
  return rc(rope_qk_inplace_table(static_cast<bf16*>(qkv), static_cast<const float2*>(cs), B, Sq, H + Hkv, (H + 2 * Hkv) * D, D, inverse,
                                  S(stream)));
}
int32_t dtx_swiglu_fwd(const void* gu, void* act, int32_t M, int32_t F, void* stream) {
  return rc(swiglu_fwd(static_cast<const bf16*>(gu), static_cast<bf16*>(act), M, F, 0, S(stream)));
}
int32_t dtx_swiglu_bwd(const void* dact, const void* gu, void* dgu, int32_t M, int32_t F, void* stream) {
  return rc(swiglu_bwd(static_cast<const bf16*>(dact), static_cast<const bf16*>(gu), static_cast<bf16*>(dgu), M, F, 0, S(stream)));
}
int32_t dtx_lora_dropout_fwd(const void* h, void* hd, int32_t M, int32_t d, int32_t nt, float p, uint64_t key, void* stream) {
  return rc(lora_dropout_fwd(static_cast<const bf16*>(h), static_cast<bf16*>(hd), M, d, nt, p, key, S(stream)));
}
int32_t dtx_swiglu_bwd_lora_dropout(const void* dact, const void* g, const void* gu, void* dgu, int32_t M, int32_t F,
                                    int32_t interleaved, float p, uint64_t key, void* stream) {
  return rc(swiglu_bwd_lora_dropout(static_cast<const bf16*>(dact), static_cast<const bf16*>(g), static_cast<const bf16*>(gu),
                                    static_cast<bf16*>(dgu), M, F, interleaved, p, key, S(stream)));
}
int32_t dtx_lora_dropout_bwd_add(void* dh, const void* g, int32_t M, int32_t d, int32_t nt, float p, uint64_t key, void* stream) {
  return rc(lora_dropout_bwd_add(static_cast<bf16*>(dh), static_cast<const bf16*>(g), M, d, nt, p, key, S(stream)));
}
int32_t dtx_nf4_roundtrip(void* w_bf16, int64_t n, void* stream) {
  return rc(nf4_roundtrip_bf16(static_cast<bf16*>(w_bf16), n, S(stream)));
}
int32_t dtx_nf4_pack(const void* w_bf16, void* packed, void* absmax, int64_t n, void* stream) {
  return rc(nf4_quantize_pack(static_cast<const bf16*>(w_bf16), static_cast<uint8_t*>(packed), static_cast<float*>(absmax), n, S(stream)));
}
int32_t dtx_nf4_dequant(const void* packed, const void* absmax, void* w_bf16, int64_t n, void* stream) {
  return rc(nf4_dequant_bf16(static_cast<const uint8_t*>(packed), static_cast<const float*>(absmax), static_cast<bf16*>(w_bf16), n, S(stream)));
}
int32_t dtx_cross_entropy(const void* logits, int64_t ldl, const void* labels, void* shifted, void* n_valid, void* row_loss,
                          void* dlogits, int64_t ldd, void* loss_out, int32_t B, int32_t Sq, int32_t V, void* stream) {
  cudaError_t e = shift_labels(static_cast<const int32_t*>(labels), static_cast<int32_t*>(shifted), static_cast<int32_t*>(n_valid), B,
                               Sq, S(stream));
  if (e != cudaSuccess) return rc(e);
  e = cross_entropy_fwd_bwd(static_cast<const float*>(logits), ldl, static_cast<const int32_t*>(shifted),
                            static_cast<const int32_t*>(n_valid), static_cast<float*>(row_loss), static_cast<bf16*>(dlogits), ldd,
                            B * Sq, V, S(stream));
  if (e != cudaSuccess) return rc(e);
  return rc(loss_reduce(static_cast<const float*>(row_loss), static_cast<const int32_t*>(n_valid), static_cast<float*>(loss_out),
                        B * Sq, S(stream)));
}
int32_t dtx_sumsq(const void* g, int64_t n, void* scratch, void* out, void* stream) {
  return rc(sumsq(static_cast<const float*>(g), n, static_cast<float*>(scratch), static_cast<float*>(out), S(stream)));
}
int32_t dtx_adamw(void* p, const void* g, void* m, void* v, int64_t n, float lr, float beta1, float beta2, float eps,
                  float weight_decay, int32_t step, float grad_scale, const void* sumsq_ptr, float max_grad_norm,
                  void* grad_norm_out, void* stream) {
  AdamWArgs a;
  a.p = static_cast<float*>(p); a.g = static_cast<const float*>(g); a.m = static_cast<float*>(m); a.v = static_cast<float*>(v);
  a.n = n; a.lr = lr; a.beta1 = beta1; a.beta2 = beta2; a.eps = eps; a.weight_decay = weight_decay;
  a.bias1 = static_cast<float>(1.0 - pow(static_cast<double>(beta1), step));
  a.bias2 = static_cast<float>(1.0 - pow(static_cast<double>(beta2), step));
  a.grad_scale = grad_scale; a.sumsq = static_cast<const float*>(sumsq_ptr); a.max_grad_norm = max_grad_norm;
  a.grad_norm_out = static_cast<float*>(grad_norm_out);
  return rc(adamw_step(a, S(stream)));
}
int32_t dtx_attn_fwd(const void* qkv, void* out, void* lse2, int32_t B, int32_t Sq, int32_t H, int32_t Hkv, float scale,
                     const void* seq_lens, int32_t window, void* stream) {
  AttnArgs a;
  a.Hkv = Hkv;
  a.qkv = static_cast<const bf16*>(qkv); a.out = static_cast<bf16*>(out); a.lse = static_cast<float*>(lse2);
  a.B = B; a.S = Sq; a.H = H; a.scale = scale;
  a.seq_lens = static_cast<const int32_t*>(seq_lens); a.window = window;
  return rc(attn_fwd(a, S(stream)));
}
int32_t dtx_attn_bwd(const void* qkv, const void* out, const void* dout, const void* lse2, void* delta, void* dqkv, int32_t B,
                     int32_t Sq, int32_t H, int32_t Hkv, float scale, const void* seq_lens, int32_t window, const void* rope_cs_t,
                     int32_t rope_stride, void* stream) {
  AttnArgs a;
  a.Hkv = Hkv;
  a.qkv = static_cast<const bf16*>(qkv); a.out = const_cast<bf16*>(static_cast<const bf16*>(out));
  a.lse = const_cast<float*>(static_cast<const float*>(lse2)); a.dout = static_cast<const bf16*>(dout);
  a.delta = static_cast<float*>(delta); a.dqkv = static_cast<bf16*>(dqkv);
  a.B = B; a.S = Sq; a.H = H; a.scale = scale;
  a.seq_lens = static_cast<const int32_t*>(seq_lens); a.window = window;
  a.rope_cs = static_cast<const float2*>(rope_cs_t); a.rope_stride = rope_stride;
  return rc(attn_bwd(a, S(stream)));
}

}  // extern "C"
