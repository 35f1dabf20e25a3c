// Internal (C++) launch API of libdtxtune's sm_100a kernels.  The public surface is include/dtxtune.h.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>

namespace dtx {

typedef __nv_bfloat16 bf16;

enum GemmEpilogue {
  EPI_BF16 = 0,      // C[bf16] = acc
  EPI_F32 = 1,       // C[f32]  = acc            (logits, split-K partials)
  EPI_BF16_ADD = 2,  // C[bf16] = acc + R[bf16]  (residual stream update)
  // fused epilogues of the CTA-pair kernel (256-wide N tiles; M > 128):
  EPI_ROPE = 3,        // C[bf16] = rotary(acc) on columns < rope_cols (head_dim 128, half-split), plain store beyond
  EPI_SWIGLU_FWD = 4,  // N tiles hold [gate 128 | up 128] (GU-interleaved layout): C[bf16] = acc, aux[M, N/2] = silu(gate)*up
  EPI_SWIGLU_BWD = 5,  // acc = d(act) [M, F]; reads gu = aux_in[M, 2F] (interleaved), writes d(gu) to C[M, 2F]; d(act) never stored
};

// C[M,N] = A[M,K] * B[N,K]^T (+ A2[M,K2] * B2[N,K2]^T), bf16 operands, fp32 accumulation in TMEM.
//   a_mn_major = 0: A is row-major [M, K]   (contraction dim contiguous)   lda = row stride (elements)
//   a_mn_major = 1: A is row-major [K, M]   (M contiguous)                 lda = row stride
//   b_mn_major = 0: B is row-major [N, K]                                   ldb = row stride
//   b_mn_major = 1: B is row-major [K, N]                                   ldb = row stride
// The optional second segment (A2,B2,K2) extends the contraction: it is how the LoRA up-projection
// is accumulated into the same TMEM tile as the frozen base projection.
struct GemmArgs {
  const bf16* A = nullptr; int64_t lda = 0; int a_mn_major = 0;
  const bf16* B = nullptr; int64_t ldb = 0; int b_mn_major = 0;
  const bf16* A2 = nullptr; int64_t lda2 = 0;
  const bf16* B2 = nullptr; int64_t ldb2 = 0;
  int K2 = 0;
  void* C = nullptr; int64_t ldc = 0;
  const bf16* R = nullptr; int64_t ldr = 0;
  void* aux = nullptr; int64_t ld_aux = 0;             // EPI_SWIGLU_FWD: act out; EPI_SWIGLU_BWD: gu in (ld = 2F)
  const float2* rope_cs = nullptr; int rope_S = 0, rope_cols = 0, rope_inverse = 0;  // EPI_ROPE
  const int32_t* rope_pos = nullptr;  // EPI_ROPE, optional [M]: position of every row inside its sequence (packed ragged batches); null: row % rope_S
  int M = 0, N = 0, K = 0;
  // optional device-side row count (<= M): the CTA-pair kernel skips 256-row tiles that start at or beyond it (rows up to the
  // end of the last live tile are still computed).  Lets the lm_head GEMMs run over the unmasked tokens only without a
  // device-to-host round trip for their number.
  const int32_t* m_eff = nullptr;
  int epilogue = EPI_BF16;
  int split_k = 1;  // >1 requires EPI_F32; C is [split_k][M][ldc] partial sums
  int block_n = 0;  // 0 = auto (256 for wide N, 64 for N <= 64)
};
cudaError_t gemm_bf16(const GemmArgs& a, cudaStream_t s);
int gemm_num_sms();
// 1 (default): wide GEMMs use the CTA-pair (cta_group::2) kernel; 0: single-CTA kernel everywhere (A/B measurements)
void gemm_set_pair_kernel(int on);
bool attn_bwd_can_rope();  // the backward kernels apply the inverse rotary themselves when AttnArgs::rope_cs is set
int attn_bwd_launches();   // kernels one attn_bwd() call launches (dQ (+ delta) and dK/dV)
// forward softmax: every N-th pair of exponentials (N = 2, 3, 4) is computed on the FMA pipe with a cubic polynomial instead of
// MUFU.EX2 (max. relative error 7.5e-5, far below bf16 resolution); 0 = all on the MUFU
void attn_set_fwd_exp_fma_every(int n);
void attn_set_dq_exp_fma_every(int n);  // dQ kernel: every n-th pair of exponentials on the FMA pipe (0 = none: default; 3, 4)
void gemm_set_pair_group_m(int tiles);  // rasterisation group height of the pair kernel, in 256-row tiles
// 1 (default): RoPE / SwiGLU run inside GEMM and attention epilogues; 0: separate HBM-bound kernels (A/B, tiny M)
void trainer_set_fused_epilogues(int on);
// 1 (default): --quantization int4 expands the next NF4 matrix on a side stream under the current GEMM; 0: inline
void trainer_set_nf4_prefetch(int on);
void trainer_set_varlen_group_cost(int permille);  // fixed cost per length group in the partition's cost model
void trainer_set_varlen_pack(int on);   // ragged LoRA micro-batches run packed in one pass (default 1; 0: length groups)
void trainer_set_varlen_split(int on);  // ragged micro-batches run as length groups (default 1)

// ---------------------------------------------------------------------------------------------
// flash attention (causal, head_dim 128), packed qkv layout [B*S, (H + 2*Hkv)*128] (q heads | k heads | v heads per token)
// ---------------------------------------------------------------------------------------------
struct AttnArgs {
  const bf16* qkv = nullptr;  // [B*S, (H + 2*Hkv)*D]
  bf16* out = nullptr;        // [B*S, H*D]
  float* lse = nullptr;       // [B, H, S]  natural-log sum-exp of scaled scores
  int B = 0, S = 0, H = 0;
  int Hkv = 0;                // kv heads; 0 = H (multi-head attention)
  float scale = 0.f;
  // Optional true row lengths (device int32 [B]): rows are right-padded beyond them.  Query / KV tiles that lie entirely in a
  // row's padding are skipped and their outputs (out, dq, dk, dv) written as zeros, the dK/dV kernel stops at the last query
  // block that holds a real token.  nullptr = every row is S long.
  const int32_t* seq_lens = nullptr;
  // Sliding-window attention (Mistral): query i sees keys j with i - window <= j <= i  (transformers 4.34.0
  // _make_sliding_window_causal_mask: triu(diagonal=-sliding_window)); 0 = plain causal.
  int window = 0;
  // PACKED ragged batch (optional, device int32 [B+1]): sequence b occupies rows row_start[b] .. row_start[b+1]) of qkv / out
  // (multiples of 128) instead of b*S .. (b+1)*S; S is then only the tile-grid extent and the stride of lse / delta per (b, h),
  // total_rows = row_start[B] (host copy, for the tensor maps).  Tiles beyond a sequence's rows do nothing.
  const int32_t* row_start = nullptr;
  int total_rows = 0;
  // backward
  int rope_stride = 0;              // row stride (positions) of the transposed rope table; 0 = S
  const float2* rope_cs = nullptr;  // backward only: TRANSPOSED table [64][S] (cos, sin); if set, dq and dk get the inverse rotary applied before the store
  const bf16* dout = nullptr;  // [B*S, H*D]
  bf16* dqkv = nullptr;        // [B*S, (H + 2*Hkv)*D]
  float* delta = nullptr;      // [B, H, S] scratch: rowsum(dO * O)
};
cudaError_t attn_fwd(const AttnArgs& a, cudaStream_t s);
cudaError_t attn_bwd(const AttnArgs& a, cudaStream_t s);

// ---------------------------------------------------------------------------------------------
// HBM-bound kernels
// ---------------------------------------------------------------------------------------------
cudaError_t embedding_fwd(const int32_t* ids, const bf16* table, bf16* out, int M, int d, int vocab, cudaStream_t s);
// y = w * x * rsqrt(mean(x^2) + eps);  rstd saved for backward.
// row_map (optional, [M]): row m of x is written to row row_map[m] of y; rows with row_map[m] < 0 are skipped (their rstd too).
cudaError_t rmsnorm_fwd(const bf16* x, const bf16* w, bf16* y, float* rstd, int M, int d, float eps, cudaStream_t s,
                        const int32_t* row_map = nullptr);
// dx = rstd * (w*dy) - x * rstd^3 * mean(w*dy*x)  (+ dres if not null)
// row_map (optional, [M]): the gradient of row m sits in row row_map[m] of dy; rows with row_map[m] < 0 get dx = dres (or 0).
cudaError_t rmsnorm_bwd(const bf16* dy, const bf16* x, const bf16* w, const float* rstd, const bf16* dres, bf16* dx,
                        int M, int d, cudaStream_t s, const int32_t* row_map = nullptr);
// half-split rotary embedding applied in place to the first n_rot_heads heads (q heads then k heads) of every row of
// packed qkv (row stride W elements). inverse=1 applies R^T (backward).  cs = [S][D/2] float2(cos, sin) table
cudaError_t rope_qk_inplace_table(bf16* qkv, const float2* cs, int B, int S, int n_rot_heads, int W, int D, int inverse,
                                  cudaStream_t s);
// gu [M, 2F]: [gate F | up F] (interleaved = 0) or the GU-interleaved layout the trainer uses (interleaved = 1: feature f
// has its gate at column (f/128)*256 + f%128 and its up 128 columns further); act[M,F] = silu(gate) * up
cudaError_t swiglu_fwd(const bf16* gu, bf16* act, int M, int F, int interleaved, cudaStream_t s);
// dgu[M,2F] from dact[M,F] and saved gu
cudaError_t swiglu_bwd(const bf16* dact, const bf16* gu, bf16* dgu, int M, int F, int interleaved, cudaStream_t s);
// labels_shift[b,t] = labels[b,t+1] (last = -100); n_valid counted into *n_valid (int32).
// With row_map / valid_idx (both or neither): row_map[m] = position of row m among the rows with a label (in order), or -1;
// valid_idx[k] = the k-th such row.
// pos (optional, [B*S]): position of every token inside its sequence (packed ragged batches: sequences of different lengths
// back to back) - a token is the last of its sequence when the next token's position is 0; null: rows of S tokens.
cudaError_t shift_labels(const int32_t* labels, int32_t* shifted, int32_t* n_valid, int B, int S, cudaStream_t s,
                         int32_t* row_map = nullptr, int32_t* valid_idx = nullptr, const int32_t* pos = nullptr);
// softmax cross-entropy over fp32 logits [M,V]; row_loss[M] (0 for ignored rows); dlogits bf16 = (p - onehot)/n_valid.
// valid_idx (optional): COMPACT mode - logits / dlogits row k belongs to token valid_idx[k] (k < *n_valid; other blocks
// return), labels and row_loss stay indexed by token; row_loss of unlabelled tokens must have been zeroed by the caller.
cudaError_t cross_entropy_fwd_bwd(const float* logits, int64_t ldl, const int32_t* labels, const int32_t* n_valid,
                                  float* row_loss, bf16* dlogits, int64_t ldd, int M, int V, cudaStream_t s,
                                  const int32_t* valid_idx = nullptr, int n_div = 0);
// loss = sum(row_loss)/n_valid, fixed summation order.  n_div > 0 (here and above): divide by this count instead of *n_valid
// (one length group of a micro-batch: the mean runs over the labelled tokens of all its groups); accumulate: add to *loss.
cudaError_t loss_reduce(const float* row_loss, const int32_t* n_valid, float* loss, int M, cudaStream_t s, int n_div = 0, int accumulate = 0);
// rows[i] of the [*, S_src] int32 matrices ids / labels -> row i of the [n, S_dst] outputs (S_dst <= S_src), lens_out[i] = lens[rows[i]]
struct RowList { int32_t n; int32_t rows[64]; };
// PACKED ragged batch: sequence b of the [B, S_src] inputs occupies rows start[b] .. start[b+1]) of the outputs (its length
// rounded up to 128; the padding inside keeps the source's padding ids / -100 labels), pos_out = position inside the sequence,
// start_out[B+1] = the same offsets on the device for the attention kernels.
struct RowStarts { int32_t n; int32_t start[65]; };
cudaError_t pack_rows(const int32_t* ids, const int32_t* labels, int S_src, RowStarts rs, int32_t* ids_out, int32_t* labels_out,
                      int32_t* pos_out, int32_t* start_out, cudaStream_t s);
cudaError_t gather_rows(const int32_t* ids, const int32_t* labels, const int32_t* lens, int S_src, RowList rows, int S_dst,
                        int32_t* ids_out, int32_t* labels_out, int32_t* lens_out, cudaStream_t s);
// out[i] = sum_s partial[s][i]  (fixed order)
cudaError_t sum_partials(const float* partial, float* out, int64_t n, int splits, cudaStream_t s);
// sumsq of a flat fp32 buffer, deterministic two-stage; result in *out (fp32)
cudaError_t sumsq(const float* g, int64_t n, float* scratch, float* out, cudaStream_t s);

struct AdamWArgs {
  float* p; const float* g; float* m; float* v; int64_t n;
  float lr, beta1, beta2, eps, weight_decay;
  float bias1, bias2;          // 1 - beta^t
  float grad_scale;            // 1/(world*grad_accum), applied before clipping
  const float* sumsq;          // device: sum of squares of the *unscaled* flat grad
  float max_grad_norm;         // <= 0 disables clipping
  float* grad_norm_out;        // device: scaled norm (pre-clip), may be null
};
cudaError_t adamw_step(const AdamWArgs& a, cudaStream_t s);

// LoRA dropout with counter-based masks (see elementwise.cu): hd[M, nt*d] = per-target dropped copies of h[M, d];
// dh[M, d] += sum_t mask_t o g[:, t*d:(t+1)*d] / (1-p)
cudaError_t lora_dropout_fwd(const bf16* h, bf16* hd, int M, int d, int nt, float p, uint64_t key, cudaStream_t s);
cudaError_t lora_dropout_bwd_add(bf16* dh, const bf16* g, int M, int d, int nt, float p, uint64_t key, cudaStream_t s);
// LoRA dropout on down_proj's input, backward: dgu[M,2F] = SwiGLU backward of d(act) = dact + mask o g / (1-p) (g [M,F] = the
// LoRA branch's input gradient; mask = target 0 of `key`, element m*F + f, as lora_dropout_fwd with d = F) in one pass
cudaError_t swiglu_bwd_lora_dropout(const bf16* dact, const bf16* g, const bf16* gu, bf16* dgu, int M, int F, int interleaved, float p,
                                    uint64_t key, cudaStream_t s);
// fp32 -> bf16 with scale, strided 2-D (used to refresh the bf16 LoRA shadows)
cudaError_t cast_f32_to_bf16_2d(const float* src, int64_t lds, bf16* dst, int64_t ldd, int rows, int cols, float scale,
                                int transpose, cudaStream_t s);
// w <- dequant(quant(w)) in place: NF4 with 64-element absmax blocks (bitsandbytes 4-bit, no double quantisation)
cudaError_t nf4_roundtrip_bf16(bf16* w, int64_t n, cudaStream_t s);
// packed NF4 storage (bitsandbytes quantize_4bit layout): q[i] = code(w[2i]) << 4 | code(w[2i+1]), absmax[b] = max |w| of block b
cudaError_t nf4_quantize_pack(const bf16* w, uint8_t* q, float* absmax, int64_t n, cudaStream_t s);
cudaError_t nf4_dequant_bf16(const uint8_t* q, const float* absmax, bf16* w, int64_t n, cudaStream_t s);
// per sequence: row_sum[b] = sum of row_loss over the S tokens of sequence b, row_valid[b] = tokens with a label >= 0
cudaError_t row_loss_stats(const float* row_loss, const int32_t* shifted_labels, int B, int S, float* row_sum, int32_t* row_valid,
                           cudaStream_t s, const int32_t* row_start = nullptr);  // row_start: packed batch ([B+1] first rows)
// ---- full-parameter SFT (BASELINE.json configs[3]) ----
// RMSNorm weight gradient: dw[c] (+)= sum_m dy[m,c] * x[m,c] * rstd[m]   (two-stage, fixed order; scratch >= 64 * d floats)
cudaError_t rmsnorm_dw(const bf16* dy, const bf16* x, const float* rstd, int M, int d, float* scratch, bf16* dw, int accumulate,
                       cudaStream_t s);
// embedding gradient: dE32[ids[m], :] += dx[m, :]  (fp32 atomics: the one reduction of the step whose order is not fixed)
cudaError_t embedding_bwd(const int32_t* ids, const bf16* dx, float* dE32, int M, int d, int vocab, cudaStream_t s);
// dst[i] = (accumulate ? dst[i] : 0) + src[i]   fp32 -> bf16
cudaError_t add_f32_into_bf16(const float* src, bf16* dst, int64_t n, int accumulate, cudaStream_t s);
// *out (+)= sum g[i]^2 over a bf16 buffer (two-stage, fixed order; first = 1 overwrites)
cudaError_t sumsq_bf16_acc(const bf16* g, int64_t n, float* scratch, float* out, int first, cudaStream_t s);
cudaError_t cast_bf16_to_f32(const bf16* src, float* dst, int64_t n, cudaStream_t s);
// AdamW on a shard of fp32 master weights fed by bf16 gradients; writes the updated weights back as bf16.
// Elements with index >= nodecay_from (RMSNorm weights at the end of a layer block) get no weight decay.
struct AdamWShardArgs {
  float* master; float* m; float* v; const bf16* g; bf16* w; int64_t n; int64_t nodecay_from;
  float lr, beta1, beta2, eps, weight_decay, bias1, bias2, grad_scale;
  const float* sumsq;  // device: sum of squares of the unscaled global gradient
  float max_grad_norm;
  float* grad_norm_out;
};
cudaError_t adamw_shard_step(const AdamWShardArgs& a, cudaStream_t s);

cudaError_t fill_normal_bf16(bf16* p, int64_t n, float std, uint64_t seed, cudaStream_t s);
cudaError_t fill_const_bf16(bf16* p, int64_t n, float v, cudaStream_t s);

}  // namespace dtx
