/* libdtxtune — C ABI of the Blackwell-native DataTunerX fine-tuning worker.
 *
 * The reference (DataTunerX/datatunerx @ 508be30) has no in-process plugin API for this path: the
 * Finetune controller launches `python /tuning/train.py <argv>` (internal/controller/finetune/
 * finetune_controller.go:451-516) and everything below that command line is Python glue around
 * third-party wheels (cmd/tuning/train.py:138-305).  This header is the boundary a replacement host
 * (Go via cgo per BASELINE.json north_star; Python/ctypes in this repo because Go is not installed)
 * binds instead.  Each entry point names the reference code it replaces.
 *
 * Conventions: plain C types only; every function returns 0 on success or a negative dtx_status;
 * dtx_last_error() returns a NUL-terminated message owned by the library (valid until the next call
 * on the same handle / thread).  The caller owns every host buffer it passes; the library owns all
 * device memory.  One host thread per handle; handles on different GPUs may be driven concurrently.
 * There is no CPU fallback: without a CUDA device every compute entry point fails with DTX_ERR_CUDA.
 */
#ifndef DTXTUNE_H_
#define DTXTUNE_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DTX_ABI_VERSION 2
#if defined(__GNUC__)
#define DTX_API __attribute__((visibility("default")))
#else
#define DTX_API
#endif

typedef enum {
  DTX_OK = 0,
  DTX_ERR_INVALID = -1,      /* bad argument / unsupported configuration */
  DTX_ERR_CUDA = -2,         /* CUDA runtime / driver error (message has details) */
  DTX_ERR_NCCL = -3,         /* NCCL error or libnccl.so.2 not loadable */
  DTX_ERR_STATE = -4,        /* call sequence error (e.g. step before weights are loaded) */
  DTX_ERR_UNSUPPORTED = -5   /* accepted by the reference's CLI but not implemented natively yet */
} dtx_status;

typedef enum { DTX_F32 = 0, DTX_BF16 = 1, DTX_F16 = 2 } dtx_dtype;
typedef enum { DTX_SCHED_LINEAR = 0, DTX_SCHED_COSINE = 1, DTX_SCHED_CONSTANT = 2,
               DTX_SCHED_CONSTANT_WITH_WARMUP = 3 } dtx_sched;

/* LoRA target bits, in HF module order (cmd/tuning/parser.py:211-213 `--lora_target`; the controller
 * hard-codes "q_proj,v_proj": finetune_controller.go:482).  Any non-empty subset works.  Bit 8 (o_proj) is reserved: its
 * adapter is not implemented and dtx_trainer_create refuses it with DTX_ERR_UNSUPPORTED.
 *   bit   module                   lora_A [r, in]   lora_B [out, r]   input of the adapter
 *   1     self_attn.q_proj         [r, hidden]      [hidden, r]       input_layernorm(x)
 *   2     self_attn.k_proj         [r, hidden]      [kv_width, r]     input_layernorm(x)      (kv_width = n_kv_heads * head_dim)
 *   4     self_attn.v_proj         [r, hidden]      [kv_width, r]     input_layernorm(x)
 *   16    mlp.gate_proj            [r, hidden]      [ffn, r]          post_attention_layernorm(x)
 *   32    mlp.up_proj              [r, hidden]      [ffn, r]          post_attention_layernorm(x)
 *   64    mlp.down_proj            [r, ffn]         [hidden, r]       silu(gate) * up
 * Tensor names are "model.layers.N.<module>.lora_A.weight" / "...lora_B.weight" (a "base_model.model." prefix is accepted).
 * A is initialised U(-1/sqrt(in), 1/sqrt(in)), B = 0; one independent dropout mask per module. */
#define DTX_TARGET_Q 1u
#define DTX_TARGET_K 2u
#define DTX_TARGET_V 4u
#define DTX_TARGET_GATE 16u
#define DTX_TARGET_UP 32u
#define DTX_TARGET_DOWN 64u

/* Architecture of the frozen base model: the fields of HF config.json that LlamaForCausalLM reads
 * (loaded by AutoConfig at cmd/tuning/train.py:221). */
typedef struct {
  int32_t vocab, hidden, n_layers, n_heads, n_kv_heads, head_dim, ffn;
  float rms_eps, rope_theta;
  int32_t max_seq;
  int32_t sliding_window;  /* Mistral `sliding_window` (0 = none); only changes the mask when train.seq_len exceeds it */
} dtx_model_cfg;

/* Everything of Seq2SeqTrainingArguments / FinetuningArguments that reaches the training step
 * (cmd/tuning/train.py:196-217, 266-280; cmd/tuning/parser.py:138-149; HF defaults for the rest:
 * beta1 .9, beta2 .999, eps 1e-8, max_grad_norm 1.0, warm-up 0). */
typedef struct {
  int32_t lora_r;
  float lora_alpha, lora_dropout;
  uint32_t target_mask;
  float lr, weight_decay, beta1, beta2, eps, max_grad_norm;
  int32_t sched;         /* dtx_sched */
  int32_t warmup_steps;  /* the reference drops --warmup_ratio: effective value 0 (train.py:204) */
  int32_t total_steps;   /* optimizer steps of the whole run (drives the LR schedule) */
  int32_t grad_accum;
  int32_t micro_batch, seq_len;
  uint64_t seed;
  /* 1 = full-parameter SFT (BASELINE.json configs[3]; beyond the reference, whose worker always wraps LoRA - train.py:277):
   * every weight trains, lora_* / target_mask are ignored.  bf16 weights and gradients, fp32 master weights + Adam moments
   * sharded over the data-parallel ranks (ZeRO-1), gradients reduce-scattered per layer while the backward pass runs,
   * updated weights all-gathered; AdamW weight decay skips the RMSNorm weights (HF Trainer.get_decay_parameter_names). */
  int32_t full_finetune;
  int32_t reserved;
} dtx_train_cfg;

typedef struct dtx_trainer dtx_trainer;

/* ---- library ---- */
DTX_API int32_t dtx_abi_version(void);
/* message of the last failure on this thread when no handle is available (dtx_trainer_create) */
DTX_API const char* dtx_last_global_error(void);
DTX_API const char* dtx_last_error(const dtx_trainer* t);

/* ---- lifecycle: replaces trainer_init_per_worker's model/LoRA/optimizer setup (train.py:138-296) ---- */
/* nccl_unique_id: 128 bytes from dtx_get_nccl_unique_id on rank 0 (world > 1), else NULL. */
DTX_API int32_t dtx_trainer_create(const dtx_model_cfg* model, const dtx_train_cfg* train, int32_t device, int32_t rank,
                           int32_t world, const void* nccl_unique_id, dtx_trainer** out);
DTX_API void dtx_trainer_destroy(dtx_trainer* t);
DTX_API int32_t dtx_get_nccl_unique_id(void* out128);

/* Upload one tensor by its HF checkpoint name (AutoModelForCausalLM.from_pretrained, train.py:236-242),
 * e.g. "model.layers.3.self_attn.q_proj.weight" [out,in], "lm_head.weight", "model.norm.weight";
 * LoRA init may be overridden with "...q_proj.lora_A.weight" [r,in] / "...lora_B.weight" [out,r]. */
DTX_API int32_t dtx_load_tensor(dtx_trainer* t, const char* hf_name, const void* host, int32_t dtype, const int64_t* shape,
                        int32_t ndim);
/* Random-init base weights on the device: N(0, 0.02), norm weights 1 (HF _init_weights), seed-driven. */
DTX_API int32_t dtx_init_random_weights(dtx_trainer* t, uint64_t seed);
/* peft 0.5.0 LoRA init on the host RNG-free path: A ~ kaiming-uniform(a=sqrt 5) from `seed`, B = 0. */
DTX_API int32_t dtx_init_lora(dtx_trainer* t, uint64_t seed);

/* `--quantization int4` (cmd/tuning/train.py:224-230, bitsandbytes BitsAndBytesConfig(load_in_4bit, nf4, fp16 compute, no
 * double quantisation)): mode 4 re-stores the decoder-layer Linear weights PACKED - two 4-bit NF4 codes per byte plus one fp32
 * absmax per 64 consecutive elements (0.5625 bytes / weight instead of 2) - and frees the bf16 copies.  Each GEMM that needs a
 * weight expands it on the fly into a per-trainer bf16 scratch right before the launch (one HBM-bound kernel, bit-identical to
 * bitsandbytes' dequantize_4bit values).  Call after the base weights are loaded.
 * mode 8 (`--quantization int8`, LLM.int8 with runtime outlier decomposition) is NOT implemented: DTX_ERR_UNSUPPORTED. */
DTX_API int32_t dtx_quantize_base(dtx_trainer* t, int32_t mode);
/* bytes of device memory currently held by the frozen base weights (bf16 or packed NF4 + absmax), for reporting */
DTX_API int64_t dtx_base_weight_bytes(const dtx_trainer* t);

/* ---- the hot path: one micro-batch of HF Trainer.training_step + (at the accumulation boundary)
 * all-reduce, clip, AdamW, scheduler (train.py:299; ds_config.json ZeRO-0).
 *   input_ids / labels : host int32 [micro_batch, seq_len_batch]; labels use -100 for ignored positions and are NOT pre-shifted.
 *   seq_len_batch      : this batch's padded length - a multiple of 128, <= train.seq_len; 0 = train.seq_len.  The reference's
 *                        DataCollatorForSeq2Seq pads every batch to its own longest row (train.py:282-286): so does the host here.
 *   seq_lens           : host int32 [micro_batch] true row lengths (right padding beyond them), or NULL = every row is full.
 *                        Attention tiles that lie entirely in a row's padding are skipped (their outputs are written as zeros).
 *   flags              : DTX_STEP_FORCE = run the optimizer step after this micro-batch even if fewer than grad_accum have been
 *                        accumulated (HF Trainer's end-of-epoch step when an epoch holds fewer batches than grad_accum).
 * Outputs (host): mean token loss of this micro-batch, global grad-norm before clipping and the lr used
 * (both only meaningful when *stepped_out == 1). */
#define DTX_STEP_FORCE 1
DTX_API int32_t dtx_step(dtx_trainer* t, const int32_t* input_ids, const int32_t* labels, const int32_t* seq_lens,
                 int32_t seq_len_batch, int32_t flags, float* loss_out, float* grad_norm_out, float* lr_out,
                 int32_t* stepped_out);
/* Same with the batch already resident on this trainer's device (int32 device pointers; d_seq_lens may be NULL). */
DTX_API int32_t dtx_step_device(dtx_trainer* t, const void* d_input_ids, const void* d_labels, const void* d_seq_lens,
                        int32_t seq_len_batch, int32_t flags, float* loss_out, float* grad_norm_out, float* lr_out,
                        int32_t* stepped_out);
/* Forward only: SFTTrainer.evaluate's eval_loss (cmd/tuning/trainer.py:324-327).  row_loss_sum_out / row_valid_out (host,
 * [micro_batch], may be NULL) receive each row's summed token loss and number of valid tokens so that the host can form HF's
 * per_device_eval_batch_size batches whatever the native micro-batch is. */
DTX_API int32_t dtx_eval_loss(dtx_trainer* t, const int32_t* input_ids, const int32_t* labels, const int32_t* seq_lens,
                      int32_t seq_len_batch, float* loss_out, float* row_loss_sum_out, int32_t* row_valid_out);
/* Sum a small host array over all ranks of this trainer's communicator (NCCL; a no-op when world == 1).  Used for the
 * evaluation mean across ranks (HF gathers the eval losses of all processes). */
DTX_API int32_t dtx_allreduce_host(dtx_trainer* t, double* inout, int32_t n);

/* ---- export: trainer.save_model writes the PEFT adapter (train.py:300).  hf_name as in
 * dtx_load_tensor ("...lora_A.weight" / "...lora_B.weight"); fp32, row-major, caller-sized. */
DTX_API int32_t dtx_export_adapter(dtx_trainer* t, const char* hf_name, void* host_out, int64_t nbytes);
/* The gradient the last optimizer step consumed, in the same naming and layout: the SUM over ranks and accumulated
 * micro-batches of d(mean token loss)/d(tensor), before the 1/(world*grad_accum) scaling and clipping (parity tests). */
DTX_API int32_t dtx_export_adapter_grad(dtx_trainer* t, const char* hf_name, void* host_out, int64_t nbytes);
/* Full-parameter SFT: one weight (grad = 0) or its accumulated gradient (grad = 1) by HF checkpoint name, as bf16 bit patterns
 * in the HF layout - what trainer.save_model writes for a full fine-tune. */
DTX_API int32_t dtx_export_weight(dtx_trainer* t, const char* hf_name, void* host_out_bf16, int64_t nbytes, int32_t grad);
/* trainable parameters: LoRA = n_layers * sum over the enabled targets of r * (in + out) (Llama-2-7B at r = 16: q,v 8 388 608;
 * gate,up,down 23 199 744; q,k,v,gate,up,down 35 782 656); full-parameter SFT = every weight */
DTX_API int64_t dtx_num_trainable(const dtx_trainer* t);
/* kernels launched by this trainer since creation (bench.py's gpu_launches) */
DTX_API int64_t dtx_launch_count(const dtx_trainer* t);
/* device time of the most recent dtx_step in ms (CUDA events on the trainer's stream) */
DTX_API float dtx_last_step_ms(const dtx_trainer* t);
/* event-timed segments of the most recent dtx_step in ms: out[0] whole step, out[1] forward + backward, out[2] gradient
 * all-reduce (0 when world == 1 or no optimizer step ran), out[3] grad-norm + clip + AdamW + adapter refresh */
DTX_API int32_t dtx_last_step_timings(const dtx_trainer* t, float* out4);
/* How the last training micro-batch was run: 0 = packed (sequences back to back, one pass), 1 = one pass at the padded shape,
 * > 1 = that many length groups (see "varlen_pack" / "varlen_split" below). */
DTX_API int32_t dtx_last_step_groups(const dtx_trainer* t);
/* The PACKED layout dtx_step uses for a ragged micro-batch (host arithmetic, no device): sequence b occupies rows
 * row_start_out[b] .. row_start_out[b+1]) - its length rounded up to 128, at least 128 - of one pass over row_start_out[micro_batch]
 * rows (array of micro_batch + 1 entries, micro_batch <= 64).  Returns 1 when that is fewer rows than micro_batch * seq_len_batch (the
 * step packs), 0 when packing saves nothing (one pass at the padded shape), or a negative status. */
DTX_API int32_t dtx_plan_packed_rows(int32_t micro_batch, const int32_t* seq_lens, int32_t seq_len_batch, int32_t* row_start_out);
/* The partition dtx_step would choose for a LoRA micro-batch of `micro_batch` rows with these true lengths, padded to
 * seq_len_batch (host arithmetic, no device; n_sms <= 0: 148).  order_out[micro_batch]: rows sorted by length, longest first;
 * group g = order_out[group_start_out[g] .. group_start_out[g+1]) run at padded length group_len_out[g] (arrays of micro_batch + 1
 * and micro_batch entries).  Returns the number of groups (1 = one pass at seq_len_batch) or a negative status. */
DTX_API int32_t dtx_plan_length_groups(const dtx_model_cfg* mc, int32_t micro_batch, int32_t n_sms, const int32_t* seq_lens,
                                       int32_t seq_len_batch, int32_t* order_out, int32_t* group_start_out, int32_t* group_len_out);
/* HF get_scheduler value: lr multiplier after `step` optimizer steps (host arithmetic, no device). */
DTX_API double dtx_lr_lambda(int32_t sched, int32_t step, int32_t warmup_steps, int32_t total_steps);

/* Tuning / diagnostics switches.  "gemm_pair_kernel" = 1 (default): wide GEMMs run the cta_group::2 CTA-pair kernel;
 * 0: the single-CTA kernel everywhere (used for A/B measurements in profiles/).  "fused_epilogues" = 1 (default): RoPE and
 * SwiGLU run inside the GEMM / attention epilogues; 0: separate HBM-bound kernels.  "gemm_group_m": rasterisation group of the
 * CTA-pair GEMM in 256-row tiles (default 16).  "attn_fwd_exp_fma_every" = N in {0, 2, 3, 4}: every N-th pair of the forward
 * softmax's exponentials is computed on the FMA pipe (cubic polynomial) instead of MUFU.EX2 (default 3; 0 = none).
 * "attn_dq_exp_fma_every" = N in {0, 3, 4}: the same for the dQ kernel's exp / dS phase (default 0).
 * "varlen_split" = 1 (default): a LoRA micro-batch that comes with row lengths is run as length groups (rows sorted by length,
 * partition chosen by a cost model; same token-mean loss and gradients up to summation order); 0: one pass at the batch's length.
 * "varlen_pack" = 1 (default): such a micro-batch (LoRA or full-parameter) is instead run PACKED - sequences back to back at their
 * 128-rounded lengths, one pass - whenever the fused RoPE epilogue applies (q|k|v width a multiple of 256); 0: length groups.
 * "varlen_group_cost" = N: fixed cost the partition's cost model charges per group, in thousandths of one wave of every GEMM of a layer.
 * "nf4_prefetch" = 1 (default): with --quantization int4 the next matrix is expanded on a side stream under the current GEMM
 * (read at dtx_quantize_base time); 0: expansion inline on the main stream.  Unknown names return DTX_ERR_INVALID. */
DTX_API int32_t dtx_set_option(const char* name, int32_t value);

/* ---- per-kernel entry points (raw device pointers, `stream` = cudaStream_t or NULL) for the parity
 * tests and for ncu captures.  Shapes are documented in datatunerx_b200/csrc/kernels.h. ---- */
DTX_API int32_t dtx_gemm_bf16(const void* A, int64_t lda, int32_t a_mn_major, const void* B, int64_t ldb, int32_t b_mn_major,
                      const void* A2, int64_t lda2, const void* B2, int64_t ldb2, int32_t K2, void* C, int64_t ldc,
                      const void* R, int64_t ldr, int32_t M, int32_t N, int32_t K, int32_t epilogue, int32_t split_k,
                      int32_t block_n, void* stream);
/* The fused epilogues of the CTA-pair GEMM as the training step runs them (M > 128, B operand K-major or MN-major):
 *   epilogue 3 (RoPE)        : C[M,N] bf16 = rotary(acc) on columns < rope_cols (head_dim 128, half-split pairs i / i+64, position =
 *                              row % rope_S), plain beyond; rope_cs = device [rope_S][64] float2 (cos, sin) from dtx_rope_table
 *   epilogue 4 (SwiGLU fwd)  : B rows in the GU-interleaved layout (128 gate rows | 128 up rows per 128 features): C[M,N] = acc
 *                              (the interleaved gate|up activations), aux[M, N/2] = silu(gate) * up
 *   epilogue 5 (SwiGLU bwd)  : acc = d(act) [M, N=F]; aux = saved gate|up [M, 2F] (interleaved, ld_aux = 2F); C[M, 2F] = d(gate|up)
 * A2/B2/K2 extend the contraction as in dtx_gemm_bf16. */
DTX_API int32_t dtx_gemm_fused(const void* A, int64_t lda, const void* B, int64_t ldb, int32_t b_mn_major, const void* A2,
                       int64_t lda2, const void* B2, int64_t ldb2, int32_t K2, void* C, int64_t ldc, void* aux, int64_t ld_aux,
                       const void* rope_cs, int32_t rope_S, int32_t rope_cols, int32_t M, int32_t N, int32_t K,
                       int32_t epilogue, void* stream);
DTX_API int32_t dtx_embedding_fwd(const void* ids, const void* table, void* out, int32_t M, int32_t d, int32_t vocab, void* stream);
DTX_API int32_t dtx_rmsnorm_fwd(const void* x, const void* w, void* y, void* rstd, int32_t M, int32_t d, float eps, void* stream);
DTX_API int32_t dtx_rmsnorm_bwd(const void* dy, const void* x, const void* w, const void* rstd, const void* dres, void* dx,
                        int32_t M, int32_t d, void* stream);
DTX_API int32_t dtx_rope_table(void* cs_out_device, int32_t S, int32_t D, float theta, void* stream);
DTX_API int32_t dtx_rope_qk(void* qkv, const void* cs_table, int32_t B, int32_t S, int32_t H, int32_t Hkv, int32_t D,
                    int32_t inverse, void* stream);
DTX_API int32_t dtx_swiglu_fwd(const void* gu, void* act, int32_t M, int32_t F, void* stream);
DTX_API int32_t dtx_swiglu_bwd(const void* dact, const void* gu, void* dgu, int32_t M, int32_t F, void* stream);
/* LoRA dropout with counter-based masks: hd[M, nt*d] = per-target dropped copies of h[M, d] (peft: lora_A(lora_dropout(x)),
 * one nn.Dropout per wrapped module); dh[M, d] += sum_t mask_t o g[:, t*d:(t+1)*d] / (1 - p) regenerates the same masks. */
DTX_API int32_t dtx_lora_dropout_fwd(const void* h, void* hd, int32_t M, int32_t d, int32_t nt, float p, uint64_t key, void* stream);
DTX_API int32_t dtx_lora_dropout_bwd_add(void* dh, const void* g, int32_t M, int32_t d, int32_t nt, float p, uint64_t key,
                                 void* stream);
/* LoRA dropout on down_proj's input, backward, in one pass: dgu[M, 2F] = SwiGLU backward (as dtx_swiglu_bwd) of
 * d(act) = dact + mask o g / (1 - p), where g [M, F] is the LoRA branch's input gradient and mask is the one
 * dtx_lora_dropout_fwd(act, ., M, F, 1, p, key) drew.  interleaved = 0: gu / dgu rows are [gate F | up F]; 1: the
 * GU-interleaved layout of the training step (feature f: gate at column (f/128)*256 + f%128, up 128 further). */
DTX_API int32_t dtx_swiglu_bwd_lora_dropout(const void* dact, const void* g, const void* gu, void* dgu, int32_t M, int32_t F,
                                            int32_t interleaved, float p, uint64_t key, void* stream);
DTX_API int32_t dtx_nf4_roundtrip(void* w_bf16, int64_t n, void* stream);
/* packed NF4 storage (bitsandbytes quantize_4bit layout: first element of a pair in the high nibble; one fp32 absmax per 64) */
DTX_API int32_t dtx_nf4_pack(const void* w_bf16, void* packed_u8, void* absmax_f32, int64_t n, void* stream);
DTX_API int32_t dtx_nf4_dequant(const void* packed_u8, const void* absmax_f32, void* w_bf16, int64_t n, void* stream);
DTX_API int32_t dtx_cross_entropy(const void* logits_f32, int64_t ldl, const void* labels_unshifted, void* shifted_scratch,
                          void* n_valid_scratch, void* row_loss, void* dlogits_bf16, int64_t ldd, void* loss_out,
                          int32_t B, int32_t S, int32_t V, void* stream);
DTX_API int32_t dtx_sumsq(const void* g, int64_t n, void* scratch, void* out, void* stream);
DTX_API int32_t dtx_adamw(void* p, const void* g, void* m, void* v, int64_t n, float lr, float beta1, float beta2, float eps,
                  float weight_decay, int32_t step, float grad_scale, const void* sumsq, float max_grad_norm,
                  void* grad_norm_out, void* stream);
/* attention: packed qkv [B*S, (H + 2*Hkv)*128]; Hkv < H = grouped-query attention (Mistral / Llama-2-70B).
 *   seq_lens : optional device int32 [B] true row lengths (right padding beyond): tiles entirely in the padding are skipped and
 *              their outputs written as zeros; NULL = all rows full.
 *   window   : sliding-window span (query i sees keys i - window .. i), 0 = plain causal.
 *   rope_cs_t (backward): optional TRANSPOSED rotary table [64][rope_stride] float2 - when given, dq and dk leave the kernel
 *              with the inverse rotary applied (what the training step does instead of a separate RoPE-backward kernel). */
DTX_API int32_t dtx_attn_fwd(const void* qkv, void* out, void* lse2, int32_t B, int32_t S, int32_t H, int32_t Hkv, float scale,
                     const void* seq_lens, int32_t window, void* stream);
DTX_API int32_t dtx_attn_bwd(const void* qkv, const void* out, const void* dout, const void* lse2, void* delta_scratch,
                     void* dqkv, int32_t B, int32_t S, int32_t H, int32_t Hkv, float scale, const void* seq_lens,
                     int32_t window, const void* rope_cs_t, int32_t rope_stride, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DTXTUNE_H_ */
