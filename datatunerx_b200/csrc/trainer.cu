// The training step of the DataTunerX fine-tuning worker, rebuilt for B200.
//
// Replaces, for the data-parallel LoRA-SFT path, what the reference reaches through
//   cmd/tuning/train.py:299  trainer.train()  ->  HF Trainer.training_step / LlamaForCausalLM.forward /
//   peft lora.Linear / DeepSpeed ZeRO-0 all-reduce / clip_grad_norm_ / torch.optim.AdamW / get_scheduler
// (SURVEY §8a rows a7-a11).  One dtx_trainer = one GPU rank.  No PyTorch, no CPU fallback.
//
// HBM layout (DESIGN.md §3): frozen base weights bf16 with q|k|v and gate|up row-concatenated so that one
// GEMM serves each pair; LoRA masters fp32 in one flat buffer (A^T[d,r] | B[d,r] per target per layer) with
// m, v and the gradient in identically laid-out flat buffers (one NCCL all-reduce, one AdamW launch);
// bf16 "shadows" of the adapters padded to a 64-wide rank block feed the tensor-core GEMMs.
// Activations needed by backward are kept (no recompute: 180 GB HBM makes gradient checkpointing pointless
// for 7B LoRA at 16K tokens/step).
#include "kernels.h"
#include "../../include/dtxtune.h"

#include <cuda.h>
#include <dlfcn.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

namespace dtx {

namespace {

// ------------------------------------------------------------------------------------------------
// NCCL, loaded lazily so that libdtxtune.so has no link-time dependency (N=1 runs never touch it)
// ------------------------------------------------------------------------------------------------
struct UidByValue {  // ncclUniqueId is passed by value
  char internal[128];
};
struct NcclApi {
  void* handle = nullptr;
  int (*GetUniqueId)(void*) = nullptr;
  int (*CommInitRank)(void**, int, UidByValue, int) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  int (*ReduceScatter)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;  // (send, recv, recvcount, dtype, op, comm, stream)
  int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;           // (send, recv, sendcount, dtype, comm, stream)
  int (*CommDestroy)(void*) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
};
NcclApi* nccl_api() {
  static NcclApi api;
  static bool tried = false;
  if (!tried) {
    tried = true;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* n : names) {
      // RTLD_LOCAL: a host that imports PyTorch AFTER this call must still resolve ITS bundled NCCL's newer symbols - with
      // RTLD_GLOBAL the system libnccl (2.27) shadowed them and `import torch` died with "undefined symbol: ncclDevCommCreate"
      api.handle = dlopen(n, RTLD_NOW | RTLD_LOCAL);
      if (api.handle) break;
    }
    if (api.handle) {
      api.GetUniqueId = reinterpret_cast<int (*)(void*)>(dlsym(api.handle, "ncclGetUniqueId"));
      api.CommInitRank = reinterpret_cast<int (*)(void**, int, UidByValue, int)>(dlsym(api.handle, "ncclCommInitRank"));
      api.AllReduce = reinterpret_cast<int (*)(const void*, void*, size_t, int, int, void*, cudaStream_t)>(
          dlsym(api.handle, "ncclAllReduce"));
      api.ReduceScatter = reinterpret_cast<int (*)(const void*, void*, size_t, int, int, void*, cudaStream_t)>(
          dlsym(api.handle, "ncclReduceScatter"));
      api.AllGather = reinterpret_cast<int (*)(const void*, void*, size_t, int, void*, cudaStream_t)>(dlsym(api.handle, "ncclAllGather"));
      api.CommDestroy = reinterpret_cast<int (*)(void*)>(dlsym(api.handle, "ncclCommDestroy"));
      api.GetErrorString = reinterpret_cast<const char* (*)(int)>(dlsym(api.handle, "ncclGetErrorString"));
    }
  }
  if (!api.handle || !api.GetUniqueId || !api.CommInitRank || !api.AllReduce || !api.CommDestroy) return nullptr;
  return &api;
}
constexpr int kNcclFloat32 = 7;
constexpr int kNcclFloat64 = 8;
constexpr int kNcclBfloat16 = 9;
constexpr int kNcclSum = 0;

thread_local std::string g_error;
int g_nf4_prefetch = 1;     // expand the next NF4 matrix on a side stream while the current GEMM runs (0: inline, for A/B runs)
int g_varlen_split = 1;     // ragged micro-batches run as length groups (rows sorted by length, partition chosen by a cost model);
                            // 2: always cut where the 128-rounded lengths differ (parity tests at shapes too small for the model to split)
int g_varlen_pack = 1;      // ragged LoRA micro-batches run PACKED: sequences back to back at 128-rounded lengths, one pass (0: length groups)
int g_varlen_fix_permille = 200;   // fixed cost charged per length group, in thousandths of "one wave of every GEMM of a layer"
int g_fused_epilogues = 1;  // RoPE / SwiGLU fused into the GEMM and attention epilogues (needs M > 128: CTA-pair GEMM)

// ------------------------------------------------------------------------------------------------
// LoRA-specific small kernels
// ------------------------------------------------------------------------------------------------
// row of output feature n of a target inside its group's weight: plain (row0 + n), or GU-interleaved (wgu: 128 gate rows, then
// the 128 up rows of the same features, ...; row0 = 0 for gate, 128 for up)
__host__ __device__ __forceinline__ int target_row(int row0, int n, int gu) { return gu ? row0 + (n >> 7) * 256 + (n & 127) : row0 + n; }

// dst[n*r + j] (+)= scale * sum_s part[s*split_stride + target_row(row0, n, gu)*ld + col0 + j]   (fixed order)
__global__ void lora_gather_kernel(const float* __restrict__ part, int splits, long long split_stride, int ld, int row0, int gu,
                                   int col0, int rows, int r, float* __restrict__ dst, int accumulate, float scale) {
  const long long total = static_cast<long long>(rows) * r;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int n = static_cast<int>(i / r), j = static_cast<int>(i % r);
    const float* src = part + static_cast<long long>(target_row(row0, n, gu)) * ld + col0 + j;
    float s = 0.f;
    for (int k = 0; k < splits; ++k) s += src[k * split_stride];
    s *= scale;
    dst[i] = accumulate ? dst[i] + s : s;
  }
}

// Adapter groups: the targets that share one input and one frozen weight, so that one LoRA down-projection GEMM serves all
// of them and their up-projection rides as a K-extension of that weight's GEMM.
enum { G_ATT = 0, G_GU = 1, G_DN = 2, N_GROUPS = 3 };  // q|k|v -> wqkv (input h1), gate|up -> wgu (h2), down -> wdown (act)
constexpr int kMaxTargets = 6;                        // q, k, v, gate, up, down (o_proj is not implemented)
// the linear modules of a decoder layer in HF module order: bit i of dtx_train_cfg.target_mask selects module i
const char* const kModules[7] = {"q_proj", "k_proj", "v_proj", "o_proj", "gate_proj", "up_proj", "down_proj"};
constexpr int kModO = 3;

// Per-target geometry of the LoRA adapters inside one layer's block of the flat parameter buffer.
struct TargetInfo {
  int group;       // G_ATT / G_GU / G_DN
  int gi;          // position inside the group: rank block gi*r of the group's shadows (and input block gi*d_in with dropout)
  int row0;        // first row of the target's output features inside the group's weight / b_ext (see target_row)
  int gu;          // rows in the GU-interleaved layout (gate_proj, up_proj)
  int d_in;        // input features: hidden, or ffn for down_proj
  int d_out;       // output features (n_heads*128 for q, n_kv_heads*128 for k, v, ffn for gate / up, hidden for down)
  long long off;   // offset of this target's [A^T (d_in x r) | B (d_out x r)] inside the layer block
};

// bf16 shadows of one group (all layers): a_cat [L][RP][KA], b_ext [L][rows][RP]
struct GroupInfo {
  int n = 0;       // enabled targets in the group
  int ti0 = 0;     // index of its first target among all enabled targets (the dropout mask's target index)
  int d_in = 0;    // input width of the group
  int rows = 0;    // output rows of the group's weight (W, 2F, d)
  int RP = 0;      // n*r rounded up to the 64-wide rank block
  int KA = 0;      // contraction length of the LoRA down-projection: d_in, or n*d_in with dropout (one dropped copy per target)
  int split_a = 1, split_b = 1;
  bf16* a_cat = nullptr;
  bf16* b_ext = nullptr;
};

// refresh bf16 shadows of all adapters from the fp32 masters; for target ti of group G:
//   G.a_cat[l][(gi*r + j)*KA + a_col0 + c]             = A^T[c*r + j]      (a_col0 = 0; with LoRA dropout gi*d_in)
//   G.b_ext[l][target_row(row0, n, gu)*RP + gi*r + j]  = scale * B[n*r + j]
struct ShadowArgs {
  const float* params;
  int L, r, nt, a_split;
  long long per_layer;
  TargetInfo tg[kMaxTargets];
  GroupInfo g[N_GROUPS];
  float scale;
};
__global__ void lora_shadow_kernel(ShadowArgs a) {
  const long long total = a.per_layer * a.L;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int l = static_cast<int>(i / a.per_layer);
    long long rem = i - l * a.per_layer;
    int ti = 0;
    while (ti + 1 < a.nt && rem >= a.tg[ti + 1].off) ++ti;
    const TargetInfo& tg = a.tg[ti];
    const GroupInfo& g = a.g[tg.group];
    rem -= tg.off;
    const float v = a.params[i];
    if (rem < static_cast<long long>(tg.d_in) * a.r) {
      const int c = static_cast<int>(rem / a.r), j = static_cast<int>(rem % a.r);
      g.a_cat[(static_cast<long long>(l) * g.RP + tg.gi * a.r + j) * g.KA + (a.a_split ? tg.gi * tg.d_in : 0) + c] = __float2bfloat16_rn(v);
    } else {
      rem -= static_cast<long long>(tg.d_in) * a.r;
      const int n = static_cast<int>(rem / a.r), j = static_cast<int>(rem % a.r);
      g.b_ext[(static_cast<long long>(l) * g.rows + target_row(tg.row0, n, tg.gu)) * g.RP + tg.gi * a.r + j] =
          __float2bfloat16_rn(v * a.scale);
    }
  }
}

struct Layer {
  // wgu: [2F, d] in the GU-interleaved layout (128 gate rows | 128 up rows per 128 features)
  bf16 *wqkv = nullptr, *wo = nullptr, *wgu = nullptr, *wdown = nullptr, *norm1 = nullptr, *norm2 = nullptr;
  bf16* a_cat[N_GROUPS] = {nullptr, nullptr, nullptr};  // shadows of the adapter groups (null: group has no target)
  bf16* b_ext[N_GROUPS] = {nullptr, nullptr, nullptr};
  bf16* t[N_GROUPS] = {nullptr, nullptr, nullptr};      // saved LoRA down-projections t_g = lora_in * A_cat^T  [M, RP_g]
  bf16 *h1 = nullptr, *qkv = nullptr, *attn = nullptr, *x_mid = nullptr, *gu = nullptr;  // saved
  bf16* hd = nullptr;  // LoRA dropout on q/k/v only: [M, n*d] dropped copies of h1, one per target (peft: one nn.Dropout per module)
  float *lse = nullptr, *rstd1 = nullptr, *rstd2 = nullptr;
  // --quantization int4: packed NF4 codes (two per byte) + one fp32 absmax per 64 elements; the bf16 pointers above are then
  // null and the GEMMs read a per-trainer scratch that dequantize() fills right before each launch
  uint8_t* q4[4] = {nullptr, nullptr, nullptr, nullptr};   // wqkv, wo, wgu, wdown
  float* absmax[4] = {nullptr, nullptr, nullptr, nullptr};
};
enum { W_QKV = 0, W_O = 1, W_GU = 2, W_DOWN = 3 };

}  // namespace
void trainer_set_fused_epilogues(int on) { g_fused_epilogues = on; }
void trainer_set_nf4_prefetch(int on) { g_nf4_prefetch = on; }
void trainer_set_varlen_split(int on) { g_varlen_split = on; }
void trainer_set_varlen_pack(int on) { g_varlen_pack = on; }
void trainer_set_varlen_group_cost(int permille) { g_varlen_fix_permille = permille < 0 ? 0 : permille; }
}  // namespace dtx

using namespace dtx;

struct dtx_trainer {
  dtx_model_cfg mc{};
  dtx_train_cfg tc{};
  int device = 0, rank = 0, world = 1;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  void* nccl_comm = nullptr;
  std::string err;
  std::vector<void*> allocs;
  size_t bytes_allocated = 0;

  int M = 0, nt = 0;            // M = micro_batch * seq_len: the largest batch this trainer was created for; nt = LoRA targets
  int cur_S = 0, cur_M = 0;     // padded length / token count of the batch being processed (<= seq_len / M)
  int cur_B = 0;                // its rows: micro_batch, or the rows of one length group (SubPlan)
  bool sub_accum = false;       // a later length group of the same micro-batch: gradients and loss add to the earlier groups'
  int sub_ndiv = 0;             // > 0: labelled tokens of the WHOLE micro-batch (the divisor of the token-mean loss of every group)
  int n_sms = 148;
  int last_groups = 1;          // length groups of the last training micro-batch (diagnostics; 0 = packed)
  bool packed = false;          // the batch in d_ids / d_labels is PACKED: sequence b owns rows d_row_start[b] .. d_row_start[b+1])
  bool use_seq_lens = false;    // d_seq_lens holds this batch's true row lengths
  int dq = 0, dkv = 0, W = 0;  // q width (= hidden), k/v width (n_kv_heads*128), packed qkv row width
  bool dropout = false;
  TargetInfo tg[kMaxTargets];   // enabled targets in HF module order
  int tg_mod[kMaxTargets] = {}; // their HF module index (kModules)
  GroupInfo grp[N_GROUPS];
  int64_t per_layer = 0, n_train = 0;
  uint64_t fwd_count = 0;      // forward passes so far: seeds the dropout masks

  bf16 *embed = nullptr, *lm_head = nullptr, *normf = nullptr;
  std::vector<Layer> layers;
  std::vector<bf16*> xs;  // residual stream, L+1 entries
  float *params = nullptr, *grads = nullptr, *adam_m = nullptr, *adam_v = nullptr;

  // transients
  bf16 *h2 = nullptr, *act = nullptr, *dact = nullptr, *dgu = nullptr, *dx_a = nullptr, *dx_b = nullptr, *dh = nullptr,
       *dattn = nullptr, *dqkv = nullptr, *dt = nullptr, *dlogits = nullptr, *glora = nullptr;
  bf16* hd_mlp = nullptr;  // LoRA dropout on MLP targets: dropped copies of h2 (gate|up) or act (down), rebuilt in the backward pass
  float *logits = nullptr, *rstdf = nullptr, *row_loss = nullptr, *delta = nullptr, *part_b = nullptr, *part_a = nullptr;
  float *d_loss = nullptr, *d_sumsq = nullptr, *d_gnorm = nullptr, *d_scratch = nullptr;
  int32_t *d_ids = nullptr, *d_labels = nullptr, *d_shift = nullptr, *d_nvalid = nullptr, *d_seq_lens = nullptr;
  int32_t *d_row_map = nullptr, *d_valid_idx = nullptr;  // token -> position among the labelled tokens (-1: none) and back
  int32_t *d_ids_full = nullptr, *d_labels_full = nullptr, *d_lens_full = nullptr;  // the whole ragged micro-batch (length groups gather from it)
  int32_t *d_pos = nullptr, *d_row_start = nullptr;  // packed batch: position of every row inside its sequence; first row of every sequence
  std::vector<int32_t> h_labels, h_lens;  // host copies of a device-resident ragged batch (the partition is planned on the host)
  std::vector<float> h_row_sum;           // per-row evaluation statistics of the length groups, in group order
  std::vector<int32_t> h_row_valid;
  float* d_row_sum = nullptr;     // [micro_batch] per-row summed token loss (evaluation)
  int32_t* d_row_valid = nullptr; // [micro_batch] per-row valid-token count
  double* d_host_red = nullptr;   // staging for dtx_allreduce_host
  int window = 0;                 // sliding-window attention span (0 = plain causal)
  // ---- full-parameter SFT (train.full_finetune): every weight trains, no adapters (BASELINE.json configs[3]) ----
  // Weights live in ONE flat bf16 buffer - L layer blocks [wqkv | wo | wgu | wdown | norm1 | norm2] then a globals block
  // [embed | lm_head | final norm], each padded to a multiple of world * 128 elements - with a gradient buffer of the same
  // layout.  Rank r owns elements [r, r + 1) * block / world of every block: the block's bf16 gradients are reduce-scattered
  // in place (NCCL, on a side stream, as soon as the backward pass has finished the layer), the fp32 master weights and Adam
  // moments exist for the owned slices only (ZeRO-1 style), and the updated bf16 slices are all-gathered in place.
  bool full = false;
  int64_t layer_elems = 0, glob_elems = 0;
  int64_t off_wo = 0, off_wgu = 0, off_wdown = 0, off_n1 = 0, off_n2 = 0, goff_lm = 0, goff_nf = 0, layer_used = 0, glob_used = 0;
  bf16 *w_flat = nullptr, *g_flat = nullptr;
  float *master = nullptr, *fm = nullptr, *fv = nullptr, *embed_g32 = nullptr, *ndw_scratch = nullptr;
  bool master_valid = false;
  bool rs_now = false;  // this backward pass ends an accumulation group: finished layers go to the reduce-scatter stream
  cudaStream_t comm_stream = nullptr;
  std::vector<cudaEvent_t> ev_layer;
  cudaEvent_t ev_comm = nullptr;
  // all-gather of the updated weights runs on the side stream, block by block in the order the NEXT forward pass needs them
  // (globals, layer 0, 1, ...); ag_pending[b] = the main stream has not yet been told to wait for block b (L = globals)
  std::vector<cudaEvent_t> ev_ag;
  std::vector<uint8_t> ag_pending;
  bool quant4 = false;
  bf16* scratch_w[4] = {nullptr, nullptr, nullptr, nullptr};  // dequantised wqkv / wo / wgu / wdown of the layer in flight
  cudaEvent_t ev_deq[4] = {nullptr, nullptr, nullptr, nullptr}, ev_scr[4] = {nullptr, nullptr, nullptr, nullptr};
  int deq_layer[4] = {-1, -1, -1, -1};       // layer whose matrix of that type sits (or is being expanded) in the scratch
  uint8_t deq_pending[4] = {0, 0, 0, 0};     // expansion launched on the side stream, main stream not yet told to wait
  int64_t base_bytes = 0;
  float2* rope_cs = nullptr;
  float2* rope_cs_t = nullptr;  // the same table transposed to [D/2][S]: coalesced when thread r needs position q0 + r (attention backward epilogues)

  // which base tensors have been uploaded: [0] embed, [1] lm_head, [2] final norm, then 9 per layer
  // (q, k, v, o, gate, up, down, norm1, norm2); a step with a hole in this map would train on uninitialised memory
  std::vector<uint8_t> loaded;
  bool all_random = false;
  bool have_lora = false;
  cudaEvent_t ev_fb = nullptr, ev_ar = nullptr;
  float seg_ms[4] = {0.f, 0.f, 0.f, 0.f};
  cudaStream_t copy_stream = nullptr;
  int micro_idx = 0;
  int opt_step = 0;
  int64_t launches = 0;
  float last_ms = 0.f;

  int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    err = buf;
    return code;
  }
  template <typename T>
  bool alloc(T** p, size_t n) {
    void* q = nullptr;
    cudaError_t e = cudaMalloc(&q, n * sizeof(T));
    if (e != cudaSuccess) {
      fail(DTX_ERR_CUDA, "cudaMalloc(%zu bytes) failed after %zu bytes: %s", n * sizeof(T), bytes_allocated,
           cudaGetErrorString(e));
      return false;
    }
    allocs.push_back(q);
    bytes_allocated += n * sizeof(T);
    *p = static_cast<T*>(q);
    return true;
  }
  void release(void* p, size_t bytes) {
    if (!p) return;
    for (size_t i = 0; i < allocs.size(); ++i)
      if (allocs[i] == p) {
        allocs[i] = allocs.back();
        allocs.pop_back();
        break;
      }
    cudaFree(p);
    bytes_allocated -= bytes;
  }
  // first base tensor that has not been loaded, or nullptr when the model is complete
  const char* missing_weight(char* buf, size_t n) const {
    if (all_random) return nullptr;
    static const char* top[3] = {"model.embed_tokens.weight", "lm_head.weight", "model.norm.weight"};
    static const char* per[9] = {"self_attn.q_proj", "self_attn.k_proj", "self_attn.v_proj", "self_attn.o_proj", "mlp.gate_proj",
                                 "mlp.up_proj", "mlp.down_proj", "input_layernorm", "post_attention_layernorm"};
    for (size_t i = 0; i < loaded.size(); ++i)
      if (!loaded[i]) {
        if (i < 3) snprintf(buf, n, "%s", top[i]);
        else snprintf(buf, n, "model.layers.%zu.%s.weight", (i - 3) / 9, per[(i - 3) % 9]);
        return buf;
      }
    return nullptr;
  }
};

namespace {

#define CK(expr, nlaunch)                                                                        \
  do {                                                                                           \
    cudaError_t _e = (expr);                                                                     \
    if (_e != cudaSuccess) return t->fail(DTX_ERR_CUDA, "%s: %s", #expr, cudaGetErrorString(_e)); \
    t->launches += (nlaunch);                                                                    \
  } while (0)

// checked copies / fills outside the hot loop (no launch counted)
#define CKM(expr)                                                                                \
  do {                                                                                           \
    cudaError_t _e = (expr);                                                                     \
    if (_e != cudaSuccess) return t->fail(DTX_ERR_CUDA, "%s: %s", #expr, cudaGetErrorString(_e)); \
  } while (0)

// Host -> device copies of weights / adapters go through the TRAINER'S stream and are waited for: cudaMemcpy() from pageable
// memory returns once the data is staged - the DMA may still be in flight - and it runs on the legacy default stream, with
// which the trainer's non-blocking stream does not synchronise.  A kernel launched right behind it (the adapter shadow
// refresh) then read stale parameters: the first step after loading adapters from the host differed from run to run
// (profiles/r02_load_race.txt).
inline cudaError_t upload_sync(void* dst, const void* src, size_t bytes, cudaStream_t s) {
  cudaError_t e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, s);
  if (e != cudaSuccess) return e;
  return cudaStreamSynchronize(s);
}

// key of the dropout masks of one (forward pass, layer): the per-element keep decision is
// splitmix64(key + target * 0x9E3779B97F4A7C15 + m * d + c) >> 40 >= p * 2^24  (restated in oracle/llama_lora.py)
uint64_t dropout_key(const dtx_trainer* t, int layer) {
  uint64_t x = t->tc.seed * 0xD1B54A32D192ED03ull + t->fwd_count * 0x100000001B3ull + static_cast<uint64_t>(layer) * 0x9E3779B1ull +
               static_cast<uint64_t>(t->rank) * 0xC2B2AE3D27D4EB4Full;
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}

int pick_split(int m_tiles, int kb_total) {
  int s = (2 * gemm_num_sms() + m_tiles - 1) / m_tiles;
  if (s < 1) s = 1;
  if (s > 16) s = 16;
  if (s > kb_total) s = kb_total;
  // every split must own at least one k-block
  while (s > 1 && (s - 1) * ((kb_total + s - 1) / s) >= kb_total) --s;
  return s;
}

int create_buffers(dtx_trainer* t) {
  const dtx_model_cfg& mc = t->mc;
  const dtx_train_cfg& tc = t->tc;
  const size_t d = mc.hidden, F = mc.ffn, V = mc.vocab, L = mc.n_layers, M = t->M, W = t->W;
  bool ok = true;
  const bool full = t->full;
  if (full) {
    // one flat weight buffer + one flat gradient buffer; every block padded so that it splits evenly over the ranks
    const size_t unit = static_cast<size_t>(t->world) * 128;
    auto pad = [&](size_t n) { return (n + unit - 1) / unit * unit; };
    t->off_wo = W * d;
    t->off_wgu = t->off_wo + d * d;
    t->off_wdown = t->off_wgu + 2 * F * d;
    t->off_n1 = t->off_wdown + d * F;
    t->off_n2 = t->off_n1 + d;
    t->layer_used = t->off_n2 + d;
    t->layer_elems = pad(t->layer_used);
    t->goff_lm = V * d;
    t->goff_nf = 2 * V * d;
    t->glob_used = 2 * V * d + d;
    t->glob_elems = pad(t->glob_used);
    const size_t total = L * t->layer_elems + t->glob_elems, shard = total / t->world;
    ok = ok && t->alloc(&t->w_flat, total) && t->alloc(&t->g_flat, total);
    ok = ok && t->alloc(&t->master, shard) && t->alloc(&t->fm, shard) && t->alloc(&t->fv, shard);
    ok = ok && t->alloc(&t->embed_g32, V * d) && t->alloc(&t->ndw_scratch, 64 * d);
    if (!ok) return DTX_ERR_CUDA;
    CKM(cudaMemset(t->w_flat, 0, total * sizeof(bf16)));
    CKM(cudaMemset(t->g_flat, 0, total * sizeof(bf16)));
    CKM(cudaMemset(t->fm, 0, shard * sizeof(float)));
    CKM(cudaMemset(t->fv, 0, shard * sizeof(float)));
    bf16* gl = t->w_flat + L * t->layer_elems;
    t->embed = gl;
    t->lm_head = gl + t->goff_lm;
    t->normf = gl + t->goff_nf;
    t->n_train = static_cast<int64_t>(L * t->layer_used + t->glob_used);
  } else {
    ok = ok && t->alloc(&t->embed, V * d) && t->alloc(&t->lm_head, V * d) && t->alloc(&t->normf, d);
    for (GroupInfo& g : t->grp) {
      if (!g.n) continue;
      const size_t na = L * g.RP * g.KA, nb = L * g.rows * g.RP;
      ok = ok && t->alloc(&g.a_cat, na) && t->alloc(&g.b_ext, nb);
      if (!ok) return DTX_ERR_CUDA;
      CKM(cudaMemset(g.a_cat, 0, na * sizeof(bf16)));
      CKM(cudaMemset(g.b_ext, 0, nb * sizeof(bf16)));
    }
  }
  t->base_bytes = static_cast<int64_t>((2 * V * d + d) * sizeof(bf16));
  t->loaded.assign(3 + 9 * L, 0);
  t->layers.resize(L);
  t->xs.resize(L + 1);
  for (size_t l = 0; l <= L; ++l) ok = ok && t->alloc(&t->xs[l], M * d);
  for (size_t l = 0; l < L && ok; ++l) {
    Layer& y = t->layers[l];
    if (full) {
      bf16* blk = t->w_flat + l * t->layer_elems;
      y.wqkv = blk; y.wo = blk + t->off_wo; y.wgu = blk + t->off_wgu; y.wdown = blk + t->off_wdown;
      y.norm1 = blk + t->off_n1; y.norm2 = blk + t->off_n2;
    } else {
      ok = ok && t->alloc(&y.wqkv, W * d) && t->alloc(&y.wo, d * d) && t->alloc(&y.wgu, 2 * F * d) &&
           t->alloc(&y.wdown, d * F) && t->alloc(&y.norm1, d) && t->alloc(&y.norm2, d);
      for (int gi = 0; gi < N_GROUPS; ++gi) {
        const GroupInfo& g = t->grp[gi];
        if (!g.n) continue;
        y.a_cat[gi] = g.a_cat + l * g.RP * g.KA;
        y.b_ext[gi] = g.b_ext + l * g.rows * g.RP;
        ok = ok && t->alloc(&y.t[gi], M * g.RP);
      }
    }
    t->base_bytes += static_cast<int64_t>((W * d + d * d + 3 * F * d + 2 * d) * sizeof(bf16));
    ok = ok && t->alloc(&y.h1, M * d) && t->alloc(&y.qkv, M * W) &&
         t->alloc(&y.attn, M * d) && t->alloc(&y.x_mid, M * d) && t->alloc(&y.gu, M * 2 * F);
    if (t->dropout && t->grp[G_ATT].n) ok = ok && t->alloc(&y.hd, M * t->grp[G_ATT].KA);
    ok = ok && t->alloc(&y.lse, static_cast<size_t>(tc.micro_batch) * mc.n_heads * tc.seq_len) && t->alloc(&y.rstd1, M) &&
         t->alloc(&y.rstd2, M);
  }
  if (!ok) return DTX_ERR_CUDA;
  if (!full) {
    ok = ok && t->alloc(&t->params, t->n_train) && t->alloc(&t->grads, t->n_train) && t->alloc(&t->adam_m, t->n_train) &&
         t->alloc(&t->adam_v, t->n_train);
    if (!ok) return DTX_ERR_CUDA;
    CKM(cudaMemset(t->params, 0, t->n_train * sizeof(float)));
    CKM(cudaMemset(t->grads, 0, t->n_train * sizeof(float)));
    CKM(cudaMemset(t->adam_m, 0, t->n_train * sizeof(float)));
    CKM(cudaMemset(t->adam_v, 0, t->n_train * sizeof(float)));
  }
  ok = ok && t->alloc(&t->h2, M * d) && t->alloc(&t->act, M * F) && t->alloc(&t->dact, M * F) && t->alloc(&t->dgu, M * 2 * F) &&
       t->alloc(&t->dx_a, M * d) && t->alloc(&t->dx_b, M * d) && t->alloc(&t->dh, M * d) && t->alloc(&t->dattn, M * d) &&
       t->alloc(&t->dqkv, M * W) && t->alloc(&t->dlogits, M * V) && t->alloc(&t->logits, M * V) &&
       t->alloc(&t->rstdf, M) && t->alloc(&t->row_loss, M) &&
       t->alloc(&t->delta, static_cast<size_t>(tc.micro_batch) * mc.n_heads * tc.seq_len);
  if (!full) {  // per-step LoRA scratch, shared by the groups (the backward pass finishes one group before it starts the next)
    const int kb_tok = (static_cast<int>(M) + 63) / 64;
    size_t n_dt = 0, n_pb = 0, n_pa = 0, n_glora = 0, n_hd = 0;
    for (int gi = 0; gi < N_GROUPS; ++gi) {
      GroupInfo& g = t->grp[gi];
      if (!g.n) continue;
      g.split_b = pick_split((g.rows + 127) / 128, kb_tok);
      g.split_a = pick_split((g.KA + 127) / 128, kb_tok);
      n_dt = std::max(n_dt, M * g.RP);
      n_pb = std::max(n_pb, static_cast<size_t>(g.split_b) * g.rows * g.RP);
      n_pa = std::max(n_pa, static_cast<size_t>(g.split_a) * g.KA * g.RP);
      n_glora = std::max(n_glora, M * g.KA);
      if (gi != G_ATT) n_hd = std::max(n_hd, M * g.KA);
    }
    ok = ok && t->alloc(&t->dt, n_dt) && t->alloc(&t->part_b, n_pb) && t->alloc(&t->part_a, n_pa);
    if (t->dropout) ok = ok && t->alloc(&t->glora, n_glora) && (n_hd == 0 || t->alloc(&t->hd_mlp, n_hd));
  }
  ok = ok && t->alloc(&t->d_loss, 4) && t->alloc(&t->d_sumsq, 4) && t->alloc(&t->d_gnorm, 4) && t->alloc(&t->d_scratch, 1024);
  ok = ok && t->alloc(&t->d_ids, M) && t->alloc(&t->d_labels, M) && t->alloc(&t->d_shift, M) && t->alloc(&t->d_nvalid, 4);
  ok = ok && t->alloc(&t->d_row_map, M) && t->alloc(&t->d_valid_idx, M);
  ok = ok && t->alloc(&t->d_ids_full, M) && t->alloc(&t->d_labels_full, M) && t->alloc(&t->d_lens_full, static_cast<size_t>(tc.micro_batch)) &&
       t->alloc(&t->d_pos, M) && t->alloc(&t->d_row_start, static_cast<size_t>(tc.micro_batch) + 1);
  ok = ok && t->alloc(&t->d_seq_lens, static_cast<size_t>(tc.micro_batch)) && t->alloc(&t->d_row_sum, static_cast<size_t>(tc.micro_batch)) &&
       t->alloc(&t->d_row_valid, static_cast<size_t>(tc.micro_batch)) && t->alloc(&t->d_host_red, 64);
  ok = ok && t->alloc(&t->rope_cs, static_cast<size_t>(tc.seq_len) * (mc.head_dim / 2));
  ok = ok && t->alloc(&t->rope_cs_t, static_cast<size_t>(tc.seq_len) * (mc.head_dim / 2));
  if (!ok) return DTX_ERR_CUDA;
  // rotary table in double precision (HF LlamaRotaryEmbedding: inv_freq = theta^(-2i/D))
  {
    const int half = mc.head_dim / 2;
    std::vector<float2> cs(static_cast<size_t>(tc.seq_len) * half);
    for (int pos = 0; pos < tc.seq_len; ++pos)
      for (int i = 0; i < half; ++i) {
        // HF computes inv_freq and the angle in fp32; reproduce that rounding, then take cos/sin accurately
        const float inv_freq = 1.0f / powf(mc.rope_theta, static_cast<float>(2 * i) / static_cast<float>(mc.head_dim));
        const float ang = static_cast<float>(pos) * inv_freq;
        cs[static_cast<size_t>(pos) * half + i] = make_float2(static_cast<float>(cos(static_cast<double>(ang))),
                                                              static_cast<float>(sin(static_cast<double>(ang))));
      }
    CKM(cudaMemcpy(t->rope_cs, cs.data(), cs.size() * sizeof(float2), cudaMemcpyHostToDevice));
    std::vector<float2> cst(cs.size());
    for (int pos = 0; pos < tc.seq_len; ++pos)
      for (int i = 0; i < half; ++i) cst[static_cast<size_t>(i) * tc.seq_len + pos] = cs[static_cast<size_t>(pos) * half + i];
    CKM(cudaMemcpy(t->rope_cs_t, cst.data(), cst.size() * sizeof(float2), cudaMemcpyHostToDevice));
  }
  return DTX_OK;
}

int refresh_shadows(dtx_trainer* t) {
  ShadowArgs a;
  a.params = t->params;
  a.L = t->mc.n_layers;
  a.r = t->tc.lora_r;
  a.nt = t->nt;
  a.a_split = t->dropout ? 1 : 0;
  a.per_layer = t->per_layer;
  for (int i = 0; i < kMaxTargets; ++i) a.tg[i] = t->tg[i];
  for (int i = 0; i < N_GROUPS; ++i) a.g[i] = t->grp[i];
  a.scale = t->tc.lora_alpha / static_cast<float>(t->tc.lora_r);
  long long total = t->n_train;
  int grid = static_cast<int>((total + 255) / 256);
  if (grid > 148 * 8) grid = 148 * 8;
  lora_shadow_kernel<<<grid, 256, 0, t->stream>>>(a);
  CK(cudaGetLastError(), 1);
  return DTX_OK;
}

// Frozen base weight `which` of layer l for the next GEMM.  bf16-resident: the pointer.  --quantization int4: the packed NF4
// codes are expanded into the per-trainer scratch of that matrix type (HBM-bound: 0.56 B read + 2 B written per weight, ~85 us
// per layer of a 7B model and direction) - the values are exactly bitsandbytes' dequantize_4bit output, so the GEMM sees what
// the reference's 4-bit matmul multiplies with.  The expansion of the NEXT matrix in program order is launched on a side
// stream as soon as the current one is handed out: its small CTAs (no shared memory) co-reside with the persistent GEMM
// CTAs and use HBM bandwidth the tensor-bound GEMM leaves idle, so that the expansion disappears from the critical path.
int nf4_expand(dtx_trainer* t, int l, int which, cudaStream_t s) {
  Layer& y = t->layers[l];
  const int64_t d = t->mc.hidden, F = t->mc.ffn;
  const int64_t n[4] = {static_cast<int64_t>(t->W) * d, d * d, 2 * F * d, d * F};
  CK(nf4_dequant_bf16(y.q4[which], y.absmax[which], t->scratch_w[which], n[which], s), 1);
  return DTX_OK;
}
// next (layer, matrix) the step will ask for after (l, which); backward = the step is in (or about to enter) its backward pass
bool next_weight(const dtx_trainer* t, int l, int which, bool backward, bool will_backward, int* nl, int* nw) {
  const int L = t->mc.n_layers;
  if (!backward) {  // forward order: qkv, o, gu, down
    if (which < W_DOWN) { *nl = l; *nw = which + 1; return true; }
    if (l + 1 < L) { *nl = l + 1; *nw = W_QKV; return true; }
    if (will_backward) { *nl = L - 1; *nw = W_DOWN; return true; }
    return false;
  }
  // backward order: down, gu, o, qkv (layer 0's qkv is never asked for: no consumer of its input gradient)
  if (which > W_QKV) {
    if (which - 1 == W_QKV && l == 0) return false;
    *nl = l; *nw = which - 1; return true;
  }
  if (l - 1 >= 0) { *nl = l - 1; *nw = W_DOWN; return true; }
  return false;
}
int base_weight(dtx_trainer* t, int l, int which, bool backward, bool will_backward, const bf16** out) {
  Layer& y = t->layers[l];
  bf16* res[4] = {y.wqkv, y.wo, y.wgu, y.wdown};
  if (!t->quant4) {
    *out = res[which];
    return DTX_OK;
  }
  if (t->deq_layer[which] == l) {  // already in the scratch (the frozen weights never change), or on its way there
    if (t->deq_pending[which]) CKM(cudaStreamWaitEvent(t->stream, t->ev_deq[which], 0));
  } else {
    int rc = nf4_expand(t, l, which, t->stream);
    if (rc) return rc;
  }
  t->deq_pending[which] = 0;
  t->deq_layer[which] = l;
  *out = t->scratch_w[which];
  int nl, nw;
  if (t->copy_stream && next_weight(t, l, which, backward, will_backward, &nl, &nw) && t->deq_layer[nw] != nl) {
    // the scratch of type nw was last read by a GEMM launched earlier on the main stream: order the overwrite behind it
    CKM(cudaEventRecord(t->ev_scr[nw], t->stream));
    CKM(cudaStreamWaitEvent(t->copy_stream, t->ev_scr[nw], 0));
    int rc = nf4_expand(t, nl, nw, t->copy_stream);
    if (rc) return rc;
    CKM(cudaEventRecord(t->ev_deq[nw], t->copy_stream));
    t->deq_pending[nw] = 1;
    t->deq_layer[nw] = nl;
  }
  return DTX_OK;
}
#define BASEW(which, ptr)                                                        \
  const bf16* ptr = nullptr;                                                     \
  do {                                                                           \
    int _rc = base_weight(t, l, which, in_backward, backward, &ptr);             \
    if (_rc) return _rc;                                                         \
  } while (0)

// full-parameter SFT, world > 1: the updated weights of block b (L = globals) are being all-gathered on the side stream;
// make the main stream wait for it right before the block's first use
inline void wait_weights(dtx_trainer* t, int b) {
  if (!t->ag_pending.empty() && t->ag_pending[b]) {
    cudaStreamWaitEvent(t->stream, t->ev_ag[b], 0);
    t->ag_pending[b] = 0;
  }
}
inline void wait_all_weights(dtx_trainer* t) {
  for (size_t b = 0; b < t->ag_pending.size(); ++b) wait_weights(t, static_cast<int>(b));
}

// full-parameter SFT, world > 1: reduce-scatter one gradient block in place on the side stream once the main stream has
// produced it (event), so that the transfer overlaps the rest of the backward pass
int reduce_scatter_block(dtx_trainer* t, bf16* block, int64_t elems, int ev_idx) {
  NcclApi* api = nccl_api();
  if (!api || !api->ReduceScatter || !t->nccl_comm) return t->fail(DTX_ERR_NCCL, "ncclReduceScatter unavailable for world=%d", t->world);
  cudaEvent_t ev = t->ev_layer[ev_idx];
  CKM(cudaEventRecord(ev, t->stream));
  CKM(cudaStreamWaitEvent(t->comm_stream, ev, 0));
  const int64_t shard = elems / t->world;
  int rc = api->ReduceScatter(block, block + static_cast<int64_t>(t->rank) * shard, static_cast<size_t>(shard), kNcclBfloat16, kNcclSum,
                              t->nccl_comm, t->comm_stream);
  if (rc != 0) return t->fail(DTX_ERR_NCCL, "ncclReduceScatter failed: %s", api->GetErrorString ? api->GetErrorString(rc) : "?");
  t->launches += 1;
  return DTX_OK;
}

// forward (+ backward) of one micro-batch whose ids / labels (/ row lengths) are already in t->d_ids / t->d_labels (/ t->d_seq_lens).
// The batch is [micro_batch, cur_S]: cur_S <= seq_len is this batch's own padded length (DataCollatorForSeq2Seq pads to the
// longest row of the batch, cmd/tuning/train.py:282-286); every buffer was sized for seq_len.
int fwd_bwd(dtx_trainer* t, bool backward) {
  const dtx_model_cfg& mc = t->mc;
  const dtx_train_cfg& tc = t->tc;
  const int d = mc.hidden, F = mc.ffn, V = mc.vocab, L = mc.n_layers, M = t->cur_M, H = mc.n_heads, D = mc.head_dim;
  const int Hkv = mc.n_kv_heads, W = t->W;
  const int B = t->cur_B, S = t->cur_S;
  const int32_t* seq_lens = t->use_seq_lens ? t->d_seq_lens : nullptr;
  const int kb_tok = (M + 63) / 64;
  cudaStream_t s = t->stream;
  const float att_scale = 1.0f / sqrtf(static_cast<float>(D));
  const bool fused = g_fused_epilogues && M > 128 && ((t->dq + t->dkv) % 256 == 0) && (W % 256 == 0);  // whole 256-column tiles
  const bool lora = !t->full;    // full-parameter SFT: no adapters, every weight gets a gradient
  const GroupInfo &ga = t->grp[G_ATT], &gg = t->grp[G_GU], &gd = t->grp[G_DN];
  const bool lora_att = lora && ga.n > 0, lora_gu = lora && gg.n > 0, lora_dn = lora && gd.n > 0;
  bool in_backward = false;      // which half of the step asks for a base weight (prefetch order of the NF4 expansion)
  const bool drop = lora && t->dropout;  // adapters laid out for per-target dropped inputs (KA = n*d_in)
  const float p_drop = backward ? tc.lora_dropout : 0.f;  // eval (model.eval()) runs the same path with p = 0
  t->fwd_count += 1;
  // dropout key of group g in layer l: the mask of a target is indexed by its position among ALL enabled targets, and the
  // kernels add (position inside the group) * G to the key - so the group's offset goes into the key
  auto group_key = [&](int l, const GroupInfo& g) { return dropout_key(t, l) + static_cast<uint64_t>(g.ti0) * 0x9E3779B97F4A7C15ull; };
  // t_g = lora_in * A_cat^T  [M, RP]: the LoRA down-projection of every target of a group in one GEMM
  auto lora_down = [&](const GroupInfo& G, const bf16* in, const bf16* a_cat, bf16* out) {
    GemmArgs g;
    g.A = in; g.lda = G.KA; g.B = a_cat; g.ldb = G.KA; g.C = out; g.ldc = G.RP;
    g.M = M; g.N = G.RP; g.K = G.KA; g.epilogue = EPI_BF16; g.block_n = 64;
    return gemm_bf16(g, s);
  };
  // dt = dY * B_ext  [M, RP]  (dY: gradient of the group's output, [M, rows])
  auto lora_dt = [&](const GroupInfo& G, const bf16* dY, const bf16* b_ext) {
    GemmArgs g;
    g.A = dY; g.lda = G.rows; g.B = b_ext; g.ldb = G.RP; g.b_mn_major = 1; g.C = t->dt; g.ldc = G.RP;
    g.M = M; g.N = G.RP; g.K = G.rows; g.epilogue = EPI_BF16; g.block_n = 64;
    return gemm_bf16(g, s);
  };
  // glora = dt * A_cat  [M, KA]: the LoRA branch's input gradient before the dropout masks (one block per target)
  auto lora_dx = [&](const GroupInfo& G, const bf16* a_cat) {
    GemmArgs g;
    g.A = t->dt; g.lda = G.RP; g.B = a_cat; g.ldb = G.KA; g.b_mn_major = 1; g.C = t->glora; g.ldc = G.KA;
    g.M = M; g.N = G.KA; g.K = G.RP; g.epilogue = EPI_BF16;
    return gemm_bf16(g, s);
  };

  wait_weights(t, L);  // globals (embedding, lm_head, final norm)
  CK(embedding_fwd(t->d_ids, t->embed, t->xs[0], M, d, V, s), 1);
  for (int l = 0; l < L; ++l) {
    Layer& y = t->layers[l];
    wait_weights(t, l);
    CK(rmsnorm_fwd(t->xs[l], y.norm1, y.h1, y.rstd1, M, d, mc.rms_eps, s), 1);
    const bf16* lora_in = y.h1;
    if (drop && lora_att) {  // peft: lora_A(lora_dropout(x)) with one nn.Dropout per wrapped module -> one dropped copy per target
      CK(lora_dropout_fwd(y.h1, y.hd, M, d, ga.n, p_drop, dropout_key(t, l), s), 1);
      lora_in = y.hd;
    }
    if (lora_att) CK(lora_down(ga, lora_in, y.a_cat[G_ATT], y.t[G_ATT]), 1);  // t = lora_in * A_cat^T   [M, RP]
    {  // qkv = h1 * Wqkv^T + t * B_ext^T : base projection and LoRA up-projection in one TMEM accumulator
      BASEW(W_QKV, wqkv);
      GemmArgs g;
      g.A = y.h1; g.lda = d; g.B = wqkv; g.ldb = d;
      if (lora_att) { g.A2 = y.t[G_ATT]; g.lda2 = ga.RP; g.B2 = y.b_ext[G_ATT]; g.ldb2 = ga.RP; g.K2 = ga.RP; }
      g.C = y.qkv; g.ldc = W; g.M = M; g.N = W; g.K = d; g.epilogue = EPI_BF16;
      if (fused) {  // rotary embedding of q and k applied to the fp32 accumulator in the epilogue
        g.epilogue = EPI_ROPE; g.rope_cs = t->rope_cs; g.rope_S = S; g.rope_cols = t->dq + t->dkv;
        g.rope_pos = t->packed ? t->d_pos : nullptr;  // packed batch: a row's position is its offset inside its own sequence
      }
      CK(gemm_bf16(g, s), 1);
    }
    if (!fused && t->packed) return t->fail(DTX_ERR_STATE, "packed batches need the fused RoPE epilogue");
    if (!fused) CK(rope_qk_inplace_table(y.qkv, t->rope_cs, B, S, H + Hkv, W, D, 0, s), 1);
    {
      AttnArgs a;
      a.qkv = y.qkv; a.out = y.attn; a.lse = y.lse; a.B = B; a.S = S; a.H = H; a.Hkv = Hkv; a.scale = att_scale;
      a.seq_lens = seq_lens; a.window = t->window;
      if (t->packed) { a.row_start = t->d_row_start; a.total_rows = M; }
      CK(attn_fwd(a, s), 1);
    }
    {  // x_mid = x + attn * Wo^T
      BASEW(W_O, wo);
      GemmArgs g;
      g.A = y.attn; g.lda = d; g.B = wo; g.ldb = d; g.C = y.x_mid; g.ldc = d; g.R = t->xs[l]; g.ldr = d;
      g.M = M; g.N = d; g.K = d; g.epilogue = EPI_BF16_ADD;
      CK(gemm_bf16(g, s), 1);
    }
    CK(rmsnorm_fwd(y.x_mid, y.norm2, t->h2, y.rstd2, M, d, mc.rms_eps, s), 1);
    if (lora_gu) {  // t_gu = h2 * A_gu^T  (h2 and its dropped copies are per-step scratch: the backward pass rebuilds them)
      const bf16* in = t->h2;
      if (drop) {
        CK(lora_dropout_fwd(t->h2, t->hd_mlp, M, d, gg.n, p_drop, group_key(l, gg), s), 1);
        in = t->hd_mlp;
      }
      CK(lora_down(gg, in, y.a_cat[G_GU], y.t[G_GU]), 1);
    }
    {  // [gate | up] = h2 * Wgu^T + t_gu * B_gu^T  (B_gu rows GU-interleaved like Wgu: gate and up of a feature share a tile)
      BASEW(W_GU, wgu);
      GemmArgs g;
      g.A = t->h2; g.lda = d; g.B = wgu; g.ldb = d; g.C = y.gu; g.ldc = 2 * F;
      if (lora_gu) { g.A2 = y.t[G_GU]; g.lda2 = gg.RP; g.B2 = y.b_ext[G_GU]; g.ldb2 = gg.RP; g.K2 = gg.RP; }
      g.M = M; g.N = 2 * F; g.K = d; g.epilogue = EPI_BF16;
      if (fused) {  // silu(gate) * up computed from the accumulator tile ([gate 128 | up 128] interleaved layout)
        g.epilogue = EPI_SWIGLU_FWD; g.aux = t->act; g.ld_aux = F;
      }
      CK(gemm_bf16(g, s), 1);
    }
    if (!fused) CK(swiglu_fwd(y.gu, t->act, M, F, 1, s), 1);
    if (lora_dn) {  // t_dn = act * A_dn^T  (K = F)
      const bf16* in = t->act;
      if (drop) {
        CK(lora_dropout_fwd(t->act, t->hd_mlp, M, F, 1, p_drop, group_key(l, gd), s), 1);
        in = t->hd_mlp;
      }
      CK(lora_down(gd, in, y.a_cat[G_DN], y.t[G_DN]), 1);
    }
    {  // x_next = x_mid + act * Wdown^T + t_dn * B_dn^T
      BASEW(W_DOWN, wdown);
      GemmArgs g;
      g.A = t->act; g.lda = F; g.B = wdown; g.ldb = F; g.C = t->xs[l + 1]; g.ldc = d; g.R = y.x_mid; g.ldr = d;
      if (lora_dn) { g.A2 = y.t[G_DN]; g.lda2 = gd.RP; g.B2 = y.b_ext[G_DN]; g.ldb2 = gd.RP; g.K2 = gd.RP; }
      g.M = M; g.N = d; g.K = F; g.epilogue = EPI_BF16_ADD;
      CK(gemm_bf16(g, s), 1);
    }
  }
  // lm_head, CE and their backward only over the tokens that carry a label (shifted label >= 0): prompt tokens and padding
  // (27 % of the synthetic batch, far more on real instruction data) have zero loss and zero gradient.  The labelled rows
  // are compacted by the final norm (row map from an ordered scan inside shift_labels), the two lm_head GEMMs take the row
  // count from device memory and skip the dead 256-row tiles, the norm backward scatters the gradient back.
  // (full-parameter SFT keeps every row: the lm_head weight gradient contracts over tokens, and its operands must then be zero
  // - not stale - on the unlabelled rows)
  int32_t* row_map = lora ? t->d_row_map : nullptr;
  int32_t* valid_idx = lora ? t->d_valid_idx : nullptr;
  const int32_t* m_eff = lora ? t->d_nvalid : nullptr;
  if (t->packed) CK(shift_labels(t->d_labels, t->d_shift, t->d_nvalid, 1, M, s, row_map, valid_idx, t->d_pos), 1);
  else CK(shift_labels(t->d_labels, t->d_shift, t->d_nvalid, B, S, s, row_map, valid_idx), 1);
  CK(rmsnorm_fwd(t->xs[L], t->normf, t->h2, t->rstdf, M, d, mc.rms_eps, s, row_map), 1);
  {  // fp32 logits (the reference patches lm_head to return fp32: cmd/tuning/train.py:256-264)
    GemmArgs g;
    g.A = t->h2; g.lda = d; g.B = t->lm_head; g.ldb = d; g.C = t->logits; g.ldc = V;
    g.M = M; g.N = V; g.K = d; g.epilogue = EPI_F32; g.m_eff = m_eff;
    CK(gemm_bf16(g, s), 1);
  }
  CKM(cudaMemsetAsync(t->row_loss, 0, static_cast<size_t>(M) * sizeof(float), s));
  // one length group of a ragged micro-batch (t->sub_ndiv > 0): the token mean runs over the labelled tokens of all its groups
  CK(cross_entropy_fwd_bwd(t->logits, V, t->d_shift, t->d_nvalid, t->row_loss, backward ? t->dlogits : nullptr, V, M, V, s, valid_idx,
                           t->sub_ndiv), 1);
  CK(loss_reduce(t->row_loss, t->d_nvalid, t->d_loss, M, s, t->sub_ndiv, t->sub_accum ? 1 : 0), 1);
  if (!backward) return DTX_OK;
  in_backward = true;

  const int accumulate = (t->micro_idx > 0 || t->sub_accum) ? 1 : 0;
  // weight gradient of a Linear: dW[out, in] (+)= dY^T X - a token-contraction GEMM with both operands MN-major
  auto dw_gemm = [&](const bf16* dY, int n_out, const bf16* X, int n_in, bf16* dW) -> cudaError_t {
    GemmArgs g;
    g.A = dY; g.lda = n_out; g.a_mn_major = 1; g.B = X; g.ldb = n_in; g.b_mn_major = 1;
    g.C = dW; g.ldc = n_in; g.M = n_out; g.N = n_in; g.K = M;
    g.epilogue = accumulate ? EPI_BF16_ADD : EPI_BF16; g.R = accumulate ? dW : nullptr; g.ldr = n_in;
    return gemm_bf16(g, s);
  };
  // adapter gradients of group gi in layer l: grad of B_ext (all rows) dY^T * t_g [rows, RP] and grad of A_cat^T lora_in^T * dt
  // [KA, RP], both split over tokens, then gathered per target into the flat gradient.  dA^T = lora_in^T (dy * sB) (the scale
  // rides in B_ext); dB = s * dy^T t (t is unscaled, so the scale is applied by the gather).
  auto lora_wgrad = [&](int l, int gi, const bf16* dY, const bf16* lora_in) -> int {
    const GroupInfo& G = t->grp[gi];
    const int split_b = std::min(G.split_b, pick_split((G.rows + 127) / 128, kb_tok));
    const int split_a = std::min(G.split_a, pick_split((G.KA + 127) / 128, kb_tok));
    {
      GemmArgs g;
      g.A = dY; g.lda = G.rows; g.a_mn_major = 1; g.B = t->layers[l].t[gi]; g.ldb = G.RP; g.b_mn_major = 1;
      g.C = t->part_b; g.ldc = G.RP; g.M = G.rows; g.N = G.RP; g.K = M; g.epilogue = EPI_F32; g.split_k = split_b;
      g.block_n = 64;
      CK(gemm_bf16(g, s), 1);
    }
    {
      GemmArgs g;
      g.A = lora_in; g.lda = G.KA; g.a_mn_major = 1; g.B = t->dt; g.ldb = G.RP; g.b_mn_major = 1;
      g.C = t->part_a; g.ldc = G.RP; g.M = G.KA; g.N = G.RP; g.K = M; g.epilogue = EPI_F32; g.split_k = split_a;
      g.block_n = 64;
      CK(gemm_bf16(g, s), 1);
    }
    const int r = tc.lora_r;
    for (int ti = G.ti0; ti < G.ti0 + G.n; ++ti) {  // the targets of a group are consecutive in HF module order
      const TargetInfo& tg = t->tg[ti];
      float* gl = t->grads + static_cast<int64_t>(l) * t->per_layer + tg.off;
      lora_gather_kernel<<<(tg.d_in * r + 255) / 256, 256, 0, s>>>(t->part_a, split_a, static_cast<long long>(G.KA) * G.RP, G.RP,
                                                                 drop ? tg.gi * tg.d_in : 0, 0, tg.gi * r, tg.d_in, r, gl, accumulate, 1.0f);
      lora_gather_kernel<<<(tg.d_out * r + 255) / 256, 256, 0, s>>>(t->part_b, split_b, static_cast<long long>(G.rows) * G.RP, G.RP,
                                                                  tg.row0, tg.gu, tg.gi * r, tg.d_out, r,
                                                                  gl + static_cast<int64_t>(tg.d_in) * r, accumulate,
                                                                  tc.lora_alpha / static_cast<float>(r));
      CK(cudaGetLastError(), 2);
    }
    return DTX_OK;
  };
  bf16* gglob = t->full ? t->g_flat + static_cast<int64_t>(L) * t->layer_elems : nullptr;
  if (t->full) {  // lm_head weight gradient (h2 still holds the final-norm output) and the final norm's weight gradient
    CK(dw_gemm(t->dlogits, V, t->h2, d, gglob + t->goff_lm), 1);
  }
  {  // d h_f = dlogits * W_lm  (compact rows in LoRA mode)
    GemmArgs g;
    g.A = t->dlogits; g.lda = V; g.B = t->lm_head; g.ldb = d; g.b_mn_major = 1; g.C = t->dh; g.ldc = d;
    g.M = M; g.N = d; g.K = V; g.epilogue = EPI_BF16; g.m_eff = m_eff;
    CK(gemm_bf16(g, s), 1);
  }
  if (t->full) CK(rmsnorm_dw(t->dh, t->xs[L], t->rstdf, M, d, t->ndw_scratch, gglob + t->goff_nf, accumulate, s), 2);
  CK(rmsnorm_bwd(t->dh, t->xs[L], t->normf, t->rstdf, nullptr, t->dx_a, M, d, s, row_map), 1);
  bf16* cur = t->dx_a;
  bf16* other = t->dx_b;
  for (int l = L - 1; l >= 0; --l) {
    Layer& y = t->layers[l];
    bf16* gl_w = t->full ? t->g_flat + static_cast<int64_t>(l) * t->layer_elems : nullptr;  // this layer's gradient block
    if (t->full) {  // dWdown = d x_out^T * act: act = silu(gate) * up is recomputed from the saved gate|up (one HBM-bound pass)
      CK(swiglu_fwd(y.gu, t->act, M, F, 1, s), 1);
      CK(dw_gemm(cur, d, t->act, F, gl_w + t->off_wdown), 1);
    }
    if (lora_dn) CK(lora_dt(gd, cur, y.b_ext[G_DN]), 1);  // dt_dn = dx * B_dn  [M, RP_dn]
    // with dropout the LoRA branch's input gradient is masked: it cannot ride in the dact GEMM's accumulator
    const bool dn_dropped = lora_dn && drop;
    {  // dact = dx * Wdown (+ dt_dn * A_dn) ; fused: d[gate|up] straight from the accumulator, dact never touches HBM
      BASEW(W_DOWN, wdown);
      GemmArgs g;
      g.A = cur; g.lda = d; g.B = wdown; g.ldb = F; g.b_mn_major = 1; g.C = t->dact; g.ldc = F;
      if (lora_dn && !drop) { g.A2 = t->dt; g.lda2 = gd.RP; g.B2 = y.a_cat[G_DN]; g.ldb2 = gd.KA; g.K2 = gd.RP; }
      g.M = M; g.N = F; g.K = d; g.epilogue = EPI_BF16;
      if (fused && !dn_dropped) {
        g.epilogue = EPI_SWIGLU_BWD; g.C = t->dgu; g.ldc = 2 * F; g.aux = y.gu; g.ld_aux = 2 * F;
      }
      CK(gemm_bf16(g, s), 1);
    }
    if (dn_dropped) {  // d(act) = dact + mask o (dt_dn * A_dn) / (1 - p) and the SwiGLU backward in one pass
      CK(lora_dx(gd, y.a_cat[G_DN]), 1);
      CK(swiglu_bwd_lora_dropout(t->dact, t->glora, y.gu, t->dgu, M, F, 1, p_drop, group_key(l, gd), s), 1);
    } else if (!fused) {
      CK(swiglu_bwd(t->dact, y.gu, t->dgu, M, F, 1, s), 1);
    }
    if (lora_dn) {  // dB_dn = dx^T t_dn, dA_dn = act^T dt_dn: act = silu(gate) * up recomputed from the saved gate|up
      CK(swiglu_fwd(y.gu, t->act, M, F, 1, s), 1);
      const bf16* in = t->act;
      if (drop) {
        CK(lora_dropout_fwd(t->act, t->hd_mlp, M, F, 1, p_drop, group_key(l, gd), s), 1);
        in = t->hd_mlp;
      }
      int rc = lora_wgrad(l, G_DN, cur, in);
      if (rc) return rc;
    }
    if (lora_gu) CK(lora_dt(gg, t->dgu, y.b_ext[G_GU]), 1);  // dt_gu = d[gate|up] * B_gu  [M, RP_gu]
    {  // dh2 = [dgate | dup] * [Wg ; Wu] (+ dt_gu * A_gu)
      BASEW(W_GU, wgu);
      GemmArgs g;
      g.A = t->dgu; g.lda = 2 * F; g.B = wgu; g.ldb = d; g.b_mn_major = 1; g.C = t->dh; g.ldc = d;
      if (lora_gu && !drop) { g.A2 = t->dt; g.lda2 = gg.RP; g.B2 = y.a_cat[G_GU]; g.ldb2 = gg.KA; g.K2 = gg.RP; }
      g.M = M; g.N = d; g.K = 2 * F; g.epilogue = EPI_BF16;
      CK(gemm_bf16(g, s), 1);
    }
    if (lora_gu && drop) {  // dh2 += sum_t mask_t o (dt_t * A_t) / (1 - p)
      CK(lora_dx(gg, y.a_cat[G_GU]), 1);
      CK(lora_dropout_bwd_add(t->dh, t->glora, M, d, gg.n, p_drop, group_key(l, gg), s), 1);
    }
    if (t->full || lora_gu)  // h2 = norm2(x_mid) recomputed: dWgu / dA_gu contract it over the tokens
      CK(rmsnorm_fwd(y.x_mid, y.norm2, t->h2, nullptr, M, d, mc.rms_eps, s), 1);
    if (t->full) {  // dWgu = d[gate|up]^T * h2 and the norm's own weight gradient
      CK(dw_gemm(t->dgu, 2 * F, t->h2, d, gl_w + t->off_wgu), 1);
      CK(rmsnorm_dw(t->dh, y.x_mid, y.rstd2, M, d, t->ndw_scratch, gl_w + t->off_n2, accumulate, s), 2);
    }
    if (lora_gu) {  // dB_gu = d[gate|up]^T t_gu (rows gathered out of the interleaved layout), dA_gu = h2^T dt_gu
      const bf16* in = t->h2;
      if (drop) {
        CK(lora_dropout_fwd(t->h2, t->hd_mlp, M, d, gg.n, p_drop, group_key(l, gg), s), 1);
        in = t->hd_mlp;
      }
      int rc = lora_wgrad(l, G_GU, t->dgu, in);
      if (rc) return rc;
    }
    CK(rmsnorm_bwd(t->dh, y.x_mid, y.norm2, y.rstd2, cur, other, M, d, s), 1);  // other = d x_mid
    {  // dattn = dx_mid * Wo
      BASEW(W_O, wo);
      GemmArgs g;
      g.A = other; g.lda = d; g.B = wo; g.ldb = d; g.b_mn_major = 1; g.C = t->dattn; g.ldc = d;
      g.M = M; g.N = d; g.K = d; g.epilogue = EPI_BF16;
      CK(gemm_bf16(g, s), 1);
    }
    if (t->full) CK(dw_gemm(other, d, y.attn, d, gl_w + t->off_wo), 1);  // dWo = d x_mid^T * attn
    {
      AttnArgs a;
      a.qkv = y.qkv; a.out = y.attn; a.lse = y.lse; a.B = B; a.S = S; a.H = H; a.Hkv = Hkv; a.scale = att_scale;
      a.dout = t->dattn; a.dqkv = t->dqkv; a.delta = t->delta;
      a.seq_lens = seq_lens; a.window = t->window; a.rope_stride = tc.seq_len;
      if (t->packed) { a.row_start = t->d_row_start; a.total_rows = M; }
      // The dQ / dK kernels apply the inverse rotary in their store epilogues from the TRANSPOSED table (thread r of a tile
      // reads position q0 + r: one coalesced 256-byte line per frequency and warp).  A first attempt with the [S][64] table
      // (32 uncoalesced 8-byte reads per thread) cost +270 us/layer, the standalone HBM-bound kernel 92 us.
      const bool rope_in_attn = fused && attn_bwd_can_rope();
      a.rope_cs = rope_in_attn ? t->rope_cs_t : nullptr;
      CK(attn_bwd(a, s), attn_bwd_launches());
      if (!rope_in_attn) CK(rope_qk_inplace_table(t->dqkv, t->rope_cs, B, S, H + Hkv, W, D, 1, s), 1);
    }
    if (lora_att) CK(lora_dt(ga, t->dqkv, y.b_ext[G_ATT]), 1);  // dt = dqkv * B_ext   [M, RP]
    if (t->full) CK(dw_gemm(t->dqkv, W, y.h1, d, gl_w), 1);  // dWqkv = dqkv^T * h1 (dqkv already carries the inverse rotary)
    // LoRA: layer 0's input gradient has no consumer (the embedding is frozen, SURVEY §8a): its dh1 GEMM, the dropout-branch
    // gradient and the norm-1 backward are skipped.  Full-parameter SFT trains the embedding and needs them.
    const bool need_dx = l > 0 || t->full;
    if (need_dx) {  // dh1 = dqkv * Wqkv (+ dt * A_cat in the same accumulator when there is no dropout between h1 and A)
      BASEW(W_QKV, wqkv);
      GemmArgs g;
      g.A = t->dqkv; g.lda = W; g.B = wqkv; g.ldb = d; g.b_mn_major = 1;
      if (lora_att && !drop) { g.A2 = t->dt; g.lda2 = ga.RP; g.B2 = y.a_cat[G_ATT]; g.ldb2 = ga.KA; g.K2 = ga.RP; }
      g.C = t->dh; g.ldc = d; g.M = M; g.N = d; g.K = W; g.epilogue = EPI_BF16;
      CK(gemm_bf16(g, s), 1);
    }
    if (lora_att && drop && need_dx) {  // dh1 += sum_t mask_t o (dt_t * A_t) / (1 - p): the masks are regenerated from the counter-based RNG
      CK(lora_dx(ga, y.a_cat[G_ATT]), 1);
      CK(lora_dropout_bwd_add(t->dh, t->glora, M, d, ga.n, p_drop, dropout_key(t, l), s), 1);
    }
    if (lora_att) {
      int rc = lora_wgrad(l, G_ATT, t->dqkv, drop ? y.hd : y.h1);
      if (rc) return rc;
    }
    if (t->full) CK(rmsnorm_dw(t->dh, t->xs[l], y.rstd1, M, d, t->ndw_scratch, gl_w + t->off_n1, accumulate, s), 2);
    if (need_dx) CK(rmsnorm_bwd(t->dh, t->xs[l], y.norm1, y.rstd1, other, cur, M, d, s), 1);  // cur = d x_in
    if (t->full && t->rs_now && t->world > 1) {  // this layer's gradients are final: reduce-scatter them while the backward pass goes on
      int rc = reduce_scatter_block(t, gl_w, t->layer_elems, l);
      if (rc) return rc;
    }
  }
  if (t->full) {  // embedding gradient: rows of d x_0 scattered by token id (fp32 atomics), then folded into the bf16 gradient block
    const size_t vd = static_cast<size_t>(V) * d;
    CKM(cudaMemsetAsync(t->embed_g32, 0, vd * sizeof(float), s));
    CK(embedding_bwd(t->d_ids, cur, t->embed_g32, M, d, V, s), 1);
    CK(add_f32_into_bf16(t->embed_g32, gglob, static_cast<int64_t>(vd), accumulate, s), 1);
  }
  return DTX_OK;
}

int optimizer_step(dtx_trainer* t, float* lr_used) {
  const dtx_train_cfg& tc = t->tc;
  cudaStream_t s = t->stream;
  if (t->world > 1) {
    NcclApi* api = nccl_api();
    if (!api || !t->nccl_comm) return t->fail(DTX_ERR_NCCL, "NCCL communicator missing for world=%d", t->world);
    int rc = api->AllReduce(t->grads, t->grads, static_cast<size_t>(t->n_train), kNcclFloat32, kNcclSum, t->nccl_comm, s);
    if (rc != 0) return t->fail(DTX_ERR_NCCL, "ncclAllReduce failed: %s", api->GetErrorString ? api->GetErrorString(rc) : "?");
    t->launches += 1;
  }
  cudaEventRecord(t->ev_ar, s);
  CK(sumsq(t->grads, t->n_train, t->d_scratch, t->d_sumsq, s), 2);
  const double lam = dtx_lr_lambda(tc.sched, t->opt_step, tc.warmup_steps, tc.total_steps);
  const float lr = static_cast<float>(static_cast<double>(tc.lr) * lam);
  const int step1 = t->opt_step + 1;
  AdamWArgs a;
  a.p = t->params; a.g = t->grads; a.m = t->adam_m; a.v = t->adam_v; a.n = t->n_train;
  a.lr = lr; a.beta1 = tc.beta1; a.beta2 = tc.beta2; a.eps = tc.eps; a.weight_decay = tc.weight_decay;
  a.bias1 = static_cast<float>(1.0 - pow(static_cast<double>(tc.beta1), step1));
  a.bias2 = static_cast<float>(1.0 - pow(static_cast<double>(tc.beta2), step1));
  // HF scales every micro-batch loss by 1/grad_accum whatever the number actually accumulated (forced end-of-epoch step)
  a.grad_scale = 1.0f / static_cast<float>(t->world * (tc.grad_accum > 0 ? tc.grad_accum : 1));
  a.sumsq = t->d_sumsq; a.max_grad_norm = tc.max_grad_norm; a.grad_norm_out = t->d_gnorm;
  CK(adamw_step(a, s), 1);
  int rc = refresh_shadows(t);
  if (rc) return rc;
  t->opt_step += 1;
  if (lr_used) *lr_used = lr;
  return DTX_OK;
}

// Full-parameter SFT: the blocks' bf16 gradients have been (or are now) reduce-scattered in place; every rank then runs
// clip + AdamW on the slices it owns (fp32 master weights + moments, ZeRO-1 style) and the updated bf16 slices are
// all-gathered in place.  HF's no-decay set (RMSNorm weights) sits at the end of every block.
int optimizer_step_full(dtx_trainer* t, float* lr_used) {
  const dtx_train_cfg& tc = t->tc;
  cudaStream_t s = t->stream;
  const int L = t->mc.n_layers, N = t->world;
  NcclApi* api = N > 1 ? nccl_api() : nullptr;
  if (N > 1 && (!api || !api->ReduceScatter || !api->AllGather || !t->nccl_comm))
    return t->fail(DTX_ERR_NCCL, "NCCL reduce-scatter / all-gather unavailable for world=%d", N);
  bf16* gglob = t->g_flat + static_cast<int64_t>(L) * t->layer_elems;
  if (N > 1) {
    if (!t->rs_now)  // gradients of earlier micro-batches only: nothing was sent during the backward pass
      for (int l = L - 1; l >= 0; --l) {
        int rc = reduce_scatter_block(t, t->g_flat + static_cast<int64_t>(l) * t->layer_elems, t->layer_elems, l);
        if (rc) return rc;
      }
    int rc = reduce_scatter_block(t, gglob, t->glob_elems, L);
    if (rc) return rc;
    CKM(cudaEventRecord(t->ev_comm, t->comm_stream));
    CKM(cudaStreamWaitEvent(s, t->ev_comm, 0));
  }
  cudaEventRecord(t->ev_ar, s);
  const int64_t lsh = t->layer_elems / N, gsh = t->glob_elems / N;  // slice lengths
  auto slice = [&](int blk, bf16* base, int64_t* n, int64_t* moff) {  // this rank's slice of block blk (L = globals)
    const int64_t sh = blk < L ? lsh : gsh;
    *n = sh;
    *moff = static_cast<int64_t>(blk) * lsh;  // offset inside the master / moment shards
    return base + (blk < L ? static_cast<int64_t>(blk) * t->layer_elems : static_cast<int64_t>(L) * t->layer_elems) + static_cast<int64_t>(t->rank) * sh;
  };
  if (!t->master_valid) {  // first step (or weights re-loaded): fp32 master copies of the owned bf16 slices
    for (int blk = 0; blk <= L; ++blk) {
      int64_t n, moff;
      bf16* w = slice(blk, t->w_flat, &n, &moff);
      CK(cast_bf16_to_f32(w, t->master + moff, n, s), 1);
    }
    t->master_valid = true;
  }
  for (int blk = 0; blk <= L; ++blk) {
    int64_t n, moff;
    bf16* g = slice(blk, t->g_flat, &n, &moff);
    CK(sumsq_bf16_acc(g, n, t->d_scratch, t->d_sumsq, blk == 0 ? 1 : 0, s), 2);
  }
  if (N > 1) {
    int rc = api->AllReduce(t->d_sumsq, t->d_sumsq, 1, kNcclFloat32, kNcclSum, t->nccl_comm, s);
    if (rc != 0) return t->fail(DTX_ERR_NCCL, "ncclAllReduce failed: %s", api->GetErrorString ? api->GetErrorString(rc) : "?");
    t->launches += 1;
  }
  const double lam = dtx_lr_lambda(tc.sched, t->opt_step, tc.warmup_steps, tc.total_steps);
  const float lr = static_cast<float>(static_cast<double>(tc.lr) * lam);
  const int step1 = t->opt_step + 1;
  for (int blk = 0; blk <= L; ++blk) {
    int64_t n, moff;
    bf16* g = slice(blk, t->g_flat, &n, &moff);
    bf16* w = slice(blk, t->w_flat, &n, &moff);
    AdamWShardArgs a;
    a.master = t->master + moff; a.m = t->fm + moff; a.v = t->fv + moff; a.g = g; a.w = w; a.n = n;
    // RMSNorm weights (no weight decay): the tail [off_n1, layer_used) of a layer block, [goff_nf, glob_used) of the globals
    const int64_t nd_begin = blk < L ? t->off_n1 : t->goff_nf, first = static_cast<int64_t>(t->rank) * n;
    a.nodecay_from = nd_begin - first < 0 ? 0 : nd_begin - first;
    a.lr = lr; a.beta1 = tc.beta1; a.beta2 = tc.beta2; a.eps = tc.eps; a.weight_decay = tc.weight_decay;
    a.bias1 = static_cast<float>(1.0 - pow(static_cast<double>(tc.beta1), step1));
    a.bias2 = static_cast<float>(1.0 - pow(static_cast<double>(tc.beta2), step1));
    a.grad_scale = 1.0f / static_cast<float>(N * (tc.grad_accum > 0 ? tc.grad_accum : 1));
    a.sumsq = t->d_sumsq; a.max_grad_norm = tc.max_grad_norm; a.grad_norm_out = t->d_gnorm;
    CK(adamw_shard_step(a, s), 1);
  }
  if (N > 1) {
    // Every rank gets every updated slice (in place: the send slice sits at its final position).  The all-gathers run on the
    // side stream in the order the next forward pass consumes the blocks, so that they overlap it: measured on 8 GPUs (13B),
    // the 26 GB all-gather was 58 of the step's 658 ms when it sat on the main stream.
    CKM(cudaEventRecord(t->ev_comm, s));
    CKM(cudaStreamWaitEvent(t->comm_stream, t->ev_comm, 0));
    for (int i = 0; i <= L; ++i) {
      const int blk = i == 0 ? L : i - 1;  // globals first, then layer 0, 1, ...
      int64_t n, moff;
      bf16* w = slice(blk, t->w_flat, &n, &moff);
      bf16* base = w - static_cast<int64_t>(t->rank) * n;
      int rc = api->AllGather(w, base, static_cast<size_t>(n), kNcclBfloat16, t->nccl_comm, t->comm_stream);
      if (rc != 0) return t->fail(DTX_ERR_NCCL, "ncclAllGather failed: %s", api->GetErrorString ? api->GetErrorString(rc) : "?");
      CKM(cudaEventRecord(t->ev_ag[blk], t->comm_stream));
      t->ag_pending[blk] = 1;
      t->launches += 1;
    }
  }
  t->opt_step += 1;
  if (lr_used) *lr_used = lr;
  return DTX_OK;
}

// validate and record the shape of the batch about to be processed
int set_batch_shape(dtx_trainer* t, int32_t seq_len_batch, bool have_lens) {
  const int S = seq_len_batch > 0 ? seq_len_batch : t->tc.seq_len;
  if (S % 128 || S > t->tc.seq_len)
    return t->fail(DTX_ERR_INVALID, "seq_len_batch %d must be a multiple of 128 and <= seq_len %d", S, t->tc.seq_len);
  t->cur_S = S;
  t->cur_B = t->tc.micro_batch;
  t->cur_M = S * t->tc.micro_batch;
  t->use_seq_lens = have_lens;
  t->packed = false;
  return DTX_OK;
}

// ---- ragged micro-batches as length groups -------------------------------------------------------------------------
// The reference pads a batch to its longest row (DataCollatorForSeq2Seq, cmd/tuning/train.py:282-286) and computes over the
// padding.  Here the attention kernels already skip padding tiles; the GEMMs, norms and CE do not - on instruction data with a
// long tail of row lengths more than half of their rows are padding.  A micro-batch with row lengths is therefore run as
// LENGTH GROUPS: rows sorted by length, cut into contiguous groups, each group padded to its own longest row (128-rounded)
// and sent through forward + backward on its own; gradients accumulate, and every group's loss and dlogits are divided by the
// labelled-token count of the WHOLE micro-batch, so the result is the same token mean (up to summation order).  The cut is
// chosen by dynamic programming over a cost model of the step's GEMMs (256-row tiles x column tiles in waves of one CTA pair
// per two SMs) plus a fixed cost per group: few long groups waste rows on padding, many short ones waste waves.
struct SubPlan {
  int n = 0;            // groups (1: run the micro-batch as it is)
  int start[65] = {0};  // group g = order[start[g] .. start[g+1])
  int S[64] = {0};      // padded length of group g
  int order[64] = {0};  // rows sorted by length, longest first
  int n_div = 0;        // labelled tokens of the whole micro-batch, counted the way the groups' shift_labels kernels will
};

// PACKED layout of a ragged micro-batch (LoRA or full-parameter): sequence b gets its length rounded up to 128 rows, sequences back to back - one
// pass over sum_b ceil128(len_b) rows instead of B * S_batch (or one pass per length group).  GEMMs, norms and CE simply see
// fewer rows; the attention kernels take the first row of every sequence from a table; RoPE takes a row's position and the
// label shift a sequence's end from a per-row position array.  Returns false when packing does not apply or saves nothing.
// the layout alone (host arithmetic): first row of every sequence; true when it is smaller than the padded rectangle
bool packed_rows(const int32_t* lens, int B, int S_batch, RowStarts* rs) {
  rs->n = B;
  rs->start[0] = 0;
  for (int b = 0; b < B; ++b) {
    const int len = std::min(std::max(lens[b], 0), S_batch);
    rs->start[b + 1] = rs->start[b] + std::min(S_batch, std::max(128, (len + 127) / 128 * 128));
  }
  return rs->start[B] < B * S_batch && rs->start[B] > 128;
}
bool plan_packed(const dtx_trainer* t, const int32_t* lens, int S_batch, RowStarts* rs) {
  const int B = t->tc.micro_batch;
  if (!g_varlen_pack || g_varlen_split == 0 || g_varlen_split == 2 || !lens || B < 1 || B > 64) return false;
  if (!g_fused_epilogues || ((t->dq + t->dkv) % 256) || (t->W % 256)) return false;  // RoPE must run in the GEMM epilogue (per-row positions)
  return packed_rows(lens, B, S_batch, rs);
}

struct PlanDims { int hidden, ffn, W, n_sms, B; };  // what the cost model needs of the model / device / batch

double group_cost(const PlanDims& t, int rows, int S) {
  const int d = t.hidden, F = t.ffn, W = t.W;
  const long long mt = (static_cast<long long>(rows) * S + 255) / 256;
  const long long slots = std::max(1, t.n_sms / 2);
  auto waves = [&](int n_cols, int k) { return static_cast<double>((mt * ((n_cols + 255) / 256) + slots - 1) / slots) * k; };
  // forward: qkv, o, gate|up, down; backward dX: through down (N = F), gate|up, o, qkv
  return waves(W, d) + waves(d, d) + waves(2 * F, d) + waves(d, F) + waves(F, d) + waves(d, 2 * F) + waves(d, d) + waves(d, W);
}

// labels may be null (planning only: n_div stays 0)
void plan_groups(const PlanDims& t, const int32_t* lens, const int32_t* labels, int S_batch, SubPlan* p) {
  const int B = t.B;
  p->n = 1;
  if (!g_varlen_split || !lens || B < 2 || B > 64) return;
  auto c128 = [&](int len) { return std::min(S_batch, std::max(128, (std::min(std::max(len, 0), S_batch) + 127) / 128 * 128)); };
  for (int i = 0; i < B; ++i) p->order[i] = i;
  std::stable_sort(p->order, p->order + B, [&](int a, int b) { return lens[a] > lens[b]; });
  const bool force = g_varlen_split == 2;  // tests: minimise padded rows, no fixed cost
  const double fix = force ? 0.0 : 0.001 * g_varlen_fix_permille * group_cost(t, 1, 256);
  auto cost = [&](int rows, int S) { return force ? static_cast<double>(rows) * S : group_cost(t, rows, S); };
  double best[65];
  int cut[65];
  best[0] = 0.0;
  for (int j = 1; j <= B; ++j) {
    best[j] = 1e300;
    for (int i = 0; i < j; ++i) {  // group = sorted rows i .. j-1, padded to the longest of them (row i); at least 256 rows of tokens
      int S = c128(lens[p->order[i]]);
      if ((j - i) * S < 256) {  // every group keeps M >= 256 (whole 256-row GEMM tiles, the fused-epilogue kernels)
        if (S_batch < 256) continue;
        S = 256;
      }
      const double c = best[i] + cost(j - i, S) + fix;
      if (c < best[j]) { best[j] = c; cut[j] = i; }
    }
  }
  if (best[B] > 1e299 || best[B] >= cost(B, S_batch) + fix) return;  // one group at the batch's own padded length is as good
  int ends[65], n = 0;
  for (int j = B; j > 0; j = cut[j]) ends[n++] = j;
  p->n = n;
  p->start[0] = 0;
  for (int g = 0; g < n; ++g) {
    p->start[g + 1] = ends[n - 1 - g];
    int S = c128(lens[p->order[p->start[g]]]);
    if ((p->start[g + 1] - p->start[g]) * S < 256) S = 256;
    p->S[g] = S;
  }
  if (n < 2) { p->n = 1; return; }
  if (!labels) return;
  long long cnt = 0;  // positions 1 .. S_g - 1 of every row carry the shifted label of the position before them
  for (int g = 0; g < n; ++g)
    for (int k = p->start[g]; k < p->start[g + 1]; ++k) {
      const int32_t* row = labels + static_cast<size_t>(p->order[k]) * S_batch;
      for (int j = 1; j < p->S[g]; ++j) cnt += row[j] >= 0 ? 1 : 0;
    }
  p->n_div = static_cast<int>(cnt);
  if (p->n_div <= 0) p->n = 1;  // nothing carries a label: the plain path handles the degenerate batch
}

int check_ready(dtx_trainer* t) {
  char buf[160];
  if (const char* m = t->missing_weight(buf, sizeof(buf)))
    return t->fail(DTX_ERR_STATE, "base weight %s was never loaded (dtx_load_tensor / dtx_init_random_weights)", m);
  if (!t->full && !t->have_lora) return t->fail(DTX_ERR_STATE, "LoRA adapters not initialised (dtx_init_lora / dtx_load_tensor)");
  return DTX_OK;
}

// plan (optional, n > 1): run the micro-batch as length groups gathered from src_* (device, [micro_batch, S_src] / [micro_batch])
int do_step(dtx_trainer* t, int32_t flags, float* loss_out, float* gnorm_out, float* lr_out, int32_t* stepped_out,
            const SubPlan* plan = nullptr, const int32_t* src_ids = nullptr, const int32_t* src_labels = nullptr,
            const int32_t* src_lens = nullptr, int S_src = 0) {
  cudaEventRecord(t->ev0, t->stream);
  const int accum = t->tc.grad_accum > 0 ? t->tc.grad_accum : 1;
  t->rs_now = t->full && (t->micro_idx + 1 >= accum || (flags & DTX_STEP_FORCE));
  int rc = DTX_OK;
  t->last_groups = t->packed ? 0 : 1;
  if (plan && plan->n > 1) {
    t->last_groups = plan->n;
    for (int g = 0; g < plan->n && rc == DTX_OK; ++g) {
      RowList rl;
      rl.n = plan->start[g + 1] - plan->start[g];
      for (int k = 0; k < rl.n; ++k) rl.rows[k] = plan->order[plan->start[g] + k];
      cudaError_t ge = gather_rows(src_ids, src_labels, src_lens, S_src, rl, plan->S[g], t->d_ids, t->d_labels, t->d_seq_lens, t->stream);
      if (ge != cudaSuccess) {
        t->sub_accum = false;
        t->sub_ndiv = 0;
        return t->fail(DTX_ERR_CUDA, "gather_rows: %s", cudaGetErrorString(ge));
      }
      t->launches += 1;
      t->cur_B = rl.n;
      t->cur_S = plan->S[g];
      t->cur_M = rl.n * plan->S[g];
      t->use_seq_lens = true;
      t->sub_accum = g > 0;
      t->sub_ndiv = plan->n_div;
      rc = fwd_bwd(t, true);
    }
    t->sub_accum = false;
    t->sub_ndiv = 0;
  } else {
    rc = fwd_bwd(t, true);
  }
  if (rc) return rc;
  cudaEventRecord(t->ev_fb, t->stream);
  t->micro_idx += 1;
  int stepped = 0;
  float lr = 0.f;
  if (t->micro_idx >= accum || (flags & DTX_STEP_FORCE)) {
    rc = t->full ? optimizer_step_full(t, &lr) : optimizer_step(t, &lr);
    if (rc) return rc;
    t->micro_idx = 0;
    stepped = 1;
  }
  cudaEventRecord(t->ev1, t->stream);
  float host[2] = {0.f, 0.f};
  cudaMemcpyAsync(&host[0], t->d_loss, sizeof(float), cudaMemcpyDeviceToHost, t->stream);
  if (stepped) cudaMemcpyAsync(&host[1], t->d_gnorm, sizeof(float), cudaMemcpyDeviceToHost, t->stream);
  cudaError_t e = cudaStreamSynchronize(t->stream);
  if (e != cudaSuccess) return t->fail(DTX_ERR_CUDA, "step failed on device: %s", cudaGetErrorString(e));
  cudaEventElapsedTime(&t->last_ms, t->ev0, t->ev1);
  t->seg_ms[0] = t->last_ms;
  cudaEventElapsedTime(&t->seg_ms[1], t->ev0, t->ev_fb);
  t->seg_ms[2] = t->seg_ms[3] = 0.f;
  if (stepped) {
    cudaEventElapsedTime(&t->seg_ms[2], t->ev_fb, t->ev_ar);
    cudaEventElapsedTime(&t->seg_ms[3], t->ev_ar, t->ev1);
  }
  if (loss_out) *loss_out = host[0];
  if (gnorm_out) *gnorm_out = host[1];
  if (lr_out) *lr_out = lr;
  if (stepped_out) *stepped_out = stepped;
  return DTX_OK;
}

// --- HF tensor-name parsing -----------------------------------------------------------------------
bool parse_layer(const char* name, int* layer, const char** rest) {
  const char* p = strstr(name, "layers.");
  if (!p) return false;
  p += 7;
  char* end = nullptr;
  long v = strtol(p, &end, 10);
  if (end == p || *end != '.') return false;
  *layer = static_cast<int>(v);
  *rest = end + 1;
  return true;
}

void to_bf16_host(const void* src, int dtype, size_t n, std::vector<bf16>& out) {
  out.resize(n);
  if (dtype == DTX_BF16) {
    memcpy(out.data(), src, n * 2);
  } else if (dtype == DTX_F32) {
    const float* f = static_cast<const float*>(src);
    for (size_t i = 0; i < n; ++i) out[i] = __float2bfloat16_rn(f[i]);
  } else {
    const __half* h = static_cast<const __half*>(src);
    for (size_t i = 0; i < n; ++i) out[i] = __float2bfloat16_rn(__half2float(h[i]));
  }
}
void to_f32_host(const void* src, int dtype, size_t n, std::vector<float>& out) {
  out.resize(n);
  if (dtype == DTX_F32) {
    memcpy(out.data(), src, n * 4);
  } else if (dtype == DTX_BF16) {
    const bf16* b = static_cast<const bf16*>(src);
    for (size_t i = 0; i < n; ++i) out[i] = __bfloat162float(b[i]);
  } else {
    const __half* h = static_cast<const __half*>(src);
    for (size_t i = 0; i < n; ++i) out[i] = __half2float(h[i]);
  }
}

// index among the enabled targets of the LoRA module named in `rest` ("self_attn.q_proj.lora_A.weight", "mlp.down_proj...."),
// or -1 when it names no enabled target
int target_index(const dtx_trainer* t, const char* rest) {
  int mod = -1;
  for (int m = 0; m < 7 && mod < 0; ++m) {
    const char* p = strstr(rest, kModules[m]);
    if (p && (p == rest || p[-1] == '.')) mod = m;  // a whole path component, not the tail of another name
  }
  for (int i = 0; i < t->nt && mod >= 0; ++i)
    if (t->tg_mod[i] == mod) return i;
  return -1;
}

}  // namespace

// ==================================================================================================
// C ABI
// ==================================================================================================
extern "C" {

int32_t dtx_abi_version(void) { return DTX_ABI_VERSION; }
const char* dtx_last_global_error(void) { return g_error.c_str(); }
const char* dtx_last_error(const dtx_trainer* t) { return t ? t->err.c_str() : g_error.c_str(); }

double dtx_lr_lambda(int32_t sched, int32_t step, int32_t warmup, int32_t total) {
  // transformers.optimization get_{linear,cosine,constant}_schedule_with_warmup lambdas
  if (sched == DTX_SCHED_CONSTANT) return 1.0;
  if (step < warmup) return static_cast<double>(step) / static_cast<double>(warmup > 1 ? warmup : 1);
  if (sched == DTX_SCHED_CONSTANT_WITH_WARMUP) return 1.0;
  if (sched == DTX_SCHED_LINEAR) {
    const double v = static_cast<double>(total - step) / static_cast<double>((total - warmup) > 1 ? (total - warmup) : 1);
    return v > 0.0 ? v : 0.0;
  }
  const double prog = static_cast<double>(step - warmup) / static_cast<double>((total - warmup) > 1 ? (total - warmup) : 1);
  const double v = 0.5 * (1.0 + cos(M_PI * 2.0 * 0.5 * prog));
  return v > 0.0 ? v : 0.0;
}

int32_t dtx_get_nccl_unique_id(void* out128) {
  NcclApi* api = nccl_api();
  if (!api) {
    g_error = "libnccl.so.2 could not be loaded";
    return DTX_ERR_NCCL;
  }
  int rc = api->GetUniqueId(out128);
  if (rc != 0) {
    g_error = std::string("ncclGetUniqueId failed: ") + (api->GetErrorString ? api->GetErrorString(rc) : "?");
    return DTX_ERR_NCCL;
  }
  return DTX_OK;
}

int32_t dtx_trainer_create(const dtx_model_cfg* mc, const dtx_train_cfg* tc, int32_t device, int32_t rank, int32_t world,
                           const void* nccl_unique_id, dtx_trainer** out) {
  if (!mc || !tc || !out) {
    g_error = "null argument";
    return DTX_ERR_INVALID;
  }
  *out = nullptr;
  auto bad = [&](const char* m) {
    g_error = m;
    return DTX_ERR_INVALID;
  };
  if (mc->head_dim != 128) return bad("only head_dim 128 is implemented (Llama-2 / Mistral family)");
  if (mc->n_kv_heads <= 0 || mc->n_heads % mc->n_kv_heads) return bad("n_heads must be a multiple of n_kv_heads");
  if (mc->n_heads * mc->head_dim != mc->hidden) return bad("hidden != n_heads * head_dim");
  if (mc->hidden % 64 || mc->ffn % 128 || mc->vocab % 8)
    return bad("hidden must be a multiple of 64, ffn a multiple of 128 (GU-interleaved layout), vocab a multiple of 8");
  if (tc->seq_len % 128 || tc->seq_len <= 0 || tc->micro_batch <= 0) return bad("seq_len must be a positive multiple of 128");
  if (tc->seq_len > mc->max_seq) return bad("seq_len exceeds max_seq");
  if (!tc->full_finetune && (tc->lora_r <= 0 || tc->lora_r % 8)) return bad("lora_r must be a positive multiple of 8");
  if (tc->lora_dropout < 0.0f || tc->lora_dropout >= 1.0f) return bad("lora_dropout must be in [0, 1)");
  const uint32_t implemented = DTX_TARGET_Q | DTX_TARGET_K | DTX_TARGET_V | DTX_TARGET_GATE | DTX_TARGET_UP | DTX_TARGET_DOWN;
  if (!tc->full_finetune && ((tc->target_mask & ~implemented) || tc->target_mask == 0)) {
    g_error = "lora_target must be a non-empty subset of q_proj,k_proj,v_proj,gate_proj,up_proj,down_proj "
              "(o_proj is the one linear module whose adapter is not implemented)";
    return DTX_ERR_UNSUPPORTED;
  }
  if (world < 1 || rank < 0 || rank >= world) return bad("bad rank/world");
  if (world > 1 && !nccl_unique_id) return bad("world > 1 needs an NCCL unique id");

  cudaError_t e = cudaSetDevice(device);
  if (e != cudaSuccess) {
    g_error = std::string("cudaSetDevice failed (no CUDA device? there is no CPU fallback): ") + cudaGetErrorString(e);
    return DTX_ERR_CUDA;
  }
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess || prop.major != 10) {
    g_error = "libdtxtune requires an sm_100 (Blackwell B200) device";
    return DTX_ERR_CUDA;
  }
  dtx_trainer* t = new dtx_trainer();
  t->mc = *mc;
  t->tc = *tc;
  t->device = device;
  t->rank = rank;
  t->world = world;
  if (prop.multiProcessorCount > 0) t->n_sms = prop.multiProcessorCount;
  t->M = tc->micro_batch * tc->seq_len;
  t->dq = mc->n_heads * mc->head_dim;
  t->dkv = mc->n_kv_heads * mc->head_dim;
  t->W = t->dq + 2 * t->dkv;
  t->full = tc->full_finetune != 0;
  t->dropout = !t->full && tc->lora_dropout > 0.0f;
  t->nt = 0;
  t->per_layer = 0;
  if (!t->full) {
    // per-layer block of the flat parameter buffer: [A^T | B] of every enabled target in HF module order
    const int d = mc->hidden, F = mc->ffn;
    struct Mod { int group, row0, gu, d_in, d_out; };
    const Mod mods[7] = {{G_ATT, 0, 0, d, t->dq},     {G_ATT, t->dq, 0, d, t->dkv}, {G_ATT, t->dq + t->dkv, 0, d, t->dkv},
                         {-1, 0, 0, 0, 0},             {G_GU, 0, 1, d, F},            {G_GU, 128, 1, d, F},
                         {G_DN, 0, 0, F, d}};
    const int rows[N_GROUPS] = {t->W, 2 * F, d};
    for (int m = 0; m < 7; ++m) {
      if (m == kModO || !(tc->target_mask & (1u << m))) continue;
      GroupInfo& g = t->grp[mods[m].group];
      if (g.n == 0) g.ti0 = t->nt;
      TargetInfo& tg = t->tg[t->nt];
      tg.group = mods[m].group;
      tg.gi = g.n++;
      tg.row0 = mods[m].row0;
      tg.gu = mods[m].gu;
      tg.d_in = mods[m].d_in;
      tg.d_out = mods[m].d_out;
      tg.off = t->per_layer;
      t->tg_mod[t->nt] = m;
      t->per_layer += static_cast<int64_t>(tg.d_in + tg.d_out) * tc->lora_r;
      ++t->nt;
    }
    for (int gi = 0; gi < N_GROUPS; ++gi) {
      GroupInfo& g = t->grp[gi];
      g.d_in = gi == G_DN ? F : d;
      g.rows = rows[gi];
      g.RP = ((g.n * tc->lora_r + 63) / 64) * 64;
      g.KA = t->dropout ? g.n * g.d_in : g.d_in;
    }
  }
  t->n_train = static_cast<int64_t>(mc->n_layers) * t->per_layer;
  t->cur_S = tc->seq_len;
  t->cur_M = t->M;
  // Mistral-style sliding window: only a different mask once the sequence is longer than the window
  // (transformers 4.34.0 _make_sliding_window_causal_mask: triu(diagonal=-sliding_window), i.e. query i sees keys i - sw .. i)
  t->window = (mc->sliding_window > 0 && tc->seq_len > mc->sliding_window + 1) ? mc->sliding_window : 0;
  cudaStreamCreateWithFlags(&t->stream, cudaStreamNonBlocking);
  cudaEventCreate(&t->ev0);
  cudaEventCreate(&t->ev1);
  cudaEventCreate(&t->ev_fb);
  cudaEventCreate(&t->ev_ar);
  if (t->full) {
    cudaStreamCreateWithFlags(&t->comm_stream, cudaStreamNonBlocking);
    cudaEventCreateWithFlags(&t->ev_comm, cudaEventDisableTiming);
    t->ev_layer.resize(mc->n_layers + 1);
    for (auto& e : t->ev_layer) cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
    t->ev_ag.resize(mc->n_layers + 1);
    for (auto& e : t->ev_ag) cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
    t->ag_pending.assign(mc->n_layers + 1, 0);
  }
  int rc = create_buffers(t);
  if (rc) {
    g_error = t->err;
    dtx_trainer_destroy(t);
    return rc;
  }
  if (world > 1) {
    NcclApi* api = nccl_api();
    if (!api) {
      g_error = "libnccl.so.2 could not be loaded";
      dtx_trainer_destroy(t);
      return DTX_ERR_NCCL;
    }
    UidByValue uid;
    memcpy(uid.internal, nccl_unique_id, 128);
    int nrc = api->CommInitRank(&t->nccl_comm, world, uid, rank);
    if (nrc != 0) {
      g_error = std::string("ncclCommInitRank failed: ") + (api->GetErrorString ? api->GetErrorString(nrc) : "?");
      dtx_trainer_destroy(t);
      return DTX_ERR_NCCL;
    }
  }
  e = cudaDeviceSynchronize();
  if (e != cudaSuccess) {
    g_error = std::string("device error during create: ") + cudaGetErrorString(e);
    dtx_trainer_destroy(t);
    return DTX_ERR_CUDA;
  }
  *out = t;
  return DTX_OK;
}

void dtx_trainer_destroy(dtx_trainer* t) {
  if (!t) return;
  cudaSetDevice(t->device);
  cudaDeviceSynchronize();  // includes the side stream's collectives
  if (t->nccl_comm) {
    NcclApi* api = nccl_api();
    if (api) api->CommDestroy(t->nccl_comm);
  }
  for (void* p : t->allocs) cudaFree(p);
  if (t->ev0) cudaEventDestroy(t->ev0);
  if (t->ev1) cudaEventDestroy(t->ev1);
  if (t->ev_fb) cudaEventDestroy(t->ev_fb);
  if (t->ev_ar) cudaEventDestroy(t->ev_ar);
  if (t->ev_comm) cudaEventDestroy(t->ev_comm);
  for (auto e : t->ev_layer) cudaEventDestroy(e);
  for (auto e : t->ev_ag) cudaEventDestroy(e);
  if (t->comm_stream) cudaStreamDestroy(t->comm_stream);
  if (t->copy_stream) cudaStreamDestroy(t->copy_stream);
  for (int i = 0; i < 4; ++i) {
    if (t->ev_deq[i]) cudaEventDestroy(t->ev_deq[i]);
    if (t->ev_scr[i]) cudaEventDestroy(t->ev_scr[i]);
  }
  if (t->stream) cudaStreamDestroy(t->stream);
  delete t;
}

int32_t dtx_load_tensor(dtx_trainer* t, const char* name, const void* host, int32_t dtype, const int64_t* shape, int32_t nd) {
  if (!t || !name || !host || !shape || nd < 1 || nd > 2) return t ? t->fail(DTX_ERR_INVALID, "bad argument") : DTX_ERR_INVALID;
  cudaSetDevice(t->device);
  wait_all_weights(t);      // full-parameter SFT: no all-gather may still be writing the weight buffer
  t->master_valid = false;  // ... and the fp32 master copies are rebuilt from the bf16 weights at the next step
  const int64_t d = t->mc.hidden, F = t->mc.ffn, V = t->mc.vocab, r = t->tc.lora_r, dq = t->dq, dkv = t->dkv;
  const int64_t rows = shape[0], cols = nd == 2 ? shape[1] : 1;
  auto expect = [&](int64_t er, int64_t ec) { return rows == er && cols == ec; };
  auto upload = [&](bf16* dst, size_t n) -> int {
    std::vector<bf16> tmp;
    to_bf16_host(host, dtype, n, tmp);
    cudaError_t e = upload_sync(dst, tmp.data(), n * sizeof(bf16), t->stream);
    if (e != cudaSuccess) return t->fail(DTX_ERR_CUDA, "upload %s: %s", name, cudaGetErrorString(e));
    return DTX_OK;
  };
  if (strstr(name, "embed_tokens.weight")) {
    if (!expect(V, d)) return t->fail(DTX_ERR_INVALID, "%s: expected [%lld,%lld]", name, (long long)V, (long long)d);
    t->loaded[0] = 1;
    return upload(t->embed, V * d);
  }
  if (strstr(name, "lm_head.weight")) {
    if (!expect(V, d)) return t->fail(DTX_ERR_INVALID, "%s: expected [%lld,%lld]", name, (long long)V, (long long)d);
    t->loaded[1] = 1;
    return upload(t->lm_head, V * d);
  }
  int layer = -1;
  const char* rest = nullptr;
  if (!parse_layer(name, &layer, &rest)) {
    if (strstr(name, "norm.weight")) {  // model.norm.weight
      if (rows != d) return t->fail(DTX_ERR_INVALID, "%s: expected [%lld]", name, (long long)d);
      t->loaded[2] = 1;
      return upload(t->normf, d);
    }
    return t->fail(DTX_ERR_INVALID, "unknown tensor name %s", name);
  }
  if (layer < 0 || layer >= t->mc.n_layers) return t->fail(DTX_ERR_INVALID, "%s: layer out of range", name);
  Layer& y = t->layers[layer];
  uint8_t* lmap = t->loaded.data() + 3 + 9 * static_cast<size_t>(layer);
  const bool is_lora_a = strstr(rest, "lora_A") != nullptr, is_lora_b = strstr(rest, "lora_B") != nullptr;
  if (is_lora_a || is_lora_b) {
    const int ti = target_index(t, rest);
    if (ti < 0) return t->fail(DTX_ERR_INVALID, "%s: module is not a LoRA target", name);
    float* base = t->params + static_cast<int64_t>(layer) * t->per_layer + t->tg[ti].off;
    const int64_t d_in = t->tg[ti].d_in, d_out = t->tg[ti].d_out;
    std::vector<float> f;
    if (is_lora_a) {  // [r, d_in] -> stored transposed [d_in, r]
      if (!expect(r, d_in)) return t->fail(DTX_ERR_INVALID, "%s: expected [%lld,%lld]", name, (long long)r, (long long)d_in);
      to_f32_host(host, dtype, r * d_in, f);
      std::vector<float> tr(d_in * r);
      for (int64_t j = 0; j < r; ++j)
        for (int64_t c = 0; c < d_in; ++c) tr[c * r + j] = f[j * d_in + c];
      CKM(upload_sync(base, tr.data(), tr.size() * 4, t->stream));
    } else {
      if (!expect(d_out, r)) return t->fail(DTX_ERR_INVALID, "%s: expected [%lld,%lld]", name, (long long)d_out, (long long)r);
      to_f32_host(host, dtype, d_out * r, f);
      CKM(upload_sync(base + d_in * r, f.data(), f.size() * 4, t->stream));
    }
    t->have_lora = true;
    int rc = refresh_shadows(t);
    if (rc) return rc;
    CKM(cudaStreamSynchronize(t->stream));
    return DTX_OK;
  }
  if (t->quant4 && !strstr(rest, "layernorm"))
    return t->fail(DTX_ERR_STATE, "%s: the base weights are already NF4-packed; load tensors before dtx_quantize_base", name);
  // gate/up rows go to the GU-interleaved layout: 128 gate rows, then the 128 up rows of the same features, ...
  for (int which = 0; which < 2; ++which) {
    if (!strstr(rest, which ? "mlp.up_proj.weight" : "mlp.gate_proj.weight")) continue;
    if (!expect(F, d)) return t->fail(DTX_ERR_INVALID, "%s: expected [%lld,%lld]", name, (long long)F, (long long)d);
    std::vector<bf16> tmp;
    to_bf16_host(host, dtype, static_cast<size_t>(F) * d, tmp);
    for (int64_t b = 0; b < F / 128; ++b) {
      cudaError_t e = cudaMemcpyAsync(y.wgu + (b * 256 + which * 128) * d, tmp.data() + b * 128 * d, 128 * d * sizeof(bf16),
                                      cudaMemcpyHostToDevice, t->stream);
      if (e != cudaSuccess) return t->fail(DTX_ERR_CUDA, "upload %s: %s", name, cudaGetErrorString(e));
    }
    CKM(cudaStreamSynchronize(t->stream));  // `tmp` dies at the end of this scope
    lmap[4 + which] = 1;
    return DTX_OK;
  }
  struct Slot { const char* key; bf16* dst; int64_t r, c; int bit; };
  const Slot slots[] = {
      {"self_attn.q_proj.weight", y.wqkv, dq, d, 0},                  {"self_attn.k_proj.weight", y.wqkv + dq * d, dkv, d, 1},
      {"self_attn.v_proj.weight", y.wqkv + (dq + dkv) * d, dkv, d, 2}, {"self_attn.o_proj.weight", y.wo, d, dq, 3},
      {"mlp.down_proj.weight", y.wdown, d, F, 6},             {"input_layernorm.weight", y.norm1, d, 1, 7},
      {"post_attention_layernorm.weight", y.norm2, d, 1, 8},
  };
  for (const Slot& sl : slots) {
    if (strstr(rest, sl.key)) {
      if (!expect(sl.r, sl.c)) return t->fail(DTX_ERR_INVALID, "%s: expected [%lld,%lld]", name, (long long)sl.r, (long long)sl.c);
      int rc = upload(sl.dst, sl.r * sl.c);
      if (rc == DTX_OK) lmap[sl.bit] = 1;  // a step with a hole in this map is refused (check_ready)
      return rc;
    }
  }
  return t->fail(DTX_ERR_INVALID, "unknown tensor name %s", name);
}

int32_t dtx_init_random_weights(dtx_trainer* t, uint64_t seed) {
  if (!t) return DTX_ERR_INVALID;
  if (t->quant4) return t->fail(DTX_ERR_STATE, "init_random_weights: the base weights are already NF4-packed");
  t->master_valid = false;
  cudaSetDevice(t->device);
  const int64_t d = t->mc.hidden, F = t->mc.ffn, V = t->mc.vocab;
  cudaStream_t s = t->stream;
  uint64_t k = seed * 1000003ull;
  CK(fill_normal_bf16(t->embed, V * d, 0.02f, ++k, s), 1);
  CK(fill_normal_bf16(t->lm_head, V * d, 0.02f, ++k, s), 1);
  CK(fill_const_bf16(t->normf, d, 1.0f, s), 1);
  for (Layer& y : t->layers) {
    CK(fill_normal_bf16(y.wqkv, static_cast<int64_t>(t->W) * d, 0.02f, ++k, s), 1);
    CK(fill_normal_bf16(y.wo, d * d, 0.02f, ++k, s), 1);
    CK(fill_normal_bf16(y.wgu, 2 * F * d, 0.02f, ++k, s), 1);
    CK(fill_normal_bf16(y.wdown, d * F, 0.02f, ++k, s), 1);
    CK(fill_const_bf16(y.norm1, d, 1.0f, s), 1);
    CK(fill_const_bf16(y.norm2, d, 1.0f, s), 1);
  }
  cudaError_t e = cudaStreamSynchronize(s);
  if (e != cudaSuccess) return t->fail(DTX_ERR_CUDA, "init_random_weights: %s", cudaGetErrorString(e));
  std::fill(t->loaded.begin(), t->loaded.end(), 1);
  return DTX_OK;
}

int32_t dtx_quantize_base(dtx_trainer* t, int32_t mode) {
  // mode 4: NF4 (--quantization int4).  Applies to the decoder-layer Linear weights (bitsandbytes skips lm_head; embeddings
  // and norms are never quantised).  The bf16 copies are replaced by packed codes + absmax and freed.
  if (!t) return DTX_ERR_INVALID;
  if (mode == 8)
    return t->fail(DTX_ERR_UNSUPPORTED, "--quantization int8 (bitsandbytes LLM.int8 with runtime outlier decomposition, "
                                         "cmd/tuning/train.py:231-232) is not implemented natively; use int4 or no quantization");
  if (mode != 4) return t->fail(DTX_ERR_INVALID, "quantize_base: mode must be 4 (nf4)");
  if (t->full) return t->fail(DTX_ERR_INVALID, "quantize_base: full-parameter SFT trains the bf16 weights themselves");
  if (t->quant4) return t->fail(DTX_ERR_STATE, "quantize_base: already quantised");
  {
    char buf[160];
    if (const char* m = t->missing_weight(buf, sizeof(buf)))
      return t->fail(DTX_ERR_STATE, "quantize_base: base weight %s is not loaded yet", m);
  }
  cudaSetDevice(t->device);
  const int64_t d = t->mc.hidden, F = t->mc.ffn, W = t->W;
  const int64_t n[4] = {W * d, d * d, 2 * F * d, d * F};
  for (int i = 0; i < 4; ++i)
    if (n[i] % 64) return t->fail(DTX_ERR_INVALID, "quantize_base: matrix sizes must be multiples of the 64-element NF4 block");
  cudaStream_t s = t->stream;
  for (Layer& y : t->layers) {
    bf16** w[4] = {&y.wqkv, &y.wo, &y.wgu, &y.wdown};
    for (int i = 0; i < 4; ++i) {
      if (!t->alloc(&y.q4[i], static_cast<size_t>(n[i] / 2)) || !t->alloc(&y.absmax[i], static_cast<size_t>(n[i] / 64))) return DTX_ERR_CUDA;
      CK(nf4_quantize_pack(*w[i], y.q4[i], y.absmax[i], n[i], s), 1);
    }
    CKM(cudaStreamSynchronize(s));
    for (int i = 0; i < 4; ++i) {
      t->release(*w[i], static_cast<size_t>(n[i]) * sizeof(bf16));
      *w[i] = nullptr;
      t->base_bytes += n[i] / 2 + (n[i] / 64) * 4 - n[i] * static_cast<int64_t>(sizeof(bf16));
    }
  }
  for (int i = 0; i < 4; ++i)
    if (!t->alloc(&t->scratch_w[i], static_cast<size_t>(n[i]))) return DTX_ERR_CUDA;
  if (g_nf4_prefetch) {
    CKM(cudaStreamCreateWithFlags(&t->copy_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 4; ++i) {
      CKM(cudaEventCreateWithFlags(&t->ev_deq[i], cudaEventDisableTiming));
      CKM(cudaEventCreateWithFlags(&t->ev_scr[i], cudaEventDisableTiming));
    }
  }
  t->quant4 = true;
  return DTX_OK;
}

int64_t dtx_base_weight_bytes(const dtx_trainer* t) { return t ? t->base_bytes : 0; }

int32_t dtx_init_lora(dtx_trainer* t, uint64_t seed) {
  if (!t) return DTX_ERR_INVALID;
  if (t->full) return t->fail(DTX_ERR_STATE, "init_lora: this trainer was created for full-parameter SFT (no adapters)");
  cudaSetDevice(t->device);
  const int64_t r = t->tc.lora_r;
  std::vector<float> host(t->n_train, 0.f);
  // peft 0.5.0 LoraLayer.reset_lora_parameters: kaiming_uniform_(A, a=sqrt(5)) => U(-1/sqrt(fan_in), +1/sqrt(fan_in)); B = 0
  uint64_t x = seed ? seed : 0x9E3779B97F4A7C15ull;
  auto next = [&]() {
    x += 0x9E3779B97F4A7C15ull;
    uint64_t z = x;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    z ^= z >> 31;
    return static_cast<float>(z >> 40) * (1.0f / 16777216.0f);
  };
  for (int64_t l = 0; l < t->mc.n_layers; ++l)
    for (int ti = 0; ti < t->nt; ++ti) {
      const int64_t d_in = t->tg[ti].d_in;
      const float bound = 1.0f / sqrtf(static_cast<float>(d_in));
      float* a = host.data() + l * t->per_layer + t->tg[ti].off;
      for (int64_t i = 0; i < d_in * r; ++i) a[i] = (2.f * next() - 1.f) * bound;
    }
  CKM(upload_sync(t->params, host.data(), host.size() * 4, t->stream));
  CKM(cudaMemsetAsync(t->adam_m, 0, t->n_train * 4, t->stream));
  CKM(cudaMemsetAsync(t->adam_v, 0, t->n_train * 4, t->stream));
  t->opt_step = 0;
  t->micro_idx = 0;
  int rc = refresh_shadows(t);
  if (rc) return rc;
  CKM(cudaStreamSynchronize(t->stream));
  t->have_lora = true;
  return DTX_OK;
}

int32_t dtx_step(dtx_trainer* t, const int32_t* ids, const int32_t* labels, const int32_t* seq_lens, int32_t seq_len_batch,
                 int32_t flags, float* loss, float* gnorm, float* lr, int32_t* stepped) {
  if (!t || !ids || !labels) return t ? t->fail(DTX_ERR_INVALID, "null batch") : DTX_ERR_INVALID;
  cudaSetDevice(t->device);
  int rc = check_ready(t);
  if (rc == DTX_OK) rc = set_batch_shape(t, seq_len_batch, seq_lens != nullptr);
  if (rc) return rc;
  RowStarts rs;
  if (plan_packed(t, seq_lens, t->cur_S, &rs)) {  // ragged batch, packed: staging buffers -> sequences back to back
    CKM(cudaMemcpyAsync(t->d_ids_full, ids, static_cast<size_t>(t->cur_M) * 4, cudaMemcpyHostToDevice, t->stream));
    CKM(cudaMemcpyAsync(t->d_labels_full, labels, static_cast<size_t>(t->cur_M) * 4, cudaMemcpyHostToDevice, t->stream));
    CKM(cudaMemcpyAsync(t->d_seq_lens, seq_lens, static_cast<size_t>(t->tc.micro_batch) * 4, cudaMemcpyHostToDevice, t->stream));
    CK(pack_rows(t->d_ids_full, t->d_labels_full, t->cur_S, rs, t->d_ids, t->d_labels, t->d_pos, t->d_row_start, t->stream), 1);
    t->cur_M = rs.start[rs.n];
    t->packed = true;
    rc = do_step(t, flags, loss, gnorm, lr, stepped);
    t->packed = false;
    return rc;
  }
  SubPlan plan;
  if (!t->full) plan_groups(PlanDims{t->mc.hidden, t->mc.ffn, t->W, t->n_sms, t->tc.micro_batch}, seq_lens, labels, t->cur_S, &plan);
  if (plan.n > 1) {  // ragged batch: the whole batch goes to the staging buffers, the length groups gather from there
    const int S_src = t->cur_S;
    CKM(cudaMemcpyAsync(t->d_ids_full, ids, static_cast<size_t>(t->cur_M) * 4, cudaMemcpyHostToDevice, t->stream));
    CKM(cudaMemcpyAsync(t->d_labels_full, labels, static_cast<size_t>(t->cur_M) * 4, cudaMemcpyHostToDevice, t->stream));
    CKM(cudaMemcpyAsync(t->d_lens_full, seq_lens, static_cast<size_t>(t->tc.micro_batch) * 4, cudaMemcpyHostToDevice, t->stream));
    return do_step(t, flags, loss, gnorm, lr, stepped, &plan, t->d_ids_full, t->d_labels_full, t->d_lens_full, S_src);
  }
  CKM(cudaMemcpyAsync(t->d_ids, ids, static_cast<size_t>(t->cur_M) * 4, cudaMemcpyHostToDevice, t->stream));
  CKM(cudaMemcpyAsync(t->d_labels, labels, static_cast<size_t>(t->cur_M) * 4, cudaMemcpyHostToDevice, t->stream));
  if (seq_lens) CKM(cudaMemcpyAsync(t->d_seq_lens, seq_lens, static_cast<size_t>(t->tc.micro_batch) * 4, cudaMemcpyHostToDevice, t->stream));
  return do_step(t, flags, loss, gnorm, lr, stepped);
}

int32_t dtx_step_device(dtx_trainer* t, const void* d_ids, const void* d_labels, const void* d_seq_lens, int32_t seq_len_batch,
                        int32_t flags, float* loss, float* gnorm, float* lr, int32_t* stepped) {
  if (!t || !d_ids || !d_labels) return t ? t->fail(DTX_ERR_INVALID, "null batch") : DTX_ERR_INVALID;
  cudaSetDevice(t->device);
  int rc = check_ready(t);
  if (rc == DTX_OK) rc = set_batch_shape(t, seq_len_batch, d_seq_lens != nullptr);
  if (rc) return rc;
  if (d_seq_lens && g_varlen_pack && g_varlen_split == 1 && t->tc.micro_batch <= 64) {
    // the packed layout is planned on the host from the row lengths (B * 4 bytes)
    t->h_lens.resize(static_cast<size_t>(t->tc.micro_batch));
    CKM(cudaMemcpyAsync(t->h_lens.data(), d_seq_lens, t->h_lens.size() * 4, cudaMemcpyDeviceToHost, t->stream));
    CKM(cudaStreamSynchronize(t->stream));
    RowStarts rs;
    if (plan_packed(t, t->h_lens.data(), t->cur_S, &rs)) {
      CKM(cudaMemcpyAsync(t->d_seq_lens, d_seq_lens, static_cast<size_t>(t->tc.micro_batch) * 4, cudaMemcpyDeviceToDevice, t->stream));
      CK(pack_rows(static_cast<const int32_t*>(d_ids), static_cast<const int32_t*>(d_labels), t->cur_S, rs, t->d_ids, t->d_labels, t->d_pos,
                   t->d_row_start, t->stream), 1);
      t->cur_M = rs.start[rs.n];
      t->packed = true;
      rc = do_step(t, flags, loss, gnorm, lr, stepped);
      t->packed = false;
      return rc;
    }
  }
  if (d_seq_lens && g_varlen_split && !t->full && t->tc.micro_batch > 1 && t->tc.micro_batch <= 64) {
    // the partition is planned on the host: fetch the row lengths and the labels (B*S*4 bytes, tens of microseconds)
    t->h_lens.resize(static_cast<size_t>(t->tc.micro_batch));
    t->h_labels.resize(static_cast<size_t>(t->cur_M));
    CKM(cudaMemcpyAsync(t->h_lens.data(), d_seq_lens, t->h_lens.size() * 4, cudaMemcpyDeviceToHost, t->stream));
    CKM(cudaMemcpyAsync(t->h_labels.data(), d_labels, t->h_labels.size() * 4, cudaMemcpyDeviceToHost, t->stream));
    CKM(cudaStreamSynchronize(t->stream));
    SubPlan plan;
    plan_groups(PlanDims{t->mc.hidden, t->mc.ffn, t->W, t->n_sms, t->tc.micro_batch}, t->h_lens.data(), t->h_labels.data(), t->cur_S, &plan);
    if (plan.n > 1)
      return do_step(t, flags, loss, gnorm, lr, stepped, &plan, static_cast<const int32_t*>(d_ids), static_cast<const int32_t*>(d_labels),
                     static_cast<const int32_t*>(d_seq_lens), t->cur_S);
  }
  CKM(cudaMemcpyAsync(t->d_ids, d_ids, static_cast<size_t>(t->cur_M) * 4, cudaMemcpyDeviceToDevice, t->stream));
  CKM(cudaMemcpyAsync(t->d_labels, d_labels, static_cast<size_t>(t->cur_M) * 4, cudaMemcpyDeviceToDevice, t->stream));
  if (d_seq_lens) CKM(cudaMemcpyAsync(t->d_seq_lens, d_seq_lens, static_cast<size_t>(t->tc.micro_batch) * 4, cudaMemcpyDeviceToDevice, t->stream));
  return do_step(t, flags, loss, gnorm, lr, stepped);
}

int32_t dtx_eval_loss(dtx_trainer* t, const int32_t* ids, const int32_t* labels, const int32_t* seq_lens, int32_t seq_len_batch,
                      float* loss_out, float* row_sum_out, int32_t* row_valid_out) {
  if (!t || !ids || !labels) return t ? t->fail(DTX_ERR_INVALID, "null batch") : DTX_ERR_INVALID;
  cudaSetDevice(t->device);
  int rc = check_ready(t);
  if (rc == DTX_OK) rc = set_batch_shape(t, seq_len_batch, seq_lens != nullptr);
  if (rc) return rc;
  const int B = t->tc.micro_batch;
  float h = 0.f;
  RowStarts rs;
  if (plan_packed(t, seq_lens, t->cur_S, &rs)) {  // ragged batch, packed: one forward pass over the sequences back to back
    CKM(cudaMemcpyAsync(t->d_ids_full, ids, static_cast<size_t>(t->cur_M) * 4, cudaMemcpyHostToDevice, t->stream));
    CKM(cudaMemcpyAsync(t->d_labels_full, labels, static_cast<size_t>(t->cur_M) * 4, cudaMemcpyHostToDevice, t->stream));
    CKM(cudaMemcpyAsync(t->d_seq_lens, seq_lens, static_cast<size_t>(B) * 4, cudaMemcpyHostToDevice, t->stream));
    CK(pack_rows(t->d_ids_full, t->d_labels_full, t->cur_S, rs, t->d_ids, t->d_labels, t->d_pos, t->d_row_start, t->stream), 1);
    t->cur_M = rs.start[rs.n];
    t->packed = true;
    rc = fwd_bwd(t, false);
    t->packed = false;
    if (rc) return rc;
    CKM(cudaMemcpyAsync(&h, t->d_loss, 4, cudaMemcpyDeviceToHost, t->stream));
    if (row_sum_out || row_valid_out) {
      CK(row_loss_stats(t->row_loss, t->d_shift, B, t->cur_S, t->d_row_sum, t->d_row_valid, t->stream, t->d_row_start), 1);
      if (row_sum_out) CKM(cudaMemcpyAsync(row_sum_out, t->d_row_sum, static_cast<size_t>(B) * 4, cudaMemcpyDeviceToHost, t->stream));
      if (row_valid_out) CKM(cudaMemcpyAsync(row_valid_out, t->d_row_valid, static_cast<size_t>(B) * 4, cudaMemcpyDeviceToHost, t->stream));
    }
    cudaError_t e = cudaStreamSynchronize(t->stream);
    if (e != cudaSuccess) return t->fail(DTX_ERR_CUDA, "eval failed on device: %s", cudaGetErrorString(e));
    if (loss_out) *loss_out = h;
    return DTX_OK;
  }
  SubPlan plan;
  if (!t->full) plan_groups(PlanDims{t->mc.hidden, t->mc.ffn, t->W, t->n_sms, B}, seq_lens, labels, t->cur_S, &plan);
  if (plan.n > 1) {
    // ragged batch as length groups (forward only): the per-row statistics come back in group order and are put back in
    // the caller's row order; the batch loss accumulates over the groups with the whole batch's labelled-token count
    const int S_src = t->cur_S;
    CKM(cudaMemcpyAsync(t->d_ids_full, ids, static_cast<size_t>(t->cur_M) * 4, cudaMemcpyHostToDevice, t->stream));
    CKM(cudaMemcpyAsync(t->d_labels_full, labels, static_cast<size_t>(t->cur_M) * 4, cudaMemcpyHostToDevice, t->stream));
    CKM(cudaMemcpyAsync(t->d_lens_full, seq_lens, static_cast<size_t>(B) * 4, cudaMemcpyHostToDevice, t->stream));
    t->h_row_sum.assign(static_cast<size_t>(B), 0.f);
    t->h_row_valid.assign(static_cast<size_t>(B), 0);
    for (int g = 0; g < plan.n && rc == DTX_OK; ++g) {
      RowList rl;
      rl.n = plan.start[g + 1] - plan.start[g];
      for (int k = 0; k < rl.n; ++k) rl.rows[k] = plan.order[plan.start[g] + k];
      cudaError_t ge = gather_rows(t->d_ids_full, t->d_labels_full, t->d_lens_full, S_src, rl, plan.S[g], t->d_ids, t->d_labels,
                                   t->d_seq_lens, t->stream);
      if (ge != cudaSuccess) rc = t->fail(DTX_ERR_CUDA, "gather_rows: %s", cudaGetErrorString(ge));
      if (rc) break;
      t->launches += 1;
      t->cur_B = rl.n;
      t->cur_S = plan.S[g];
      t->cur_M = rl.n * plan.S[g];
      t->use_seq_lens = true;
      t->sub_accum = g > 0;
      t->sub_ndiv = plan.n_div;
      rc = fwd_bwd(t, false);
      if (rc == DTX_OK && (row_sum_out || row_valid_out)) {
        cudaError_t e2 = row_loss_stats(t->row_loss, t->d_shift, rl.n, t->cur_S, t->d_row_sum, t->d_row_valid, t->stream);
        if (e2 == cudaSuccess) e2 = cudaMemcpyAsync(t->h_row_sum.data() + plan.start[g], t->d_row_sum, static_cast<size_t>(rl.n) * 4, cudaMemcpyDeviceToHost, t->stream);
        if (e2 == cudaSuccess) e2 = cudaMemcpyAsync(t->h_row_valid.data() + plan.start[g], t->d_row_valid, static_cast<size_t>(rl.n) * 4, cudaMemcpyDeviceToHost, t->stream);
        // d_row_sum / d_row_valid are reused by the next group: the copies above are stream-ordered in front of its kernels
        if (e2 != cudaSuccess) rc = t->fail(DTX_ERR_CUDA, "eval row statistics: %s", cudaGetErrorString(e2));
        t->launches += 1;
      }
    }
    t->sub_accum = false;
    t->sub_ndiv = 0;
    if (rc) return rc;
    CKM(cudaMemcpyAsync(&h, t->d_loss, 4, cudaMemcpyDeviceToHost, t->stream));
    cudaError_t e = cudaStreamSynchronize(t->stream);
    if (e != cudaSuccess) return t->fail(DTX_ERR_CUDA, "eval failed on device: %s", cudaGetErrorString(e));
    for (int k = 0; k < B; ++k) {
      if (row_sum_out) row_sum_out[plan.order[k]] = t->h_row_sum[static_cast<size_t>(k)];
      if (row_valid_out) row_valid_out[plan.order[k]] = t->h_row_valid[static_cast<size_t>(k)];
    }
    if (loss_out) *loss_out = h;
    return DTX_OK;
  }
  CKM(cudaMemcpyAsync(t->d_ids, ids, static_cast<size_t>(t->cur_M) * 4, cudaMemcpyHostToDevice, t->stream));
  CKM(cudaMemcpyAsync(t->d_labels, labels, static_cast<size_t>(t->cur_M) * 4, cudaMemcpyHostToDevice, t->stream));
  if (seq_lens) CKM(cudaMemcpyAsync(t->d_seq_lens, seq_lens, static_cast<size_t>(B) * 4, cudaMemcpyHostToDevice, t->stream));
  rc = fwd_bwd(t, false);
  if (rc) return rc;
  CKM(cudaMemcpyAsync(&h, t->d_loss, 4, cudaMemcpyDeviceToHost, t->stream));
  if (row_sum_out || row_valid_out) {
    CK(row_loss_stats(t->row_loss, t->d_shift, B, t->cur_S, t->d_row_sum, t->d_row_valid, t->stream), 1);
    if (row_sum_out) CKM(cudaMemcpyAsync(row_sum_out, t->d_row_sum, static_cast<size_t>(B) * 4, cudaMemcpyDeviceToHost, t->stream));
    if (row_valid_out) CKM(cudaMemcpyAsync(row_valid_out, t->d_row_valid, static_cast<size_t>(B) * 4, cudaMemcpyDeviceToHost, t->stream));
  }
  cudaError_t e = cudaStreamSynchronize(t->stream);
  if (e != cudaSuccess) return t->fail(DTX_ERR_CUDA, "eval failed on device: %s", cudaGetErrorString(e));
  if (loss_out) *loss_out = h;
  return DTX_OK;
}

int32_t dtx_allreduce_host(dtx_trainer* t, double* inout, int32_t n) {
  if (!t || !inout || n < 0 || n > 64) return t ? t->fail(DTX_ERR_INVALID, "allreduce_host: n must be in [0, 64]") : DTX_ERR_INVALID;
  if (t->world == 1 || n == 0) return DTX_OK;
  cudaSetDevice(t->device);
  NcclApi* api = nccl_api();
  if (!api || !t->nccl_comm) return t->fail(DTX_ERR_NCCL, "NCCL communicator missing for world=%d", t->world);
  CKM(cudaMemcpyAsync(t->d_host_red, inout, static_cast<size_t>(n) * 8, cudaMemcpyHostToDevice, t->stream));
  int rc = api->AllReduce(t->d_host_red, t->d_host_red, static_cast<size_t>(n), kNcclFloat64, kNcclSum, t->nccl_comm, t->stream);
  if (rc != 0) return t->fail(DTX_ERR_NCCL, "ncclAllReduce failed: %s", api->GetErrorString ? api->GetErrorString(rc) : "?");
  CKM(cudaMemcpyAsync(inout, t->d_host_red, static_cast<size_t>(n) * 8, cudaMemcpyDeviceToHost, t->stream));
  CKM(cudaStreamSynchronize(t->stream));
  return DTX_OK;
}

static int32_t export_lora_tensor(dtx_trainer* t, const float* flat, const char* name, void* host_out, int64_t nbytes) {
  if (!t || !name || !host_out) return t ? t->fail(DTX_ERR_INVALID, "null argument") : DTX_ERR_INVALID;
  if (t->full || !flat) return t->fail(DTX_ERR_STATE, "no adapters: this trainer was created for full-parameter SFT");
  cudaSetDevice(t->device);
  const int64_t r = t->tc.lora_r;
  int layer = -1;
  const char* rest = nullptr;
  if (!parse_layer(name, &layer, &rest) || layer < 0 || layer >= t->mc.n_layers)
    return t->fail(DTX_ERR_INVALID, "bad adapter tensor name %s", name);
  const int ti = target_index(t, rest);
  if (ti < 0) return t->fail(DTX_ERR_INVALID, "%s: module is not a LoRA target", name);
  const int64_t d_in = t->tg[ti].d_in, d_out = t->tg[ti].d_out;
  const bool is_a = strstr(rest, "lora_A") != nullptr;
  if (nbytes < (is_a ? d_in : d_out) * r * 4) return t->fail(DTX_ERR_INVALID, "%s: output buffer too small", name);
  const float* base = flat + static_cast<int64_t>(layer) * t->per_layer + t->tg[ti].off;
  CKM(cudaStreamSynchronize(t->stream));
  std::vector<float> tmp(d_in * r);
  float* out = static_cast<float*>(host_out);
  if (strstr(rest, "lora_A")) {
    CKM(cudaMemcpyAsync(tmp.data(), base, d_in * r * 4, cudaMemcpyDeviceToHost, t->stream));
    CKM(cudaStreamSynchronize(t->stream));
    for (int64_t c = 0; c < d_in; ++c)
      for (int64_t j = 0; j < r; ++j) out[j * d_in + c] = tmp[c * r + j];
  } else if (strstr(rest, "lora_B")) {
    CKM(cudaMemcpyAsync(out, base + d_in * r, d_out * r * 4, cudaMemcpyDeviceToHost, t->stream));
    CKM(cudaStreamSynchronize(t->stream));
  } else {
    return t->fail(DTX_ERR_INVALID, "%s: expected lora_A or lora_B", name);
  }
  return DTX_OK;
}

int32_t dtx_export_adapter(dtx_trainer* t, const char* name, void* host_out, int64_t nbytes) {
  return export_lora_tensor(t, t ? t->params : nullptr, name, host_out, nbytes);
}
int32_t dtx_export_adapter_grad(dtx_trainer* t, const char* name, void* host_out, int64_t nbytes) {
  return export_lora_tensor(t, t ? t->grads : nullptr, name, host_out, nbytes);
}

// Full-parameter SFT: one weight (grad = 0) or its accumulated gradient (grad = 1) by HF name, as bf16 bit patterns in the HF
// layout (gate / up rows taken back out of the GU-interleaved storage).  Gradients are only complete on a single rank.
int32_t dtx_export_weight(dtx_trainer* t, const char* name, void* host_out, int64_t nbytes, int32_t grad) {
  if (!t || !name || !host_out) return t ? t->fail(DTX_ERR_INVALID, "null argument") : DTX_ERR_INVALID;
  if (!t->full) return t->fail(DTX_ERR_STATE, "export_weight: only for full-parameter SFT trainers (LoRA: dtx_export_adapter)");
  cudaSetDevice(t->device);
  wait_all_weights(t);
  CKM(cudaStreamSynchronize(t->stream));
  const int64_t d = t->mc.hidden, F = t->mc.ffn, V = t->mc.vocab, dq = t->dq, dkv = t->dkv, L = t->mc.n_layers;
  const bf16* flat = grad ? t->g_flat : t->w_flat;
  const bf16* gl = flat + L * t->layer_elems;
  auto copy = [&](const bf16* src, int64_t n) -> int32_t {
    if (nbytes < n * 2) return t->fail(DTX_ERR_INVALID, "%s: output buffer too small", name);
    CKM(cudaMemcpyAsync(host_out, src, n * 2, cudaMemcpyDeviceToHost, t->stream));
    CKM(cudaStreamSynchronize(t->stream));
    return DTX_OK;
  };
  if (strstr(name, "embed_tokens.weight")) return copy(gl, V * d);
  if (strstr(name, "lm_head.weight")) return copy(gl + t->goff_lm, V * d);
  int layer = -1;
  const char* rest = nullptr;
  if (!parse_layer(name, &layer, &rest)) {
    if (strstr(name, "norm.weight")) return copy(gl + t->goff_nf, d);
    return t->fail(DTX_ERR_INVALID, "unknown tensor name %s", name);
  }
  if (layer < 0 || layer >= L) return t->fail(DTX_ERR_INVALID, "%s: layer out of range", name);
  const bf16* blk = flat + layer * t->layer_elems;
  for (int which = 0; which < 2; ++which) {
    if (!strstr(rest, which ? "mlp.up_proj.weight" : "mlp.gate_proj.weight")) continue;
    if (nbytes < F * d * 2) return t->fail(DTX_ERR_INVALID, "%s: output buffer too small", name);
    for (int64_t b = 0; b < F / 128; ++b)
      CKM(cudaMemcpyAsync(static_cast<bf16*>(host_out) + b * 128 * d, blk + t->off_wgu + (b * 256 + which * 128) * d, 128 * d * 2,
                          cudaMemcpyDeviceToHost, t->stream));
    CKM(cudaStreamSynchronize(t->stream));
    return DTX_OK;
  }
  struct Slot { const char* key; int64_t off, n; };
  const Slot slots[] = {
      {"self_attn.q_proj.weight", 0, dq * d}, {"self_attn.k_proj.weight", dq * d, dkv * d},
      {"self_attn.v_proj.weight", (dq + dkv) * d, dkv * d}, {"self_attn.o_proj.weight", t->off_wo, d * d},
      {"mlp.down_proj.weight", t->off_wdown, d * F}, {"input_layernorm.weight", t->off_n1, d},
      {"post_attention_layernorm.weight", t->off_n2, d},
  };
  for (const Slot& sl : slots)
    if (strstr(rest, sl.key)) return copy(blk + sl.off, sl.n);
  return t->fail(DTX_ERR_INVALID, "unknown tensor name %s", name);
}

int64_t dtx_num_trainable(const dtx_trainer* t) { return t ? t->n_train : 0; }
int64_t dtx_launch_count(const dtx_trainer* t) { return t ? t->launches : 0; }
float dtx_last_step_ms(const dtx_trainer* t) { return t ? t->last_ms : 0.f; }
int32_t dtx_last_step_groups(const dtx_trainer* t) { return t ? t->last_groups : 0; }

int32_t dtx_plan_packed_rows(int32_t micro_batch, const int32_t* seq_lens, int32_t seq_len_batch, int32_t* row_start_out) {
  if (!seq_lens || !row_start_out || micro_batch < 1 || micro_batch > 64 || seq_len_batch < 128 || seq_len_batch % 128) return DTX_ERR_INVALID;
  RowStarts rs;
  const bool saves = packed_rows(seq_lens, micro_batch, seq_len_batch, &rs);
  for (int b = 0; b <= micro_batch; ++b) row_start_out[b] = rs.start[b];
  return saves ? 1 : 0;
}

int32_t dtx_plan_length_groups(const dtx_model_cfg* mc, int32_t micro_batch, int32_t n_sms, const int32_t* seq_lens, int32_t seq_len_batch,
                               int32_t* order_out, int32_t* group_start_out, int32_t* group_len_out) {
  if (!mc || !seq_lens || !order_out || !group_start_out || !group_len_out || micro_batch < 1 || seq_len_batch < 128 || seq_len_batch % 128)
    return DTX_ERR_INVALID;
  const int hkv = mc->n_kv_heads > 0 ? mc->n_kv_heads : mc->n_heads;
  SubPlan plan;
  plan_groups(PlanDims{mc->hidden, mc->ffn, (mc->n_heads + 2 * hkv) * mc->head_dim, n_sms > 0 ? n_sms : 148, micro_batch}, seq_lens, nullptr,
              seq_len_batch, &plan);
  if (plan.n <= 1) {  // one pass at the batch's padded length, rows in their own order
    for (int i = 0; i < micro_batch; ++i) order_out[i] = i;
    group_start_out[0] = 0;
    group_start_out[1] = micro_batch;
    group_len_out[0] = seq_len_batch;
    return 1;
  }
  for (int i = 0; i < micro_batch; ++i) order_out[i] = plan.order[i];
  for (int g = 0; g <= plan.n; ++g) group_start_out[g] = plan.start[g];
  for (int g = 0; g < plan.n; ++g) group_len_out[g] = plan.S[g];
  return plan.n;
}

int32_t dtx_last_step_timings(const dtx_trainer* t, float* out4) {
  if (!t || !out4) return DTX_ERR_INVALID;
  for (int i = 0; i < 4; ++i) out4[i] = t->seg_ms[i];
  return DTX_OK;
}

}  // extern "C"
