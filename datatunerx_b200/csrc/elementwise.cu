// HBM-bound kernels of the LoRA-SFT step (SURVEY §2.3 K1,K2,K5,K9,K11,K13 + SwiGLU elementwise).
// All of them are single-pass over their algorithmic bytes with 16-byte vector accesses, fp32 math,
// warp-shuffle reductions and fixed (deterministic) summation orders.  None uses tensor cores:
// they are bandwidth-bound and are measured against the HBM roofline (DESIGN.md §4).
#include "common.cuh"
#include "kernels.h"

namespace dtx {

namespace {

__device__ __forceinline__ void bf16x8_to_f32(const uint4& u, float (&f)[8]) {
  float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y), c = unpack_bf16x2(u.z), d = unpack_bf16x2(u.w);
  f[0] = a.x; f[1] = a.y; f[2] = b.x; f[3] = b.y; f[4] = c.x; f[5] = c.y; f[6] = d.x; f[7] = d.y;
}
__device__ __forceinline__ uint4 f32_to_bf16x8(const float (&f)[8]) {
  uint4 o;
  o.x = pack_bf16x2(f[0], f[1]); o.y = pack_bf16x2(f[2], f[3]);
  o.z = pack_bf16x2(f[4], f[5]); o.w = pack_bf16x2(f[6], f[7]);
  return o;
}
__device__ __forceinline__ uint4 ldg_stream(const uint4* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}

// block-wide sum, result broadcast to all threads. blockDim.x multiple of 32, <= 1024.
__device__ __forceinline__ float block_sum(float v, float* sh) {
  v = warp_sum(v);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31, nw = blockDim.x >> 5;
  __syncthreads();
  if (l == 0) sh[w] = v;
  __syncthreads();
  float t = 0.f;
  for (int i = 0; i < nw; ++i) t += sh[i];  // fixed order
  return t;
}

// ------------------------------------------------------------------------------------------
// K1: embedding gather.  HF nn.Embedding forward (transformers LlamaModel.embed_tokens).
// ------------------------------------------------------------------------------------------
__global__ void embedding_kernel(const int32_t* __restrict__ ids, const bf16* __restrict__ table, bf16* __restrict__ out,
                                 int d, int vocab) {
  const int m = blockIdx.x;
  int id = ids[m];
  if (id < 0 || id >= vocab) id = 0;
  const uint4* src = reinterpret_cast<const uint4*>(table + static_cast<size_t>(id) * d);
  uint4* dst = reinterpret_cast<uint4*>(out + static_cast<size_t>(m) * d);
  for (int i = threadIdx.x; i < d / 8; i += blockDim.x) dst[i] = __ldg(src + i);
}

// ------------------------------------------------------------------------------------------
// K2: RMSNorm.  One 128-thread block per row; the row lives in registers between the reduce and the scale
// (NCH 16-byte chunks per thread), so each element is read from HBM exactly once.  Many small blocks per SM
// (16 x 4 warps) keep enough loads in flight to saturate HBM; r01's one-warp-per-row version held 32 chunks per
// thread in 150 registers, ran 8 warps/SM and reached only 31% of HBM bandwidth (profiles/r01_launches_bwd.txt).
//   y = w * (x * rsqrt(mean(x^2) + eps)), all math fp32 (HF LlamaRMSNorm computes in fp32).
// ------------------------------------------------------------------------------------------
constexpr int RMS_THREADS = 128;

__device__ __forceinline__ float block_sum_128(float v, float* sh4) {
  v = warp_sum(v);
  if ((threadIdx.x & 31) == 0) sh4[threadIdx.x >> 5] = v;
  __syncthreads();
  return (sh4[0] + sh4[1]) + (sh4[2] + sh4[3]);  // fixed order
}

template <int NCH>
__global__ void __launch_bounds__(RMS_THREADS) rmsnorm_fwd_kernel(const bf16* __restrict__ x, const bf16* __restrict__ w,
                                                                  bf16* __restrict__ y, float* __restrict__ rstd, int d,
                                                                  float eps, const int32_t* __restrict__ row_map) {
  __shared__ float sh[4];
  const int row = blockIdx.x;
  const int out_row = row_map ? row_map[row] : row;
  if (out_row < 0) return;  // this token is not needed downstream (block-uniform)
  const uint4* xr = reinterpret_cast<const uint4*>(x + static_cast<size_t>(row) * d);
  const int nvec = d >> 3;
  uint4 buf[NCH];
  float ss = 0.f;
#pragma unroll
  for (int i = 0; i < NCH; ++i) {
    const int v = i * RMS_THREADS + threadIdx.x;
    if (v < nvec) buf[i] = ldg_stream(xr + v);
  }
#pragma unroll
  for (int i = 0; i < NCH; ++i) {
    const int v = i * RMS_THREADS + threadIdx.x;
    if (v < nvec) {
      float f[8];
      bf16x8_to_f32(buf[i], f);
#pragma unroll
      for (int j = 0; j < 8; ++j) ss += f[j] * f[j];
    }
  }
  ss = block_sum_128(ss, sh);
  const float r = rsqrtf(ss / static_cast<float>(d) + eps);
  if (threadIdx.x == 0 && rstd) rstd[row] = r;
  const uint4* wr = reinterpret_cast<const uint4*>(w);
  uint4* yr = reinterpret_cast<uint4*>(y + static_cast<size_t>(out_row) * d);
#pragma unroll
  for (int i = 0; i < NCH; ++i) {
    const int v = i * RMS_THREADS + threadIdx.x;
    if (v < nvec) {
      float f[8], g[8];
      bf16x8_to_f32(buf[i], f);
      bf16x8_to_f32(__ldg(wr + v), g);
#pragma unroll
      for (int j = 0; j < 8; ++j) f[j] = f[j] * r * g[j];
      yr[v] = f32_to_bf16x8(f);
    }
  }
}

// dx = rstd * (w*dy) - x * rstd^3 * mean(w*dy*x) (+ dres).  Base weights are frozen: no dw.
template <int NCH>
__global__ void __launch_bounds__(RMS_THREADS) rmsnorm_bwd_kernel(const bf16* __restrict__ dy, const bf16* __restrict__ x,
                                                                  const bf16* __restrict__ w, const float* __restrict__ rstd,
                                                                  const bf16* __restrict__ dres, bf16* __restrict__ dx, int d,
                                                                  const int32_t* __restrict__ row_map) {
  __shared__ float sh[4];
  const int row = blockIdx.x;
  const size_t off = static_cast<size_t>(row) * d;
  const int src_row = row_map ? row_map[row] : row;
  if (src_row < 0) {  // no gradient arrives for this token: dx = dres (or 0)
    const int nv = d >> 3;
    for (int v = threadIdx.x; v < nv; v += RMS_THREADS)
      reinterpret_cast<uint4*>(dx + off)[v] = dres ? ldg_stream(reinterpret_cast<const uint4*>(dres + off) + v) : make_uint4(0u, 0u, 0u, 0u);
    return;
  }
  const uint4* dyr = reinterpret_cast<const uint4*>(dy + static_cast<size_t>(src_row) * d);
  const uint4* xr = reinterpret_cast<const uint4*>(x + off);
  const uint4* wr = reinterpret_cast<const uint4*>(w);
  const uint4* rr = dres ? reinterpret_cast<const uint4*>(dres + off) : nullptr;
  const int nvec = d >> 3;
  uint4 bx[NCH], bg[NCH], br[NCH];
#pragma unroll
  for (int i = 0; i < NCH; ++i) {
    const int v = i * RMS_THREADS + threadIdx.x;
    if (v < nvec) {
      bx[i] = ldg_stream(xr + v);
      bg[i] = ldg_stream(dyr + v);
      if (rr) br[i] = ldg_stream(rr + v);
    }
  }
  float dot = 0.f;
#pragma unroll
  for (int i = 0; i < NCH; ++i) {
    const int v = i * RMS_THREADS + threadIdx.x;
    if (v < nvec) {
      float fx[8], fg[8], fw[8];
      bf16x8_to_f32(bx[i], fx);
      bf16x8_to_f32(bg[i], fg);
      bf16x8_to_f32(__ldg(wr + v), fw);
#pragma unroll
      for (int j = 0; j < 8; ++j) dot += fg[j] * fw[j] * fx[j];
    }
  }
  dot = block_sum_128(dot, sh);
  const float r = rstd[row];
  const float c = dot * r * r * r / static_cast<float>(d);
  uint4* dxr = reinterpret_cast<uint4*>(dx + off);
#pragma unroll
  for (int i = 0; i < NCH; ++i) {
    const int v = i * RMS_THREADS + threadIdx.x;
    if (v < nvec) {
      float fx[8], fg[8], fw[8], o[8];
      bf16x8_to_f32(bx[i], fx);
      bf16x8_to_f32(bg[i], fg);
      bf16x8_to_f32(__ldg(wr + v), fw);
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = fg[j] * fw[j] * r - fx[j] * c;
      if (rr) {
        float fr[8];
        bf16x8_to_f32(br[i], fr);
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] += fr[j];
      }
      dxr[v] = f32_to_bf16x8(o);
    }
  }
}

// ------------------------------------------------------------------------------------------
// K5: rotary embedding, half-split convention (HF rotate_half), in place on q and k of packed qkv.
//   out[i] = x[i] cos - x[i+D/2] sin ; out[i+D/2] = x[i+D/2] cos + x[i] sin ; inverse flips sin.
// cs table: [S][D/2] float2(cos, sin), built in double precision on the host.
// ------------------------------------------------------------------------------------------
__global__ void rope_kernel(bf16* __restrict__ qkv, const float2* __restrict__ cs, int S, int NH, int W, int D, int inverse,
                            long long total_vec) {
  // one thread handles 8 consecutive i (one uint4 from each half) of one (token, head); heads 0..NH-1 = q heads then k heads
  const int half = D >> 1;
  const int vec_per_head = half >> 3;
  for (long long t = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; t < total_vec;
       t += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int iv = static_cast<int>(t % vec_per_head);
    long long r = t / vec_per_head;
    const int h = static_cast<int>(r % NH);
    const long long m = r / NH;
    const int pos = static_cast<int>(m % S);
    bf16* base = qkv + m * static_cast<long long>(W) + static_cast<long long>(h) * D + iv * 8;
    uint4 lo = *reinterpret_cast<uint4*>(base);
    uint4 hi = *reinterpret_cast<uint4*>(base + half);
    float a[8], b[8];
    bf16x8_to_f32(lo, a);
    bf16x8_to_f32(hi, b);
    const float2* c = cs + static_cast<size_t>(pos) * half + iv * 8;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float2 v = __ldg(c + j);
      const float sn = inverse ? -v.y : v.y;
      const float x0 = a[j], x1 = b[j];
      a[j] = x0 * v.x - x1 * sn;
      b[j] = x1 * v.x + x0 * sn;
    }
    *reinterpret_cast<uint4*>(base) = f32_to_bf16x8(a);
    *reinterpret_cast<uint4*>(base + half) = f32_to_bf16x8(b);
  }
}

// ------------------------------------------------------------------------------------------
// SwiGLU elementwise (HF LlamaMLP: down(silu(gate(x)) * up(x))) on packed [gate | up].
// ------------------------------------------------------------------------------------------
__global__ void swiglu_fwd_kernel(const bf16* __restrict__ gu, bf16* __restrict__ act, int M, int F, int il) {
  const int vecF = F >> 3;
  const long long total = static_cast<long long>(M) * vecF;
  for (long long t = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; t < total;
       t += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long m = t / vecF;
    const int v = static_cast<int>(t % vecF);
    // il: GU-interleaved layout, feature f -> gate at (f/128)*256 + f%128, up 128 further; else [gate F | up F]
    const int f = v << 3;
    const long long gpos = il ? (static_cast<long long>(f >> 7) * 256 + (f & 127)) : f;
    const uint4* g = reinterpret_cast<const uint4*>(gu + m * 2LL * F + gpos);
    const uint4* u = reinterpret_cast<const uint4*>(gu + m * 2LL * F + gpos + (il ? 128 : F));
    float fg[8], fu[8];
    bf16x8_to_f32(ldg_stream(g), fg);
    bf16x8_to_f32(ldg_stream(u), fu);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float s = 1.f / (1.f + __expf(-fg[j]));
      fg[j] = fg[j] * s * fu[j];
    }
    reinterpret_cast<uint4*>(act + m * static_cast<long long>(F))[v] = f32_to_bf16x8(fg);
  }
}
__device__ __forceinline__ bool drop_keep(uint64_t key, int target, long long idx, uint32_t thresh);
// glora (optional): LoRA dropout on down_proj's input - d(act) = dact + mask o glora / (1 - p), the mask regenerated (target 0
// of `key`, element m*F + f), so that the masked LoRA-branch gradient joins the SwiGLU backward without another pass over HBM
__global__ void swiglu_bwd_kernel(const bf16* __restrict__ dact, const bf16* __restrict__ gu, bf16* __restrict__ dgu,
                                  int M, int F, int il, const bf16* __restrict__ glora = nullptr, uint32_t thresh = 0,
                                  float inv_keep = 1.f, uint64_t key = 0) {
  const int vecF = F >> 3;
  const long long total = static_cast<long long>(M) * vecF;
  for (long long t = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; t < total;
       t += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long m = t / vecF;
    const int v = static_cast<int>(t % vecF);
    float fg[8], fu[8], fd[8], og[8], ou[8];
    const int f = v << 3;
    const long long gpos = il ? (static_cast<long long>(f >> 7) * 256 + (f & 127)) : f;
    const long long upos = gpos + (il ? 128 : F);
    bf16x8_to_f32(ldg_stream(reinterpret_cast<const uint4*>(gu + m * 2LL * F + gpos)), fg);
    bf16x8_to_f32(ldg_stream(reinterpret_cast<const uint4*>(gu + m * 2LL * F + upos)), fu);
    bf16x8_to_f32(ldg_stream(reinterpret_cast<const uint4*>(dact + m * static_cast<long long>(F)) + v), fd);
    if (glora) {
      float fl[8];
      bf16x8_to_f32(ldg_stream(reinterpret_cast<const uint4*>(glora + m * static_cast<long long>(F)) + v), fl);
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (drop_keep(key, 0, m * F + f + j, thresh)) fd[j] += fl[j] * inv_keep;
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float s = 1.f / (1.f + __expf(-fg[j]));
      const float silu = fg[j] * s;
      ou[j] = fd[j] * silu;
      og[j] = fd[j] * fu[j] * (s + silu * (1.f - s));  // d/dg [g*sigmoid(g)] = s + g*s*(1-s)
    }
    *reinterpret_cast<uint4*>(dgu + m * 2LL * F + gpos) = f32_to_bf16x8(og);
    *reinterpret_cast<uint4*>(dgu + m * 2LL * F + upos) = f32_to_bf16x8(ou);
  }
}

// ------------------------------------------------------------------------------------------
// K9: shifted-label cross entropy (HF ForCausalLMLoss: logits[..., :-1] vs labels[..., 1:],
// ignore_index -100, mean over valid tokens).
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) shift_labels_kernel(const int32_t* __restrict__ labels, int32_t* __restrict__ shifted,
                                                            int32_t* __restrict__ n_valid, int B, int S,
                                                            int32_t* __restrict__ row_map, int32_t* __restrict__ valid_idx,
                                                            const int32_t* __restrict__ pos) {
  // one block; thread t owns the contiguous token range [t*c, (t+1)*c): counts, block-wide exclusive scan, ordered positions
  __shared__ int sh[1024];
  const int total = B * S;
  const int c = (total + blockDim.x - 1) / blockDim.x;
  const int lo = min(total, static_cast<int>(threadIdx.x) * c), hi = min(total, lo + c);
  int cnt = 0;
  for (int i = lo; i < hi; ++i) {
    // last token of its sequence: nothing to predict.  Packed ragged batch: the next token starts a new sequence (position 0)
    const bool last = pos ? (i + 1 >= total || pos[i + 1] == 0) : (i % S == S - 1);
    const int v = last ? -100 : labels[i + 1];
    shifted[i] = v;
    cnt += (v >= 0) ? 1 : 0;
  }
  sh[threadIdx.x] = cnt;
  __syncthreads();
  for (int o = 1; o < static_cast<int>(blockDim.x); o <<= 1) {  // Hillis-Steele inclusive scan
    const int add = (static_cast<int>(threadIdx.x) >= o) ? sh[threadIdx.x - o] : 0;
    __syncthreads();
    sh[threadIdx.x] += add;
    __syncthreads();
  }
  if (threadIdx.x == blockDim.x - 1) *n_valid = sh[threadIdx.x];
  if (row_map) {
    int pos = sh[threadIdx.x] - cnt;
    for (int i = lo; i < hi; ++i) {
      if (shifted[i] >= 0) {
        row_map[i] = pos;
        valid_idx[pos] = i;
        ++pos;
      } else {
        row_map[i] = -1;
      }
    }
  }
}

// one block per row: online (max, sum-exp) in one read, then p - onehot scaled by 1/n_valid.
__global__ void __launch_bounds__(256) ce_kernel(const float* __restrict__ logits, long long ldl,
                                                 const int32_t* __restrict__ labels, const int32_t* __restrict__ n_valid,
                                                 float* __restrict__ row_loss, bf16* __restrict__ dlogits, long long ldd,
                                                 int V, const int32_t* __restrict__ valid_idx, int n_div) {
  __shared__ float shm[8], shs[8];
  __shared__ float s_max, s_sum;
  const int row = blockIdx.x;  // row of logits / dlogits
  if (valid_idx && row >= *n_valid) return;
  const int tok = valid_idx ? valid_idx[row] : row;  // token whose label / row_loss this is
  const int label = labels[tok];
  bf16* drow = dlogits ? dlogits + static_cast<long long>(row) * ldd : nullptr;
  const int nv4 = V >> 2;
  if (label < 0 || label >= V) {  // ignored token: zero gradient row, zero loss
    if (threadIdx.x == 0) row_loss[tok] = 0.f;
    if (drow) {
      uint2 z = make_uint2(0u, 0u);
      for (int i = threadIdx.x; i < nv4; i += blockDim.x) reinterpret_cast<uint2*>(drow)[i] = z;
      for (int i = (nv4 << 2) + threadIdx.x; i < V; i += blockDim.x) drow[i] = __float2bfloat16_rn(0.f);
    }
    return;
  }
  const float* lrow = logits + static_cast<long long>(row) * ldl;
  float mx = -INFINITY, sm = 0.f;
  for (int i = threadIdx.x; i < nv4; i += blockDim.x) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(lrow) + i);
    const float m4 = fmaxf(fmaxf(v.x, v.y), fmaxf(v.z, v.w));
    if (m4 > mx) { sm *= __expf(mx - m4); mx = m4; }
    sm += __expf(v.x - mx) + __expf(v.y - mx) + __expf(v.z - mx) + __expf(v.w - mx);
  }
  for (int i = (nv4 << 2) + threadIdx.x; i < V; i += blockDim.x) {
    const float v = lrow[i];
    if (v > mx) { sm *= __expf(mx - v); mx = v; }
    sm += __expf(v - mx);
  }
  // warp then block combine of (max, sum)
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float om = __shfl_xor_sync(0xffffffffu, mx, o), os = __shfl_xor_sync(0xffffffffu, sm, o);
    const float nm = fmaxf(mx, om);
    // a lane with no elements (V < 4 * blockDim) holds (-inf, 0): (-inf) - (-inf) would be NaN
    sm = (mx == -INFINITY ? 0.f : sm * __expf(mx - nm)) + (om == -INFINITY ? 0.f : os * __expf(om - nm));
    mx = nm;
  }
  if ((threadIdx.x & 31) == 0) { shm[threadIdx.x >> 5] = mx; shs[threadIdx.x >> 5] = sm; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float M0 = shm[0], S0 = shs[0];
    for (int i = 1; i < (blockDim.x >> 5); ++i) {
      const float nm = fmaxf(M0, shm[i]);
      S0 = (M0 == -INFINITY ? 0.f : S0 * __expf(M0 - nm)) + (shm[i] == -INFINITY ? 0.f : shs[i] * __expf(shm[i] - nm));
      M0 = nm;
    }
    s_max = M0;
    s_sum = S0;
    row_loss[tok] = (M0 + logf(S0)) - lrow[label];
  }
  __syncthreads();
  if (!drow) return;
  const float M0 = s_max;
  const float inv = 1.f / s_sum;
  // n_div > 0: this launch covers one length group of a micro-batch; the mean runs over the labelled tokens of ALL its groups
  const float scale = 1.f / static_cast<float>(max(n_div > 0 ? n_div : *n_valid, 1));
  for (int i = threadIdx.x; i < nv4; i += blockDim.x) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(lrow) + i);
    float p0 = __expf(v.x - M0) * inv, p1 = __expf(v.y - M0) * inv, p2 = __expf(v.z - M0) * inv, p3 = __expf(v.w - M0) * inv;
    const int c = i << 2;
    if (label >= c && label < c + 4) {
      if (label == c) p0 -= 1.f; else if (label == c + 1) p1 -= 1.f; else if (label == c + 2) p2 -= 1.f; else p3 -= 1.f;
    }
    uint2 o;
    o.x = pack_bf16x2(p0 * scale, p1 * scale);
    o.y = pack_bf16x2(p2 * scale, p3 * scale);
    reinterpret_cast<uint2*>(drow)[i] = o;
  }
  for (int i = (nv4 << 2) + threadIdx.x; i < V; i += blockDim.x) {
    float p = __expf(lrow[i] - M0) * inv;
    if (i == label) p -= 1.f;
    drow[i] = __float2bfloat16_rn(p * scale);
  }
}

__global__ void loss_reduce_kernel(const float* __restrict__ row_loss, const int32_t* __restrict__ n_valid,
                                   float* __restrict__ loss, int M, int n_div, int accumulate) {
  __shared__ float sh[32];
  // fixed assignment of rows to threads + fixed-order combine => bitwise reproducible
  double acc = 0.0;
  for (int i = threadIdx.x; i < M; i += blockDim.x) acc += static_cast<double>(row_loss[i]);
  float v = static_cast<float>(acc);
  v = block_sum(v, sh);
  if (threadIdx.x == 0) *loss = (accumulate ? *loss : 0.f) + v / static_cast<float>(max(n_div > 0 ? n_div : *n_valid, 1));
}

__global__ void sum_partials_kernel(const float* __restrict__ partial, float* __restrict__ out, long long n, int splits) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    float s = 0.f;
    for (int k = 0; k < splits; ++k) s += partial[k * n + i];
    out[i] = s;
  }
}

// ------------------------------------------------------------------------------------------
// K11: gradient norm (deterministic two-stage) and K13: fused clip + AdamW
// ------------------------------------------------------------------------------------------
constexpr int SUMSQ_BLOCKS = 296;
__global__ void sumsq_stage1(const float* __restrict__ g, long long n, float* __restrict__ scratch) {
  __shared__ float sh[32];
  float acc = 0.f;
  const long long n4 = n >> 2;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(g) + i);
    acc += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
  }
  if (blockIdx.x == 0)
    for (long long i = (n4 << 2) + threadIdx.x; i < n; i += blockDim.x) acc += g[i] * g[i];
  acc = block_sum(acc, sh);
  if (threadIdx.x == 0) scratch[blockIdx.x] = acc;
}
__global__ void sumsq_stage2(const float* __restrict__ scratch, int nblocks, float* __restrict__ out) {
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int i = 0; i < nblocks; ++i) s += static_cast<double>(scratch[i]);
    *out = static_cast<float>(s);
  }
}

// torch.optim.AdamW (decoupled weight decay, no amsgrad) fused with torch.nn.utils.clip_grad_norm_:
//   clip = min(1, max_norm / (||g|| + 1e-6));  p *= 1 - lr*wd;  m,v update;  p -= lr/bias1 * m / (sqrt(v)/sqrt(bias2) + eps)
__global__ void adamw_kernel(AdamWArgs a) {
  float gs = a.grad_scale;
  if (a.sumsq) {
    const float norm = sqrtf(*a.sumsq) * a.grad_scale;
    if (a.grad_norm_out && blockIdx.x == 0 && threadIdx.x == 0) *a.grad_norm_out = norm;
    if (a.max_grad_norm > 0.f) {
      const float coef = a.max_grad_norm / (norm + 1e-6f);
      if (coef < 1.f) gs *= coef;
    }
  }
  const float step = a.lr / a.bias1;
  const float rs2 = rsqrtf(a.bias2);
  const float decay = 1.f - a.lr * a.weight_decay;
  const long long n4 = a.n >> 2;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    float4 p = reinterpret_cast<float4*>(a.p)[i];
    const float4 g4 = __ldg(reinterpret_cast<const float4*>(a.g) + i);
    float4 m = reinterpret_cast<float4*>(a.m)[i];
    float4 v = reinterpret_cast<float4*>(a.v)[i];
    float* pp = &p.x; const float* gp = &g4.x; float* mp = &m.x; float* vp = &v.x;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float g = gp[j] * gs;
      pp[j] *= decay;
      mp[j] = a.beta1 * mp[j] + (1.f - a.beta1) * g;
      vp[j] = a.beta2 * vp[j] + (1.f - a.beta2) * g * g;
      const float denom = sqrtf(vp[j]) * rs2 + a.eps;
      pp[j] -= step * (mp[j] / denom);
    }
    reinterpret_cast<float4*>(a.p)[i] = p;
    reinterpret_cast<float4*>(a.m)[i] = m;
    reinterpret_cast<float4*>(a.v)[i] = v;
  }
  if (blockIdx.x == 0) {
    for (long long i = (n4 << 2) + threadIdx.x; i < a.n; i += blockDim.x) {
      const float g = a.g[i] * gs;
      float p = a.p[i] * decay;
      const float m = a.beta1 * a.m[i] + (1.f - a.beta1) * g;
      const float v = a.beta2 * a.v[i] + (1.f - a.beta2) * g * g;
      p -= step * (m / (sqrtf(v) * rs2 + a.eps));
      a.p[i] = p; a.m[i] = m; a.v[i] = v;
    }
  }
}

// ------------------------------------------------------------------------------------------
// LoRA dropout (peft lora.Linear: lora_A(lora_dropout(x)), one nn.Dropout per wrapped module).  Counter-based masks:
// keep(m, c, target) = splitmix64(key + target * G + m * d + c) >> 40 >= p * 2^24 ; kept values are scaled by 1/(1-p).
// The backward kernel regenerates the same decisions instead of storing masks.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ bool drop_keep(uint64_t key, int target, long long idx, uint32_t thresh) {
  uint64_t x = key + static_cast<uint64_t>(target) * 0x9E3779B97F4A7C15ull + static_cast<uint64_t>(idx);
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  x ^= x >> 31;
  return static_cast<uint32_t>(x >> 40) >= thresh;
}
__global__ void lora_dropout_fwd_kernel(const bf16* __restrict__ h, bf16* __restrict__ hd, long long M, int d, int nt,
                                        uint32_t thresh, float inv_keep, uint64_t key) {
  const int vec = d >> 3;
  const long long total = M * vec;
  for (long long t = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; t < total;
       t += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long m = t / vec;
    const int c0 = static_cast<int>(t % vec) << 3;
    float f[8];
    bf16x8_to_f32(ldg_stream(reinterpret_cast<const uint4*>(h + m * d + c0)), f);
    for (int ti = 0; ti < nt; ++ti) {
      float o[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = drop_keep(key, ti, m * d + c0 + j, thresh) ? f[j] * inv_keep : 0.f;
      *reinterpret_cast<uint4*>(hd + m * static_cast<long long>(nt) * d + static_cast<long long>(ti) * d + c0) = f32_to_bf16x8(o);
    }
  }
}
__global__ void lora_dropout_bwd_kernel(bf16* __restrict__ dh, const bf16* __restrict__ g, long long M, int d, int nt,
                                        uint32_t thresh, float inv_keep, uint64_t key) {
  const int vec = d >> 3;
  const long long total = M * vec;
  for (long long t = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; t < total;
       t += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long m = t / vec;
    const int c0 = static_cast<int>(t % vec) << 3;
    float acc[8];
    uint4* dst = reinterpret_cast<uint4*>(dh + m * d + c0);
    bf16x8_to_f32(*dst, acc);
    for (int ti = 0; ti < nt; ++ti) {
      float gv[8];
      bf16x8_to_f32(ldg_stream(reinterpret_cast<const uint4*>(g + m * static_cast<long long>(nt) * d + static_cast<long long>(ti) * d + c0)), gv);
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (drop_keep(key, ti, m * d + c0 + j, thresh)) acc[j] += gv[j] * inv_keep;
    }
    *dst = f32_to_bf16x8(acc);
  }
}

__global__ void cast2d_kernel(const float* __restrict__ src, long long lds, bf16* __restrict__ dst, long long ldd, int rows,
                              int cols, float scale, int transpose) {
  const long long total = static_cast<long long>(rows) * cols;
  for (long long t = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; t < total;
       t += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int r = static_cast<int>(t / cols), c = static_cast<int>(t % cols);
    const float v = src[r * lds + c] * scale;
    if (transpose) dst[c * ldd + r] = __float2bfloat16_rn(v);
    else dst[r * ldd + c] = __float2bfloat16_rn(v);
  }
}

// ------------------------------------------------------------------------------------------
// QLoRA base weights (cmd/tuning/train.py:224-230: BitsAndBytesConfig(load_in_4bit, nf4, no double quant), bitsandbytes
// 0.41.3).  Block-wise: 64 consecutive elements share one fp32 absmax; codes are the 16 NF4 levels.  The trainer keeps the
// decoder weights PACKED (nf4_pack_kernel: 0.5625 B per weight) and expands a matrix into a bf16 scratch right before the
// GEMM that needs it (nf4_dequant_kernel); nf4_roundtrip_kernel (quantise + dequantise in place) is the same arithmetic in
// one kernel, kept for the per-kernel parity test.
// ------------------------------------------------------------------------------------------
__constant__ float kNF4[16] = {-1.0f, -0.6961928009986877f, -0.5250730514526367f, -0.39491748809814453f,
                               -0.28444138169288635f, -0.18477343022823334f, -0.09105003625154495f, 0.0f,
                               0.07958029955625534f, 0.16093020141124725f, 0.24611230194568634f, 0.33791524171829224f,
                               0.44070982933044434f, 0.5626170039176941f, 0.7229568362236023f, 1.0f};
__device__ __forceinline__ int nf4_code(float x) {  // nearest level (bitsandbytes dQuantizeNF4 decision tree = midpoints)
  int c = 0;
#pragma unroll
  for (int i = 0; i < 15; ++i) c += (x > 0.5f * (kNF4[i] + kNF4[i + 1])) ? 1 : 0;
  return c;
}
__global__ void nf4_roundtrip_kernel(bf16* __restrict__ w, long long nblocks) {
  for (long long b = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; b < nblocks;
       b += static_cast<long long>(gridDim.x) * blockDim.x) {
    uint4* p = reinterpret_cast<uint4*>(w + b * 64);
    float v[64];
    float amax = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      float f[8];
      bf16x8_to_f32(p[i], f);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        v[i * 8 + j] = f[j];
        amax = fmaxf(amax, fabsf(f[j]));
      }
    }
    const float inv = amax > 0.f ? 1.0f / amax : 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      float f[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) f[j] = kNF4[nf4_code(v[i * 8 + j] * inv)] * amax;
      p[i] = f32_to_bf16x8(f);
    }
  }
}
// Packed storage: one thread per 64-element block.  Byte layout as bitsandbytes kQuantizeBlockwise<..., NF4>: the first
// element of a pair sits in the high nibble.
__global__ void nf4_pack_kernel(const bf16* __restrict__ w, uint8_t* __restrict__ q, float* __restrict__ absmax, long long nblocks) {
  for (long long b = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; b < nblocks;
       b += static_cast<long long>(gridDim.x) * blockDim.x) {
    const uint4* p = reinterpret_cast<const uint4*>(w + b * 64);
    float v[64];
    float amax = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      float f[8];
      bf16x8_to_f32(p[i], f);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        v[i * 8 + j] = f[j];
        amax = fmaxf(amax, fabsf(f[j]));
      }
    }
    const float inv = amax > 0.f ? 1.0f / amax : 0.f;
    absmax[b] = amax;
    uint32_t words[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      uint32_t wd = 0;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const uint32_t byte = (static_cast<uint32_t>(nf4_code(v[i * 8 + 2 * j] * inv)) << 4) |
                              static_cast<uint32_t>(nf4_code(v[i * 8 + 2 * j + 1] * inv));
        wd |= byte << (8 * j);
      }
      words[i] = wd;
    }
    uint4* dst = reinterpret_cast<uint4*>(q + b * 32);
    dst[0] = make_uint4(words[0], words[1], words[2], words[3]);
    dst[1] = make_uint4(words[4], words[5], words[6], words[7]);
  }
}
// Expansion: one thread per 16 packed bytes (32 weights, half a block): 16 B + 4 B read, 64 B written; the 16 levels
// live in shared memory as bf16-rounded-on-store fp32 products (level * absmax, rounded to bf16 = what bitsandbytes'
// dequantize_4bit yields after the cast to the compute dtype).
__global__ void __launch_bounds__(256) nf4_dequant_kernel(const uint8_t* __restrict__ q, const float* __restrict__ absmax,
                                                          bf16* __restrict__ w, long long nhalf) {
  __shared__ float lv[16];
  if (threadIdx.x < 16) lv[threadIdx.x] = kNF4[threadIdx.x];
  __syncthreads();
  for (long long t = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; t < nhalf;
       t += static_cast<long long>(gridDim.x) * blockDim.x) {
    const uint4 pk = ldg_stream(reinterpret_cast<const uint4*>(q) + t);
    const float am = __ldg(absmax + (t >> 1));
    const uint32_t words[4] = {pk.x, pk.y, pk.z, pk.w};
    uint4* dst = reinterpret_cast<uint4*>(w + t * 32);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float f[8];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const uint32_t byte = (words[i] >> (8 * j)) & 0xFFu;
        f[2 * j] = lv[byte >> 4] * am;
        f[2 * j + 1] = lv[byte & 15u] * am;
      }
      dst[i] = f32_to_bf16x8(f);
    }
  }
}

// per-sequence loss sum / valid-token count (evaluation: lets the host form HF's eval batches of any size)
__global__ void row_loss_stats_kernel(const float* __restrict__ row_loss, const int32_t* __restrict__ labels, int S,
                                      float* __restrict__ row_sum, int32_t* __restrict__ row_valid, const int32_t* __restrict__ row_start) {
  __shared__ float sh[32];
  __shared__ int shc[32];
  const int b = blockIdx.x;
  // packed batch: sequence b owns rows row_start[b] .. row_start[b+1]); otherwise rows b*S .. (b+1)*S
  const size_t r0 = row_start ? static_cast<size_t>(row_start[b]) : static_cast<size_t>(b) * S;
  const int n = row_start ? row_start[b + 1] - row_start[b] : S;
  double acc = 0.0;
  int cnt = 0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    acc += static_cast<double>(row_loss[r0 + i]);
    cnt += labels[r0 + i] >= 0 ? 1 : 0;
  }
  float v = block_sum(static_cast<float>(acc), sh);
  for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) shc[threadIdx.x >> 5] = cnt;
  __syncthreads();
  if (threadIdx.x == 0) {
    int c = 0;
    for (int i = 0; i < (blockDim.x >> 5); ++i) c += shc[i];
    row_sum[b] = v;
    row_valid[b] = c;
  }
}

__device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}
__global__ void fill_normal_kernel(bf16* __restrict__ p, long long n, float std, uint64_t seed) {
  const long long n2 = (n + 1) >> 1;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n2;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const uint64_t h = splitmix64(seed * 0x100000001B3ull + static_cast<uint64_t>(i));
    const float u1 = (static_cast<float>(h >> 40) + 1.f) * (1.f / 16777217.f);
    const float u2 = static_cast<float>((h >> 8) & 0xFFFFFFull) * (1.f / 16777216.f);
    const float r = sqrtf(-2.f * logf(u1));
    float s, c;
    sincosf(6.283185307179586f * u2, &s, &c);
    p[2 * i] = __float2bfloat16_rn(r * c * std);
    if (2 * i + 1 < n) p[2 * i + 1] = __float2bfloat16_rn(r * s * std);
  }
}
__global__ void fill_const_kernel(bf16* __restrict__ p, long long n, float v) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x)
    p[i] = __float2bfloat16_rn(v);
}

// ------------------------------------------------------------------------------------------
// full-parameter SFT: RMSNorm weight gradient, embedding gradient, sharded AdamW on bf16 gradients
// ------------------------------------------------------------------------------------------
constexpr int NDW_ROWBLOCKS = 64;
// stage 1: block (cb, rb) sums columns [64*cb, +64) over its row range: 256 threads = 64 columns x 4 row lanes
__global__ void __launch_bounds__(256) rmsnorm_dw_stage1(const bf16* __restrict__ dy, const bf16* __restrict__ x,
                                                          const float* __restrict__ rstd, int M, int d, float* __restrict__ part) {
  __shared__ float sh[4][64];
  const int c = blockIdx.x * 64 + (threadIdx.x & 63), lane_r = threadIdx.x >> 6;
  const int rows_per = (M + NDW_ROWBLOCKS - 1) / NDW_ROWBLOCKS;
  const int r0 = blockIdx.y * rows_per, r1 = min(M, r0 + rows_per);
  float acc = 0.f;
  if (c < d)
    for (int m = r0 + lane_r; m < r1; m += 4)
      acc += __bfloat162float(dy[static_cast<size_t>(m) * d + c]) * __bfloat162float(x[static_cast<size_t>(m) * d + c]) * rstd[m];
  sh[lane_r][threadIdx.x & 63] = acc;
  __syncthreads();
  if (lane_r == 0 && c < d) part[static_cast<size_t>(blockIdx.y) * d + c] = (sh[0][threadIdx.x] + sh[1][threadIdx.x]) + (sh[2][threadIdx.x] + sh[3][threadIdx.x]);
}
__global__ void rmsnorm_dw_stage2(const float* __restrict__ part, int d, bf16* __restrict__ dw, int accumulate) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= d) return;
  float s = 0.f;
  for (int r = 0; r < NDW_ROWBLOCKS; ++r) s += part[static_cast<size_t>(r) * d + c];
  if (accumulate) s += __bfloat162float(dw[c]);
  dw[c] = __float2bfloat16_rn(s);
}
__global__ void embedding_bwd_kernel(const int32_t* __restrict__ ids, const bf16* __restrict__ dx, float* __restrict__ dE, int d, int vocab) {
  const int m = blockIdx.x;
  const int id = ids[m];
  if (id < 0 || id >= vocab) return;
  const bf16* src = dx + static_cast<size_t>(m) * d;
  float* dst = dE + static_cast<size_t>(id) * d;
  for (int c = threadIdx.x; c < d; c += blockDim.x) atomicAdd(dst + c, __bfloat162float(src[c]));
}
__global__ void add_f32_into_bf16_kernel(const float* __restrict__ src, bf16* __restrict__ dst, long long n, int accumulate) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n; i += static_cast<long long>(gridDim.x) * blockDim.x) {
    float v = src[i];
    if (accumulate) v += __bfloat162float(dst[i]);
    dst[i] = __float2bfloat16_rn(v);
  }
}
__global__ void cast_bf16_to_f32_kernel(const bf16* __restrict__ src, float* __restrict__ dst, long long n) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n; i += static_cast<long long>(gridDim.x) * blockDim.x)
    dst[i] = __bfloat162float(src[i]);
}
__global__ void sumsq_bf16_stage1(const bf16* __restrict__ g, long long n, float* __restrict__ scratch) {
  __shared__ float sh[32];
  float acc = 0.f;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n; i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float v = __bfloat162float(g[i]);
    acc += v * v;
  }
  acc = block_sum(acc, sh);
  if (threadIdx.x == 0) scratch[blockIdx.x] = acc;
}
__global__ void sumsq_acc_stage2(const float* __restrict__ scratch, int nblocks, float* __restrict__ out, int first) {
  if (threadIdx.x == 0) {
    double s = first ? 0.0 : static_cast<double>(*out);
    for (int i = 0; i < nblocks; ++i) s += static_cast<double>(scratch[i]);
    *out = static_cast<float>(s);
  }
}
// torch.optim.AdamW + clip_grad_norm_ as adamw_kernel, on fp32 master weights with bf16 gradients; the bf16 working copy of the
// weights is refreshed in the same pass (DeepSpeed bf16 optimizer semantics: fp32 master + state, bf16 model weights)
__global__ void adamw_shard_kernel(AdamWShardArgs a) {
  float gs = a.grad_scale;
  if (a.sumsq) {
    const float norm = sqrtf(*a.sumsq) * a.grad_scale;
    if (a.grad_norm_out && blockIdx.x == 0 && threadIdx.x == 0) *a.grad_norm_out = norm;
    if (a.max_grad_norm > 0.f) {
      const float coef = a.max_grad_norm / (norm + 1e-6f);
      if (coef < 1.f) gs *= coef;
    }
  }
  const float step = a.lr / a.bias1;
  const float rs2 = rsqrtf(a.bias2);
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < a.n; i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float g = __bfloat162float(a.g[i]) * gs;
    const float decay = (i >= a.nodecay_from) ? 1.f : 1.f - a.lr * a.weight_decay;
    float p = a.master[i] * decay;
    const float m = a.beta1 * a.m[i] + (1.f - a.beta1) * g;
    const float v = a.beta2 * a.v[i] + (1.f - a.beta2) * g * g;
    p -= step * (m / (sqrtf(v) * rs2 + a.eps));
    a.master[i] = p;
    a.m[i] = m;
    a.v[i] = v;
    a.w[i] = __float2bfloat16_rn(p);
  }
}

inline int grid_for(long long work, int block, int max_blocks = 148 * 16) {
  long long g = (work + block - 1) / block;
  if (g < 1) g = 1;
  if (g > max_blocks) g = max_blocks;
  return static_cast<int>(g);
}

}  // namespace

cudaError_t embedding_fwd(const int32_t* ids, const bf16* table, bf16* out, int M, int d, int vocab, cudaStream_t s) {
  if (d % 8) return cudaErrorInvalidValue;
  embedding_kernel<<<M, 256, 0, s>>>(ids, table, out, d, vocab);
  return cudaGetLastError();
}

cudaError_t rmsnorm_fwd(const bf16* x, const bf16* w, bf16* y, float* rstd, int M, int d, float eps, cudaStream_t s,
                        const int32_t* row_map) {
  if (d % 8 || d > 8192) return cudaErrorInvalidValue;
  const int nch = (d / 8 + RMS_THREADS - 1) / RMS_THREADS;
  if (nch <= 1) rmsnorm_fwd_kernel<1><<<M, RMS_THREADS, 0, s>>>(x, w, y, rstd, d, eps, row_map);
  else if (nch <= 2) rmsnorm_fwd_kernel<2><<<M, RMS_THREADS, 0, s>>>(x, w, y, rstd, d, eps, row_map);
  else if (nch <= 4) rmsnorm_fwd_kernel<4><<<M, RMS_THREADS, 0, s>>>(x, w, y, rstd, d, eps, row_map);
  else rmsnorm_fwd_kernel<8><<<M, RMS_THREADS, 0, s>>>(x, w, y, rstd, d, eps, row_map);
  return cudaGetLastError();
}

cudaError_t rmsnorm_bwd(const bf16* dy, const bf16* x, const bf16* w, const float* rstd, const bf16* dres, bf16* dx, int M,
                        int d, cudaStream_t s, const int32_t* row_map) {
  if (d % 8 || d > 8192) return cudaErrorInvalidValue;
  const int nch = (d / 8 + RMS_THREADS - 1) / RMS_THREADS;
  if (nch <= 1) rmsnorm_bwd_kernel<1><<<M, RMS_THREADS, 0, s>>>(dy, x, w, rstd, dres, dx, d, row_map);
  else if (nch <= 2) rmsnorm_bwd_kernel<2><<<M, RMS_THREADS, 0, s>>>(dy, x, w, rstd, dres, dx, d, row_map);
  else if (nch <= 4) rmsnorm_bwd_kernel<4><<<M, RMS_THREADS, 0, s>>>(dy, x, w, rstd, dres, dx, d, row_map);
  else rmsnorm_bwd_kernel<8><<<M, RMS_THREADS, 0, s>>>(dy, x, w, rstd, dres, dx, d, row_map);
  return cudaGetLastError();
}

cudaError_t rope_qk_inplace_table(bf16* qkv, const float2* cs, int B, int S, int n_rot_heads, int W, int D, int inverse,
                                  cudaStream_t s) {
  if (D % 16) return cudaErrorInvalidValue;
  const long long total = static_cast<long long>(B) * S * n_rot_heads * (D / 16);
  rope_kernel<<<grid_for(total, 256), 256, 0, s>>>(qkv, cs, S, n_rot_heads, W, D, inverse, total);
  return cudaGetLastError();
}

cudaError_t swiglu_fwd(const bf16* gu, bf16* act, int M, int F, int interleaved, cudaStream_t s) {
  if (F % 8 || (interleaved && F % 128)) return cudaErrorInvalidValue;
  swiglu_fwd_kernel<<<grid_for(static_cast<long long>(M) * (F / 8), 256), 256, 0, s>>>(gu, act, M, F, interleaved);
  return cudaGetLastError();
}
cudaError_t swiglu_bwd(const bf16* dact, const bf16* gu, bf16* dgu, int M, int F, int interleaved, cudaStream_t s) {
  if (F % 8 || (interleaved && F % 128)) return cudaErrorInvalidValue;
  swiglu_bwd_kernel<<<grid_for(static_cast<long long>(M) * (F / 8), 256), 256, 0, s>>>(dact, gu, dgu, M, F, interleaved);
  return cudaGetLastError();
}

cudaError_t shift_labels(const int32_t* labels, int32_t* shifted, int32_t* n_valid, int B, int S, cudaStream_t s,
                         int32_t* row_map, int32_t* valid_idx, const int32_t* pos) {
  if ((row_map == nullptr) != (valid_idx == nullptr)) return cudaErrorInvalidValue;
  shift_labels_kernel<<<1, 1024, 0, s>>>(labels, shifted, n_valid, B, S, row_map, valid_idx, pos);
  return cudaGetLastError();
}

cudaError_t cross_entropy_fwd_bwd(const float* logits, int64_t ldl, const int32_t* labels, const int32_t* n_valid,
                                  float* row_loss, bf16* dlogits, int64_t ldd, int M, int V, cudaStream_t s,
                                  const int32_t* valid_idx, int n_div) {
  if ((ldl & 3) || (ldd & 3)) return cudaErrorInvalidValue;
  ce_kernel<<<M, 256, 0, s>>>(logits, ldl, labels, n_valid, row_loss, dlogits, ldd, V, valid_idx, n_div);
  return cudaGetLastError();
}

cudaError_t loss_reduce(const float* row_loss, const int32_t* n_valid, float* loss, int M, cudaStream_t s, int n_div, int accumulate) {
  loss_reduce_kernel<<<1, 1024, 0, s>>>(row_loss, n_valid, loss, M, n_div, accumulate);
  return cudaGetLastError();
}

__global__ void gather_rows_kernel(const int32_t* __restrict__ ids, const int32_t* __restrict__ labels, const int32_t* __restrict__ lens,
                                   int S_src, RowList rows, int S_dst, int32_t* __restrict__ ids_out, int32_t* __restrict__ labels_out,
                                   int32_t* __restrict__ lens_out) {
  const int i = blockIdx.y, src = rows.rows[i];
  for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < S_dst; c += gridDim.x * blockDim.x) {
    ids_out[static_cast<long long>(i) * S_dst + c] = ids[static_cast<long long>(src) * S_src + c];
    labels_out[static_cast<long long>(i) * S_dst + c] = labels[static_cast<long long>(src) * S_src + c];
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) lens_out[i] = lens[src];
}

__global__ void pack_rows_kernel(const int32_t* __restrict__ ids, const int32_t* __restrict__ labels, int S_src, RowStarts rs,
                                 int32_t* __restrict__ ids_out, int32_t* __restrict__ labels_out, int32_t* __restrict__ pos_out,
                                 int32_t* __restrict__ start_out) {
  const int b = blockIdx.y, r0 = rs.start[b], cap = rs.start[b + 1] - r0;
  for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < cap; c += gridDim.x * blockDim.x) {
    ids_out[r0 + c] = ids[static_cast<long long>(b) * S_src + c];
    labels_out[r0 + c] = labels[static_cast<long long>(b) * S_src + c];
    pos_out[r0 + c] = c;
  }
  if (blockIdx.x == 0 && blockIdx.y == 0)
    for (int i = threadIdx.x; i <= rs.n; i += blockDim.x) start_out[i] = rs.start[i];
}

cudaError_t pack_rows(const int32_t* ids, const int32_t* labels, int S_src, RowStarts rs, int32_t* ids_out, int32_t* labels_out,
                      int32_t* pos_out, int32_t* start_out, cudaStream_t s) {
  if (rs.n <= 0 || rs.n > 64 || S_src <= 0) return cudaErrorInvalidValue;
  int max_cap = 0;
  for (int b = 0; b < rs.n; ++b) {
    const int cap = rs.start[b + 1] - rs.start[b];
    if (cap <= 0 || cap > S_src || (cap & 127) || (rs.start[b] & 127)) return cudaErrorInvalidValue;
    max_cap = cap > max_cap ? cap : max_cap;
  }
  pack_rows_kernel<<<dim3((max_cap + 255) / 256, rs.n), 256, 0, s>>>(ids, labels, S_src, rs, ids_out, labels_out, pos_out, start_out);
  return cudaGetLastError();
}

cudaError_t gather_rows(const int32_t* ids, const int32_t* labels, const int32_t* lens, int S_src, RowList rows, int S_dst,
                        int32_t* ids_out, int32_t* labels_out, int32_t* lens_out, cudaStream_t s) {
  if (rows.n <= 0 || rows.n > 64 || S_dst > S_src || S_dst <= 0) return cudaErrorInvalidValue;
  gather_rows_kernel<<<dim3((S_dst + 255) / 256, rows.n), 256, 0, s>>>(ids, labels, lens, S_src, rows, S_dst, ids_out, labels_out, lens_out);
  return cudaGetLastError();
}

cudaError_t sum_partials(const float* partial, float* out, int64_t n, int splits, cudaStream_t s) {
  sum_partials_kernel<<<grid_for(n, 256), 256, 0, s>>>(partial, out, n, splits);
  return cudaGetLastError();
}

cudaError_t sumsq(const float* g, int64_t n, float* scratch, float* out, cudaStream_t s) {
  sumsq_stage1<<<SUMSQ_BLOCKS, 256, 0, s>>>(g, n, scratch);
  sumsq_stage2<<<1, 32, 0, s>>>(scratch, SUMSQ_BLOCKS, out);
  return cudaGetLastError();
}

cudaError_t adamw_step(const AdamWArgs& a, cudaStream_t s) {
  if ((reinterpret_cast<uintptr_t>(a.p) | reinterpret_cast<uintptr_t>(a.g) | reinterpret_cast<uintptr_t>(a.m) |
       reinterpret_cast<uintptr_t>(a.v)) & 15)
    return cudaErrorInvalidValue;
  adamw_kernel<<<grid_for(a.n / 4 + 1, 256, 148 * 8), 256, 0, s>>>(a);
  return cudaGetLastError();
}

cudaError_t nf4_roundtrip_bf16(bf16* w, int64_t n, cudaStream_t s) {
  if (n % 64) return cudaErrorInvalidValue;
  nf4_roundtrip_kernel<<<grid_for(n / 64, 128), 128, 0, s>>>(w, n / 64);
  return cudaGetLastError();
}
cudaError_t nf4_quantize_pack(const bf16* w, uint8_t* q, float* absmax, int64_t n, cudaStream_t s) {
  if (n % 64) return cudaErrorInvalidValue;
  nf4_pack_kernel<<<grid_for(n / 64, 128), 128, 0, s>>>(w, q, absmax, n / 64);
  return cudaGetLastError();
}
cudaError_t nf4_dequant_bf16(const uint8_t* q, const float* absmax, bf16* w, int64_t n, cudaStream_t s) {
  if (n % 64) return cudaErrorInvalidValue;
  nf4_dequant_kernel<<<grid_for(n / 32, 256), 256, 0, s>>>(q, absmax, w, n / 32);
  return cudaGetLastError();
}
cudaError_t row_loss_stats(const float* row_loss, const int32_t* shifted_labels, int B, int S, float* row_sum, int32_t* row_valid,
                           cudaStream_t s, const int32_t* row_start) {
  row_loss_stats_kernel<<<B, 256, 0, s>>>(row_loss, shifted_labels, S, row_sum, row_valid, row_start);
  return cudaGetLastError();
}

static uint32_t drop_thresh(float p) {
  double v = static_cast<double>(p) * 16777216.0;
  if (v < 0) v = 0;
  if (v > 16777215.0) v = 16777215.0;
  return static_cast<uint32_t>(v);
}
cudaError_t lora_dropout_fwd(const bf16* h, bf16* hd, int M, int d, int nt, float p, uint64_t key, cudaStream_t s) {
  if (d % 8) return cudaErrorInvalidValue;
  lora_dropout_fwd_kernel<<<grid_for(static_cast<long long>(M) * (d / 8), 256), 256, 0, s>>>(h, hd, M, d, nt, drop_thresh(p),
                                                                                          1.0f / (1.0f - p), key);
  return cudaGetLastError();
}
cudaError_t lora_dropout_bwd_add(bf16* dh, const bf16* g, int M, int d, int nt, float p, uint64_t key, cudaStream_t s) {
  if (d % 8) return cudaErrorInvalidValue;
  lora_dropout_bwd_kernel<<<grid_for(static_cast<long long>(M) * (d / 8), 256), 256, 0, s>>>(dh, g, M, d, nt, drop_thresh(p),
                                                                                          1.0f / (1.0f - p), key);
  return cudaGetLastError();
}
cudaError_t swiglu_bwd_lora_dropout(const bf16* dact, const bf16* g, const bf16* gu, bf16* dgu, int M, int F, int interleaved, float p,
                                    uint64_t key, cudaStream_t s) {
  if (!g || F % 8 || (interleaved && F % 128)) return cudaErrorInvalidValue;
  swiglu_bwd_kernel<<<grid_for(static_cast<long long>(M) * (F / 8), 256), 256, 0, s>>>(dact, gu, dgu, M, F, interleaved, g, drop_thresh(p),
                                                                                    1.0f / (1.0f - p), key);
  return cudaGetLastError();
}

cudaError_t cast_f32_to_bf16_2d(const float* src, int64_t lds, bf16* dst, int64_t ldd, int rows, int cols, float scale,
                                int transpose, cudaStream_t s) {
  cast2d_kernel<<<grid_for(static_cast<long long>(rows) * cols, 256), 256, 0, s>>>(src, lds, dst, ldd, rows, cols, scale,
                                                                                  transpose);
  return cudaGetLastError();
}

cudaError_t rmsnorm_dw(const bf16* dy, const bf16* x, const float* rstd, int M, int d, float* scratch, bf16* dw, int accumulate,
                       cudaStream_t s) {
  rmsnorm_dw_stage1<<<dim3((d + 63) / 64, NDW_ROWBLOCKS), 256, 0, s>>>(dy, x, rstd, M, d, scratch);
  rmsnorm_dw_stage2<<<(d + 255) / 256, 256, 0, s>>>(scratch, d, dw, accumulate);
  return cudaGetLastError();
}
cudaError_t embedding_bwd(const int32_t* ids, const bf16* dx, float* dE32, int M, int d, int vocab, cudaStream_t s) {
  embedding_bwd_kernel<<<M, 256, 0, s>>>(ids, dx, dE32, d, vocab);
  return cudaGetLastError();
}
cudaError_t add_f32_into_bf16(const float* src, bf16* dst, int64_t n, int accumulate, cudaStream_t s) {
  add_f32_into_bf16_kernel<<<grid_for(n, 256), 256, 0, s>>>(src, dst, n, accumulate);
  return cudaGetLastError();
}
cudaError_t cast_bf16_to_f32(const bf16* src, float* dst, int64_t n, cudaStream_t s) {
  cast_bf16_to_f32_kernel<<<grid_for(n, 256), 256, 0, s>>>(src, dst, n);
  return cudaGetLastError();
}
cudaError_t sumsq_bf16_acc(const bf16* g, int64_t n, float* scratch, float* out, int first, cudaStream_t s) {
  sumsq_bf16_stage1<<<SUMSQ_BLOCKS, 256, 0, s>>>(g, n, scratch);
  sumsq_acc_stage2<<<1, 32, 0, s>>>(scratch, SUMSQ_BLOCKS, out, first);
  return cudaGetLastError();
}
cudaError_t adamw_shard_step(const AdamWShardArgs& a, cudaStream_t s) {
  if (a.n <= 0) return cudaSuccess;
  adamw_shard_kernel<<<grid_for(a.n, 256, 148 * 8), 256, 0, s>>>(a);
  return cudaGetLastError();
}

cudaError_t fill_normal_bf16(bf16* p, int64_t n, float std, uint64_t seed, cudaStream_t s) {
  fill_normal_kernel<<<grid_for((n + 1) / 2, 256), 256, 0, s>>>(p, n, std, seed);
  return cudaGetLastError();
}
cudaError_t fill_const_bf16(bf16* p, int64_t n, float v, cudaStream_t s) {
  fill_const_kernel<<<grid_for(n, 256), 256, 0, s>>>(p, n, v);
  return cudaGetLastError();
}

}  // namespace dtx
