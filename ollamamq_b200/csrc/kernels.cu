// Non-GEMM kernels of the transformer forward pass, hand-written for sm_100a.
//
// These are the HBM/latency-bound pieces around the tcgen05 GEMMs (gemm.cuh).  Together they stand in for
// the arithmetic the reference delegates to a remote Ollama server (/root/reference/src/dispatcher.rs:287-290).
// All of them call griddepcontrol.wait first and griddepcontrol.launch_dependents right after, so a whole
// decode step can be chained with programmatic dependent launch without ever reading stale data.
//
//   embed            gather rows of the embedding table into the fp32 residual stream
//   add_rmsnorm      residual += sum(split-K partial planes); x = RMSNorm(residual) * gamma   (fused)
//   rope_kv          sum QKV partials (+bias), rotate q/k (rotate-half RoPE), write K/V into the paged cache
//   paged_attn       FlashAttention-2 style online softmax over the paged KV cache; GQA group fused into
//                    the M dimension (row = token x head-in-group), 128-bit cp.async loads, mma.sync QK^T/PV,
//                    quad warp-shuffle softmax; decode variant is split-KV with one warp per CTA
//   attn_combine     merge the split-KV partials
//   argmax           greedy sampler + device-side advance of (cur_token, pos) so decode steps chain on the GPU
#include "kernels.cuh"
#include <cfloat>
#include <type_traits>
#include <cstdlib>
#include <algorithm>
#include "ptx.cuh"

namespace mq {

// ------------------------------------------------------------------------------------------------
// launch helper
// ------------------------------------------------------------------------------------------------
template <typename... KArgs, typename... Args>
static void launch_k(const LaunchCfg& lc, void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = lc.stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = lc.pdl ? 1 : 0;
  cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}

// ------------------------------------------------------------------------------------------------
// embedding gather
// ------------------------------------------------------------------------------------------------
// gamma != nullptr (decode chain): also emit xg = bf16(h * gamma) - the activation operand of the first QKV GEMM - and
// ssq[t] = sum h^2, the single "partial" of the first RMSNorm fold (RstdIn with parts = 1; see gemm.cuh).
__global__ void __launch_bounds__(128) embed_kernel(const int* __restrict__ token_ids, const __nv_bfloat16* __restrict__ embed,
                                                    float* __restrict__ h, int H, const __nv_bfloat16* __restrict__ gamma,
                                                    __nv_bfloat16* __restrict__ xg, float* __restrict__ ssq) {
  pdl_launch_dependents();  // let the next kernel start its prologue (weight prefetch) right away
  pdl_wait();
  const int t = blockIdx.x;
  const int tok = token_ids[t];
  const uint4* src = reinterpret_cast<const uint4*>(embed + (size_t)tok * H);
  float4* dst = reinterpret_cast<float4*>(h + (size_t)t * H);
  float ss = 0.f;
  for (int i = threadIdx.x; i < H / 8; i += blockDim.x) {
    const uint4 v = src[i];
    const float e[8] = {bf16_lo(v.x), bf16_hi(v.x), bf16_lo(v.y), bf16_hi(v.y), bf16_lo(v.z), bf16_hi(v.z), bf16_lo(v.w), bf16_hi(v.w)};
    dst[2 * i] = make_float4(e[0], e[1], e[2], e[3]);
    dst[2 * i + 1] = make_float4(e[4], e[5], e[6], e[7]);
    if (gamma) {
      const uint4 g = reinterpret_cast<const uint4*>(gamma)[i];
      uint4 o;
      o.x = pack_bf16(e[0] * bf16_lo(g.x), e[1] * bf16_hi(g.x));
      o.y = pack_bf16(e[2] * bf16_lo(g.y), e[3] * bf16_hi(g.y));
      o.z = pack_bf16(e[4] * bf16_lo(g.z), e[5] * bf16_hi(g.z));
      o.w = pack_bf16(e[6] * bf16_lo(g.w), e[7] * bf16_hi(g.w));
      reinterpret_cast<uint4*>(xg + (size_t)t * H)[i] = o;
#pragma unroll
      for (int k = 0; k < 8; ++k) ss += e[k] * e[k];
    }
  }
  if (gamma) {
    __shared__ float red[4];
    ss = warp_sum(ss);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ss;
    __syncthreads();
    if (threadIdx.x == 0) ssq[t] = (red[0] + red[1]) + (red[2] + red[3]);
  }
}
void launch_embed(const LaunchCfg& lc, const int* token_ids, const __nv_bfloat16* embed, float* h, int T, int H,
                  const __nv_bfloat16* gamma, __nv_bfloat16* xg, float* ssq) {
  launch_k(lc, embed_kernel, dim3(T), dim3(128), 0, token_ids, embed, h, H, gamma, xg, ssq);
}

// ------------------------------------------------------------------------------------------------
// fused residual-add + RMSNorm.  One CTA per row, blockDim = H/16, every thread keeps 16 values in registers.
// ------------------------------------------------------------------------------------------------
// NP = number of split-K planes, a compile-time constant so that EVERY load of the thread (residual, planes,
// gamma) is issued before the first use: with a run-time plane loop the kernel was a chain of ~20 dependent L2
// round trips (r01 timeline: 4.7 - 6 us busy per launch, three launches per layer).
template <bool F32, int NP>
__global__ void add_rmsnorm_kernel(float* __restrict__ h, const void* __restrict__ partial, long long plane_stride,
                                   const __nv_bfloat16* __restrict__ gamma, __nv_bfloat16* __restrict__ x,
                                   const int* __restrict__ row_idx, int H, float eps, Trace tr) {
  pdl_launch_dependents();  // let the next kernel start its prologue (weight prefetch) right away
  if (threadIdx.x == 0) trace_begin(tr);
  const int row = blockIdx.x;
  const int nthr = blockDim.x;
  uint2 gm[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) gm[j] = reinterpret_cast<const uint2*>(gamma)[threadIdx.x + j * nthr];  // weights: no dependency
  pdl_wait();
  if (threadIdx.x == 0) trace_waited(tr);
  const int src = row_idx ? row_idx[row] : row;
  const float4* h4 = reinterpret_cast<const float4*>(h + (size_t)src * H);
  float4 v[4];
  float4 b[4][F32 ? (NP > 0 ? NP : 1) : 1];
  uint2 bb[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) v[j] = h4[threadIdx.x + j * nthr];
  if constexpr (F32) {
    const float* pp = reinterpret_cast<const float*>(partial) + (size_t)src * H;
#pragma unroll
    for (int s = 0; s < NP; ++s)
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j][s] = reinterpret_cast<const float4*>(pp + s * plane_stride)[threadIdx.x + j * nthr];
  } else if constexpr (NP > 0) {
#pragma unroll
    for (int j = 0; j < 4; ++j)
      bb[j] = reinterpret_cast<const uint2*>(reinterpret_cast<const __nv_bfloat16*>(partial) + (size_t)src * H)[threadIdx.x + j * nthr];
  }
  float ss = 0.f;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    float4 a = v[j];
    if constexpr (F32) {
#pragma unroll
      for (int s = 0; s < NP; ++s) { a.x += b[j][s].x; a.y += b[j][s].y; a.z += b[j][s].z; a.w += b[j][s].w; }
    } else if constexpr (NP > 0) {
      a.x += bf16_lo(bb[j].x); a.y += bf16_hi(bb[j].x); a.z += bf16_lo(bb[j].y); a.w += bf16_hi(bb[j].y);
    }
    v[j] = a;
    ss += a.x * a.x + a.y * a.y + a.z * a.z + a.w * a.w;
    if (!row_idx) reinterpret_cast<float4*>(h + (size_t)src * H)[threadIdx.x + j * nthr] = a;
  }
  __shared__ float red[32];
  ss = warp_sum(ss);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ss;
  __syncthreads();
  float tot = 0.f;
  for (int w = 0; w < (nthr + 31) / 32; ++w) tot += red[w];
  const float rstd = rsqrtf(tot / (float)H + eps);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    uint2 o;
    o.x = pack_bf16(v[j].x * rstd * bf16_lo(gm[j].x), v[j].y * rstd * bf16_hi(gm[j].x));
    o.y = pack_bf16(v[j].z * rstd * bf16_lo(gm[j].y), v[j].w * rstd * bf16_hi(gm[j].y));
    reinterpret_cast<uint2*>(x + (size_t)row * H)[threadIdx.x + j * nthr] = o;
  }
  if (threadIdx.x == 0) trace_end(tr);
}
void launch_add_rmsnorm(const LaunchCfg& lc, float* h, const void* partial, bool partial_is_f32, int n_planes,
                        long long plane_stride, const __nv_bfloat16* gamma, __nv_bfloat16* x, const int* row_idx,
                        int rows, int H, float eps, Trace tr) {
  const int thr = H / 16;  // H % 512 == 0 is checked at model load
  // (r01 A/B: a 4-CTA cluster per row with a DSMEM exchange of the partial sums was SLOWER at decode width -
  //  4.1 / 5.0 us busy against 3.3 / 4.3 us - the cluster barrier costs more than the narrower loads save.)
  auto go = [&](auto f32tag, auto nptag) {
    launch_k(lc, add_rmsnorm_kernel<decltype(f32tag)::value, decltype(nptag)::value>, dim3(rows), dim3(thr), 0, h,
             partial, plane_stride, gamma, x, row_idx, H, eps, tr);
  };
  using T = std::true_type;
  using F = std::false_type;
  if (!partial_is_f32) {
    if (n_planes > 0) go(F{}, std::integral_constant<int, 1>{}); else go(F{}, std::integral_constant<int, 0>{});
    return;
  }
  switch (n_planes) {  // 0 .. kMaxSplitPlanes
    case 0: go(T{}, std::integral_constant<int, 0>{}); break;
    case 1: go(T{}, std::integral_constant<int, 1>{}); break;
    case 2: go(T{}, std::integral_constant<int, 2>{}); break;
    case 3: go(T{}, std::integral_constant<int, 3>{}); break;
    case 4: go(T{}, std::integral_constant<int, 4>{}); break;
    case 5: go(T{}, std::integral_constant<int, 5>{}); break;
    case 6: go(T{}, std::integral_constant<int, 6>{}); break;
    case 7: go(T{}, std::integral_constant<int, 7>{}); break;
    default: go(T{}, std::integral_constant<int, 8>{}); break;
  }
}

// ------------------------------------------------------------------------------------------------
// RoPE + paged KV write (v1: one CTA per token = 64 CTAs at decode, 30 us of pure load latency per layer;
// v2: (token, 4 heads) CTAs with 2-byte accesses; v3 below: 8/16-byte accesses).
// ------------------------------------------------------------------------------------------------
// 4 consecutive qkv values of token t starting at columns col and col + half: sum of the NP split-K planes
// (+ bias).  NP is a compile-time constant so that all 2 * NP loads are in flight together.
template <bool F32, int NP>
__device__ __forceinline__ void qkv_pair4(const RopeKvParams& p, int t, int col, int half, int qkv_dim, float4& va,
                                          float4& vb) {
  if constexpr (F32) {
    const float* pp = reinterpret_cast<const float*>(p.qkv) + (size_t)t * qkv_dim + col;
    float4 a[NP], b[NP];
#pragma unroll
    for (int s = 0; s < NP; ++s) {
      a[s] = *reinterpret_cast<const float4*>(pp + s * p.plane_stride);
      b[s] = *reinterpret_cast<const float4*>(pp + s * p.plane_stride + half);
    }
    va = a[0]; vb = b[0];
#pragma unroll
    for (int s = 1; s < NP; ++s) {
      va.x += a[s].x; va.y += a[s].y; va.z += a[s].z; va.w += a[s].w;
      vb.x += b[s].x; vb.y += b[s].y; vb.z += b[s].z; vb.w += b[s].w;
    }
  } else {
    const __nv_bfloat16* pp = reinterpret_cast<const __nv_bfloat16*>(p.qkv) + (size_t)t * qkv_dim + col;
    const uint2 a = *reinterpret_cast<const uint2*>(pp);
    const uint2 b = *reinterpret_cast<const uint2*>(pp + half);
    va = make_float4(bf16_lo(a.x), bf16_hi(a.x), bf16_lo(a.y), bf16_hi(a.y));
    vb = make_float4(bf16_lo(b.x), bf16_hi(b.x), bf16_lo(b.y), bf16_hi(b.y));
  }
}
__device__ __forceinline__ void add_bias4(float4& v, const __nv_bfloat16* bias) {
  const uint2 b = *reinterpret_cast<const uint2*>(bias);
  v.x += bf16_lo(b.x); v.y += bf16_hi(b.x); v.z += bf16_lo(b.y); v.w += bf16_hi(b.y);
}
__device__ __forceinline__ uint2 pack4_bf16(float a, float b, float c, float d) {
  uint2 o;
  o.x = pack_bf16(a, b);
  o.y = pack_bf16(c, d);
  return o;
}

// One CTA (256 threads) per (token, 16 heads); a thread owns 4 consecutive rotation pairs (i..i+3, i+64..i+67)
// of one head, so every access is 8 B (bf16) or 16 B (fp32 planes).
// head_dim is a compile-time constant of the rope / attention kernels; 128 (Llama-3, Qwen2.5), 96 (Phi-3) and 64 are built
template <typename F>
static void dispatch_head_dim(int d, F&& f) {
  switch (d) {
    case 128: f(std::integral_constant<int, 128>{}); break;
    case 96: f(std::integral_constant<int, 96>{}); break;
    case 64: f(std::integral_constant<int, 64>{}); break;
    case 32: f(std::integral_constant<int, 32>{}); break;  // BERT-small heads (encoder path)
    default: break;  // rejected at mq_worker_open / by the debug ABI before any launch
  }
}

template <bool F32, int D, int NP>
__global__ void __launch_bounds__(256) rope_kv_kernel(const RopeKvParams p) {
  pdl_launch_dependents();  // let the next kernel start its prologue (weight prefetch) right away
  if (threadIdx.x == 0) trace_begin(p.tr);
  constexpr int HALF = D / 2;  // 16 threads per head x 4 pairs cover HALF <= 64 (threads beyond HALF idle: d = 96, 64)
  const int t = blockIdx.x;
  const int hd = blockIdx.y * 16 + (threadIdx.x >> 4);  // q heads, then k heads, then v heads
  const int n_heads = p.n_q + 2 * p.n_kv;
  const bool live = hd < n_heads && (int)(threadIdx.x & 15) * 4 < HALF;
  const int qkv_dim = n_heads * D;
  const int i = (threadIdx.x & 15) * 4;  // first of 4 pair indices
  const int col = hd * D + i;
  // Everything that does not depend on the QKV GEMM happens BEFORE the dependency wait: positions, the block-table
  // walk, the bias and the four sin/cos pairs (positions / slot tables are written by the host or by the previous
  // step's sampler, never by a kernel of this pass).
  float sn[4] = {0.f, 0.f, 0.f, 0.f}, cs[4] = {1.f, 1.f, 1.f, 1.f};
  float4 bias_a = make_float4(0.f, 0.f, 0.f, 0.f), bias_b = bias_a;
  __nv_bfloat16* dst = nullptr;
  if (live) {
    const int pos = p.pos[t];
    if (hd < p.n_q + p.n_kv) {
      if (p.rope_table) {  // (cos, sin) per (position, pair), built once with the sincosf below
        const float4 t0 = *reinterpret_cast<const float4*>(p.rope_table + (size_t)pos * HALF + i);
        const float4 t1 = *reinterpret_cast<const float4*>(p.rope_table + (size_t)pos * HALF + i + 2);
        cs[0] = t0.x; sn[0] = t0.y; cs[1] = t0.z; sn[1] = t0.w; cs[2] = t1.x; sn[2] = t1.y; cs[3] = t1.z; sn[3] = t1.w;
      } else {
        const float4 fr = *reinterpret_cast<const float4*>(p.inv_freq + i);
        sincosf((float)pos * fr.x, &sn[0], &cs[0]);
        sincosf((float)pos * fr.y, &sn[1], &cs[1]);
        sincosf((float)pos * fr.z, &sn[2], &cs[2]);
        sincosf((float)pos * fr.w, &sn[3], &cs[3]);
      }
    }
    if (p.bias) { add_bias4(bias_a, p.bias + col); add_bias4(bias_b, p.bias + col + HALF); }
    if (hd < p.n_q) {
      dst = p.q_out + (size_t)t * p.n_q * D + hd * D;
    } else {
      const int slot = p.slot_of_tok[t];
      const int page = p.block_table[(size_t)slot * p.max_pages + pos / kPageSize];
      const bool is_k = hd < p.n_q + p.n_kv;
      const int kvh = is_k ? hd - p.n_q : hd - p.n_q - p.n_kv;
      dst = (is_k ? p.k_cache : p.v_cache) + (((size_t)page * p.n_kv + kvh) * kPageSize + pos % kPageSize) * D;
    }
  }
  pdl_wait();
  if (threadIdx.x == 0) trace_waited(p.tr);
  if (!live) return;
  float4 a, b;
  qkv_pair4<F32, NP>(p, t, col, HALF, qkv_dim, a, b);
  a.x += bias_a.x; a.y += bias_a.y; a.z += bias_a.z; a.w += bias_a.w;
  b.x += bias_b.x; b.y += bias_b.y; b.z += bias_b.z; b.w += bias_b.w;
  // v heads keep sin = 0, cos = 1: the rotation degenerates to a copy
  const uint2 lo = pack4_bf16(a.x * cs[0] - b.x * sn[0], a.y * cs[1] - b.y * sn[1], a.z * cs[2] - b.z * sn[2],
                              a.w * cs[3] - b.w * sn[3]);
  const uint2 hi = pack4_bf16(b.x * cs[0] + a.x * sn[0], b.y * cs[1] + a.y * sn[1], b.z * cs[2] + a.z * sn[2],
                              b.w * cs[3] + a.w * sn[3]);
  *reinterpret_cast<uint2*>(dst + i) = lo;
  *reinterpret_cast<uint2*>(dst + i + HALF) = hi;
  if (threadIdx.x == 0) trace_end(p.tr);  // thread 0 always owns a live (head, pair) of its CTA
}
// table[pos][i] = (cos, sin)(pos * inv_freq[i]) - the very values rope_kv_kernel computes on the fly without a table
__global__ void rope_table_kernel(float2* __restrict__ table, const float* __restrict__ inv_freq, int n_pos, int half) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n_pos * half) return;
  float s, c;
  sincosf((float)(idx / half) * inv_freq[idx % half], &s, &c);
  table[idx] = make_float2(c, s);
}
void launch_rope_table(cudaStream_t st, float2* table, const float* inv_freq, int n_pos, int half) {
  const int n = n_pos * half;
  rope_table_kernel<<<(n + 255) / 256, 256, 0, st>>>(table, inv_freq, n_pos, half);
}
void launch_rope_kv(const LaunchCfg& lc, const RopeKvParams& p) {
  const dim3 grid(p.T, (p.n_q + 2 * p.n_kv + 15) / 16);
  auto go = [&](auto dtag) {
    constexpr int D = decltype(dtag)::value;
    if (!p.qkv_is_f32) { launch_k(lc, rope_kv_kernel<false, D, 1>, grid, dim3(256), 0, p); return; }
    switch (p.n_planes) {  // 1 .. kMaxSplitPlanes
      case 1: launch_k(lc, rope_kv_kernel<true, D, 1>, grid, dim3(256), 0, p); break;
      case 2: launch_k(lc, rope_kv_kernel<true, D, 2>, grid, dim3(256), 0, p); break;
      case 3: launch_k(lc, rope_kv_kernel<true, D, 3>, grid, dim3(256), 0, p); break;
      case 4: launch_k(lc, rope_kv_kernel<true, D, 4>, grid, dim3(256), 0, p); break;
      case 5: launch_k(lc, rope_kv_kernel<true, D, 5>, grid, dim3(256), 0, p); break;
      case 6: launch_k(lc, rope_kv_kernel<true, D, 6>, grid, dim3(256), 0, p); break;
      case 7: launch_k(lc, rope_kv_kernel<true, D, 7>, grid, dim3(256), 0, p); break;
      default: launch_k(lc, rope_kv_kernel<true, D, 8>, grid, dim3(256), 0, p); break;
    }
  };
  dispatch_head_dim(p.head_dim, go);
}

// ------------------------------------------------------------------------------------------------
// paged flash attention (prefill + decode)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc, int src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(src_bytes)
               : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3)
               : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3)
               : "r"(addr));
}
__device__ __forceinline__ void mma_bf16_16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// Rows of Q/K/V tiles are 256 B (128 bf16) = 16 chunks of 16 B; chunk index is XOR-swizzled with (row & 7)
// so ldmatrix (8 rows x 16 B at one logical chunk column) is bank-conflict free.  head_dim 96 / 64 keep the
// 256-byte pitch (chunks >= head_dim / 8 are never written nor read), so one swizzle serves all three.
constexpr int kTilePitch = 128;  // elements per smem tile row, whatever the head_dim
__device__ __forceinline__ uint32_t tile_off(int row, int chunk) { return (uint32_t)(row * 16 + (chunk ^ (row & 7))) * 16u; }

// Prefill / encoder attention: one CTA per (tile of <= NW*16 query rows, kv head).
template <int NW, int TN, int STAGES, int D>
__global__ void __launch_bounds__(NW * 32) paged_attn_kernel(const AttnParams p) {
  constexpr int P = kTilePitch;  // smem row pitch in elements (256 B for every head_dim: keeps the XOR swizzle valid)
  constexpr int CH = D / 8;      // 16-byte chunks per row that hold data
  constexpr int R = NW * 16;
  constexpr int NT = TN / 8;  // score n-tiles per kv tile
  static_assert(TN % 16 == 0 && STAGES >= 2, "tile shape");
  extern __shared__ __align__(128) uint8_t smem[];
  uint8_t* Qs = smem;
  uint8_t* Ks = Qs + R * P * 2;
  uint8_t* Vs = Ks + STAGES * TN * P * 2;

  pdl_launch_dependents();  // let the next kernel start its prologue (weight prefetch) right away
  pdl_wait();

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, c = lane & 3;
  const int kvh = blockIdx.y;
  const int G = p.n_q / p.n_kv;
  const int4 tile = p.tiles[blockIdx.x];
  const int tok0 = tile.x, ntok = tile.y, slot = tile.z, pos0 = tile.w;
  const int n_rows = ntok * G;
  const int kv_begin = 0, kv_end = p.bidirectional ? p.seq_len[slot] : pos0 + ntok;  // encoder rows see the whole sequence
  const int* btab = p.block_table + (size_t)slot * p.max_pages;
  const int seq0 = p.seq_start ? p.seq_start[slot] : 0;
  const int n_tiles = kv_begin < kv_end ? (kv_end - kv_begin + TN - 1) / TN : 0;

  float o[D / 8][4];
#pragma unroll
  for (int i = 0; i < D / 8; ++i) o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f;
  float m_run[2] = {-INFINITY, -INFINITY};
  float l_run[2] = {0.f, 0.f};
  const int row_a = warp * 16 + g, row_b = row_a + 8;

  if (n_tiles > 0) {
    // ---- Q tile -> smem (zero-filled beyond the valid rows)
    for (int i = tid; i < R * CH; i += NW * 32) {
      const int r = i / CH, ch = i % CH;
      const bool ok = r < n_rows;
      const int rr = ok ? r : 0;
      const int tok = tok0 + rr / G, head = kvh * G + rr % G;
      const size_t qrow = p.seq_start ? (size_t)tok * p.row_stride : (size_t)tok * p.n_q * D;
      cp_async16(Qs + tile_off(r, ch), p.q + qrow + head * D + ch * 8, ok ? 16 : 0);
    }
    auto load_kv = [&](int stage, int t0) {
      uint8_t* kst = Ks + stage * TN * P * 2;
      uint8_t* vst = Vs + stage * TN * P * 2;
      for (int i = tid; i < TN * CH; i += NW * 32) {
        const int j = i / CH, ch = i % CH;
        const int kvpos = t0 + j;
        const bool ok = kvpos < kv_end;
        const int pp = ok ? kvpos : kv_end - 1;
        size_t off;
        if (p.seq_start) {
          off = (size_t)(seq0 + pp) * p.row_stride + kvh * D + ch * 8;
        } else {
          const int page = btab[pp / kPageSize];
          off = (((size_t)page * p.n_kv + kvh) * kPageSize + pp % kPageSize) * D + ch * 8;
        }
        cp_async16(kst + tile_off(j, ch), p.k_cache + off, ok ? 16 : 0);
        cp_async16(vst + tile_off(j, ch), p.v_cache + off, ok ? 16 : 0);
      }
    };
    // prologue: STAGES-1 tiles in flight (one commit group per tile slot, empty groups keep the count uniform)
#pragma unroll
    for (int s0 = 0; s0 < STAGES - 1; ++s0) {
      if (s0 < n_tiles) load_kv(s0, kv_begin + s0 * TN);
      cp_async_commit();
    }
    uint32_t qf[D / 16][4];
    const int qpos_a = pos0 + row_a / G, qpos_b = pos0 + row_b / G;

    for (int it = 0; it < n_tiles; ++it) {
      const int t0 = kv_begin + it * TN;
      if (it + STAGES - 1 < n_tiles) load_kv((it + STAGES - 1) % STAGES, t0 + (STAGES - 1) * TN);
      cp_async_commit();
      cp_async_wait<STAGES - 1>();
      __syncthreads();
      if (it == 0) {
        const uint32_t qbase = smem_u32(Qs);
#pragma unroll
        for (int ks = 0; ks < D / 16; ++ks) {
          const int r = warp * 16 + (lane & 7) + 8 * ((lane >> 3) & 1);
          ldsm_x4(qbase + tile_off(r, ks * 2 + (lane >> 4)), qf[ks][0], qf[ks][1], qf[ks][2], qf[ks][3]);
        }
      }
      const uint32_t kbase = smem_u32(Ks + (it % STAGES) * TN * P * 2);
      const uint32_t vbase = smem_u32(Vs + (it % STAGES) * TN * P * 2);

      // ---- S = Q K^T
      float s[NT][4];
#pragma unroll
      for (int n2 = 0; n2 < NT / 2; ++n2) {
#pragma unroll
        for (int e = 0; e < 4; ++e) s[2 * n2][e] = s[2 * n2 + 1][e] = 0.f;
#pragma unroll
        for (int ks = 0; ks < D / 16; ++ks) {
          const int r = n2 * 16 + (lane & 7) + 8 * (lane >> 4);
          uint32_t b0, b1, b2, b3;
          ldsm_x4(kbase + tile_off(r, ks * 2 + ((lane >> 3) & 1)), b0, b1, b2, b3);
          mma_bf16_16816(s[2 * n2], qf[ks], b0, b1);
          mma_bf16_16816(s[2 * n2 + 1], qf[ks], b2, b3);
        }
      }
      // ---- mask + online softmax (rows g and g+8 of this warp's 16-row slab)
      float mx_a = -INFINITY, mx_b = -INFINITY;
#pragma unroll
      for (int n = 0; n < NT; ++n) {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int col = t0 + n * 8 + 2 * c + (e & 1);
          const int qpos = (e < 2) ? qpos_a : qpos_b;
          const bool ok = (p.bidirectional || col <= qpos) && (col < kv_end);
          const float v = ok ? s[n][e] * p.scale_log2 : -INFINITY;
          s[n][e] = v;
          if (e < 2) mx_a = fmaxf(mx_a, v); else mx_b = fmaxf(mx_b, v);
        }
      }
      mx_a = fmaxf(mx_a, __shfl_xor_sync(0xffffffffu, mx_a, 1));
      mx_a = fmaxf(mx_a, __shfl_xor_sync(0xffffffffu, mx_a, 2));
      mx_b = fmaxf(mx_b, __shfl_xor_sync(0xffffffffu, mx_b, 1));
      mx_b = fmaxf(mx_b, __shfl_xor_sync(0xffffffffu, mx_b, 2));
      const float mn_a = fmaxf(m_run[0], mx_a), mn_b = fmaxf(m_run[1], mx_b);
      const float mu_a = (mn_a == -INFINITY) ? 0.f : mn_a;
      const float mu_b = (mn_b == -INFINITY) ? 0.f : mn_b;
      const float al_a = exp2f(m_run[0] - mu_a), al_b = exp2f(m_run[1] - mu_b);
      m_run[0] = mn_a; m_run[1] = mn_b;
      float sum_a = 0.f, sum_b = 0.f;
#pragma unroll
      for (int n = 0; n < NT; ++n) {
        s[n][0] = exp2f(s[n][0] - mu_a); s[n][1] = exp2f(s[n][1] - mu_a);
        s[n][2] = exp2f(s[n][2] - mu_b); s[n][3] = exp2f(s[n][3] - mu_b);
        sum_a += s[n][0] + s[n][1];
        sum_b += s[n][2] + s[n][3];
      }
      l_run[0] = l_run[0] * al_a + sum_a;
      l_run[1] = l_run[1] * al_b + sum_b;
#pragma unroll
      for (int i = 0; i < D / 8; ++i) { o[i][0] *= al_a; o[i][1] *= al_a; o[i][2] *= al_b; o[i][3] *= al_b; }
      // ---- O += P V
#pragma unroll
      for (int kt = 0; kt < TN / 16; ++kt) {
        uint32_t a[4];
        a[0] = pack_bf16(s[2 * kt][0], s[2 * kt][1]);
        a[1] = pack_bf16(s[2 * kt][2], s[2 * kt][3]);
        a[2] = pack_bf16(s[2 * kt + 1][0], s[2 * kt + 1][1]);
        a[3] = pack_bf16(s[2 * kt + 1][2], s[2 * kt + 1][3]);
#pragma unroll
        for (int d2 = 0; d2 < D / 16; ++d2) {
          const int r = kt * 16 + (lane & 7) + 8 * ((lane >> 3) & 1);
          uint32_t b0, b1, b2, b3;
          ldsm_x4_t(vbase + tile_off(r, d2 * 2 + (lane >> 4)), b0, b1, b2, b3);
          mma_bf16_16816(o[2 * d2], a, b0, b1);
          mma_bf16_16816(o[2 * d2 + 1], a, b2, b3);
        }
      }
      __syncthreads();
    }
  }

  // ---- finalize
  float l_a = l_run[0], l_b = l_run[1];
  l_a += __shfl_xor_sync(0xffffffffu, l_a, 1); l_a += __shfl_xor_sync(0xffffffffu, l_a, 2);
  l_b += __shfl_xor_sync(0xffffffffu, l_b, 1); l_b += __shfl_xor_sync(0xffffffffu, l_b, 2);
#pragma unroll
  for (int half = 0; half < 2; ++half) {
    const int row = half ? row_b : row_a;
    if (row >= n_rows) continue;
    const int tok = tok0 + row / G, head = kvh * G + row % G;
    const float l = half ? l_b : l_a;
    {
      const float inv = l > 0.f ? 1.f / l : 0.f;
      __nv_bfloat16* po = p.out + ((size_t)tok * p.n_q + head) * D;
#pragma unroll
      for (int n = 0; n < D / 8; ++n)
        *reinterpret_cast<uint32_t*>(po + n * 8 + 2 * c) = pack_bf16(o[n][2 * half] * inv, o[n][2 * half + 1] * inv);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// decode attention (one query token per sequence): one warp per (slot, kv head, kv split)
//
//   S   [16 x 16 tokens] = Q [16 rows: G real heads, rest zero] . K^T      mma.m16n8k16 x 16 per page
//   O^T [128 dims x 8 heads] += V^T [128 x 16 tokens] . P^T [16 tokens x 8 heads]
// The C fragments of S are exactly the B fragments of P^T, so the probabilities never leave registers, and the
// transposed second product needs half the accumulators / MMAs of the row-major form.  A KV tile is one 16-token
// page = one contiguous 4 KiB block per tensor: one block-table lookup and 16 trivially addressed cp.async per
// lane per tile.  Masking only happens on the boundary tile.  (r01 v2 capture: the generic kernel was issue-bound
// at 7 warps/SM, 37% issue-active, 3.5 TB/s.)
// ------------------------------------------------------------------------------------------------
//
// NW > 1 (small batches): the NW warps of a CTA each take one KV split of the same (slot, kv head) and merge through
// SHARED memory - no partial rows in global memory, no fence, no arrival counter (r01 timeline at 8 slots: the
// global-memory split path spent ~12 us per layer on a 3 us stream).  NW == 1 keeps the grid-level split
// (blockIdx.z) with the in-kernel global combine for shapes where one warp per CTA already fills the GPU.
template <int STAGES, int D, int NW>
__global__ void __launch_bounds__(32 * NW) decode_attn_kernel(const AttnParams p) {
  constexpr int TN = kPageSize, P = kTilePitch, CH = D / 8, KS = D / 16;
  constexpr int RING = 2 * STAGES * TN * P * 2;  // bytes of one warp's K + V ring
  static_assert(TN == 16, "a KV tile is one page");
  static_assert(NW == 1 || RING >= (8 * D + 16) * 4, "the ring doubles as the warp's partial-result buffer");
  extern __shared__ __align__(128) uint8_t smem[];
  const int warp = threadIdx.x >> 5;
  uint8_t* Ks = smem + warp * RING;
  uint8_t* Vs = Ks + STAGES * TN * P * 2;

  pdl_launch_dependents();
  if (threadIdx.x == 0) trace_begin(p.tr);

  const int lane = threadIdx.x & 31;
  const int g = lane >> 2, c = lane & 3;
  const int slot = blockIdx.x, kvh = blockIdx.y;
  const int G = p.n_q / p.n_kv;  // <= 8 (checked on the host)
  const int kv_len = p.pos[slot] + 1;
  int kv_begin = 0, kv_end = kv_len;
  const bool split = NW == 1 && p.n_splits > 1;   // grid-level split with the global-memory combine
  const int n_parts = NW > 1 ? NW : p.n_splits;
  if (n_parts > 1) {
    const int chunk = (((kv_len + n_parts - 1) / n_parts) + 15) & ~15;
    kv_begin = (NW > 1 ? warp : (int)blockIdx.z) * chunk;
    kv_end = min(kv_len, kv_begin + chunk);
  }
  const int* btab = p.block_table + (size_t)slot * p.max_pages;
  const int n_tiles = kv_begin < kv_end ? (kv_end - kv_begin + TN - 1) / TN : 0;

  float ot[KS][4];  // O^T: [m-tile of 16 dims][rows g / g+8, heads 2c / 2c+1]
#pragma unroll
  for (int i = 0; i < KS; ++i) ot[i][0] = ot[i][1] = ot[i][2] = ot[i][3] = 0.f;
  float m_run = -INFINITY, l_run = 0.f;  // softmax state of head g (replicated over the quad)

  if (n_tiles > 0) {
    auto load_kv = [&](int stage, int t0) {
      const int page = btab[t0 / kPageSize];
      const size_t base = ((size_t)page * p.n_kv + kvh) * kPageSize * D;  // contiguous [16][D] block
      const int valid = kv_end - t0;                                       // rows >= valid are zero-filled
      uint8_t* kst = Ks + stage * TN * P * 2;
      uint8_t* vst = Vs + stage * TN * P * 2;
#pragma unroll
      for (int k = 0; k < TN * CH / 32; ++k) {
        const int i = lane + 32 * k, j = i / CH, ch = i % CH;
        const int nb = j < valid ? 16 : 0;
        cp_async16(kst + tile_off(j, ch), p.k_cache + base + (size_t)i * 8, nb);
        cp_async16(vst + tile_off(j, ch), p.v_cache + base + (size_t)i * 8, nb);
      }
    };
    // The first STAGES-1 pages are requested BEFORE the dependency wait whenever they hold only tokens of earlier
    // steps (everything but the row the rope kernel of this very step is writing): this CTA is usually resident a
    // few us before the wait returns, and the r01 timeline shows ~6 us of prologue + first-load latency per layer.
    const bool early = kv_begin + min(STAGES - 1, n_tiles) * TN <= kv_len - 1;
    if (early) {
#pragma unroll
      for (int s0 = 0; s0 < STAGES - 1; ++s0) {
        if (s0 < n_tiles) load_kv(s0, kv_begin + s0 * TN);
        cp_async_commit();
      }
    }
    pdl_wait();
    if (threadIdx.x == 0) trace_waited(p.tr);
    if (!early) {
#pragma unroll
      for (int s0 = 0; s0 < STAGES - 1; ++s0) {
        if (s0 < n_tiles) load_kv(s0, kv_begin + s0 * TN);
        cp_async_commit();
      }
    }
    // Q fragments: row g = head g of the group (zero for g >= G), rows 8..15 zero
    uint32_t qf[KS][2];
    {
      const bool ok = g < G;
      const __nv_bfloat16* qp = p.q + ((size_t)slot * p.n_q + kvh * G + (ok ? g : 0)) * D + 2 * c;
#pragma unroll
      for (int ks = 0; ks < KS; ++ks) {
        qf[ks][0] = ok ? *reinterpret_cast<const uint32_t*>(qp + ks * 16) : 0u;
        qf[ks][1] = ok ? *reinterpret_cast<const uint32_t*>(qp + ks * 16 + 8) : 0u;
      }
    }
    for (int it = 0; it < n_tiles; ++it) {
      const int t0 = kv_begin + it * TN;
      if (it + STAGES - 1 < n_tiles) load_kv((it + STAGES - 1) % STAGES, t0 + (STAGES - 1) * TN);
      cp_async_commit();
      cp_async_wait<STAGES - 1>();
      __syncwarp();
      const uint32_t kbase = smem_u32(Ks + (it % STAGES) * TN * P * 2);
      const uint32_t vbase = smem_u32(Vs + (it % STAGES) * TN * P * 2);
      // ---- S = Q K^T for the 16 tokens of this page
      float s0[4] = {0.f, 0.f, 0.f, 0.f}, s1[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int ks = 0; ks < KS; ++ks) {
        const int r = (lane & 7) + 8 * (lane >> 4);
        uint32_t b0, b1, b2, b3;
        ldsm_x4(kbase + tile_off(r, ks * 2 + ((lane >> 3) & 1)), b0, b1, b2, b3);
        const uint32_t a[4] = {qf[ks][0], 0u, qf[ks][1], 0u};
        mma_bf16_16816(s0, a, b0, b1);
        mma_bf16_16816(s1, a, b2, b3);
      }
      float v0 = s0[0] * p.scale_log2, v1 = s0[1] * p.scale_log2, v2 = s1[0] * p.scale_log2, v3 = s1[1] * p.scale_log2;
      if (t0 + TN > kv_end) {  // boundary page (warp-uniform)
        const int col = t0 + 2 * c;
        if (col >= kv_end) v0 = -INFINITY;
        if (col + 1 >= kv_end) v1 = -INFINITY;
        if (col + 8 >= kv_end) v2 = -INFINITY;
        if (col + 9 >= kv_end) v3 = -INFINITY;
      }
      float mx = fmaxf(fmaxf(v0, v1), fmaxf(v2, v3));
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
      const float mn = fmaxf(m_run, mx);            // finite: every tile holds at least one valid token
      const float al = exp2f(m_run - mn);
      m_run = mn;
      v0 = exp2f(v0 - mn); v1 = exp2f(v1 - mn); v2 = exp2f(v2 - mn); v3 = exp2f(v3 - mn);
      l_run = l_run * al + (v0 + v1) + (v2 + v3);   // quad-partial sum
      // rescale O^T: this thread holds heads 2c, 2c+1; their factors live in the lanes with g == head
      const float al_a = __shfl_sync(0xffffffffu, al, (2 * c) * 4);
      const float al_b = __shfl_sync(0xffffffffu, al, ((2 * c + 1) & 7) * 4);
      if (__any_sync(0xffffffffu, al != 1.f)) {
#pragma unroll
        for (int i = 0; i < KS; ++i) { ot[i][0] *= al_a; ot[i][1] *= al_b; ot[i][2] *= al_a; ot[i][3] *= al_b; }
      }
      // ---- O^T += V^T P^T   (B fragments = the probabilities just computed)
      const uint32_t pb0 = pack_bf16(v0, v1), pb1 = pack_bf16(v2, v3);
#pragma unroll
      for (int mt = 0; mt < KS; ++mt) {
        const int r = (lane & 7) + 8 * (lane >> 4);
        uint32_t a[4];
        ldsm_x4_t(vbase + tile_off(r, mt * 2 + ((lane >> 3) & 1)), a[0], a[1], a[2], a[3]);
        mma_bf16_16816(ot[mt], a, pb0, pb1);
      }
      __syncwarp();
    }
  }

  if (n_tiles == 0) {  // empty split: still order this CTA's writes after the previous kernel
    pdl_wait();
    if (threadIdx.x == 0) trace_waited(p.tr);
  }
  // ---- finalize: l of head g -> full row sum; this thread needs the sums of heads 2c, 2c+1
  l_run += __shfl_xor_sync(0xffffffffu, l_run, 1);
  l_run += __shfl_xor_sync(0xffffffffu, l_run, 2);
  const int h_a = 2 * c, h_b = 2 * c + 1;
  const float l_a = __shfl_sync(0xffffffffu, l_run, h_a * 4), l_b = __shfl_sync(0xffffffffu, l_run, (h_b & 7) * 4);
  if constexpr (NW > 1) {
    // ---- in-CTA combine: every warp parks (m, l) and its O^T partial in its own (now idle) ring, then all
    // threads merge the NW partials; item = (head, 4 consecutive dims)
    cp_async_wait<0>();
    __syncwarp();
    float* part = reinterpret_cast<float*>(Ks);        // [8 heads][D]
    float2* pml = reinterpret_cast<float2*>(part + 8 * D);  // [8 heads]
    if (c == 0) pml[g] = make_float2(m_run, l_run);     // rows g >= G hold zeros / -inf: never read
#pragma unroll
    for (int hh = 0; hh < 2; ++hh) {
      const int head = hh ? h_b : h_a;
#pragma unroll
      for (int mt = 0; mt < KS; ++mt) {
        part[head * D + mt * 16 + g] = ot[mt][hh];
        part[head * D + mt * 16 + g + 8] = ot[mt][2 + hh];
      }
    }
    __syncthreads();
    for (int item = threadIdx.x; item < G * (D / 4); item += 32 * NW) {
      const int hg = item / (D / 4), d4 = item % (D / 4);
      float M = -INFINITY;
#pragma unroll
      for (int w = 0; w < NW; ++w) M = fmaxf(M, reinterpret_cast<const float2*>(smem + w * RING + 8 * D * 4)[hg].x);
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
      float L = 0.f;
#pragma unroll
      for (int w = 0; w < NW; ++w) {
        const float2 e = reinterpret_cast<const float2*>(smem + w * RING + 8 * D * 4)[hg];
        const float wgt = e.x == -INFINITY ? 0.f : exp2f(e.x - M);
        const float4 v = reinterpret_cast<const float4*>(smem + w * RING)[hg * (D / 4) + d4];
        L += e.y * wgt;
        acc.x += v.x * wgt; acc.y += v.y * wgt; acc.z += v.z * wgt; acc.w += v.w * wgt;
      }
      const float inv = L > 0.f ? 1.f / L : 0.f;
      uint2 ov;
      ov.x = pack_bf16(acc.x * inv, acc.y * inv);
      ov.y = pack_bf16(acc.z * inv, acc.w * inv);
      *reinterpret_cast<uint2*>(p.out + ((size_t)slot * p.n_q + kvh * G + hg) * D + d4 * 4) = ov;
    }
    if (threadIdx.x == 0) trace_end(p.tr);
    return;
  }
  if (split) {
    if (c == 0 && g < G) {
      const size_t base = ((size_t)blockIdx.z * p.T + slot) * p.n_q + kvh * G + g;
      p.part_ml[base * 2] = m_run;
      p.part_ml[base * 2 + 1] = l_run;
    }
#pragma unroll
    for (int hh = 0; hh < 2; ++hh) {
      const int head = hh ? h_b : h_a;
      if (head >= G) continue;
      float* po = p.part_o + (((size_t)blockIdx.z * p.T + slot) * p.n_q + kvh * G + head) * D;
#pragma unroll
      for (int mt = 0; mt < KS; ++mt) {
        po[mt * 16 + g] = ot[mt][hh];
        po[mt * 16 + g + 8] = ot[mt][2 + hh];
      }
    }
    // ---- in-kernel combine: the split that arrives last merges all partials of this (slot, kv head).
    // r01 timeline: the first version walked head by head with three dependent L2 round trips each (~8 us of
    // tail per layer); here the (m, l) pairs of all heads x splits arrive in one round trip, the weights are
    // formed from shared memory, and every head's partial rows are requested before the first one is consumed.
    __threadfence();
    int old = 0;
    if (lane == 0) old = atomicAdd(p.split_counter + slot * p.n_kv + kvh, 1);
    old = __shfl_sync(0xffffffffu, old, 0);
    if (old == p.n_splits - 1) {
      __threadfence();
      const int S = p.n_splits;  // <= kMaxDecodeSplits
      float2* ml = reinterpret_cast<float2*>(smem);  // [G][S]; the KV ring is idle by now
      __syncwarp();
      for (int i = lane; i < G * S; i += 32) {
        const int hg = i / S, sp = i % S;
        const size_t base = ((size_t)sp * p.T + slot) * p.n_q + kvh * G + hg;
        ml[i] = __ldcg(reinterpret_cast<const float2*>(p.part_ml + base * 2));
      }
      __syncwarp();
      const bool act = lane * 4 < D;
      for (int hg = 0; hg < G; ++hg) {
        const int head = kvh * G + hg;
        float4 v[kMaxDecodeSplits];
#pragma unroll
        for (int sp = 0; sp < kMaxDecodeSplits; ++sp) {
          v[sp] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (sp < S && act)
            v[sp] = __ldcg(reinterpret_cast<const float4*>(p.part_o + (((size_t)sp * p.T + slot) * p.n_q + head) * D) + lane);
        }
        float M = -INFINITY;
        for (int sp = 0; sp < S; ++sp) M = fmaxf(M, ml[hg * S + sp].x);
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        float L = 0.f;
#pragma unroll
        for (int sp = 0; sp < kMaxDecodeSplits; ++sp) {
          if (sp < S) {
            const float2 e = ml[hg * S + sp];
            const float wgt = e.x == -INFINITY ? 0.f : exp2f(e.x - M);
            L += e.y * wgt;
            acc.x += v[sp].x * wgt; acc.y += v[sp].y * wgt; acc.z += v[sp].z * wgt; acc.w += v[sp].w * wgt;
          }
        }
        const float inv = L > 0.f ? 1.f / L : 0.f;
        uint2 ov;
        ov.x = pack_bf16(acc.x * inv, acc.y * inv);
        ov.y = pack_bf16(acc.z * inv, acc.w * inv);
        if (act) *reinterpret_cast<uint2*>(p.out + ((size_t)slot * p.n_q + head) * D + lane * 4) = ov;
      }
      if (lane == 0) p.split_counter[slot * p.n_kv + kvh] = 0;  // self-resetting for the next launch
    }
  } else {
#pragma unroll
    for (int hh = 0; hh < 2; ++hh) {
      const int head = hh ? h_b : h_a;
      if (head >= G) continue;
      const float l = hh ? l_b : l_a;
      const float inv = l > 0.f ? 1.f / l : 0.f;
      __nv_bfloat16* po = p.out + ((size_t)slot * p.n_q + kvh * G + head) * D;
#pragma unroll
      for (int mt = 0; mt < KS; ++mt) {
        po[mt * 16 + g] = __float2bfloat16(ot[mt][hh] * inv);
        po[mt * 16 + g + 8] = __float2bfloat16(ot[mt][2 + hh] * inv);
      }
    }
  }  if (threadIdx.x == 0) trace_end(p.tr);
}

constexpr int kPrefillNW = kPrefillTileRows / 16, kPrefillTN = 64, kPrefillStages = 2;
constexpr int kDecodeStages = 6;
constexpr int attn_smem(int nw, int tn, int stages) { return (nw * 16 + 2 * stages * tn) * kTilePitch * 2; }
constexpr int kDecodeSmem = 2 * kDecodeStages * kPageSize * kTilePitch * 2;

void attn_set_attrs() {
  auto go = [&](auto dtag) {
    constexpr int D = decltype(dtag)::value;
    cudaFuncSetAttribute(paged_attn_kernel<kPrefillNW, kPrefillTN, kPrefillStages, D>,
                         cudaFuncAttributeMaxDynamicSharedMemorySize, attn_smem(kPrefillNW, kPrefillTN, kPrefillStages));
    cudaFuncSetAttribute(decode_attn_kernel<2, D, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
    cudaFuncSetAttribute(decode_attn_kernel<3, D, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
    cudaFuncSetAttribute(decode_attn_kernel<4, D, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
    cudaFuncSetAttribute(decode_attn_kernel<6, D, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
    cudaFuncSetAttribute(decode_attn_kernel<7, D, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
    cudaFuncSetAttribute(decode_attn_kernel<6, D, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
    cudaFuncSetAttribute(decode_attn_kernel<3, D, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
    cudaFuncSetAttribute(decode_attn_kernel<3, D, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 192 * 1024);
  };
  go(std::integral_constant<int, 128>{});
  go(std::integral_constant<int, 96>{});
  go(std::integral_constant<int, 64>{});
  go(std::integral_constant<int, 32>{});
}
void launch_attn_prefill(const LaunchCfg& lc, const AttnParams& p, int n_tiles) {
  dispatch_head_dim(p.head_dim, [&](auto dtag) {
    constexpr int D = decltype(dtag)::value;
    launch_k(lc, paged_attn_kernel<kPrefillNW, kPrefillTN, kPrefillStages, D>, dim3(n_tiles, p.n_kv, 1),
             dim3(kPrefillNW * 32), attn_smem(kPrefillNW, kPrefillTN, kPrefillStages), p);
  });
}
// one-warp decode CTAs that can be resident at once on this GPU (occupancy query, cached per process; the
// three head_dim instantiations use the same shared-memory footprint, registers never bind before it does)
int attn_decode_resident_ctas() {
  static int cached = 0;
  if (!cached) {
    int per_sm = 0, dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, decode_attn_kernel<kDecodeStages, 128, 1>, 32,
                                                      kDecodeSmem) != cudaSuccess || per_sm < 1)
      per_sm = 4;
    cached = per_sm * sms;
  }
  return cached;
}
// Pipeline depth of the decode kernel.  r01 live timelines (profiles/r01_decode_timeline_v*.txt, 64 slots x 8 kv
// heads, ctx 576): 1024 CTAs (2 KV splits) x 3 stages 33.1 us per layer; 512 CTAs (no split) x 3 stages 26.2 us,
// x 6 stages 24.6 us (floor 21 us).  What hurt was not bytes in flight but the split epilogue (partials ->
// fence -> counter -> serial combine) and the extra CTAs; so: few, long CTAs with a deep ring, and KV splits only
// when the batch alone cannot fill the GPU (engine.cu: launch_decode).  MQ_ATTN_STAGES=2..7 overrides (experiments).
static int decode_stages() {
  static const int st = [] {
    const char* e = getenv("MQ_ATTN_STAGES");
    const int v = e ? atoi(e) : kDecodeStages;
    return (v == 2 || v == 3 || v == 4 || v == 6 || v == 7) ? v : kDecodeStages;
  }();
  return st;
}
static int decode_smem() { return 2 * decode_stages() * kPageSize * kTilePitch * 2; }
constexpr int decode_ring_bytes(int stages) { return 2 * stages * kPageSize * kTilePitch * 2; }
void launch_attn_decode(const LaunchCfg& lc, const AttnParams& p, int n_slots) {
  dispatch_head_dim(p.head_dim, [&](auto dtag) {
    constexpr int D = decltype(dtag)::value;
    if (p.n_warps > 1) {  // in-CTA split: warps = KV splits, shared-memory combine, no grid-level split
      const dim3 grid(n_slots, p.n_kv, 1);
      switch (p.n_warps) {
        case 2: launch_k(lc, decode_attn_kernel<6, D, 2>, grid, dim3(64), 2 * decode_ring_bytes(6), p); break;
        case 4: launch_k(lc, decode_attn_kernel<3, D, 4>, grid, dim3(128), 4 * decode_ring_bytes(3), p); break;
        default: launch_k(lc, decode_attn_kernel<3, D, 8>, grid, dim3(256), 8 * decode_ring_bytes(3), p); break;
      }
      return;
    }
    static const bool env_stages = getenv("MQ_ATTN_STAGES") != nullptr;
    const int st = (!env_stages && (p.stages == 2 || p.stages == 3 || p.stages == 4 || p.stages == 6)) ? p.stages : decode_stages();
    const int smem = decode_ring_bytes(st);
    const dim3 grid(n_slots, p.n_kv, p.n_splits);
    switch (st) {
      case 2: launch_k(lc, decode_attn_kernel<2, D, 1>, grid, dim3(32), smem, p); break;
      case 3: launch_k(lc, decode_attn_kernel<3, D, 1>, grid, dim3(32), smem, p); break;
      case 4: launch_k(lc, decode_attn_kernel<4, D, 1>, grid, dim3(32), smem, p); break;
      case 7: launch_k(lc, decode_attn_kernel<7, D, 1>, grid, dim3(32), smem, p); break;
      default: launch_k(lc, decode_attn_kernel<kDecodeStages, D, 1>, grid, dim3(32), smem, p); break;
    }
  });
}

// ------------------------------------------------------------------------------------------------
// greedy sampler: argmax over the vocabulary (lowest index wins ties), then advance the slot state
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) argmax_kernel(const float* __restrict__ logits, int V, int ldl,
                                                      int* __restrict__ out_tokens, const int* __restrict__ dst_slot,
                                                      int* __restrict__ cur_token, int* __restrict__ pos_inc,
                                                      const int* __restrict__ active) {
  pdl_launch_dependents();  // let the next kernel start its prologue (weight prefetch) right away
  pdl_wait();
  const int row = blockIdx.x;
  const float4* lp = reinterpret_cast<const float4*>(logits + (size_t)row * ldl);
  float best = -INFINITY;
  int bi = 0x7fffffff;
  for (int i = threadIdx.x; i < V / 4; i += blockDim.x) {
    const float4 v = lp[i];
    const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int idx = i * 4 + e;
      if (vv[e] > best || (vv[e] == best && idx < bi)) { best = vv[e]; bi = idx; }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ob = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ob > best || (ob == best && oi < bi)) { best = ob; bi = oi; }
  }
  __shared__ float sb[32];
  __shared__ int si[32];
  if ((threadIdx.x & 31) == 0) { sb[threadIdx.x >> 5] = best; si[threadIdx.x >> 5] = bi; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w)
      if (sb[w] > best || (sb[w] == best && si[w] < bi)) { best = sb[w]; bi = si[w]; }
    out_tokens[row] = bi;
    const int slot = dst_slot ? dst_slot[row] : row;
    if (cur_token) cur_token[slot] = bi;
    if (pos_inc && (!active || active[slot])) pos_inc[slot] += 1;
  }
}
void launch_argmax(const LaunchCfg& lc, const float* logits, int rows, int V, int ldl, int* out_tokens,
                   const int* dst_slot, int* cur_token, int* pos_inc, const int* active) {
  launch_k(lc, argmax_kernel, dim3(rows), dim3(1024), 0, logits, V, ldl, out_tokens, dst_slot, cur_token, pos_inc,
           active);
}

// ------------------------------------------------------------------------------------------------
// stochastic sampler: temperature, top-k, top-p, seed (the "sample" step of the backend's forward pass).
//
// One CTA per row.  temperature <= 0 (the default) is the greedy path above, bit for bit.  Otherwise:
//   1. top-k:  radix select (4 passes of 256-bin counts over the order-preserving uint image of the logits) finds the
//      value of the k-th largest logit; ties at the threshold stay in (the kept set is {l >= thr}).
//   2. top-p over what top-k kept: the same radix walk with MASS histograms - fixed-point 2^40 * exp((l - max) / T)
//      in 64-bit integer atomics, so the result does not depend on the order threads arrive in - finds the largest
//      threshold whose kept mass reaches p * Z.
//   3. the draw is a Gumbel-max: argmax over the kept set of l / T - log(-log u), u from a counter-based generator
//      keyed by (seed, position, token id) - an exact sample of softmax(l / T) restricted to the kept set, with no
//      sort, no prefix sum and no state carried between steps (restated in oracle/sampler_ref.py).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t f32_key(float f) {  // order-preserving: a < b  <=>  key(a) < key(b)
  const uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key_f32(uint32_t k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}
__device__ __forceinline__ uint64_t mix64(uint64_t x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}
__device__ __forceinline__ float gumbel_noise(uint64_t seed, int counter, int idx) {
  const uint64_t r = mix64(seed ^ ((uint64_t)(uint32_t)counter * 0xD1342543DE82EF95ull) ^ ((uint64_t)(uint32_t)idx * 0xA24BAED4963EE407ull));
  const float u = ((float)(uint32_t)(r >> 40) + 0.5f) * (1.0f / 16777216.0f);  // (0, 1)
  return -logf(-logf(u));
}
constexpr float kMassScale = 1099511627776.0f;  // 2^40

// Radix walk from the most significant byte: afterwards `prefix` is the key of the threshold element.
//   MASS == false: the K-th largest key (count walk).   MASS == true: the largest key t with mass{key >= t} >= target.
// Only keys >= floor_key take part.  All threads of the block call this; the result is returned to all of them.
// `hist` holds kHistCopies private copies of the 256 bins, picked by lane: the top byte of a float (sign + 7 exponent
// bits) sends a whole row into a handful of bins, and with one copy every atomic of a warp hit the same address
// (r01: 1.78 ms per step for this walk; the copies are folded before the bins are read).
constexpr int kHistCopies = 16;
template <bool MASS>
__device__ uint32_t radix_threshold(const float* __restrict__ lp, int V, uint32_t floor_key, unsigned long long target,
                                    float mx, float inv_t, unsigned long long* hist /* smem [kHistCopies][256] */,
                                    uint32_t* bcast) {
  uint32_t prefix = 0, mask = 0;
  unsigned long long* mine = hist + (threadIdx.x & (kHistCopies - 1)) * 256;
  for (int shift = 24; shift >= 0; shift -= 8) {
    for (int i = threadIdx.x; i < 256 * kHistCopies; i += blockDim.x) hist[i] = 0ull;
    __syncthreads();
    for (int i = threadIdx.x; i < V; i += blockDim.x) {
      const float l = lp[i];
      const uint32_t k = f32_key(l);
      if (k >= floor_key && (k & mask) == prefix) {
        unsigned long long w = 1ull;
        if (MASS) w = (unsigned long long)(kMassScale * __expf((l - mx) * inv_t));
        atomicAdd(&mine[(k >> shift) & 255u], w);
      }
    }
    __syncthreads();
    if (threadIdx.x < 256) {
      unsigned long long sum = 0ull;
#pragma unroll
      for (int c = 0; c < kHistCopies; ++c) sum += hist[c * 256 + threadIdx.x];
      hist[threadIdx.x] = sum;  // copy 0 now holds the folded bins (each thread reads its column before writing it)
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      unsigned long long acc = 0ull;
      int bin = 255;
      for (; bin > 0; --bin) {
        if (acc + hist[bin] >= target) break;
        acc += hist[bin];
      }
      bcast[0] = (uint32_t)bin;
      // what is still to be found inside the chosen bin
      reinterpret_cast<unsigned long long*>(bcast + 2)[0] = target - acc;
    }
    __syncthreads();
    prefix |= bcast[0] << shift;
    mask |= 255u << shift;
    target = reinterpret_cast<unsigned long long*>(bcast + 2)[0];
    __syncthreads();
  }
  return prefix;
}


// ---- fast top-k path (0 < k <= 1024): two passes over the row instead of the radix walk's eight.
//   a. every thread keeps the maximum of its strided share of the row; the k-th largest of those 1024 maxima, T0, is a
//      lower bound of the k-th largest logit (k distinct elements are >= T0);
//   b. elements >= T0 are compacted into shared memory (a few times k of them for any distribution that is not flat),
//   c. sorted there (bitonic, value descending / token id ascending, so the result does not depend on arrival order),
//   d. cut at k (ties at the cut stay in), then at the top-p mass, and the Gumbel-max draw runs over what is left.
// More candidates than kSampleCand (a nearly constant row) falls back to the radix walk.
constexpr int kSampleCand = 4096;
__device__ __forceinline__ bool cand_before(float va, int ia, float vb, int ib) { return va > vb || (va == vb && ia < ib); }
__device__ void bitonic_desc(float* val, int* idx, int n /* power of two */) {
  for (int size = 2; size <= n; size <<= 1)
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int t = threadIdx.x; t < n / 2; t += blockDim.x) {
        const int pos = 2 * t - (t & (stride - 1)), q = pos + stride;
        const bool desc = (pos & size) == 0;
        const float va = val[pos], vb = val[q];
        const int ia = idx[pos], ib = idx[q];
        if (cand_before(va, ia, vb, ib) != desc) { val[pos] = vb; val[q] = va; idx[pos] = ib; idx[q] = ia; }
      }
      __syncthreads();
    }
}

// Steps a - c: elements >= the k-th largest of the 1024 thread maxima (0 < k <= 1024) are compacted into cval / cidx
// and, when they fit (return value <= kSampleCand), sorted value descending / id ascending; a larger return value is
// the count of a pool that overflowed.  want_z: *z_part = this thread's share of sum exp((l - mx) * inv_t) over the row.
// Shared by the top-k path and the log-probability record.
__device__ int gather_candidates(const float* __restrict__ lp, int V, float thread_max, int k, float* cval, int* cidx,
                                 int* n_cand, bool want_z, float mx, float inv_t, float* z_part) {
  cval[threadIdx.x] = thread_max;
  cidx[threadIdx.x] = threadIdx.x;
  if (threadIdx.x == 0) *n_cand = 0;
  __syncthreads();
  bitonic_desc(cval, cidx, 1024);
  const float t0 = cval[k - 1];
  __syncthreads();
  float z = 0.f;  // fixed order per thread (the caller sums the threads in a fixed tree)
  for (int i = threadIdx.x; i < V; i += blockDim.x) {
    const float l = lp[i];
    if (want_z) z += __expf((l - mx) * inv_t);
    if (l >= t0) {
      const int at = atomicAdd(n_cand, 1);
      if (at < kSampleCand) { cval[at] = l; cidx[at] = i; }
    }
  }
  *z_part = z;
  __syncthreads();
  const int nc = *n_cand;
  if (nc <= kSampleCand) {
    int n2 = 2;
    while (n2 < nc) n2 <<= 1;
    for (int i = nc + threadIdx.x; i < n2; i += blockDim.x) { cval[i] = -INFINITY; cidx[i] = 0x7fffffff; }
    __syncthreads();
    bitonic_desc(cval, cidx, n2);
  }
  return nc;
}

// The log-probability record of a row (see LogprobRec), before the draw while the pool is free: lse, then the n
// (<= min(kTopLogprobsMax, V)) most probable tokens into rec->id / rec->lp.  Returns lse to every thread; the drawn
// token's own entry is written beside the token.
__device__ float logprob_record(const float* __restrict__ lp, int V, int n, LogprobRec* rec, float* cval, int* cidx,
                                unsigned long long* hist, uint32_t* bcast, int* n_cand) {
  __shared__ float wm[32], ws[32];
  __shared__ int wc[32];
  // per-thread online (max, sum exp(l - max)) over the thread's strided share, in a fixed order
  float m = -FLT_MAX, s = 0.f;
  for (int i = threadIdx.x; i < V; i += blockDim.x) {
    const float l = lp[i];
    if (l > m) { s = s * __expf(m - l) + 1.f; m = l; }
    else s += __expf(l - m);
  }
  const float thread_max = m;
  // fixed tree: xor butterfly inside the warp (both lanes of a pair compute the same bits), then the warps in order
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float om = __shfl_xor_sync(0xffffffffu, m, o), os = __shfl_xor_sync(0xffffffffu, s, o);
    const float mm = fmaxf(m, om);
    s = s * __expf(m - mm) + os * __expf(om - mm);
    m = mm;
  }
  if ((threadIdx.x & 31) == 0) { wm[threadIdx.x >> 5] = m; ws[threadIdx.x >> 5] = s; }
  __syncthreads();
  m = wm[0];
  s = ws[0];
  for (int w = 1; w < (int)(blockDim.x >> 5); ++w) {
    const float mm = fmaxf(m, wm[w]);
    s = s * __expf(m - mm) + ws[w] * __expf(wm[w] - mm);
    m = mm;
  }
  const float lse = m + logf(s);
  if (n > 0) {
    float unused;
    const int nc = gather_candidates(lp, V, thread_max, n, cval, cidx, n_cand, false, 0.f, 1.f, &unused);
    if (nc > kSampleCand) {
      // a nearly flat row: the n-th largest key by the radix walk; every element above it (fewer than n) plus the
      // lowest ids equal to it, collected in id order one block-wide chunk at a time
      const uint32_t thr = radix_threshold<false>(lp, V, 0u, (unsigned long long)n, 0.f, 1.f, hist, bcast);
      if (threadIdx.x == 0) *n_cand = 0;
      __syncthreads();
      for (int i = threadIdx.x; i < V; i += blockDim.x) {
        const float l = lp[i];
        if (f32_key(l) > thr) {
          const int at = atomicAdd(n_cand, 1);
          cval[at] = l; cidx[at] = i;
        }
      }
      __syncthreads();
      int have = *n_cand;
      for (int base = 0; base < V && have < n; base += blockDim.x) {
        const int i = base + threadIdx.x;
        const bool eq = i < V && f32_key(lp[i]) == thr;
        const unsigned bal = __ballot_sync(0xffffffffu, eq);
        if ((threadIdx.x & 31) == 0) wc[threadIdx.x >> 5] = __popc(bal);
        __syncthreads();
        int before = 0, tot = 0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) {
          if (w < (int)(threadIdx.x >> 5)) before += wc[w];
          tot += wc[w];
        }
        const int at = have + before + __popc(bal & ((1u << (threadIdx.x & 31)) - 1u));
        if (eq && at < n) { cval[at] = lp[i]; cidx[at] = i; }
        have += tot;
        __syncthreads();
      }
      for (int i = n + threadIdx.x; i < 32; i += blockDim.x) { cval[i] = -INFINITY; cidx[i] = 0x7fffffff; }
      __syncthreads();
      bitonic_desc(cval, cidx, 32);
    }
    if ((int)threadIdx.x < n) { rec->id[threadIdx.x] = cidx[threadIdx.x]; rec->lp[threadIdx.x] = cval[threadIdx.x] - lse; }
    __syncthreads();  // the draw reuses the pool
  }
  return lse;
}

__global__ void __launch_bounds__(1024) sample_kernel(const float* __restrict__ logits, int V, int ldl,
                                                      int* __restrict__ out_tokens, const int* __restrict__ dst_slot,
                                                      int* __restrict__ cur_token, int* __restrict__ pos_inc,
                                                      const int* __restrict__ active, const SampleCtl ctl) {
  pdl_launch_dependents();
  pdl_wait();
  // one 32 KiB pool: the candidate arrays of the fast path, or the kHistCopies histograms of the radix walk
  __shared__ __align__(16) unsigned char pool[kSampleCand * 8];
  static_assert(kSampleCand * 8 >= kHistCopies * 256 * 8, "the histogram copies alias the candidate arrays");
  float* cval = reinterpret_cast<float*>(pool);
  int* cidx = reinterpret_cast<int*>(pool + kSampleCand * 4);
  unsigned long long* hist = reinterpret_cast<unsigned long long*>(pool);
  __shared__ __align__(8) uint32_t bcast[4];
  __shared__ float sb[32];
  __shared__ int si[32];
  __shared__ int n_cand, n_keep_s;
  const int row = blockIdx.x;
  const int slot = dst_slot ? dst_slot[row] : row;
  const float* lp = logits + (size_t)row * ldl;
  const int n_top = ctl.top_logprobs && ctl.lp_out ? ctl.top_logprobs[slot] : -1;
  LogprobRec* rec = n_top >= 0 ? ctl.lp_out + row : nullptr;
  float lse = 0.f;
  if (rec) lse = logprob_record(lp, V, min(min(n_top, kTopLogprobsMax), V), rec, cval, cidx, hist, bcast, &n_cand);
  const float temp = ctl.temperature ? ctl.temperature[slot] : 0.f;
  const bool greedy = !(temp > 0.f);
  const float inv_t = greedy ? 1.f : 1.f / temp;
  uint32_t thr_key = 0u;  // keep everything
  uint64_t seed = 0;
  int counter = 0;
  if (!greedy) {
    seed = ctl.seed ? ctl.seed[slot] : 0ull;
    counter = ctl.counter ? ctl.counter[slot] : 0;
    // row maximum (for the mass scale)
    float mx = -INFINITY;
    for (int i = threadIdx.x; i < V; i += blockDim.x) mx = fmaxf(mx, lp[i]);
    const float thread_max = mx;  // maximum of this thread's strided share (fast top-k path)
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 16));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 8));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 4));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
    if ((threadIdx.x & 31) == 0) sb[threadIdx.x >> 5] = mx;
    __syncthreads();
    mx = sb[0];
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) mx = fmaxf(mx, sb[w]);
    __syncthreads();
    const int k = ctl.top_k ? ctl.top_k[slot] : 0;
    const float p = ctl.top_p ? ctl.top_p[slot] : 1.f;
    bool fast_done = false;
    // k_eff: the cut used to bound the candidate set.  With top-p alone (OpenAI-style requests) the 256 largest
    // thread maxima bound it: the candidates are then the largest elements of the row in order, so if the nucleus
    // p * Z (Z over the WHOLE row) closes inside them it is exact; otherwise the radix walk below takes over.
    const bool p_on = p > 0.f && p < 1.f;
    // (256, not 1024: the 1024-th largest of 1024 thread maxima is the SMALLEST one and admits ~7 % of the row)
    const int k_eff = (k > 0 && k <= 1024 && k < V) ? k : ((k <= 0 || k >= V) && p_on && V > 1024 ? 256 : 0);
    const bool p_only = k_eff > 0 && !(k > 0 && k < V);
    if (k_eff > 0 && blockDim.x == 1024) {
      float zpart;  // top-p alone: mass of the whole row
      const int nc = gather_candidates(lp, V, thread_max, k_eff, cval, cidx, &n_cand, p_only, mx, inv_t, &zpart);
      zpart = warp_sum(zpart);
      if ((threadIdx.x & 31) == 0) sb[threadIdx.x >> 5] = zpart;
      __syncthreads();
      float z_row = 0.f;
      for (int w = 0; w < (int)(blockDim.x >> 5); ++w) z_row += sb[w];
      __syncthreads();
      if (nc <= kSampleCand) {
        if (threadIdx.x == 0) {
          int nk = nc;
          if (!p_only) {
            nk = k;                                                      // nc >= k by construction
            while (nk < nc && cval[nk] == cval[k - 1]) ++nk;             // ties at the cut stay in
          }
          n_keep_s = nk;
        }
        __syncthreads();
        if (p_on) {
          // nucleus edge by a block-wide prefix sum over the sorted candidates: thread t owns `per` consecutive ones,
          // partial sums meet through a warp scan + one shared-memory step (fixed order: reproducible)
          const int nk0 = n_keep_s;
          const int per = (nk0 + (int)blockDim.x - 1) / (int)blockDim.x;  // <= kSampleCand / 1024
          float loc[kSampleCand / 1024];
          float mine = 0.f;
#pragma unroll
          for (int j = 0; j < kSampleCand / 1024; ++j) {
            const int at = threadIdx.x * per + j;
            loc[j] = (j < per && at < nk0) ? __expf((cval[at] - mx) * inv_t) : 0.f;
            mine += loc[j];
          }
          float inc = mine;  // inclusive scan inside the warp
#pragma unroll
          for (int o = 1; o < 32; o <<= 1) {
            const float v = __shfl_up_sync(0xffffffffu, inc, o);
            if ((int)(threadIdx.x & 31) >= o) inc += v;
          }
          __syncthreads();  // sb is free again
          if ((threadIdx.x & 31) == 31) sb[threadIdx.x >> 5] = inc;
          __syncthreads();
          float before = 0.f, total = 0.f;
          for (int w = 0; w < (int)(blockDim.x >> 5); ++w) {
            if (w < (int)(threadIdx.x >> 5)) before += sb[w];
            total += sb[w];
          }
          const float target = p * (p_only ? z_row : total);
          float cum = before + inc - mine;  // mass of everything in front of this thread's share
          __syncthreads();
          if (threadIdx.x == 0) n_keep_s = 0x7fffffff;
          __syncthreads();
#pragma unroll
          for (int j = 0; j < kSampleCand / 1024; ++j) {
            const int at = threadIdx.x * per + j;
            if (j < per && at < nk0) {
              if (cum < target && cum + loc[j] >= target) atomicMin(&n_keep_s, at + 1);
              cum += loc[j];
            }
          }
          __syncthreads();
          if (threadIdx.x == 0) {
            int n = n_keep_s;
            if (n == 0x7fffffff) {
              n = p_only ? -1 : nk0;                                      // top-p alone and the nucleus is wider: radix walk
            } else {
              while (n < nk0 && cval[n] == cval[n - 1]) ++n;              // ties at the nucleus edge stay in
            }
            n_keep_s = n;
          }
          __syncthreads();
        }
        const int nk = n_keep_s;
        if (nk >= 0) {
        float best = -INFINITY;
        int bi = 0x7fffffff;
        for (int j = threadIdx.x; j < nk; j += blockDim.x) {
          const float sc = cval[j] * inv_t + gumbel_noise(seed, counter, cidx[j]);
          if (sc > best || (sc == best && cidx[j] < bi)) { best = sc; bi = cidx[j]; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          const float ob = __shfl_xor_sync(0xffffffffu, best, o);
          const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
          if (ob > best || (ob == best && oi < bi)) { best = ob; bi = oi; }
        }
        if ((threadIdx.x & 31) == 0) { sb[threadIdx.x >> 5] = best; si[threadIdx.x >> 5] = bi; }
        __syncthreads();
        if (threadIdx.x == 0) {
          for (int w = 1; w < (int)(blockDim.x >> 5); ++w)
            if (sb[w] > best || (sb[w] == best && si[w] < bi)) { best = sb[w]; bi = si[w]; }
          out_tokens[row] = bi;
          if (rec) rec->logprob = lp[bi] - lse;
          if (cur_token) cur_token[slot] = bi;
          if (pos_inc && (!active || active[slot])) pos_inc[slot] += 1;
        }
        fast_done = true;
        }
      }
      __syncthreads();
    }
    if (fast_done) return;
    if (k > 0 && k < V) thr_key = radix_threshold<false>(lp, V, 0u, (unsigned long long)k, mx, inv_t, hist, bcast);
    if (p_on) {
      // total mass of what top-k kept, in the same fixed point
      for (int i = threadIdx.x; i < 256; i += blockDim.x) hist[i] = 0ull;
      __syncthreads();
      unsigned long long part = 0ull;
      for (int i = threadIdx.x; i < V; i += blockDim.x) {
        const float l = lp[i];
        if (f32_key(l) >= thr_key) part += (unsigned long long)(kMassScale * __expf((l - mx) * inv_t));
      }
      atomicAdd(&hist[0], part);
      __syncthreads();
      const unsigned long long Z = hist[0];
      __syncthreads();
      unsigned long long target = (unsigned long long)((double)Z * (double)p);
      if (target < 1ull) target = 1ull;
      const uint32_t tp = radix_threshold<true>(lp, V, thr_key, target, mx, inv_t, hist, bcast);
      thr_key = tp > thr_key ? tp : thr_key;
    }
  }
  // ---- the draw (greedy: plain argmax, lowest index wins ties)
  float best = -INFINITY;
  int bi = 0x7fffffff;
  if (greedy) {  // the benchmark path: 16-byte loads, exactly the argmax kernel (V % 4 == 0 is checked at model load)
    const float4* lp4 = reinterpret_cast<const float4*>(lp);
    for (int i = threadIdx.x; i < V / 4; i += blockDim.x) {
      const float4 v = lp4[i];
      const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int idx = i * 4 + e;
        if (vv[e] > best || (vv[e] == best && idx < bi)) { best = vv[e]; bi = idx; }
      }
    }
  } else {
    for (int i = threadIdx.x; i < V; i += blockDim.x) {
      const float l = lp[i];
      if (f32_key(l) < thr_key) continue;
      const float sc = l * inv_t + gumbel_noise(seed, counter, i);
      if (sc > best || (sc == best && i < bi)) { best = sc; bi = i; }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ob = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ob > best || (ob == best && oi < bi)) { best = ob; bi = oi; }
  }
  if ((threadIdx.x & 31) == 0) { sb[threadIdx.x >> 5] = best; si[threadIdx.x >> 5] = bi; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w)
      if (sb[w] > best || (sb[w] == best && si[w] < bi)) { best = sb[w]; bi = si[w]; }
    if (bi == 0x7fffffff) bi = 0;  // (cannot happen: the maximum is always kept)
    out_tokens[row] = bi;
    if (rec) rec->logprob = lp[bi] - lse;
    if (cur_token) cur_token[slot] = bi;
    if (pos_inc && (!active || active[slot])) pos_inc[slot] += 1;
  }
}
void launch_sample(const LaunchCfg& lc, const float* logits, int rows, int V, int ldl, int* out_tokens,
                   const int* dst_slot, int* cur_token, int* pos_inc, const int* active, const SampleCtl& ctl) {
  launch_k(lc, sample_kernel, dim3(rows), dim3(1024), 0, logits, V, ldl, out_tokens, dst_slot, cur_token, pos_inc, active,
           ctl);
}

// ------------------------------------------------------------------------------------------------
// deterministic weight init (counter-based; the oracle restates it in numpy: oracle/weights.py)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}
__global__ void init_normal_kernel(__nv_bfloat16* w, size_t n, uint64_t seed, float std) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const uint64_t r = splitmix64(seed ^ (i * 0xD1342543DE82EF95ull));
    const float u1 = ((float)(uint32_t)(r >> 40) + 0.5f) * (1.0f / 16777216.0f);         // (0,1)
    const float u2 = ((float)(uint32_t)((r >> 16) & 0xFFFFFF)) * (1.0f / 16777216.0f);   // [0,1)
    const float z = sqrtf(-2.0f * __logf(u1)) * __cosf(6.2831853071795864f * u2);
    w[i] = __float2bfloat16(z * std);
  }
}
void launch_init_normal(cudaStream_t st, __nv_bfloat16* w, size_t n, uint64_t seed, float std) {
  init_normal_kernel<<<148 * 8, 256, 0, st>>>(w, n, seed, std);
}
__global__ void fill_bf16_kernel(__nv_bfloat16* w, size_t n, float v) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) w[i] = __float2bfloat16(v);
}
void launch_fill_bf16(cudaStream_t st, __nv_bfloat16* w, size_t n, float v) {
  fill_bf16_kernel<<<148, 256, 0, st>>>(w, n, v);
}


// ------------------------------------------------------------------------------------------------
// BERT-style encoder pieces (/api/embed path, BASELINE configs[4]): embeddings + LayerNorm, residual + bias +
// post-LayerNorm, [CLS] pooling with L2 normalisation.  One CTA per row, H / 4 threads, one float4 per thread.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float block_sum(float v, float* red) {
  v = warp_sum(v);
  __syncthreads();  // red may still be read by the previous reduction
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float tot = 0.f;
  for (int w = 0; w < (int)(blockDim.x + 31) / 32; ++w) tot += red[w];
  return tot;
}
__device__ __forceinline__ float4 ld_bf16x4(const __nv_bfloat16* p) {
  const uint2 a = *reinterpret_cast<const uint2*>(p);
  return make_float4(bf16_lo(a.x), bf16_hi(a.x), bf16_lo(a.y), bf16_hi(a.y));
}
// LayerNorm of the thread-distributed row value v (mean and variance over H), written as fp32 h and bf16 x
__device__ __forceinline__ void ln_store(float4 v, int H, float eps, const __nv_bfloat16* g, const __nv_bfloat16* b,
                                         float* h_row, __nv_bfloat16* x_row, float* red) {
  const int i = threadIdx.x * 4;
  const float mean = block_sum(v.x + v.y + v.z + v.w, red) / (float)H;
  const float4 d = make_float4(v.x - mean, v.y - mean, v.z - mean, v.w - mean);
  const float var = block_sum(d.x * d.x + d.y * d.y + d.z * d.z + d.w * d.w, red) / (float)H;
  const float rstd = rsqrtf(var + eps);
  const float4 gg = ld_bf16x4(g + i), bb = ld_bf16x4(b + i);
  const float4 o = make_float4(d.x * rstd * gg.x + bb.x, d.y * rstd * gg.y + bb.y, d.z * rstd * gg.z + bb.z,
                               d.w * rstd * gg.w + bb.w);
  *reinterpret_cast<float4*>(h_row + i) = o;
  *reinterpret_cast<uint2*>(x_row + i) = pack4_bf16(o.x, o.y, o.z, o.w);
}
__global__ void enc_embed_ln_kernel(const int* __restrict__ tok, const int* __restrict__ pos,
                                    const __nv_bfloat16* __restrict__ word, const __nv_bfloat16* __restrict__ pos_emb,
                                    const __nv_bfloat16* __restrict__ type_emb, const __nv_bfloat16* __restrict__ g,
                                    const __nv_bfloat16* __restrict__ b, float* __restrict__ h,
                                    __nv_bfloat16* __restrict__ x, int H, float eps) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float red[32];
  const int t = blockIdx.x, i = threadIdx.x * 4;
  const float4 a = ld_bf16x4(word + (size_t)tok[t] * H + i), c = ld_bf16x4(pos_emb + (size_t)pos[t] * H + i),
               e = ld_bf16x4(type_emb + i);  // token type 0 everywhere (single-segment inputs)
  ln_store(make_float4(a.x + c.x + e.x, a.y + c.y + e.y, a.z + c.z + e.z, a.w + c.w + e.w), H, eps, g, b,
           h + (size_t)t * H, x + (size_t)t * H, red);
}
void launch_enc_embed_ln(const LaunchCfg& lc, const int* tok, const int* pos, const __nv_bfloat16* word,
                         const __nv_bfloat16* pos_emb, const __nv_bfloat16* type_emb, const __nv_bfloat16* g,
                         const __nv_bfloat16* b, float* h, __nv_bfloat16* x, int T, int H, float eps) {
  launch_k(lc, enc_embed_ln_kernel, dim3(T), dim3(H / 4), 0, tok, pos, word, pos_emb, type_emb, g, b, h, x, H, eps);
}
// h = LayerNorm(h + sub + bias) * g + b   (BertSelfOutput / BertOutput: dense output + residual, post-LN)
__global__ void enc_add_ln_kernel(float* __restrict__ h, const __nv_bfloat16* __restrict__ sub,
                                  const __nv_bfloat16* __restrict__ bias, const __nv_bfloat16* __restrict__ g,
                                  const __nv_bfloat16* __restrict__ b, __nv_bfloat16* __restrict__ x, int H, float eps) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float red[32];
  const int t = blockIdx.x, i = threadIdx.x * 4;
  const float4 r = *reinterpret_cast<const float4*>(h + (size_t)t * H + i), s = ld_bf16x4(sub + (size_t)t * H + i),
               bi = ld_bf16x4(bias + i);
  ln_store(make_float4(r.x + s.x + bi.x, r.y + s.y + bi.y, r.z + s.z + bi.z, r.w + s.w + bi.w), H, eps, g, b,
           h + (size_t)t * H, x + (size_t)t * H, red);
}
void launch_enc_add_ln(const LaunchCfg& lc, float* h, const __nv_bfloat16* sub, const __nv_bfloat16* bias,
                       const __nv_bfloat16* g, const __nv_bfloat16* b, __nv_bfloat16* x, int T, int H, float eps) {
  launch_k(lc, enc_add_ln_kernel, dim3(T), dim3(H / 4), 0, h, sub, bias, g, b, x, H, eps);
}
// Warp-per-token form for hidden sizes that are multiples of 128 (<= 1024): the residual is the previous LayerNorm's
// OUTPUT, which the GEMMs already read as bf16 x - so x is also the residual stream and no fp32 copy is read or written
// (r02: the one-block-per-token kernel above moved 150 MB per call for bge-small at 32 768 tokens and ran at 63 % of
// the HBM rate; this one moves 75 MB, keeps the row in registers and reduces with shuffles only).  `h32` (nullable):
// fp32 copy of the result, written only by the last LayerNorm of the model for the pooling kernel.
template <int NV>  // 4-element vectors per lane: H = 128 * NV
__global__ void __launch_bounds__(256) enc_add_ln_warp_kernel(__nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ sub,
                                                              const __nv_bfloat16* __restrict__ bias,
                                                              const __nv_bfloat16* __restrict__ g,
                                                              const __nv_bfloat16* __restrict__ b, float* __restrict__ h32,
                                                              int T, float eps) {
  pdl_launch_dependents();
  pdl_wait();
  constexpr int H = 128 * NV;
  const int lane = threadIdx.x & 31;
  const int t = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (t >= T) return;
  __nv_bfloat16* xr = x + (size_t)t * H;
  const __nv_bfloat16* sr = sub + (size_t)t * H;
  float4 v[NV];
  float sum = 0.f;
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    const int i = (k * 32 + lane) * 4;
    const float4 r = ld_bf16x4(xr + i), s4 = ld_bf16x4(sr + i), bi = ld_bf16x4(bias + i);
    v[k] = make_float4(r.x + s4.x + bi.x, r.y + s4.y + bi.y, r.z + s4.z + bi.z, r.w + s4.w + bi.w);
    sum += (v[k].x + v[k].y) + (v[k].z + v[k].w);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  const float mean = sum * (1.0f / H);
  float sq = 0.f;
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    v[k] = make_float4(v[k].x - mean, v[k].y - mean, v[k].z - mean, v[k].w - mean);
    sq += (v[k].x * v[k].x + v[k].y * v[k].y) + (v[k].z * v[k].z + v[k].w * v[k].w);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
  const float rstd = rsqrtf(sq * (1.0f / H) + eps);
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    const int i = (k * 32 + lane) * 4;
    const float4 gg = ld_bf16x4(g + i), bb = ld_bf16x4(b + i);
    const float4 o = make_float4(v[k].x * rstd * gg.x + bb.x, v[k].y * rstd * gg.y + bb.y, v[k].z * rstd * gg.z + bb.z,
                                 v[k].w * rstd * gg.w + bb.w);
    *reinterpret_cast<uint2*>(xr + i) = pack4_bf16(o.x, o.y, o.z, o.w);
    if (h32) *reinterpret_cast<float4*>(h32 + (size_t)t * H + i) = o;
  }
}
bool enc_add_ln_warp_supported(int H) { return H % 128 == 0 && H >= 128 && H <= 1024; }
void launch_enc_add_ln_warp(const LaunchCfg& lc, __nv_bfloat16* x, const __nv_bfloat16* sub, const __nv_bfloat16* bias,
                            const __nv_bfloat16* g, const __nv_bfloat16* b, float* h32, int T, int H, float eps) {
  const dim3 grid((T + 7) / 8), block(256);
  switch (H / 128) {
#define MQ_LN_CASE(n) case n: launch_k(lc, enc_add_ln_warp_kernel<n>, grid, block, 0, x, sub, bias, g, b, h32, T, eps); break;
    MQ_LN_CASE(1) MQ_LN_CASE(2) MQ_LN_CASE(3) MQ_LN_CASE(4) MQ_LN_CASE(5) MQ_LN_CASE(6) MQ_LN_CASE(7) MQ_LN_CASE(8)
#undef MQ_LN_CASE
    default: break;
  }
}
// out[s, :] = h[first_tok[s], :] / ||.||_2   ([CLS] pooling + L2 normalisation, the bge recipe)
__global__ void enc_pool_kernel(const float* __restrict__ h, const int* __restrict__ first_tok, float* __restrict__ out,
                                int H) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float red[32];
  const int s = blockIdx.x, i = threadIdx.x * 4;
  const float4 v = *reinterpret_cast<const float4*>(h + (size_t)first_tok[s] * H + i);
  const float n = sqrtf(block_sum(v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w, red));
  const float inv = 1.0f / fmaxf(n, 1e-12f);
  *reinterpret_cast<float4*>(out + (size_t)s * H + i) = make_float4(v.x * inv, v.y * inv, v.z * inv, v.w * inv);
}
void launch_enc_pool(const LaunchCfg& lc, const float* h, const int* first_tok, float* out, int n_seq, int H) {
  launch_k(lc, enc_pool_kernel, dim3(n_seq), dim3(H / 4), 0, h, first_tok, out, H);
}

}  // namespace mq
