// Launch wrappers for the non-GEMM kernels of the forward pass (see kernels.cu for the designs).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include "ptx.cuh"

namespace mq {

constexpr int kPageSize = 16;  // tokens per KV page
constexpr int kMaxSplitPlanes = 8;  // split-K planes a reduce kernel (add_rmsnorm / rope_kv) may have to sum
inline bool head_dim_supported(int d) { return d == 128 || d == 96 || d == 64; }  // Llama-3 / Qwen2.5, Phi-3, small models
// (the rope / attention kernels also have a head_dim 32 instance, used by the BERT encoder path only)

struct LaunchCfg {
  cudaStream_t stream;
  bool pdl;  // launch with programmatic stream serialization
};

// h_f32[t,:] = embed[token_ids[t], :];  with gamma (decode chain): xg[t,:] = bf16(h * gamma), ssq[t] = sum h^2
void launch_embed(const LaunchCfg& lc, const int* token_ids, const __nv_bfloat16* embed, float* h, int T, int H,
                  const __nv_bfloat16* gamma = nullptr, __nv_bfloat16* xg = nullptr, float* ssq = nullptr);

// v = h[src,:] + sum_s partial[s][src,:];  if (!row_idx) h[src,:] = v;  x[row,:] = bf16(v * rsqrt(mean v^2 + eps) * gamma)
// partial_is_f32: planes are fp32 (decode split-K) else one bf16 plane (prefill).
void launch_add_rmsnorm(const LaunchCfg& lc, float* h, const void* partial, bool partial_is_f32, int n_planes,
                        long long plane_stride, const __nv_bfloat16* gamma, __nv_bfloat16* x, const int* row_idx,
                        int rows, int H, float eps, Trace tr = Trace{nullptr, 0});

struct RopeKvParams {
  const void* qkv;        // partial planes [S][T][qkv_dim] fp32, or one bf16 plane
  bool qkv_is_f32;
  int n_planes;
  long long plane_stride;
  const __nv_bfloat16* bias;  // nullable, [qkv_dim]
  const int* pos;             // [T] position of each token
  const int* slot_of_tok;     // [T] sequence slot of each token
  const int* block_table;     // [slots][max_pages]
  int max_pages;
  const float* inv_freq;      // [d/2]
  const float2* rope_table;   // optional [positions][d/2] (cos, sin) of pos * inv_freq: replaces the in-kernel sincosf
  __nv_bfloat16* q_out;       // [T][n_q*d]
  __nv_bfloat16* k_cache;     // layer base: [pages][n_kv][kPageSize][d]
  __nv_bfloat16* v_cache;
  int T, n_q, n_kv;
  int head_dim;               // 128, 96 or 64
  Trace tr;                   // optional timeline stamps (MQ_TRACE=1)
};
void launch_rope_kv(const LaunchCfg& lc, const RopeKvParams& p);
void launch_rope_table(cudaStream_t st, float2* table, const float* inv_freq, int n_pos, int half);

struct AttnParams {
  const __nv_bfloat16* q;        // [T][n_q*d]
  const __nv_bfloat16* k_cache;  // layer base
  const __nv_bfloat16* v_cache;
  const int* block_table;
  int max_pages;
  const int4* tiles;   // prefill: {tok0, ntok, slot, pos0} per q tile
  const int* pos;      // decode: pos[slot] (kv length = pos+1)
  __nv_bfloat16* out;  // [T][n_q*d]
  float* part_o;       // decode split partials [splits][T][n_q][d]
  float* part_ml;      // [splits][T][n_q][2]
  int n_q, n_kv, T;
  int head_dim;        // 128, 96 or 64 (32: encoder)
  int bidirectional;   // prefill only: 1 = no causal mask (encoder self-attention); needs seq_len
  const int* seq_len;  // prefill, bidirectional: [slots] total length of each sequence
  // prefill, packed mode (encoder): q / k / v are column blocks of ONE row-major activation matrix instead of a paged
  // cache - row (seq_start[slot] + position), `row_stride` elements apart; q, k_cache, v_cache point at the blocks
  const int* seq_start;  // [slots] first row of each sequence; nullptr = paged cache
  int row_stride;
  int n_splits;        // decode only: every sequence is cut into n_splits equal 16-aligned ranges (grid-level)
  int n_warps;         // decode only: 1, or 2 / 4 / 8 = in-CTA split over that many warps (then n_splits == 1)
  int stages;          // decode, n_warps == 1: ring depth 2 / 3 / 4 / 6 (0 = default 6); short contexts want MORE resident
                       // CTAs rather than a deep ring (a 6-stage CTA holds 48 KiB: 4 per SM)
  int* split_counter;  // decode only: [slots][n_kv] arrival counters (zero between launches)
  float scale_log2;    // softmax scale * log2(e)
  Trace tr;            // optional timeline stamps (MQ_TRACE=1)
};
void launch_attn_prefill(const LaunchCfg& lc, const AttnParams& p, int n_tiles);
// ---- prefill attention on tcgen05 (attn_tc.cu): head_dim 128, GQA group 1 / 2 / 4 / 8, query tiles of 128 rows
// (= 128 / G tokens x G heads).  Tensor maps: q = the [rows][n_q][128] activation, k / v = one layer of the paged cache.
constexpr int kPrefillTileRowsTc = 128;
bool attn_tc_supported(int head_dim, int n_q, int n_kv);
bool attn_tc_encode_q(CUtensorMap* out, const void* q, int rows, int n_q, int G);
bool attn_tc_encode_kv(CUtensorMap* out, const void* cache, int n_pages, int n_kv);
void attn_tc_set_attrs();
cudaError_t launch_attn_prefill_tc(const LaunchCfg& lc, const CUtensorMap& tmQ, const CUtensorMap& tmK, const CUtensorMap& tmV,
                                   const AttnParams& a, int n_tiles);
// ---- encoder attention on tcgen05 (enc_attn_tc.cu): head_dim 32, bidirectional, sequences <= 512 tokens packed in one
// [rows][3H] activation.  items = {row0, n_rows <= 256, first row of the sequence, its length} per CTA column.
constexpr int kEncAttnItemRows = 256;
bool enc_attn_tc_supported(int head_dim, int max_seq, int hidden);
bool enc_attn_tc_encode(CUtensorMap* out, const void* qkv, int rows, int H);
void enc_attn_tc_set_attrs();
cudaError_t launch_enc_attn_tc(const LaunchCfg& lc, const CUtensorMap& tm, const int4* items, int n_items, int n_heads, int H,
                               __nv_bfloat16* out, float scale_log2);
void launch_attn_decode(const LaunchCfg& lc, const AttnParams& p, int n_slots);
void attn_set_attrs();
int attn_decode_resident_ctas();
constexpr int kMaxDecodeSplits = 8;
constexpr int kPrefillTileRows = 64;  // q rows (token x group-head) per prefill CTA (r01: 128 rows / 8 warps was 20% slower: 1 CTA/SM by registers)

// next[b] = argmax_v logits[b][v]; optional: cur_token[slot]=next, pos[slot]+=1 for active slots
void launch_argmax(const LaunchCfg& lc, const float* logits, int rows, int V, int ldl, int* out_tokens,
                   const int* dst_slot, int* cur_token, int* pos_inc, const int* active);

// ---- encoder (BERT) pieces: H % 128 == 0, H / 4 <= 1024 threads
void launch_enc_embed_ln(const LaunchCfg& lc, const int* tok, const int* pos, const __nv_bfloat16* word,
                         const __nv_bfloat16* pos_emb, const __nv_bfloat16* type_emb, const __nv_bfloat16* g,
                         const __nv_bfloat16* b, float* h, __nv_bfloat16* x, int T, int H, float eps);
void launch_enc_add_ln(const LaunchCfg& lc, float* h, const __nv_bfloat16* sub, const __nv_bfloat16* bias,
                       const __nv_bfloat16* g, const __nv_bfloat16* b, __nv_bfloat16* x, int T, int H, float eps);
// warp-per-token form, bf16 residual stream (x is read as the residual and overwritten); h32 nullable
bool enc_add_ln_warp_supported(int H);
void launch_enc_add_ln_warp(const LaunchCfg& lc, __nv_bfloat16* x, const __nv_bfloat16* sub, const __nv_bfloat16* bias,
                            const __nv_bfloat16* g, const __nv_bfloat16* b, float* h32, int T, int H, float eps);
void launch_enc_pool(const LaunchCfg& lc, const float* h, const int* first_tok, float* out, int n_seq, int H);

// Log-probability record of one drawn token (MQ_TOP_LOGPROBS_MAX alternatives at most).  For the logits row l the token
// was drawn from: logprob(i) = l[i] - lse(l), lse(l) = m + log sum_j exp(l[j] - m), m = max l - the log-softmax of the
// raw logits (temperature 1, before top-k / top-p), whatever the request's sampling settings.  `logprob` is the drawn
// token's; id[0..n) / lp[0..n) are the n most probable tokens, logit descending then id ascending (ties at the cut go
// to the lower id), entries from n on are not written.  Fixed-order reductions: the same row gives the same bits.
constexpr int kTopLogprobsMax = 20;
struct LogprobRec {
  float logprob;
  int id[kTopLogprobsMax];
  float lp[kTopLogprobsMax];
};
static_assert(sizeof(LogprobRec) == 4 + 8 * kTopLogprobsMax, "LogprobRec is the raw-token record layout");

// Per-slot sampling controls (device arrays indexed by slot; a null array = the default): temperature <= 0 -> greedy;
// top_k <= 0 or >= V -> off; top_p <= 0 or >= 1 -> off; counter = position of the token being drawn (RNG stream).
// top_logprobs: -1 (or a null array) -> no record; 0..20 -> row r writes lp_out[r] with that many alternatives.  The
// switch never changes the drawn token.
struct SampleCtl {
  const float* temperature;
  const int* top_k;
  const float* top_p;
  const unsigned long long* seed;
  const int* counter;
  const int* top_logprobs;
  LogprobRec* lp_out;
};
// like launch_argmax, but rows whose slot has temperature > 0 are drawn from softmax(logits / T) restricted by
// top-k / top-p (Gumbel-max with a counter-based generator: no state, reproducible per (seed, position))
void launch_sample(const LaunchCfg& lc, const float* logits, int rows, int V, int ldl, int* out_tokens,
                   const int* dst_slot, int* cur_token, int* pos_inc, const int* active, const SampleCtl& ctl);

// deterministic counter-based N(0, std^2) fill (splitmix64 + Box-Muller), bf16
void launch_init_normal(cudaStream_t st, __nv_bfloat16* w, size_t n, uint64_t seed, float std);
void launch_fill_bf16(cudaStream_t st, __nv_bfloat16* w, size_t n, float v);

}  // namespace mq
