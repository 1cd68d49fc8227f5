// Kernel-level test ABI (SURVEY.md 8b: "plus a kernel-level test ABI, not on the serving path").
// Plain C symbols taking raw DEVICE pointers so tests/ can compare every kernel with a torch reference
// without going through the serving engine.  Nothing here is used by mq_submit().
#include "../../include/ollamamq_b200.h"
#include "gemm_host.cuh"
#include "kernels.cuh"
#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <cmath>
#include <vector>

using namespace mq;

namespace mq {
void set_last_error(const char* fmt, ...);
}

static int check_cuda(const char* what) {
  cudaError_t e = cudaDeviceSynchronize();
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) {
    mq::set_last_error("%s: %s", what, cudaGetErrorString(e));
    return MQ_ERR_CUDA;
  }
  return MQ_OK;
}

template <typename F>
static int timed_launches(const char* what, F&& launch, int reps, float* ms_out) {
  cudaError_t e = launch();
  if (e != cudaSuccess) {
    mq::set_last_error("%s: %s", what, cudaGetErrorString(e));
    return MQ_ERR_CUDA;
  }
  int rc = check_cuda(what);
  if (rc != MQ_OK || reps <= 0 || !ms_out) return rc;
  cudaEvent_t a, b;
  cudaEventCreate(&a);
  cudaEventCreate(&b);
  cudaEventRecord(a, 0);
  for (int i = 0; i < reps; ++i) launch();
  cudaEventRecord(b, 0);
  cudaEventSynchronize(b);
  float ms = 0.f;
  cudaEventElapsedTime(&ms, a, b);
  *ms_out = ms / reps;
  cudaEventDestroy(a);
  cudaEventDestroy(b);
  return check_cuda(what);
}

extern "C" {

int mq_debug_gemm(const void* W, int w_rows, int n_out, int K, const void* X, int x_rows_alloc, int T, int epi,
                  void* out, int ldo, int splits, long long split_stride, int a2_row_off, int pdl, int reps,
                  float* ms_out) {
  GemmPlan g;
  gemm_set_attrs();
  // splits < 0 selects the persistent stream-K kernel (decode tile widths only); the scratch lives for the process
  static StreamKWorkspace sk_ws;
  const bool want_sk = splits < 0;
  if (want_sk && !sk_ws.ws && streamk_workspace_alloc(&sk_ws) != 0) {
    mq::set_last_error("stream-K workspace allocation failed");
    return MQ_ERR_NOMEM;
  }
  if (want_sk) splits = 1;
  sk_ws.force = true;
  if (!gemm_plan(&g, W, w_rows, n_out, K, X, x_rows_alloc, T, epi, out, ldo, splits, split_stride, a2_row_off,
                 want_sk ? &sk_ws : nullptr)) {
    mq::set_last_error("gemm_plan failed (K%%64, splits, or cuTensorMapEncodeTiled)");
    return MQ_ERR_INVAL;
  }
  LaunchCfg lc{0, pdl != 0};
  cudaError_t e = gemm_launch(g, lc);
  if (e != cudaSuccess) {
    mq::set_last_error("gemm_launch: %s", cudaGetErrorString(e));
    return MQ_ERR_CUDA;
  }
  int rc = check_cuda("mq_debug_gemm");
  if (rc != MQ_OK) return rc;
  if (reps > 0 && ms_out) {
    cudaEvent_t a, b;
    cudaEventCreate(&a);
    cudaEventCreate(&b);
    cudaEventRecord(a, 0);
    for (int i = 0; i < reps; ++i) gemm_launch(g, lc);
    cudaEventRecord(b, 0);
    cudaEventSynchronize(b);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, a, b);
    *ms_out = ms / reps;
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    return check_cuda("mq_debug_gemm(timed)");
  }
  return MQ_OK;
}

int mq_debug_embed(const int* token_ids, const void* embed, float* h, int T, int H) {
  launch_embed(LaunchCfg{0, false}, token_ids, (const __nv_bfloat16*)embed, h, T, H);
  return check_cuda("mq_debug_embed");
}

int mq_debug_embed_chain(const int* token_ids, const void* embed, float* h, int T, int H, const void* gamma, void* xg,
                         float* ssq) {
  launch_embed(LaunchCfg{0, false}, token_ids, (const __nv_bfloat16*)embed, h, T, H, (const __nv_bfloat16*)gamma,
               (__nv_bfloat16*)xg, ssq);
  return check_cuda("mq_debug_embed_chain");
}

int mq_debug_cluster_info(int* out8) {
  if (!out8) return MQ_ERR_INVAL;
  gemm_set_attrs();
  for (int c = 1; c <= 8; ++c) out8[c - 1] = dk_max_clusters(c);
  return MQ_OK;
}

int mq_debug_gemm_fold(const void* W, int w_rows, int n_out, int K, const void* X, int x_rows_alloc, int T, int epi,
                       void* out, int ldo, int a2_row_off, int tile_rows, int streamk, const float* ssq, int parts,
                       int stride, float inv_h, float eps, int reps, float* ms_out) {
  GemmPlan g;
  gemm_set_attrs();
  static StreamKWorkspace sk_ws;
  if (streamk && !sk_ws.ws && streamk_workspace_alloc(&sk_ws) != 0) {
    mq::set_last_error("stream-K workspace allocation failed");
    return MQ_ERR_NOMEM;
  }
  sk_ws.force = true;
  if (tile_rows < 0) tile_rows = gemm_balanced_rows(n_out);
  if (!gemm_plan(&g, W, w_rows, n_out, K, X, x_rows_alloc, T, epi, out, ldo, 1, 0, a2_row_off, streamk ? &sk_ws : nullptr,
                 tile_rows)) {
    mq::set_last_error("gemm_plan failed");
    return MQ_ERR_INVAL;
  }
  gemm_plan_set_rstd(&g, RstdIn{ssq, parts, stride, inv_h, eps});
  LaunchCfg lc{0, false};
  return timed_launches("mq_debug_gemm_fold", [&] { return gemm_launch(g, lc); }, reps, ms_out);
}

int mq_debug_gemm_resid_prefill(const void* W, int n_out, int K, const void* X, int x_rows_alloc, int T, float* h,
                                const void* gamma_next, void* xg, float* ssq_out, int ssq_stride, const float* ssq_in, int parts,
                                int stride_in, float inv_h, float eps, int reps, float* ms_out) {
  GemmPlan g;
  gemm_set_attrs();
  if (!gemm_plan(&g, W, n_out, n_out, K, X, x_rows_alloc, T, EPI_RESID, h, n_out, 1, 0, 0, nullptr) ||
      !gemm_plan_set_resid(&g, gamma_next, xg, n_out, ssq_out, ssq_stride)) {
    mq::set_last_error("EPI_RESID needs the 2-CTA kernel: T > 128, n_out %% 256 == 0, K %% 64 == 0");
    return MQ_ERR_INVAL;
  }
  if (ssq_in) gemm_plan_set_rstd(&g, RstdIn{ssq_in, parts, stride_in, inv_h, eps});
  LaunchCfg lc{0, false};
  return timed_launches("mq_debug_gemm_resid_prefill", [&] { return gemm_launch(g, lc); }, reps, ms_out);
}

int mq_debug_gemm_dk_resid(const void* W, int n_out, int K, const void* X, int x_rows_alloc, int T, int cs, float* h,
                           const void* gamma_next, void* xg, float* ssq_out, int ssq_stride, int reps, float* ms_out) {
  DkPlan g;
  gemm_set_attrs();
  if (!dk_plan(&g, W, n_out, n_out, K, X, x_rows_alloc, T, 128, cs)) {
    mq::set_last_error("dk_plan failed (T > 64, K %% 64, cluster size / tokens per rank)");
    return MQ_ERR_INVAL;
  }
  g.p.h = h; g.p.ldh = n_out; g.p.gamma_next = (const __nv_bfloat16*)gamma_next; g.p.xg = (__nv_bfloat16*)xg;
  g.p.ldx = n_out; g.p.ssq_out = ssq_out; g.p.ssq_stride = ssq_stride;
  LaunchCfg lc{0, false};
  unsigned long long* dbg = nullptr;
  if (getenv("MQ_DK_DBG")) { cudaMalloc((void**)&dbg, 16 * 8); cudaMemset(dbg, 0, 16 * 8); g.p.dbg = dbg; }
  const int rc = timed_launches("mq_debug_gemm_dk_resid", [&] { return dk_launch(g, lc); }, reps, ms_out);
  if (dbg) {
    unsigned long long hst[16];
    cudaMemcpy(hst, dbg, sizeof hst, cudaMemcpyDeviceToHost);
    const char* nm[14] = {"epi entry", "epi waited", "phase0 done", "tmem full", "copies issued", "recv+bar", "finalize done", "", "producer done", "mma committed", "tok loop done", "bar2", "cpasync waited", "recv waited"};
    fprintf(stderr, "[dk dbg] T=%d n_out=%d K=%d cs=%d bn=%d:", T, n_out, K, g.cs, g.bn);
    for (int i = 0; i < 14; ++i) if (hst[i]) fprintf(stderr, " %s +%.2fus;", nm[i], (double)((long long)hst[i] - (long long)hst[0]) / 1e3);
    fprintf(stderr, "\n");
    cudaFree(dbg);
  }
  return rc;
}

// Encoder GEMM epilogues (EPI_BIAS_BF16 = 4, EPI_GELU_BF16 = 3): out[t][f] = act(sum_k X[t][k] W[f][k] + bias[f]); T > 128
// takes the persistent 2-CTA kernel with the staged epilogue, smaller T the one-tile-per-CTA kernel.
int mq_debug_gemm_bias(const void* W, int n_out, int K, const void* X, int x_rows_alloc, int T, int epi, const void* bias,
                       void* out, int ldo) {
  if (epi != EPI_BIAS_BF16 && epi != EPI_GELU_BF16) { mq::set_last_error("mq_debug_gemm_bias: epi must be 3 or 4"); return MQ_ERR_INVAL; }
  GemmPlan g;
  gemm_set_attrs();
  if (!gemm_plan(&g, W, n_out, n_out, K, X, x_rows_alloc, T, epi, out, ldo, 1, 0, 0)) {
    mq::set_last_error("mq_debug_gemm_bias: unsupported shape");
    return MQ_ERR_INVAL;
  }
  gemm_plan_set_bias(&g, bias);
  const LaunchCfg lc{0, false};
  if (gemm_launch(g, lc) != cudaSuccess) { mq::set_last_error("mq_debug_gemm_bias: launch failed"); return MQ_ERR_CUDA; }
  return check_cuda("mq_debug_gemm_bias");
}

// x = LayerNorm(x + X W^T + bias) * gamma + beta in one kernel (gemm_rowln.cuh): x = device bf16 [T][n_out] residual in /
// result out, n_out in {256, 384}; h32 (nullable) = fp32 copy of the result.
int mq_debug_gemm_rowln(const void* W, int n_out, int K, const void* X, int x_rows_alloc, int T, void* x, const void* bias,
                        const void* gamma, const void* beta, float eps, float* h32) {
  gemm_set_attrs();
  RowLnPlan g;
  if (!rowln_plan(&g, W, n_out, K, X, x_rows_alloc, T, x, bias, gamma, beta, eps, h32)) {
    mq::set_last_error("mq_debug_gemm_rowln: unsupported shape (n_out in {256, 384}, K %% 64 == 0)");
    return MQ_ERR_INVAL;
  }
  const LaunchCfg lc{0, false};
  if (rowln_launch(g, lc) != cudaSuccess) { mq::set_last_error("mq_debug_gemm_rowln: launch failed"); return MQ_ERR_CUDA; }
  return check_cuda("mq_debug_gemm_rowln");
}

// Encoder attention on tcgen05 (enc_attn_tc.cu): qkv = [rows_alloc][3H] bf16 (q | k | v column blocks), sequences packed
// back to back: sequence s = rows seq_first[s] .. + seq_len[s] (host arrays); out = [rows][H] bf16.  head_dim = H / n_heads = 32.
int mq_debug_enc_attn(const void* qkv, int rows_alloc, int H, int n_heads, const int* seq_first, const int* seq_len, int n_seq,
                      void* out) {
  if (n_heads < 1 || H % n_heads != 0 || !enc_attn_tc_supported(H / n_heads, 512, H)) {
    mq::set_last_error("mq_debug_enc_attn: needs head_dim 32");
    return MQ_ERR_INVAL;
  }
  std::vector<int> items;
  for (int s = 0; s < n_seq; ++s) {
    if (seq_len[s] < 1 || seq_len[s] > 512) { mq::set_last_error("mq_debug_enc_attn: sequence length must be 1..512"); return MQ_ERR_INVAL; }
    for (int i = 0; i < seq_len[s]; i += kEncAttnItemRows) {
      items.push_back(seq_first[s] + i);
      items.push_back(std::min(kEncAttnItemRows, seq_len[s] - i));
      items.push_back(seq_first[s]);
      items.push_back(seq_len[s]);
    }
  }
  int4* d_items = nullptr;
  if (cudaMalloc(&d_items, items.size() * sizeof(int)) != cudaSuccess) return MQ_ERR_NOMEM;
  cudaMemcpy(d_items, items.data(), items.size() * sizeof(int), cudaMemcpyHostToDevice);
  CUtensorMap tm;
  int rc = MQ_OK;
  if (!enc_attn_tc_encode(&tm, qkv, rows_alloc, H)) { mq::set_last_error("mq_debug_enc_attn: tensor map"); rc = MQ_ERR_CUDA; }
  if (rc == MQ_OK) {
    enc_attn_tc_set_attrs();
    const LaunchCfg lc{0, false};
    const float scale_log2 = (1.0f / sqrtf((float)(H / n_heads))) * 1.4426950408889634f;
    if (launch_enc_attn_tc(lc, tm, d_items, (int)items.size() / 4, n_heads, H, (__nv_bfloat16*)out, scale_log2) != cudaSuccess) {
      mq::set_last_error("mq_debug_enc_attn: launch failed");
      rc = MQ_ERR_CUDA;
    } else {
      rc = check_cuda("mq_debug_enc_attn");
    }
  }
  cudaFree(d_items);
  return rc;
}

int mq_debug_add_rmsnorm(float* h, const void* partial, int partial_is_f32, int n_planes, long long plane_stride,
                         const void* gamma, void* x, const int* row_idx, int rows, int H, float eps) {
  if (H % 512 != 0) {
    mq::set_last_error("H must be a multiple of 512");
    return MQ_ERR_INVAL;
  }
  if (n_planes < 0 || n_planes > kMaxSplitPlanes) {
    mq::set_last_error("n_planes must be 0..%d", kMaxSplitPlanes);
    return MQ_ERR_INVAL;
  }
  launch_add_rmsnorm(LaunchCfg{0, false}, h, partial, partial_is_f32 != 0, n_planes, plane_stride,
                     (const __nv_bfloat16*)gamma, (__nv_bfloat16*)x, row_idx, rows, H, eps);
  return check_cuda("mq_debug_add_rmsnorm");
}

int mq_debug_rope_kv(const void* qkv, int qkv_is_f32, int n_planes, long long plane_stride, const void* bias,
                     const int* pos, const int* slot_of_tok, const int* block_table, int max_pages,
                     const float* inv_freq, void* q_out, void* k_cache, void* v_cache, int T, int n_q, int n_kv,
                     int head_dim) {
  if (!head_dim_supported(head_dim)) { mq::set_last_error("head_dim must be 128, 96 or 64"); return MQ_ERR_INVAL; }
  if (n_planes < 1 || n_planes > kMaxSplitPlanes) {
    mq::set_last_error("n_planes must be 1..%d", kMaxSplitPlanes);
    return MQ_ERR_INVAL;
  }
  RopeKvParams p = {};
  p.qkv = qkv; p.qkv_is_f32 = qkv_is_f32 != 0; p.n_planes = n_planes; p.plane_stride = plane_stride;
  p.bias = (const __nv_bfloat16*)bias; p.pos = pos; p.slot_of_tok = slot_of_tok; p.block_table = block_table;
  p.max_pages = max_pages; p.inv_freq = inv_freq; p.q_out = (__nv_bfloat16*)q_out;
  p.k_cache = (__nv_bfloat16*)k_cache; p.v_cache = (__nv_bfloat16*)v_cache; p.T = T; p.n_q = n_q; p.n_kv = n_kv;
  p.head_dim = head_dim;
  launch_rope_kv(LaunchCfg{0, false}, p);
  return check_cuda("mq_debug_rope_kv");
}

int mq_debug_attn_prefill(const void* q, const void* k_cache, const void* v_cache, const int* block_table,
                          int max_pages, const int* tiles /* int4 per tile */, int n_tiles, void* out, int n_q,
                          int n_kv, int T, float scale, int head_dim) {
  if (!head_dim_supported(head_dim)) { mq::set_last_error("head_dim must be 128, 96 or 64"); return MQ_ERR_INVAL; }
  AttnParams p = {};
  p.head_dim = head_dim;
  p.q = (const __nv_bfloat16*)q; p.k_cache = (const __nv_bfloat16*)k_cache; p.v_cache = (const __nv_bfloat16*)v_cache;
  p.block_table = block_table; p.max_pages = max_pages; p.tiles = (const int4*)tiles; p.out = (__nv_bfloat16*)out;
  p.n_q = n_q; p.n_kv = n_kv; p.T = T; p.n_splits = 1;
  p.scale_log2 = scale * 1.4426950408889634f;
  attn_set_attrs();
  launch_attn_prefill(LaunchCfg{0, false}, p, n_tiles);
  return check_cuda("mq_debug_attn_prefill");
}

int mq_debug_attn_prefill_tc(const void* q, int q_rows, const void* k_cache, const void* v_cache, int n_pages, const int* block_table,
                             int max_pages, const int* tiles /* int4 per tile, <= 128 / G tokens each */, int n_tiles, void* out,
                             int n_q, int n_kv, float scale) {
  if (!attn_tc_supported(128, n_q, n_kv)) { mq::set_last_error("tcgen05 attention: head_dim 128, GQA group 1 / 2 / 4 / 8"); return MQ_ERR_INVAL; }
  CUtensorMap tq, tk, tv;
  if (!attn_tc_encode_q(&tq, q, q_rows, n_q, n_q / n_kv) || !attn_tc_encode_kv(&tk, k_cache, n_pages, n_kv) ||
      !attn_tc_encode_kv(&tv, v_cache, n_pages, n_kv)) {
    mq::set_last_error("cuTensorMapEncodeTiled failed");
    return MQ_ERR_CUDA;
  }
  AttnParams p = {};
  p.head_dim = 128;
  p.block_table = block_table; p.max_pages = max_pages; p.tiles = (const int4*)tiles; p.out = (__nv_bfloat16*)out;
  p.n_q = n_q; p.n_kv = n_kv; p.scale_log2 = scale * 1.4426950408889634f;
  attn_tc_set_attrs();
  cudaError_t e = launch_attn_prefill_tc(LaunchCfg{0, false}, tq, tk, tv, p, n_tiles);
  if (e != cudaSuccess) { mq::set_last_error("launch: %s", cudaGetErrorString(e)); return MQ_ERR_CUDA; }
  return check_cuda("mq_debug_attn_prefill_tc");
}

int mq_debug_attn_decode(const void* q, const void* k_cache, const void* v_cache, const int* block_table,
                         int max_pages, const int* pos, void* out, float* part_o, float* part_ml, int* split_counter,
                         int n_q, int n_kv, int n_slots, int n_splits, float scale, int head_dim) {
  if (!head_dim_supported(head_dim)) { mq::set_last_error("head_dim must be 128, 96 or 64"); return MQ_ERR_INVAL; }
  AttnParams p = {};
  p.head_dim = head_dim;
  p.q = (const __nv_bfloat16*)q; p.k_cache = (const __nv_bfloat16*)k_cache; p.v_cache = (const __nv_bfloat16*)v_cache;
  p.block_table = block_table; p.max_pages = max_pages; p.pos = pos; p.out = (__nv_bfloat16*)out;
  p.part_o = part_o; p.part_ml = part_ml; p.split_counter = split_counter; p.n_q = n_q; p.n_kv = n_kv; p.T = n_slots;
  if (n_splits < 0) {  // -2 / -4 / -8: in-CTA split over that many warps
    if (n_splits != -2 && n_splits != -4 && n_splits != -8) { mq::set_last_error("n_splits: 1..8, or -2 / -4 / -8"); return MQ_ERR_INVAL; }
    p.n_warps = -n_splits; n_splits = 1;
  } else {
    p.n_warps = 1;
  }
  p.n_splits = n_splits; p.scale_log2 = scale * 1.4426950408889634f;
  attn_set_attrs();
  launch_attn_decode(LaunchCfg{0, false}, p, n_slots);
  return check_cuda("mq_debug_attn_decode");
}

int mq_debug_sample(const float* logits, int rows, int V, int ldl, int* out_tokens, const float* temperature,
                    const int* top_k, const float* top_p, const unsigned long long* seed, const int* counter) {
  SampleCtl ctl{temperature, top_k, top_p, seed, counter};
  launch_sample(LaunchCfg{0, false}, logits, rows, V, ldl, out_tokens, nullptr, nullptr, nullptr, nullptr, ctl);
  return check_cuda("mq_debug_sample");
}

int mq_debug_sample_logprobs(const float* logits, int rows, int V, int ldl, int* out_tokens, const float* temperature,
                             const int* top_k, const float* top_p, const unsigned long long* seed, const int* counter,
                             const int* top_logprobs, void* lp_out) {
  SampleCtl ctl{temperature, top_k, top_p, seed, counter, top_logprobs, (LogprobRec*)lp_out};
  launch_sample(LaunchCfg{0, false}, logits, rows, V, ldl, out_tokens, nullptr, nullptr, nullptr, nullptr, ctl);
  return check_cuda("mq_debug_sample_logprobs");
}

int mq_debug_argmax(const float* logits, int rows, int V, int ldl, int* out_tokens, const int* dst_slot,
                    int* cur_token, int* pos_inc, const int* active) {
  launch_argmax(LaunchCfg{0, false}, logits, rows, V, ldl, out_tokens, dst_slot, cur_token, pos_inc, active);
  return check_cuda("mq_debug_argmax");
}

int mq_debug_init_normal(void* w, unsigned long long n, unsigned long long seed, float std) {
  launch_init_normal(0, (__nv_bfloat16*)w, (size_t)n, seed, std);
  return check_cuda("mq_debug_init_normal");
}

}  // extern "C"
