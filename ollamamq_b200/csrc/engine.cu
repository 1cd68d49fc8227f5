// GPU worker runtime (see engine.hpp).  Reference seam: /root/reference/src/dispatcher.rs:287-312.
#include "engine.hpp"
#include "framing.hpp"
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>

namespace mq {
void set_last_error(const char* fmt, ...);

constexpr int kRing = 16;        // output-token ring (decode steps / prefill passes in flight)
constexpr int kStageSlots = 32;  // metadata staging ring
constexpr int kMaxFlightsDecode = 4;
constexpr int kMaxFlightsPrefill = 2;

#define CUDA_TRY(expr)                                                                   \
  do {                                                                                   \
    cudaError_t _e = (expr);                                                             \
    if (_e != cudaSuccess) {                                                             \
      set_last_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return MQ_ERR_CUDA;                                                                \
    }                                                                                    \
  } while (0)

static int round_up(int a, int b) { return (a + b - 1) / b * b; }

// ------------------------------------------------------------------------------------------------
// allocation / weights
// ------------------------------------------------------------------------------------------------
int Allocations::alloc(void** p, size_t bytes, bool pinned_host) {
  void* q = nullptr;
  const cudaError_t e = pinned_host ? cudaMallocHost(&q, bytes) : cudaMalloc(&q, bytes);
  if (e != cudaSuccess) {
    set_last_error("%s(%zu bytes): %s", pinned_host ? "cudaMallocHost" : "cudaMalloc", bytes, cudaGetErrorString(e));
    return MQ_ERR_NOMEM;
  }
  (pinned_host ? host_ptrs : dev_ptrs).push_back(q);
  *p = q;
  return MQ_OK;
}

void Allocations::free_all() {
  for (void* p : dev_ptrs) cudaFree(p);
  for (void* p : host_ptrs) cudaFreeHost(p);
  dev_ptrs.clear();
  host_ptrs.clear();
}

static int add_tensor(mq_worker* w, const std::string& name, size_t n_elems, __nv_bfloat16** out) {
  int rc = w->allocs.dev(out, n_elems);
  if (rc) return rc;
  w->tensors[name] = DevTensor{*out, n_elems * 2};
  return MQ_OK;
}

// points views[0..] at consecutive sections of n entries each, starting at `at`; returns the end of the last section
template <typename... T>
static uint8_t* carve(uint8_t* at, size_t n, T**... views) {
  ((*views = reinterpret_cast<T*>(at), at += n * sizeof(T)), ...);
  return at;
}

// a slot's sampling entry in the slot table's host mirror
static void set_slot_sampling(mq_worker* w, int s, const SamplingParams& p) {
  w->h_temp[s] = p.temperature;
  w->h_topk[s] = p.top_k;
  w->h_topp[s] = p.top_p;
  w->h_seed[s] = p.seed;
  w->h_lp_top[s] = p.top_logprobs;
}

static int decode_splits(int m_tiles, int k_blocks) {
  int s = std::min(148 / m_tiles, kMaxSplitPlanes);  // the reduce kernels sum at most kMaxSplitPlanes planes
  if (s < 1) s = 1;
  while (s > 1 && (k_blocks + s - 1) / s < 8) --s;       // keep >= 8 k-blocks (32 KiB of weights per row tile)
  while (s > 1 && (s - 1) * ((k_blocks + s - 1) / s) >= k_blocks) --s;  // every split non-empty
  return s;
}

static int worker_alloc(mq_worker* w) {
  const mq_model_cfg& c = w->cfg;
  const int H = c.hidden, I = c.ffn, V = c.vocab, L = c.n_layers, D = c.head_dim;
  w->qkv_dim = (c.n_q_heads + 2 * c.n_kv_heads) * D;
  w->MB = c.max_batch;
  w->MT = std::max(c.max_prefill_tokens, c.max_batch);
  w->max_pages = (c.max_seq + kPageSize - 1) / kPageSize;
  w->n_pages = c.kv_pages > 0 ? c.kv_pages : w->MB * w->max_pages + 1;
  int rc;
  if ((rc = add_tensor(w, "embed", (size_t)V * H, &w->embed))) return rc;
  if ((rc = add_tensor(w, "final_norm", H, &w->final_norm))) return rc;
  if ((rc = add_tensor(w, "lm_head", (size_t)V * H, &w->lm_head))) return rc;
  w->layers.resize(L);
  for (int l = 0; l < L; ++l) {
    const std::string p = "layers." + std::to_string(l) + ".";
    LayerWeights& lw = w->layers[l];
    if ((rc = add_tensor(w, p + "attn_norm", H, &lw.attn_norm))) return rc;
    if ((rc = add_tensor(w, p + "wqkv", (size_t)w->qkv_dim * H, &lw.wqkv))) return rc;
    lw.bqkv = nullptr;
    if (c.qkv_bias && (rc = add_tensor(w, p + "bqkv", w->qkv_dim, &lw.bqkv))) return rc;
    if ((rc = add_tensor(w, p + "wo", (size_t)H * c.n_q_heads * D, &lw.wo))) return rc;
    if ((rc = add_tensor(w, p + "mlp_norm", H, &lw.mlp_norm))) return rc;
    if ((rc = add_tensor(w, p + "w_gate_up", (size_t)2 * I * H, &lw.w_gate_up))) return rc;
    if ((rc = add_tensor(w, p + "w_down", (size_t)H * I, &lw.w_down))) return rc;
  }
  // algorithmic bytes (SURVEY 8d): matmul weights incl. LM head, excl. embedding table
  const double p_mm = (double)L * ((double)w->qkv_dim * H + (double)H * c.n_q_heads * D + 3.0 * I * H) + (double)V * H;
  w->p_mm_bytes = 2.0 * p_mm;
  w->kv_bytes_per_tok = 2.0 * L * c.n_kv_heads * D * 2.0;

  w->cache_layer_stride = (size_t)w->n_pages * c.n_kv_heads * kPageSize * D;
  Allocations& m = w->allocs;
  if ((rc = m.dev(&w->k_cache, w->cache_layer_stride * L))) return rc;
  if ((rc = m.dev(&w->v_cache, w->cache_layer_stride * L))) return rc;
  cudaMemsetAsync(w->k_cache, 0, w->cache_layer_stride * L * 2, w->stream);
  cudaMemsetAsync(w->v_cache, 0, w->cache_layer_stride * L * 2, w->stream);

  const int MT = w->MT, MB = w->MB;
  const int qd = c.n_q_heads * D;
  // split-K plane counts for decode (fixed per model shape)
  const int kbH = H / 64, kbI = I / 64, kbQ = qd / 64;
  const int s_qkv = decode_splits((w->qkv_dim + 127) / 128, kbH);
  const int s_o = decode_splits((H + 127) / 128, kbQ);
  const int s_d = decode_splits((H + 127) / 128, kbI);
  const int MBp = round_up(MB, 16);
  if ((rc = m.dev(&w->h, (size_t)MT * H))) return rc;
  if ((rc = m.dev(&w->x, (size_t)MT * H))) return rc;
  if ((rc = m.dev(&w->q, (size_t)MT * qd))) return rc;
  if ((rc = m.dev(&w->attn, (size_t)MT * qd))) return rc;
  if ((rc = m.dev(&w->act, (size_t)MT * I))) return rc;
  if ((rc = m.dev(&w->x_last, (size_t)MBp * H))) return rc;
  const size_t qkv_bytes = std::max((size_t)MT * w->qkv_dim * 2, (size_t)s_qkv * MBp * w->qkv_dim * 4);
  const size_t proj_bytes = std::max((size_t)MT * H * 2, (size_t)std::max(s_o, s_d) * MBp * H * 4);
  uint8_t* tmp;
  if ((rc = m.dev(&tmp, qkv_bytes))) return rc;
  w->qkv_part = tmp;
  if ((rc = m.dev(&tmp, proj_bytes))) return rc;
  w->proj_part = tmp;
  if ((rc = m.dev(&w->logits, (size_t)MBp * V))) return rc;
  if ((rc = m.dev(&w->part_o, (size_t)kMaxDecodeSplits * MBp * c.n_q_heads * D))) return rc;
  if ((rc = m.dev(&w->part_ml, (size_t)kMaxDecodeSplits * MBp * c.n_q_heads * 2))) return rc;
  {
    const size_t tiles_h = (size_t)(H + 127) / 128;
    w->ssq_stride = round_up(std::max(MT, MBp), 16);
    const size_t st = (size_t)w->ssq_stride;
    if ((rc = m.dev(&w->ssq_e, st)) || (rc = m.dev(&w->ssq_o, tiles_h * st)) || (rc = m.dev(&w->ssq_d, tiles_h * st)))
      return rc;
    const char* e = getenv("MQ_DECODE_CHAIN");
    w->chain = !(e && e[0] == '0');
    // MQ_TRACE=1: per-launch %globaltimer stamps of the most recent pass (tools/decode_timeline.py)
    const char* e3 = getenv("MQ_TRACE");
    if (e3 && e3[0] == '1') {
      if (8 * c.n_layers + 1 > kTraceSlots - 2) {
        set_last_error("MQ_TRACE: more launches per pass than trace slots");
        return MQ_ERR_INVAL;
      }
      if ((rc = m.dev(&w->d_trace, (size_t)kTraceSlots * 4))) return rc;
      CUDA_TRY(cudaMemsetAsync(w->d_trace, 0xFF, (size_t)kTraceSlots * 4 * 8, w->stream));
    }
  }
  if ((rc = m.dev(&w->d_split_counter, (size_t)MBp * c.n_kv_heads))) return rc;
  CUDA_TRY(cudaMemsetAsync(w->d_split_counter, 0, (size_t)MBp * c.n_kv_heads * 4, w->stream));
  if ((rc = m.dev(&w->inv_freq, D / 2))) return rc;
  if ((rc = m.dev(&w->d_tok, MT))) return rc;
  if ((rc = m.dev(&w->d_pos_tok, MT))) return rc;
  if ((rc = m.dev(&w->d_slot_tok, MT))) return rc;
  if ((rc = m.dev(&w->d_last_idx, MBp))) return rc;
  if ((rc = m.dev(&w->d_dst_slot, MBp))) return rc;
  if ((rc = m.dev(&w->d_tiles, MT + MB))) return rc;
  if ((rc = m.dev(&w->d_cur_token, MBp))) return rc;
  CUDA_TRY(cudaMemsetAsync(w->d_cur_token, 0, MBp * 4, w->stream));
  if ((rc = m.dev(&w->d_identity, MBp))) return rc;
  if ((rc = m.dev(&w->d_out_ring, (size_t)kRing * MBp)) || (rc = m.dev(&w->d_lp_ring, (size_t)kRing * MBp))) return rc;
  if ((rc = m.host(&w->h_out_ring, (size_t)kRing * MBp)) || (rc = m.host(&w->h_lp_ring, (size_t)kRing * MBp))) return rc;

  // slot table (MBp % 16 == 0 keeps every section 64-byte aligned); every slot starts idle on scratch page 0
  w->slot_bytes = (size_t)MBp * (6 * 4 + 8 + (size_t)w->max_pages * 4);
  if ((rc = m.dev(&w->d_slots, w->slot_bytes)) || (rc = m.host(&w->h_slots, w->slot_bytes))) return rc;
  carve(carve(w->h_slots, MBp, &w->h_pos, &w->h_active, &w->h_temp, &w->h_topk, &w->h_topp, &w->h_seed, &w->h_lp_top),
        (size_t)MBp * w->max_pages, &w->h_block_table);
  carve(carve(w->d_slots, MBp, &w->d_pos, &w->d_active, &w->d_temp, &w->d_topk, &w->d_topp, &w->d_seed, &w->d_lp_top),
        (size_t)MBp * w->max_pages, &w->d_block_table);
  memset(w->h_slots, 0, w->slot_bytes);
  for (int s = 0; s < MBp; ++s) set_slot_sampling(w, s, SamplingParams{});
  CUDA_TRY(cudaMemcpyAsync(w->d_slots, w->h_slots, w->slot_bytes, cudaMemcpyHostToDevice, w->stream));
  // one staging area holds either a prefill pass's token metadata (launch_prefill) or a copy of the slot table
  w->stage_ints = std::max((size_t)3 * MT + 4 * (size_t)(MT + MB) + 2 * (size_t)MBp, w->slot_bytes / 4);
  if ((rc = m.host(&w->h_stage, w->stage_ints * kStageSlots))) return rc;
  w->stage_ev.resize(kStageSlots);
  for (auto& e : w->stage_ev) CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));

  std::vector<int> ident(MBp);
  for (int i = 0; i < MBp; ++i) ident[i] = i;
  CUDA_TRY(cudaMemcpyAsync(w->d_identity, ident.data(), MBp * 4, cudaMemcpyHostToDevice, w->stream));
  std::vector<float> invf(D / 2);
  for (int i = 0; i < D / 2; ++i)  // HF: 1.0 / (base ** (arange(0, dim, 2).float() / dim)), fp32
    invf[i] = 1.0f / powf(c.rope_theta, (float)(2 * i) / (float)D);
  CUDA_TRY(cudaMemcpyAsync(w->inv_freq, invf.data(), D / 2 * 4, cudaMemcpyHostToDevice, w->stream));
  // (cos, sin) of every (position, frequency): computed once by the GPU's own sincosf so the rope kernel and the fused
  // decode attention read exactly the values the table-less kernel would compute
  {
    const size_t n_pos = (size_t)w->max_pages * kPageSize;
    if ((rc = m.dev(&w->rope_table, n_pos * (D / 2)))) return rc;
    launch_rope_table(w->stream, w->rope_table, w->inv_freq, (int)n_pos, D / 2);
  }
  CUDA_TRY(cudaStreamSynchronize(w->stream));

  {
    const char* e = getenv("MQ_ATTN_TC");
    w->attn_tc = attn_tc_supported(D, c.n_q_heads, c.n_kv_heads) && !(e && e[0] == '0');
    if (w->attn_tc) {
      const int G = c.n_q_heads / c.n_kv_heads;
      w->tm_k.resize(L); w->tm_v.resize(L);
      bool ok = attn_tc_encode_q(&w->tm_q, w->q, MT, c.n_q_heads, G);
      for (int l = 0; l < L && ok; ++l)
        ok = attn_tc_encode_kv(&w->tm_k[l], w->k_cache + (size_t)l * w->cache_layer_stride, w->n_pages, c.n_kv_heads) &&
             attn_tc_encode_kv(&w->tm_v[l], w->v_cache + (size_t)l * w->cache_layer_stride, w->n_pages, c.n_kv_heads);
      if (!ok) {
        set_last_error("cuTensorMapEncodeTiled failed for the attention tensor maps");
        return MQ_ERR_CUDA;
      }
      w->prefill_tile_rows = kPrefillTileRowsTc;
    }
  }
  if (streamk_enabled() && streamk_workspace_alloc(&w->sk_ws) != 0) {
    set_last_error("stream-K workspace allocation failed");
    return MQ_ERR_NOMEM;
  }
  w->slot_req.assign(MB, nullptr);
  w->free_pages.clear();
  for (int p = w->n_pages - 1; p >= 1; --p) w->free_pages.push_back(p);  // page 0 = scratch
  return MQ_OK;
}

// ------------------------------------------------------------------------------------------------
// GEMM plans
// ------------------------------------------------------------------------------------------------
static int build_plans(mq_worker* w, PassPlans* pp, int T, bool decode) {
  const mq_model_cfg& c = w->cfg;
  const int H = c.hidden, I = c.ffn, D = c.head_dim, qd = c.n_q_heads * D;
  pp->T = T;
  pp->decode = decode;
  const int MBp = round_up(w->MB, 16);
  // per-layer GEMMs: stream-K only when forced (MQ_STREAMK=1); auto mode reserves it for the LM head
  const char* sk_env = getenv("MQ_STREAMK");
  const StreamKWorkspace* sk = (decode && T <= 64 && w->sk_ws.ws && sk_env && sk_env[0] == '1') ? &w->sk_ws : nullptr;
  w->sk_ws.force = sk != nullptr;
  if (decode && !sk) {
    pp->s_qkv = decode_splits((w->qkv_dim + 127) / 128, H / 64);
    pp->s_o = decode_splits((H + 127) / 128, qd / 64);
    pp->s_down = decode_splits((H + 127) / 128, I / 64);
  } else {
    pp->s_qkv = pp->s_o = pp->s_down = 1;
  }
  const int epi_part = decode ? EPI_F32 : EPI_BF16;
  const int x_rows = w->MT;
  // ---- decode chain: servable when every GEMM of the layer fits the cluster kernel (T <= 64, one head per QKV tile)
  const int tiles_h = (H + 127) / 128;
  pp->chain = decode && !sk && w->chain && T <= 64 && dk_pick_cluster(tiles_h, qd / 64, T) > 0 &&
              dk_pick_cluster(tiles_h, I / 64, T) > 0;
  if (pp->chain) {
    pp->qkv.resize(c.n_layers); pp->o_dk.resize(c.n_layers); pp->down_dk.resize(c.n_layers); pp->gate_up.resize(c.n_layers);
    pp->s_qkv = decode_splits((w->qkv_dim + 127) / 128, H / 64);
    const RstdIn rs_o{w->ssq_o, tiles_h, w->ssq_stride, 1.0f / (float)H, c.rms_eps};
    const RstdIn rs_d{w->ssq_d, tiles_h, w->ssq_stride, 1.0f / (float)H, c.rms_eps};
    const RstdIn rs_e{w->ssq_e, 1, w->ssq_stride, 1.0f / (float)H, c.rms_eps};
    for (int l = 0; l < c.n_layers; ++l) {
      const LayerWeights& lw = w->layers[l];
      DkPlan& o = pp->o_dk[l];
      DkPlan& d = pp->down_dk[l];
      // QKV stays a plane-writing split-K GEMM on all SMs (48 head tiles x 3 splits; a cluster kernel fits only 45
      // clusters of 3, and 48 x 2 CTAs measured 4.3 us per layer slower) with the RMSNorm fold in its epilogue; the
      // small rope kernel sums the planes, rotates and writes q / the paged KV
      bool ok = gemm_plan(&pp->qkv[l], lw.wqkv, w->qkv_dim, w->qkv_dim, H, w->x, x_rows, T, EPI_F32, w->qkv_part, w->qkv_dim,
                          pp->s_qkv, (long long)MBp * w->qkv_dim, 0, nullptr);
      ok &= dk_plan(&o, lw.wo, H, H, qd, w->attn, x_rows, T, 128, 0);
      ok &= dk_plan(&d, lw.w_down, H, H, I, w->act, x_rows, T, 128, 0);
      ok &= gemm_plan(&pp->gate_up[l], lw.w_gate_up, 2 * I, I, H, w->x, x_rows, T, EPI_SILU_BF16, w->act, I, 1, 0, I,
                      nullptr, gemm_balanced_rows(I));
      if (!ok) {
        set_last_error("decode-chain plan failed (layer %d, T=%d)", l, T);
        return MQ_ERR_CUDA;
      }
      gemm_plan_set_rstd(&pp->qkv[l], l == 0 ? rs_e : rs_d);
      o.p.h = w->h; o.p.ldh = H; o.p.gamma_next = lw.mlp_norm; o.p.xg = w->x; o.p.ldx = H; o.p.ssq_out = w->ssq_o;
      o.p.ssq_stride = w->ssq_stride;
      d.p.h = w->h; d.p.ldh = H; d.p.gamma_next = l + 1 < c.n_layers ? w->layers[l + 1].attn_norm : w->final_norm;
      d.p.xg = w->x; d.p.ldx = H; d.p.ssq_out = w->ssq_d; d.p.ssq_stride = w->ssq_stride;
      gemm_plan_set_rstd(&pp->gate_up[l], rs_o);
    }
    return MQ_OK;
  }
  pp->qkv.resize(c.n_layers); pp->o.resize(c.n_layers); pp->gate_up.resize(c.n_layers); pp->down.resize(c.n_layers);
  // ---- prefill with the RMSNorm fold: servable when all four GEMMs run on the persistent 2-CTA kernel
  if (!decode && w->chain && T > 128) {
    const RstdIn rs_o{w->ssq_o, tiles_h, w->ssq_stride, 1.0f / (float)H, c.rms_eps};
    const RstdIn rs_d{w->ssq_d, tiles_h, w->ssq_stride, 1.0f / (float)H, c.rms_eps};
    const RstdIn rs_e{w->ssq_e, 1, w->ssq_stride, 1.0f / (float)H, c.rms_eps};
    bool ok = true;
    for (int l = 0; l < c.n_layers && ok; ++l) {
      const LayerWeights& lw = w->layers[l];
      ok &= gemm_plan(&pp->qkv[l], lw.wqkv, w->qkv_dim, w->qkv_dim, H, w->x, x_rows, T, EPI_BF16, w->qkv_part, w->qkv_dim, 1, 0, 0, nullptr);
      ok &= gemm_plan(&pp->o[l], lw.wo, H, H, qd, w->attn, x_rows, T, EPI_RESID, w->h, H, 1, 0, 0, nullptr);
      ok &= gemm_plan(&pp->gate_up[l], lw.w_gate_up, 2 * I, I, H, w->x, x_rows, T, EPI_SILU_BF16, w->act, I, 1, 0, I, nullptr);
      ok &= gemm_plan(&pp->down[l], lw.w_down, H, H, I, w->act, x_rows, T, EPI_RESID, w->h, H, 1, 0, 0, nullptr);
      ok = ok && pp->qkv[l].twocta && pp->gate_up[l].twocta &&
           gemm_plan_set_resid(&pp->o[l], lw.mlp_norm, w->x, H, w->ssq_o, w->ssq_stride) &&
           gemm_plan_set_resid(&pp->down[l], l + 1 < c.n_layers ? w->layers[l + 1].attn_norm : w->final_norm, w->x, H, w->ssq_d,
                               w->ssq_stride);
      if (ok) {
        gemm_plan_set_rstd(&pp->qkv[l], l == 0 ? rs_e : rs_d);
        gemm_plan_set_rstd(&pp->gate_up[l], rs_o);
      }
    }
    if (ok) {
      pp->pfold = true;
      pp->s_qkv = pp->s_o = pp->s_down = 1;
      return MQ_OK;
    }
  }
  for (int l = 0; l < c.n_layers; ++l) {
    const LayerWeights& lw = w->layers[l];
    bool ok = true;
    ok &= gemm_plan(&pp->qkv[l], lw.wqkv, w->qkv_dim, w->qkv_dim, H, w->x, x_rows, T, epi_part, w->qkv_part,
                    w->qkv_dim, pp->s_qkv, (long long)MBp * w->qkv_dim, 0, sk);
    ok &= gemm_plan(&pp->o[l], lw.wo, H, H, qd, w->attn, x_rows, T, epi_part, w->proj_part, H, pp->s_o,
                    (long long)MBp * H, 0, sk);
    ok &= gemm_plan(&pp->gate_up[l], lw.w_gate_up, 2 * I, I, H, w->x, x_rows, T, EPI_SILU_BF16, w->act, I, 1, 0, I, sk);
    ok &= gemm_plan(&pp->down[l], lw.w_down, H, H, I, w->act, x_rows, T, epi_part, w->proj_part, H, pp->s_down,
                    (long long)MBp * H, 0, sk);
    if (!ok) {
      set_last_error("gemm_plan failed (layer %d, T=%d)", l, T);
      return MQ_ERR_CUDA;
    }
  }
  return MQ_OK;
}

static PassPlans* get_plans(mq_worker* w, int T, bool decode) {
  auto& m = decode ? w->plans_decode : w->plans_prefill;
  auto it = m.find(T);
  if (it != m.end()) return &it->second;
  PassPlans pp;
  if (build_plans(w, &pp, T, decode) != MQ_OK) return nullptr;
  return &(m[T] = std::move(pp));
}

// chain: the activation operand is the decode chain's xg = bf16(h * final_norm) (rows 0..rows-1 of w->x) and the
// final RMSNorm is the per-token scale of the epilogue (ssq_d of the last down projection)
static GemmPlan* get_lm_plan(mq_worker* w, int rows, bool chain = false) {
  const int key = rows + (chain ? (1 << 20) : 0);
  auto it = w->lm_plans.find(key);
  if (it != w->lm_plans.end()) return &it->second;
  GemmPlan g;
  const int MBp = round_up(w->MB, 16);
  if (!gemm_plan(&g, w->lm_head, w->cfg.vocab, w->cfg.vocab, w->cfg.hidden, chain ? w->x : w->x_last, chain ? w->MT : MBp,
                 rows, EPI_F32, w->logits, w->cfg.vocab, 1, 0, 0, (rows <= 64 && w->sk_ws.ws) ? &w->sk_ws : nullptr)) {
    set_last_error("gemm_plan(lm_head) failed");
    return nullptr;
  }
  if (chain)
    gemm_plan_set_rstd(&g, RstdIn{w->ssq_d, (w->cfg.hidden + 127) / 128, w->ssq_stride, 1.0f / (float)w->cfg.hidden, w->cfg.rms_eps});
  return &(w->lm_plans[key] = g);
}

// ------------------------------------------------------------------------------------------------
// one forward pass over T activation rows (all launches on w->stream; capturable when decode)
// ------------------------------------------------------------------------------------------------
struct PassArgs {
  int T;
  bool decode;
  int n_splits;                // decode
  int n_tiles;                 // prefill
  const int* tok;              // [T] token ids (device)
  const int* pos;              // [T]
  const int* slot_of_tok;      // [T]
  int attn_stages = 0;         // decode: ring depth of the one-warp attention CTAs (0 = default)
};


static void fill_attn_params(mq_worker* w, const PassArgs& a, int l, AttnParams* ap, Trace tr) {
  const mq_model_cfg& c = w->cfg;
  *ap = AttnParams{};
  ap->head_dim = c.head_dim;
  ap->q = w->q;
  ap->k_cache = w->k_cache + (size_t)l * w->cache_layer_stride;
  ap->v_cache = w->v_cache + (size_t)l * w->cache_layer_stride;
  ap->block_table = w->d_block_table;
  ap->max_pages = w->max_pages; ap->tiles = w->d_tiles; ap->pos = a.pos; ap->out = w->attn; ap->part_o = w->part_o;
  ap->part_ml = w->part_ml; ap->n_q = c.n_q_heads; ap->n_kv = c.n_kv_heads; ap->T = a.T;
  ap->n_splits = a.n_splits < 0 ? 1 : a.n_splits; ap->n_warps = a.n_splits < 0 ? -a.n_splits : 1;
  ap->stages = a.attn_stages;
  ap->tr = tr;
  ap->split_counter = w->d_split_counter; ap->scale_log2 = (1.0f / sqrtf((float)c.head_dim)) * 1.4426950408889634f;
}

// Decode chain: 6 launches per layer (no RMSNorm kernels).  Timeline slots (tools/decode_timeline.py): 1 + 8 * layer +
// {1 qkv, 2 rope, 3 attention, 4 o, 6 gate/up, 7 down}; slots 0 / 5 (norm1, norm2 of the plane-based path) stay unused.
static int run_layers_chain(mq_worker* w, const PassArgs& a, PassPlans* pp, uint64_t* n_launch) {
  const mq_model_cfg& c = w->cfg;
  const LaunchCfg lc{w->stream, c.use_pdl != 0};
  uint64_t nl = 0;
  launch_embed(lc, a.tok, w->embed, w->h, a.T, c.hidden, w->layers[0].attn_norm, w->x, w->ssq_e); ++nl;
  for (int l = 0; l < c.n_layers; ++l) {
    auto tr = [&](int k) { return Trace{w->d_trace, 1 + 8 * l + k}; };
    pp->qkv[l].p.tr = tr(1);
    if (gemm_launch(pp->qkv[l], lc) != cudaSuccess) return MQ_ERR_CUDA; ++nl;
    RopeKvParams rp;
    rp.qkv = w->qkv_part; rp.qkv_is_f32 = true; rp.n_planes = pp->s_qkv; rp.plane_stride = (long long)round_up(w->MB, 16) * w->qkv_dim;
    rp.bias = w->layers[l].bqkv; rp.pos = a.pos; rp.slot_of_tok = a.slot_of_tok; rp.block_table = w->d_block_table;
    rp.max_pages = w->max_pages; rp.inv_freq = w->inv_freq; rp.rope_table = w->rope_table; rp.q_out = w->q;
    rp.k_cache = w->k_cache + (size_t)l * w->cache_layer_stride;
    rp.v_cache = w->v_cache + (size_t)l * w->cache_layer_stride;
    rp.T = a.T; rp.n_q = c.n_q_heads; rp.n_kv = c.n_kv_heads; rp.head_dim = c.head_dim;
    rp.tr = tr(2);
    launch_rope_kv(lc, rp); ++nl;
    AttnParams ap;
    fill_attn_params(w, a, l, &ap, tr(3));
    launch_attn_decode(lc, ap, a.T); ++nl;
    pp->o_dk[l].p.tr = tr(4);
    if (dk_launch(pp->o_dk[l], lc) != cudaSuccess) return MQ_ERR_CUDA; ++nl;
    pp->gate_up[l].p.tr = tr(6);
    if (gemm_launch(pp->gate_up[l], lc) != cudaSuccess) return MQ_ERR_CUDA; ++nl;
    pp->down_dk[l].p.tr = tr(7);
    if (dk_launch(pp->down_dk[l], lc) != cudaSuccess) return MQ_ERR_CUDA; ++nl;
  }
  *n_launch += nl;
  return MQ_OK;
}

static int run_layers(mq_worker* w, const PassArgs& a, PassPlans* pp, uint64_t* n_launch) {
  if (a.decode && pp->chain) return run_layers_chain(w, a, pp, n_launch);
  const mq_model_cfg& c = w->cfg;
  const LaunchCfg lc{w->stream, c.use_pdl != 0};
  const int H = c.hidden;
  const int MBp = round_up(w->MB, 16);
  const bool f32p = a.decode;
  uint64_t nl = 0;
  const bool pfold = !a.decode && pp->pfold;
  if (pfold) launch_embed(lc, a.tok, w->embed, w->h, a.T, H, w->layers[0].attn_norm, w->x, w->ssq_e);
  else launch_embed(lc, a.tok, w->embed, w->h, a.T, H);
  ++nl;
  int prev_planes = 0;
  for (int l = 0; l < c.n_layers; ++l) {
    const LayerWeights& lw = w->layers[l];
    // timeline slots: 1 + 8 * layer + {0 norm1, 1 qkv, 2 rope, 3 attention, 4 o, 5 norm2, 6 gate/up, 7 down}
    auto tr = [&](int k) { return Trace{w->d_trace, 1 + 8 * l + k}; };
    auto tr_gemm = [&](GemmPlan& g, int k) { g.p.tr = tr(k); g.sk.tr = tr(k); };
    if (!pfold) {
      launch_add_rmsnorm(lc, w->h, w->proj_part, f32p, prev_planes, (long long)MBp * H, lw.attn_norm, w->x, nullptr, a.T,
                         H, c.rms_eps, tr(0)); ++nl;
    }
    tr_gemm(pp->qkv[l], 1);
    if (gemm_launch(pp->qkv[l], lc) != cudaSuccess) return MQ_ERR_CUDA; ++nl;
    RopeKvParams rp;
    rp.qkv = w->qkv_part; rp.qkv_is_f32 = f32p; rp.n_planes = pp->s_qkv; rp.plane_stride = (long long)MBp * w->qkv_dim;
    rp.bias = lw.bqkv; rp.pos = a.pos; rp.slot_of_tok = a.slot_of_tok; rp.block_table = w->d_block_table;
    rp.max_pages = w->max_pages; rp.inv_freq = w->inv_freq; rp.rope_table = w->rope_table; rp.q_out = w->q;
    rp.k_cache = w->k_cache + (size_t)l * w->cache_layer_stride;
    rp.v_cache = w->v_cache + (size_t)l * w->cache_layer_stride;
    rp.T = a.T; rp.n_q = c.n_q_heads; rp.n_kv = c.n_kv_heads; rp.head_dim = c.head_dim;
    rp.tr = tr(2);
    launch_rope_kv(lc, rp); ++nl;
    AttnParams ap;
    fill_attn_params(w, a, l, &ap, tr(3));
    if (a.decode) { launch_attn_decode(lc, ap, a.T); ++nl; }
    else if (w->attn_tc) { if (launch_attn_prefill_tc(lc, w->tm_q, w->tm_k[l], w->tm_v[l], ap, a.n_tiles) != cudaSuccess) return MQ_ERR_CUDA; ++nl; }
    else { launch_attn_prefill(lc, ap, a.n_tiles); ++nl; }
    tr_gemm(pp->o[l], 4);
    if (gemm_launch(pp->o[l], lc) != cudaSuccess) return MQ_ERR_CUDA; ++nl;
    if (!pfold) {
      launch_add_rmsnorm(lc, w->h, w->proj_part, f32p, pp->s_o, (long long)MBp * H, lw.mlp_norm, w->x, nullptr, a.T, H,
                         c.rms_eps, tr(5)); ++nl;
    }
    tr_gemm(pp->gate_up[l], 6);
    if (gemm_launch(pp->gate_up[l], lc) != cudaSuccess) return MQ_ERR_CUDA; ++nl;
    tr_gemm(pp->down[l], 7);
    if (gemm_launch(pp->down[l], lc) != cudaSuccess) return MQ_ERR_CUDA; ++nl;
    prev_planes = pp->s_down;
  }
  *n_launch += nl;
  return MQ_OK;
}

// final norm (+ last partial) on `rows` gathered rows -> lm head -> logits[rows][V]
static int run_head(mq_worker* w, bool decode, const int* row_idx, int rows, PassPlans* pp, uint64_t* n_launch) {
  const mq_model_cfg& c = w->cfg;
  const LaunchCfg lc{w->stream, c.use_pdl != 0};
  const int MBp = round_up(w->MB, 16);
  const bool chain = decode && pp->chain;  // final norm folded into the LM head (rows are the batch rows themselves)
  if (!chain) {
    // (prefill with the fold: the last down projection already added into h - nothing left to sum)
    launch_add_rmsnorm(lc, w->h, w->proj_part, decode, (!decode && pp->pfold) ? 0 : pp->s_down, (long long)MBp * c.hidden, w->final_norm, w->x_last,
                       row_idx, rows, c.hidden, c.rms_eps, Trace{w->d_trace, kTraceSlots - 2});
    *n_launch += 1;
  }
  GemmPlan* g = get_lm_plan(w, rows, chain);
  if (!g) return MQ_ERR_CUDA;
  g->p.tr = g->sk.tr = Trace{w->d_trace, kTraceSlots - 1};
  if (gemm_launch(*g, lc) != cudaSuccess) return MQ_ERR_CUDA;
  *n_launch += 1;
  return MQ_OK;
}

// ------------------------------------------------------------------------------------------------
// staging ring for metadata uploads
// ------------------------------------------------------------------------------------------------
static int* stage_acquire(mq_worker* w, int* slot_out) {
  const int s = w->stage_next;
  w->stage_next = (s + 1) % kStageSlots;
  cudaEventSynchronize(w->stage_ev[s]);  // no-op unless we lapped the GPU
  *slot_out = s;
  return w->h_stage + (size_t)s * w->stage_ints;
}
static void stage_release(mq_worker* w, int slot) { cudaEventRecord(w->stage_ev[slot], w->stream); }

static cudaEvent_t ev_get(mq_worker* w) {
  if (!w->ev_pool.empty()) {
    cudaEvent_t e = w->ev_pool.back();
    w->ev_pool.pop_back();
    return e;
  }
  cudaEvent_t e;
  cudaEventCreate(&e);
  return e;
}

// upload the slot table's host mirror when it changed (through a staging area: the mirror keeps changing while the copy
// is still queued)
static void upload_slots(mq_worker* w) {
  if (!w->slots_dirty) return;
  int ss;
  int* st = stage_acquire(w, &ss);
  memcpy(st, w->h_slots, w->slot_bytes);
  cudaMemcpyAsync(w->d_slots, st, w->slot_bytes, cudaMemcpyHostToDevice, w->stream);
  stage_release(w, ss);
  w->slots_dirty = false;
}

// sampler controls of a pass: the slot table's sampling sections, the per-slot RNG counter (nullptr: position 0) and the
// pass's row of the log-probability ring
static SampleCtl sample_ctl(mq_worker* w, const int* counter, int ring) {
  return SampleCtl{w->d_temp, w->d_topk, w->d_topp, w->d_seed, counter, w->d_lp_top,
                   w->d_lp_ring + (size_t)ring * round_up(w->MB, 16)};
}

// ------------------------------------------------------------------------------------------------
// request lifecycle helpers (worker thread only)
// ------------------------------------------------------------------------------------------------
static void req_unref(mq_req* r) {
  if (r->refs.fetch_sub(1) == 1) delete r;
}

static void free_slot(mq_worker* w, mq_req* r) {
  if (r->slot < 0) return;
  const int s = r->slot;
  for (int p : r->pages) w->free_pages.push_back(p);
  r->pages.clear();
  w->slot_req[s] = nullptr;
  w->h_active[s] = 0;
  w->h_pos[s] = 0;
  set_slot_sampling(w, s, SamplingParams{});
  for (int i = 0; i < w->max_pages; ++i) w->h_block_table[(size_t)s * w->max_pages + i] = 0;  // scratch page
  w->slots_dirty = true;
  r->slot = -1;
}

static void send_status(mq_req* r) {
  if (r->status_sent) return;
  r->status_sent = true;
  if (r->cb.on_status) r->cb.on_status(r->user, 200, content_type_for(r->rq.endpoint, r->rq.stream));
}

static void finish_req(mq_worker* w, mq_req* r, int rc, const char* msg) {
  if (r->finished) return;
  r->finished = true;
  r->done_rc = rc;
  r->t_last = Clock::now();
  free_slot(w, r);
  if (rc == 0) {
    send_status(r);
    std::string tail = frame_final(r->rq.endpoint, r->rq.stream, w->cfg.model_name, r->agg, (int)r->prompt.size(),
                                   r->n_emitted, r->stopped, r->sp.top_logprobs >= 0 ? &r->agg_lp : nullptr);
    if (!tail.empty() && r->cb.on_chunk) r->cb.on_chunk(r->user, (const uint8_t*)tail.data(), tail.size());
  }
  if (r->cb.on_done) r->cb.on_done(r->user, rc, msg ? msg : "");
  req_unref(r);
}

// rec: the token's log-probability record (read only when the request asked for one)
static void emit_token(mq_worker* w, mq_req* r, int tok, const LogprobRec* rec) {
  if (r->finished) return;
  if (!r->rq.ignore_eos && w->cfg.eos_token_id > 0 && tok == w->cfg.eos_token_id) {
    // end of sequence: the EOS token itself is not relayed; steps already in flight for this slot are discarded
    // (their tokens arrive for a finished request) and the slot / pages are free for the next admission
    r->stopped = true;
    finish_req(w, r, 0, nullptr);
    return;
  }
  if (r->n_emitted == 0) r->t_first = Clock::now();
  r->n_emitted++;
  send_status(r);
  if (r->sp.top_logprobs >= 0) {
    TokenLogprobs e;
    e.id = tok;
    e.logprob = rec->logprob;
    for (int j = 0; j < r->sp.top_logprobs; ++j) e.top.push_back({rec->id[j], rec->lp[j]});
    std::string s;
    if (r->rq.endpoint == MQ_EP_RAW_TOKENS) append_raw_record(r->rq.stream ? &s : &r->agg, e);
    else if (r->rq.stream) s = frame_token(r->rq.endpoint, w->cfg.model_name, tok, &e, r->text_len);
    else r->agg += token_text(tok);
    r->text_len += token_text(tok).size();
    if (r->rq.stream) {
      if (r->cb.on_chunk && r->cb.on_chunk(r->user, (const uint8_t*)s.data(), s.size()) != 0) r->cancel.store(true);
    } else if (r->rq.endpoint != MQ_EP_RAW_TOKENS) {
      r->agg_lp.push_back(std::move(e));
    }
  } else if (r->rq.stream) {
    uint8_t raw[4];
    std::string s;
    const uint8_t* data;
    size_t len;
    if (r->rq.endpoint == MQ_EP_RAW_TOKENS) {
      memcpy(raw, &tok, 4);
      data = raw; len = 4;
    } else {
      s = frame_token(r->rq.endpoint, w->cfg.model_name, tok);
      data = (const uint8_t*)s.data(); len = s.size();
    }
    if (r->cb.on_chunk && r->cb.on_chunk(r->user, data, len) != 0) r->cancel.store(true);  // client gone (:305-308)
  } else {
    if (r->rq.endpoint == MQ_EP_RAW_TOKENS) r->agg.append((const char*)&tok, 4);
    else r->agg += token_text(tok);
  }
  if (r->n_emitted >= r->max_new) finish_req(w, r, 0, nullptr);
}

// ------------------------------------------------------------------------------------------------
// prefill pass
// ------------------------------------------------------------------------------------------------
struct PrefillItem { mq_req* r; int n_tok; bool completes; };

static int launch_prefill(mq_worker* w, std::vector<PrefillItem>& items) {
  const mq_model_cfg& c = w->cfg;
  const int G = c.n_q_heads / c.n_kv_heads;
  const int tok_per_tile = w->prefill_tile_rows / G;
  int T = 0;
  for (auto& it : items) T += it.n_tok;
  int ss;
  int* st = stage_acquire(w, &ss);
  int* s_tok = st;
  int* s_pos = st + w->MT;
  int* s_slot = st + 2 * w->MT;
  int* s_tiles = st + 3 * w->MT;                 // int4 per tile
  int* s_last = s_tiles + 4 * (w->MT + w->MB);
  int* s_dst = s_last + round_up(w->MB, 16);
  int n_tiles = 0, n_last = 0, row = 0;
  for (auto& it : items) {
    mq_req* r = it.r;
    const int p0 = r->n_prefilled;
    for (int i = 0; i < it.n_tok; ++i) {
      s_tok[row + i] = r->prompt[p0 + i];
      s_pos[row + i] = p0 + i;
      s_slot[row + i] = r->slot;
    }
    for (int i = 0; i < it.n_tok; i += tok_per_tile) {
      int* t = s_tiles + 4 * n_tiles++;
      t[0] = row + i; t[1] = std::min(tok_per_tile, it.n_tok - i); t[2] = r->slot; t[3] = p0 + i;
    }
    if (it.completes) {
      s_last[n_last] = row + it.n_tok - 1;
      s_dst[n_last] = r->slot;
      ++n_last;
    }
    row += it.n_tok;
    r->n_prefilled += it.n_tok;
  }
  cudaMemcpyAsync(w->d_tok, s_tok, T * 4, cudaMemcpyHostToDevice, w->stream);
  cudaMemcpyAsync(w->d_pos_tok, s_pos, T * 4, cudaMemcpyHostToDevice, w->stream);
  cudaMemcpyAsync(w->d_slot_tok, s_slot, T * 4, cudaMemcpyHostToDevice, w->stream);
  cudaMemcpyAsync(w->d_tiles, s_tiles, (size_t)n_tiles * 16, cudaMemcpyHostToDevice, w->stream);
  if (n_last) {
    cudaMemcpyAsync(w->d_last_idx, s_last, n_last * 4, cudaMemcpyHostToDevice, w->stream);
    cudaMemcpyAsync(w->d_dst_slot, s_dst, n_last * 4, cudaMemcpyHostToDevice, w->stream);
  }
  stage_release(w, ss);
  upload_slots(w);

  PassPlans* pp = get_plans(w, T, false);
  if (!pp) return MQ_ERR_CUDA;
  mq_worker::Flight f;
  f.timed = w->timing;
  if (f.timed) { f.ev_begin = ev_get(w); cudaEventRecord(f.ev_begin, w->stream); }
  PassArgs a{T, false, 1, n_tiles, w->d_tok, w->d_pos_tok, w->d_slot_tok};
  uint64_t nl = 0;
  int rc = run_layers(w, a, pp, &nl);
  if (rc) return rc;
  const int ring = w->ring_next;
  w->ring_next = (ring + 1) % (kRing - 1);  // row kRing-1 is the fixed output row of captured graphs
  const int MBp = round_up(w->MB, 16);
  if (n_last) {
    rc = run_head(w, false, w->d_last_idx, n_last, pp, &nl);
    if (rc) return rc;
    const LaunchCfg lc{w->stream, c.use_pdl != 0};
    // first generated token of each finished prompt: RNG position 0 (decode steps use the token position >= 1)
    launch_sample(lc, w->logits, n_last, c.vocab, c.vocab, w->d_out_ring + (size_t)ring * MBp, w->d_dst_slot,
                  w->d_cur_token, nullptr, nullptr, sample_ctl(w, nullptr, ring));
    ++nl;
    cudaMemcpyAsync(w->h_out_ring + (size_t)ring * MBp, w->d_out_ring + (size_t)ring * MBp, n_last * 4,
                    cudaMemcpyDeviceToHost, w->stream);
    bool want_lp = false;
    for (auto& it : items) want_lp |= it.completes && it.r->sp.top_logprobs >= 0;
    if (want_lp)
      cudaMemcpyAsync(w->h_lp_ring + (size_t)ring * MBp, w->d_lp_ring + (size_t)ring * MBp, n_last * sizeof(LogprobRec),
                      cudaMemcpyDeviceToHost, w->stream);
  }
  f.ev = ev_get(w);
  cudaEventRecord(f.ev, w->stream);
  f.decode = false;
  f.ring = ring;
  int k = 0;
  for (auto& it : items)
    if (it.completes) {
      // the sequence joins the decode batch: first generated token sits in cur_token[slot], pos = prompt length
      mq_req* r = it.r;
      r->n_sched = 1;
      w->h_pos[r->slot] = (int)r->prompt.size();
      w->h_active[r->slot] = r->max_new > 1 ? 1 : 0;
      w->slots_dirty = true;
      f.emits.push_back({r, k++});
    }
  w->flights.push_back(std::move(f));
  {
    std::lock_guard<std::mutex> g(w->stats_mu);
    w->stats.kernel_launches += nl;
    w->stats.prefill_passes += 1;
    w->stats.prefill_tokens += T;
  }
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_last_error("prefill launch: %s", cudaGetErrorString(e));
    return MQ_ERR_CUDA;
  }
  return MQ_OK;
}

// ------------------------------------------------------------------------------------------------
// decode step
// ------------------------------------------------------------------------------------------------
static int decode_body(mq_worker* w, int Bcap, int n_splits, int attn_stages, int ring, uint64_t* nl) {
  const mq_model_cfg& c = w->cfg;
  PassPlans* pp = get_plans(w, Bcap, true);
  if (!pp) return MQ_ERR_CUDA;
  PassArgs a{Bcap, true, n_splits, 0, w->d_cur_token, w->d_pos, w->d_identity};
  a.attn_stages = attn_stages;
  int rc = run_layers(w, a, pp, nl);
  if (rc) return rc;
  rc = run_head(w, true, w->d_identity, Bcap, pp, nl);
  if (rc) return rc;
  const LaunchCfg lc{w->stream, c.use_pdl != 0};
  const int MBp = round_up(w->MB, 16);
  // NOTE: the ring slot is baked into a captured graph, so graphs write to a fixed staging row (ring 0 of the
  // graph area) and the copy-out below moves it into the real ring slot.
  launch_sample(lc, w->logits, Bcap, c.vocab, c.vocab, w->d_out_ring + (size_t)ring * MBp, nullptr, w->d_cur_token,
                w->d_pos, w->d_active, sample_ctl(w, w->d_pos, ring));
  *nl += 1;
  return MQ_OK;
}

static int launch_decode(mq_worker* w) {
  const int MBp = round_up(w->MB, 16);
  int hi = -1, max_ctx = 1, n_active = 0;
  double kv_tokens = 0;
  bool want_lp = false;  // some emitted slot asked for logprobs: copy the record row out beside the tokens
  for (int s = 0; s < w->MB; ++s)
    if (w->h_active[s]) {
      hi = s;
      want_lp |= w->slot_req[s]->sp.top_logprobs >= 0;
      ++n_active;
      max_ctx = std::max(max_ctx, w->h_pos[s] + 1);
      kv_tokens += w->h_pos[s] + 1;
    }
  if (hi < 0) return MQ_OK;
  const int Bcap = std::min(MBp, round_up(hi + 1, 16));
  // KV splits only when (active slots x kv heads) alone leaves SMs idle (r01 timelines, 64 slots x 8 kv heads:
  // unsplit 25 us per layer, 2-way grid split 33 us).  Small batches split INSIDE the CTA - 2 / 4 / 8 warps, each
  // one KV range, merged through shared memory (encoded as a negative count); the grid-level split with its
  // global-memory combine is the fallback for very long contexts on few slots.
  const int base_ctas = std::max(1, n_active) * w->cfg.n_kv_heads, sms = w->sm_count;
  int n_splits = 1;
  if (base_ctas < 2 * sms) {
    int nw = base_ctas > sms ? 4 : 8;  // r01 sweep: 8 / 16 slots -> 8 warps (5.3 / 6.4 us), 24 / 32 slots -> 4 warps (10.4 / 12.3 us)
    while (nw > 1 && max_ctx / nw < 64) nw >>= 1;  // keep >= 4 pages per warp
    n_splits = nw > 1 ? -nw : 1;
  }
  // ring depth of the one-warp CTAs: a warp that walks only a few pages gains nothing from a 6-stage (48 KiB) ring and
  // loses residency (4 CTAs per SM); with many (slot, kv head) pairs and short contexts - Phi-3-mini, 256 users x 32
  // tokens: 8192 CTAs of 3 pages - the kernel is a latency chain per CTA, so residency is what counts
  const int pages_per_cta = (max_ctx + kPageSize - 1) / kPageSize;
  // (Phi-3-mini, 256 slots, 3-4 pages: 2 / 3 / 4 / 6 stages -> 4.05 / 4.15 / 4.31 / 4.80 ms per step)
  const int attn_stages = pages_per_cta <= 4 ? 2 : pages_per_cta <= 8 ? 3 : pages_per_cta <= 16 ? 4 : 6;
  if (const char* e = getenv("MQ_ATTN_SPLITS")) {  // experiments: 1..8 grid-level, -2 / -4 / -8 in-CTA
    const int v = atoi(e);
    if (v == -2 || v == -4 || v == -8 || (v >= 1 && v <= kMaxDecodeSplits)) n_splits = v;
  }
  upload_slots(w);
  if (w->d_trace) cudaMemsetAsync(w->d_trace, 0xFF, (size_t)kTraceSlots * 4 * 8, w->stream);  // re-arm the timeline

  mq_worker::Flight f;
  f.timed = w->timing;
  if (f.timed) { f.ev_begin = ev_get(w); cudaEventRecord(f.ev_begin, w->stream); }
  const int ring = w->ring_next;
  w->ring_next = (ring + 1) % (kRing - 1);  // row kRing-1 is the fixed output row of captured graphs
  uint64_t nl = 0;
  bool graph_launched = false;
  if (w->cfg.use_graphs) {
    // graphs always write their tokens to ring row 0's alias at the end of the ring buffer (fixed address)
    const long long key = ((long long)Bcap * 1024 + (n_splits + 16)) * 8 + attn_stages;
    auto it = w->graphs.find(key);
    if (it == w->graphs.end()) {
      PassPlans* pp0 = get_plans(w, Bcap, true);
      if (!pp0 || !get_lm_plan(w, Bcap, pp0->chain)) return MQ_ERR_CUDA;
      // warm-up launch outside capture so every kernel's attributes are set before capturing
      uint64_t tmp = 0;
      cudaGraph_t g = nullptr;
      cudaError_t e = cudaStreamBeginCapture(w->stream, cudaStreamCaptureModeThreadLocal);
      int rc = e == cudaSuccess ? decode_body(w, Bcap, n_splits, attn_stages, kRing - 1, &tmp) : MQ_ERR_CUDA;
      cudaError_t e2 = cudaStreamEndCapture(w->stream, &g);
      if (rc != MQ_OK || e2 != cudaSuccess || !g) {
        set_last_error("graph capture failed: %s", cudaGetErrorString(e2 != cudaSuccess ? e2 : cudaGetLastError()));
        return MQ_ERR_CUDA;
      }
      cudaGraphExec_t ge = nullptr;
      e = cudaGraphInstantiate(&ge, g, 0);
      cudaGraphDestroy(g);
      if (e != cudaSuccess) {
        set_last_error("cudaGraphInstantiate: %s", cudaGetErrorString(e));
        return MQ_ERR_CUDA;
      }
      it = w->graphs.emplace(key, ge).first;
      std::lock_guard<std::mutex> gl(w->stats_mu);
      w->stats.kernel_launches += 0;
    }
    cudaError_t e = cudaGraphLaunch(it->second, w->stream);
    if (e != cudaSuccess) {
      set_last_error("cudaGraphLaunch: %s", cudaGetErrorString(e));
      return MQ_ERR_CUDA;
    }
    graph_launched = true;
    // graph wrote to the fixed row kRing-1; move it to this step's ring slot on the host side copy
    cudaMemcpyAsync(w->h_out_ring + (size_t)ring * MBp, w->d_out_ring + (size_t)(kRing - 1) * MBp, Bcap * 4,
                    cudaMemcpyDeviceToHost, w->stream);
    if (want_lp)
      cudaMemcpyAsync(w->h_lp_ring + (size_t)ring * MBp, w->d_lp_ring + (size_t)(kRing - 1) * MBp,
                      Bcap * sizeof(LogprobRec), cudaMemcpyDeviceToHost, w->stream);
    nl = get_plans(w, Bcap, true)->chain ? (uint64_t)(1 + w->cfg.n_layers * 6 + 2) : (uint64_t)(1 + w->cfg.n_layers * 8 + 3);
  } else {
    int rc = decode_body(w, Bcap, n_splits, attn_stages, ring, &nl);
    if (rc) return rc;
    cudaMemcpyAsync(w->h_out_ring + (size_t)ring * MBp, w->d_out_ring + (size_t)ring * MBp, Bcap * 4,
                    cudaMemcpyDeviceToHost, w->stream);
    if (want_lp)
      cudaMemcpyAsync(w->h_lp_ring + (size_t)ring * MBp, w->d_lp_ring + (size_t)ring * MBp, Bcap * sizeof(LogprobRec),
                      cudaMemcpyDeviceToHost, w->stream);
  }
  f.ev = ev_get(w);
  cudaEventRecord(f.ev, w->stream);
  f.decode = true;
  f.ring = ring;
  f.bytes = w->p_mm_bytes + (kv_tokens + n_active) * w->kv_bytes_per_tok;
  for (int s = 0; s < w->MB; ++s)
    if (w->h_active[s]) {
      mq_req* r = w->slot_req[s];
      f.emits.push_back({r, s});
      w->h_pos[s] += 1;  // mirrors the device-side pos++ of the sampler kernel
      r->n_sched += 1;
      if (r->n_sched >= r->max_new) {  // last token scheduled: slot leaves the batch at the next step
        w->h_active[s] = 0;
        w->slots_dirty = true;
      }
    }
  w->flights.push_back(std::move(f));
  {
    std::lock_guard<std::mutex> g(w->stats_mu);
    w->stats.kernel_launches += nl;
    w->stats.graph_launches += graph_launched ? 1 : 0;
    w->stats.decode_steps += 1;
    w->stats.decode_tokens += n_active;
  }
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_last_error("decode launch: %s", cudaGetErrorString(e));
    return MQ_ERR_CUDA;
  }
  return MQ_OK;
}

// ------------------------------------------------------------------------------------------------
// completion of GPU work -> callbacks
// ------------------------------------------------------------------------------------------------
static void retire_flight(mq_worker* w, mq_worker::Flight& f) {
  const int MBp = round_up(w->MB, 16);
  if (f.timed) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, f.ev_begin, f.ev);
    std::lock_guard<std::mutex> g(w->stats_mu);
    if (f.decode) { w->stats.decode_ms += ms; w->stats.decode_bytes += f.bytes; }
    else w->stats.prefill_ms += ms;
    w->ev_pool.push_back(f.ev_begin);
  }
  w->ev_pool.push_back(f.ev);
  const int* row = w->h_out_ring + (size_t)f.ring * MBp;
  const LogprobRec* lp_row = w->h_lp_ring + (size_t)f.ring * MBp;
  for (auto& em : f.emits) {
    mq_req* r = em.first;
    if (r->finished) continue;
    if (r->cancel.load()) continue;  // handled by the cancel sweep
    emit_token(w, r, row[em.second], lp_row + em.second);
  }
  for (auto& em : f.emits) req_unref(em.first);
}

static void poll_flights(mq_worker* w, bool block_oldest) {
  while (!w->flights.empty()) {
    mq_worker::Flight& f = w->flights.front();
    cudaError_t e = block_oldest ? cudaEventSynchronize(f.ev) : cudaEventQuery(f.ev);
    block_oldest = false;
    if (e == cudaErrorNotReady) return;
    if (e != cudaSuccess) {
      w->fatal = std::string("GPU fault: ") + cudaGetErrorString(e);
      w->healthy.store(false);
      return;
    }
    mq_worker::Flight done = std::move(f);
    w->flights.pop_front();
    retire_flight(w, done);
  }
}

// ------------------------------------------------------------------------------------------------
// the worker thread
// ------------------------------------------------------------------------------------------------
static void fail_all(mq_worker* w, const char* msg) {
  auto kill = [&](mq_req* r) { if (r && !r->finished) finish_req(w, r, MQ_ERR_CUDA, msg); };
  for (auto& f : w->flights) for (auto& em : f.emits) req_unref(em.first);
  w->flights.clear();
  for (mq_req* r : w->waiting) kill(r);
  w->waiting.clear();
  for (mq_req* r : w->prefilling) kill(r);
  w->prefilling.clear();
  for (int s = 0; s < w->MB; ++s) kill(w->slot_req[s]);
}

static bool admit(mq_worker* w, mq_req* r) {
  int slot = -1;
  for (int s = 0; s < w->MB; ++s)
    if (!w->slot_req[s]) { slot = s; break; }
  if (slot < 0) return false;
  const int need = ((int)r->prompt.size() + r->max_new + kPageSize - 1) / kPageSize;
  if ((int)w->free_pages.size() < need) return false;
  r->slot = slot;
  w->slot_req[slot] = r;
  r->pages.resize(need);
  for (int i = 0; i < need; ++i) {
    r->pages[i] = w->free_pages.back();
    w->free_pages.pop_back();
    w->h_block_table[(size_t)slot * w->max_pages + i] = r->pages[i];
  }
  w->h_pos[slot] = 0;
  w->h_active[slot] = 0;
  set_slot_sampling(w, slot, r->sp);
  w->slots_dirty = true;
  return true;
}

static void sweep_cancels(mq_worker* w) {
  const auto now = Clock::now();
  // returns true when the request was finished here (the pointer may be dangling afterwards)
  auto check = [&](mq_req* r) -> bool {
    if (!r || r->finished) return false;
    if (r->cancel.load()) { finish_req(w, r, MQ_ERR_CANCELED, "canceled"); return true; }
    if (r->has_deadline && now > r->deadline) { finish_req(w, r, MQ_ERR_TIMEOUT, "request timed out"); return true; }
    return false;
  };
  for (auto it = w->waiting.begin(); it != w->waiting.end();) it = check(*it) ? w->waiting.erase(it) : it + 1;
  for (auto it = w->prefilling.begin(); it != w->prefilling.end();) it = check(*it) ? w->prefilling.erase(it) : it + 1;
  for (int s = 0; s < w->MB; ++s) check(w->slot_req[s]);
}

static void worker_main(mq_worker* w) {
  cudaSetDevice(w->gpu);
  Clock::time_point last_arrival = Clock::now(), window_start = last_arrival;
  bool in_window = false;
  std::vector<mq_req*> others;
  for (;;) {
    for (mq_req* r : others) {  // non-generation routes: immediate answer, same Status/Chunk/Done sequence
      int status = 200;
      std::string ctype, body;
      if (r->bad_request) { status = 400; ctype = "application/json"; body = "{\"error\":\"invalid JSON request body\"}"; }
      else other_route_response(r->path, w->cfg.model_name, &status, &ctype, &body);
      r->t_first = r->t_last = Clock::now();
      r->finished = true;
      if (r->cb.on_status) r->cb.on_status(r->user, status, ctype.c_str());
      if (r->cb.on_chunk) r->cb.on_chunk(r->user, (const uint8_t*)body.data(), body.size());
      if (r->cb.on_done) r->cb.on_done(r->user, 0, "");
      req_unref(r);
    }
    others.clear();
    // ---- intake
    {
      std::unique_lock<std::mutex> lk(w->mu);
      const bool idle = w->flights.empty() && w->waiting.empty() && w->prefilling.empty() &&
                        std::none_of(w->h_active, w->h_active + w->MB, [](int a) { return a != 0; });
      if (idle && w->inbox.empty() && w->jobs.empty() && !w->stop)
        w->cv.wait_for(lk, std::chrono::milliseconds(50));
      if (w->stop) break;
      if (!w->inbox.empty()) last_arrival = Clock::now();
      while (!w->inbox.empty()) {
        mq_req* r = w->inbox.front();
        w->inbox.pop_front();
        if (r->rq.endpoint == MQ_EP_OTHER || r->bad_request) others.push_back(r);
        else w->waiting.push_back(r);
      }
      if (idle && !w->jobs.empty()) {
        auto job = std::move(w->jobs.front());
        w->jobs.pop_front();
        lk.unlock();
        job();
        continue;
      }
    }
    if (!w->healthy.load()) { fail_all(w, w->fatal.c_str()); continue; }
    sweep_cancels(w);

    // ---- admit + build one prefill pass (prefill has priority: it grows the decode batch)
    while (!w->waiting.empty() && admit(w, w->waiting.front())) {
      w->prefilling.push_back(w->waiting.front());
      w->waiting.pop_front();
    }
    // Batching window: a burst of arrivals on an idle GPU (64 users hitting "send" together) is prefilled as
    // full passes instead of a lone first prompt.  Wait while requests keep arriving <500 us apart, 4 ms at most.
    if (!w->prefilling.empty() && w->flights.empty()) {
      const auto now = Clock::now();
      if (!in_window) { in_window = true; window_start = now; }
      int queued_tokens = 0;
      for (mq_req* r : w->prefilling) queued_tokens += (int)r->prompt.size() - r->n_prefilled;
      if (queued_tokens < w->cfg.max_prefill_tokens && now - last_arrival < std::chrono::microseconds(500) &&
          now - window_start < std::chrono::milliseconds(4)) {
        std::this_thread::sleep_for(std::chrono::microseconds(30));
        continue;
      }
    }
    in_window = false;
    bool launched = false;
    int n_prefill_flights = 0, n_decode_flights = 0;
    for (auto& f : w->flights) (f.decode ? n_decode_flights : n_prefill_flights)++;
    if (!w->prefilling.empty()) {
      if (n_prefill_flights < kMaxFlightsPrefill) {
        std::vector<PrefillItem> items;
        int budget = w->cfg.max_prefill_tokens;
        while (!w->prefilling.empty() && budget > 0 && (int)items.size() < w->MB) {
          mq_req* r = w->prefilling.front();
          const int remaining = (int)r->prompt.size() - r->n_prefilled;
          if (remaining > budget && !items.empty()) break;  // keep whole prompts together when possible
          const int n = std::min(remaining, budget);
          const bool completes = n == remaining;
          items.push_back({r, n, completes});
          budget -= n;
          if (completes) { w->prefilling.pop_front(); r->refs.fetch_add(1); }
          else break;  // a chunked prompt owns the rest of this pass
        }
        if (!items.empty()) {
          if (launch_prefill(w, items) != MQ_OK) { w->fatal = mq_last_error(); w->healthy.store(false); continue; }
          launched = true;
        }
      }
    } else if (n_decode_flights < kMaxFlightsDecode) {
      bool any = false;
      for (int s = 0; s < w->MB; ++s) any |= w->h_active[s] != 0;
      if (any) {
        for (int s = 0; s < w->MB; ++s)
          if (w->h_active[s]) w->slot_req[s]->refs.fetch_add(1);
        if (launch_decode(w) != MQ_OK) { w->fatal = mq_last_error(); w->healthy.store(false); continue; }
        launched = true;
      }
    }
    // ---- completions: block only when nothing else can be launched
    poll_flights(w, !launched && !w->flights.empty());
  }
  // shutdown: drain
  cudaStreamSynchronize(w->stream);
  poll_flights(w, false);
  fail_all(w, "worker closed");
}

// ------------------------------------------------------------------------------------------------
// debug forward (kernel-level test ABI): runs on the worker thread when idle
// ------------------------------------------------------------------------------------------------
int engine_forward_logits(mq_worker* w, const int32_t* tokens, int n, int all_positions, float* out) {
  const mq_model_cfg& c = w->cfg;
  if (n < 1 || n > c.max_seq) {
    set_last_error("mq_debug_forward: n=%d out of range (max_seq %d)", n, c.max_seq);
    return MQ_ERR_INVAL;
  }
  const int MBp = round_up(w->MB, 16);
  const int G = c.n_q_heads / c.n_kv_heads, tok_per_tile = w->prefill_tile_rows / G;
  const int need = (n + kPageSize - 1) / kPageSize;
  if ((int)w->free_pages.size() < need || w->slot_req[0]) {
    set_last_error("mq_debug_forward: worker busy");
    return MQ_ERR_BUSY;
  }
  // temporary block table for slot 0
  std::vector<int> pages(need);
  for (int i = 0; i < need; ++i) { pages[i] = w->free_pages.back(); w->free_pages.pop_back(); }
  for (int i = 0; i < need; ++i) w->h_block_table[i] = pages[i];
  w->slots_dirty = true;
  uint64_t nl = 0;
  int rc = MQ_OK;
  for (int p0 = 0; p0 < n && rc == MQ_OK; p0 += c.max_prefill_tokens) {
    const int T = std::min(c.max_prefill_tokens, n - p0);
    std::vector<int> tok(T), pos(T), slot(T, 0), tiles;
    for (int i = 0; i < T; ++i) { tok[i] = tokens[p0 + i]; pos[i] = p0 + i; }
    for (int i = 0; i < T; i += tok_per_tile) {
      tiles.push_back(i); tiles.push_back(std::min(tok_per_tile, T - i)); tiles.push_back(0); tiles.push_back(p0 + i);
    }
    cudaMemcpyAsync(w->d_tok, tok.data(), T * 4, cudaMemcpyHostToDevice, w->stream);
    cudaMemcpyAsync(w->d_pos_tok, pos.data(), T * 4, cudaMemcpyHostToDevice, w->stream);
    cudaMemcpyAsync(w->d_slot_tok, slot.data(), T * 4, cudaMemcpyHostToDevice, w->stream);
    cudaMemcpyAsync(w->d_tiles, tiles.data(), tiles.size() * 4, cudaMemcpyHostToDevice, w->stream);
    upload_slots(w);
    cudaStreamSynchronize(w->stream);  // host vectors above go out of scope
    PassPlans* pp = get_plans(w, T, false);
    if (!pp) { rc = MQ_ERR_CUDA; break; }
    PassArgs a{T, false, 1, (int)tiles.size() / 4, w->d_tok, w->d_pos_tok, w->d_slot_tok};
    rc = run_layers(w, a, pp, &nl);
    if (rc) break;
    // logits for the requested rows, MBp rows at a time
    const int first = all_positions ? 0 : (p0 + T == n ? T - 1 : T);
    for (int r0 = first; r0 < T && rc == MQ_OK; r0 += MBp) {
      const int rows = std::min(MBp, T - r0);
      std::vector<int> idx(rows);
      for (int i = 0; i < rows; ++i) idx[i] = r0 + i;
      cudaMemcpyAsync(w->d_last_idx, idx.data(), rows * 4, cudaMemcpyHostToDevice, w->stream);
      cudaStreamSynchronize(w->stream);
      rc = run_head(w, false, w->d_last_idx, rows, pp, &nl);
      if (rc) break;
      float* dst = all_positions ? out + (size_t)(p0 + r0) * c.vocab : out;
      if (cudaMemcpyAsync(dst, w->logits, (size_t)rows * c.vocab * 4, cudaMemcpyDeviceToHost, w->stream) != cudaSuccess)
        rc = MQ_ERR_CUDA;
      cudaStreamSynchronize(w->stream);
    }
  }
  cudaError_t e = cudaStreamSynchronize(w->stream);
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) { set_last_error("mq_debug_forward: %s", cudaGetErrorString(e)); rc = MQ_ERR_CUDA; }
  for (int i = 0; i < need; ++i) { w->free_pages.push_back(pages[i]); w->h_block_table[i] = 0; }
  w->slots_dirty = true;
  return rc;
}

static int run_job(mq_worker* w, std::function<int()> fn) {
  std::mutex m;
  std::condition_variable cv;
  bool done = false;
  int rc = 0;
  std::string err;
  {
    std::lock_guard<std::mutex> g(w->mu);
    w->jobs.push_back([&] {
      rc = fn();
      err = mq_last_error();
      std::lock_guard<std::mutex> g2(m);
      done = true;
      cv.notify_all();
    });
  }
  w->cv.notify_all();
  std::unique_lock<std::mutex> lk(m);
  cv.wait(lk, [&] { return done; });
  if (rc != MQ_OK) set_last_error("%s", err.c_str());
  return rc;
}

}  // namespace mq

// ================================================================================================ C ABI
using namespace mq;

extern "C" {

int mq_worker_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  int ok = 0;
  for (int i = 0; i < n; ++i) {
    cudaDeviceProp p;
    if (cudaGetDeviceProperties(&p, i) == cudaSuccess && p.major == 10) ++ok;
  }
  return ok;
}

int mq_worker_open(int32_t gpu, const mq_model_cfg* cfg, mq_worker** out) {
  if (!cfg || !out) return MQ_ERR_INVAL;
  *out = nullptr;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || gpu < 0 || gpu >= n) {
    cudaGetLastError();
    set_last_error("no CUDA device %d (this library has no CPU fallback)", gpu);
    return MQ_ERR_NODEV;
  }
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, gpu));
  if (prop.major != 10) {
    set_last_error("device %d is sm_%d%d; this library is built for sm_100a only", gpu, prop.major, prop.minor);
    return MQ_ERR_NODEV;
  }
  const mq_model_cfg& c = *cfg;
  if (!head_dim_supported(c.head_dim) || (c.n_q_heads * c.head_dim) % 64 != 0 || c.hidden % 512 != 0 || c.hidden % 64 != 0 || c.ffn % 128 != 0 ||
      c.n_q_heads % c.n_kv_heads != 0 || c.n_q_heads / c.n_kv_heads > 8 || kPrefillTileRows / (c.n_q_heads / c.n_kv_heads) < 1 || c.vocab % 4 != 0 ||
      c.max_batch < 1 || c.max_batch > 256 || c.max_seq < 1 || c.max_prefill_tokens < 16 || c.n_layers < 1) {
    set_last_error("unsupported model geometry (need head_dim 128 / 96 / 64, hidden %% 512 == 0, ffn %% 128 == 0, "
                   "vocab %% 4 == 0, GQA group <= 8, 1 <= max_batch <= 256)");
    return MQ_ERR_INVAL;
  }
  CUDA_TRY(cudaSetDevice(gpu));
  mq_worker* w = new (std::nothrow) mq_worker();
  if (!w) return MQ_ERR_NOMEM;
  w->cfg = c;
  w->cfg.model_name[sizeof(w->cfg.model_name) - 1] = 0;
  w->gpu = gpu;
  w->sm_count = prop.multiProcessorCount;
  CUDA_TRY(cudaStreamCreateWithFlags(&w->stream, cudaStreamNonBlocking));
  gemm_set_attrs();
  attn_set_attrs();
  attn_tc_set_attrs();
  int rc = worker_alloc(w);
  if (rc != MQ_OK) {
    mq_worker_close(w);
    return rc;
  }
  w->thr = std::thread(worker_main, w);
  *out = w;
  return MQ_OK;
}

void mq_worker_close(mq_worker* w) {
  if (!w) return;
  if (w->thr.joinable()) {
    { std::lock_guard<std::mutex> g(w->mu); w->stop = true; }
    w->cv.notify_all();
    w->thr.join();
  }
  cudaSetDevice(w->gpu);
  {
    std::lock_guard<std::mutex> g(w->mu);
    for (mq_req* r : w->inbox) {
      if (r->cb.on_done) r->cb.on_done(r->user, MQ_ERR_CANCELED, "worker closed");
      req_unref(r);
    }
    w->inbox.clear();
  }
  if (w->stream) cudaStreamSynchronize(w->stream);
  for (auto& kv : w->graphs) cudaGraphExecDestroy(kv.second);
  streamk_workspace_free(&w->sk_ws);
  w->allocs.free_all();
  for (auto e : w->stage_ev) cudaEventDestroy(e);
  for (auto e : w->ev_pool) cudaEventDestroy(e);
  if (w->stream) cudaStreamDestroy(w->stream);
  delete w;
}

static DevTensor* find_tensor(mq_worker* w, const char* name) {
  if (!w || !name) return nullptr;
  auto it = w->tensors.find(name);
  if (it == w->tensors.end()) {
    set_last_error("unknown tensor '%s'", name);
    return nullptr;
  }
  return &it->second;
}

int mq_worker_load_tensor(mq_worker* w, const char* name, const void* src, size_t nbytes) {
  DevTensor* t = find_tensor(w, name);
  if (!t) return MQ_ERR_NOENT;
  if (nbytes != t->bytes) {
    set_last_error("tensor '%s': got %zu bytes, expected %zu", name, nbytes, t->bytes);
    return MQ_ERR_INVAL;
  }
  cudaSetDevice(w->gpu);
  CUDA_TRY(cudaMemcpy(t->ptr, src, nbytes, cudaMemcpyDefault));
  return MQ_OK;
}

int mq_worker_read_tensor(mq_worker* w, const char* name, void* dst, size_t nbytes) {
  DevTensor* t = find_tensor(w, name);
  if (!t) return MQ_ERR_NOENT;
  if (nbytes != t->bytes) {
    set_last_error("tensor '%s': asked %zu bytes, tensor has %zu", name, nbytes, t->bytes);
    return MQ_ERR_INVAL;
  }
  cudaSetDevice(w->gpu);
  CUDA_TRY(cudaMemcpy(dst, t->ptr, nbytes, cudaMemcpyDefault));
  return MQ_OK;
}

int mq_worker_init_random(mq_worker* w, uint64_t seed, float std) {
  if (!w) return MQ_ERR_INVAL;
  cudaSetDevice(w->gpu);
  uint64_t k = 0;
  for (auto& kv : w->tensors) {  // std::map: deterministic name order
    const bool is_norm = kv.first.find("norm") != std::string::npos;
    const bool is_bias = kv.first.find("bqkv") != std::string::npos;
    __nv_bfloat16* p = (__nv_bfloat16*)kv.second.ptr;
    const size_t n = kv.second.bytes / 2;
    if (is_norm) launch_fill_bf16(0, p, n, 1.0f);
    else if (is_bias) launch_fill_bf16(0, p, n, 0.0f);
    else launch_init_normal(0, p, n, seed * 0x9E3779B97F4A7C15ull + (++k) * 0xD6E8FEB86659FD93ull, std);
  }
  CUDA_TRY(cudaDeviceSynchronize());
  return MQ_OK;
}

int mq_worker_capacity(mq_worker* w) { return w ? w->MB : 0; }
int mq_worker_healthy(mq_worker* w) { return w && w->healthy.load() && !w->probe_fail.load() ? 1 : 0; }
int mq_debug_worker_set_probe_fail(mq_worker* w, int32_t probe_fail) {
  if (!w) return MQ_ERR_INVAL;
  w->probe_fail.store(probe_fail != 0);
  return MQ_OK;
}
int mq_debug_worker_inject_fault(mq_worker* w, const char* msg) {
  if (!w) return MQ_ERR_INVAL;
  {
    std::lock_guard<std::mutex> g(w->mu);  // w->fatal is read by the worker thread after it sees healthy == false
    w->fatal = std::string("GPU fault: ") + (msg ? msg : "injected");
  }
  w->healthy.store(false);
  w->cv.notify_all();
  return MQ_OK;
}

int mq_submit(mq_worker* w, const mq_request* rq, const mq_callbacks* cb, void* user, mq_req** out) {
  if (!w || !rq || !cb) return MQ_ERR_INVAL;
  if (!w->healthy.load()) {
    set_last_error("worker unhealthy: %s", w->fatal.c_str());
    return MQ_ERR_CUDA;
  }
  mq_req* r = new (std::nothrow) mq_req();
  if (!r) return MQ_ERR_NOMEM;
  r->w = w;
  r->rq = *rq;
  r->cb = *cb;
  r->user = user;
  r->t_submit = Clock::now();
  if (rq->body && rq->body_len) r->body.assign((const char*)rq->body, rq->body_len);
  if (rq->path) r->path = rq->path;
  r->rq.path = nullptr;
  if (rq->endpoint == MQ_EP_OTHER) {  // answered on the worker thread without touching the GPU
    r->rq.body = nullptr; r->rq.prompt_tokens = nullptr;
    if (out) *out = r; else r->refs.store(1);
    { std::lock_guard<std::mutex> g(w->mu); w->inbox.push_back(r); }
    w->cv.notify_all();
    return MQ_OK;
  }
  ParsedBody pb;
  const bool text_body = rq->body_kind == MQ_BODY_TEXT;  // the front parsed the JSON already (dispatcher.cpp)
  if (!r->body.empty() && !text_body && !(rq->prompt_tokens && rq->n_prompt_tokens > 0) &&
      !parse_body(r->body, rq->endpoint, &pb)) {
    // what the backend of the reference answers to a malformed body: 400 + {"error": ...}, relayed like any response
    r->bad_request = true;
    r->rq.body = nullptr; r->rq.prompt_tokens = nullptr;
    if (out) *out = r; else r->refs.store(1);
    { std::lock_guard<std::mutex> g(w->mu); w->inbox.push_back(r); }
    w->cv.notify_all();
    return MQ_OK;
  }
  if (rq->prompt_tokens && rq->n_prompt_tokens > 0)
    r->prompt.assign(rq->prompt_tokens, rq->prompt_tokens + rq->n_prompt_tokens);
  else if (!pb.tokens.empty())
    r->prompt = pb.tokens;
  else
    r->prompt = byte_tokenize(text_body ? r->body : pb.text, w->cfg.vocab);
  if (r->prompt.empty()) r->prompt.push_back(0);
  for (int32_t& t : r->prompt) if (t < 0 || t >= w->cfg.vocab) t = 0;
  r->rq.body = nullptr; r->rq.prompt_tokens = nullptr;
  apply_body(pb, &r->rq);  // a no-op when there was no JSON body to parse; from here on only r->rq is read
  if (r->rq.stream < 0) r->rq.stream = 1;
  // generation length: validated BEFORE any arithmetic with the prompt length ("num_predict": 2147483647 used to wrap
  // prompt + max_new negative, pass both checks below and die in vector::resize on the worker thread)
  long long want = r->rq.max_new_tokens > 0 ? r->rq.max_new_tokens : 128;
  if (want > (long long)w->cfg.max_seq - (long long)r->prompt.size()) {
    const int n = (int)r->prompt.size();
    delete r;
    set_last_error("prompt (%d) + max_new_tokens (%lld) exceeds max_seq %d", n, want, w->cfg.max_seq);
    return MQ_ERR_INVAL;
  }
  r->max_new = (int)want;
  // sampling: everything unset = greedy (what BASELINE measures); NaN from a C-ABI caller is greedy / off too
  SamplingParams& sp = r->sp;
  sp.temperature = r->rq.temperature == r->rq.temperature ? r->rq.temperature : 0.f;
  sp.top_k = r->rq.top_k;
  sp.top_p = r->rq.top_p == r->rq.top_p ? r->rq.top_p : 0.f;
  sp.seed = r->rq.seed;
  if (r->rq.logprobs) sp.top_logprobs = std::max(0, std::min<int>(r->rq.top_logprobs, MQ_TOP_LOGPROBS_MAX));
  if (((long long)r->prompt.size() + r->max_new + kPageSize - 1) / kPageSize > w->n_pages - 1) {
    delete r;
    set_last_error("request needs more KV pages than the worker owns (%d)", w->n_pages - 1);
    return MQ_ERR_NOMEM;
  }
  if (r->rq.timeout_ms) {
    r->has_deadline = true;
    r->deadline = r->t_submit + std::chrono::milliseconds(r->rq.timeout_ms);
  }
  if (out) *out = r; else r->refs.store(1);
  {
    std::lock_guard<std::mutex> g(w->mu);
    w->inbox.push_back(r);
  }
  w->cv.notify_all();
  return MQ_OK;
}

void mq_cancel(mq_req* r) {
  if (!r) return;
  r->cancel.store(true);
  if (r->w) r->w->cv.notify_all();
}

void mq_req_release(mq_req* r) {
  if (r) req_unref(r);
}

int mq_req_get_stats(mq_req* r, mq_req_stats* out) {
  if (!r || !out) return MQ_ERR_INVAL;
  using us = std::chrono::microseconds;
  out->n_prompt = (int)r->prompt.size();
  out->n_generated = r->n_emitted;
  out->ttft_us = r->n_emitted > 0 ? (uint64_t)std::chrono::duration_cast<us>(r->t_first - r->t_submit).count() : 0;
  out->total_us = r->finished ? (uint64_t)std::chrono::duration_cast<us>(r->t_last - r->t_submit).count() : 0;
  return MQ_OK;
}

int mq_worker_get_stats(mq_worker* w, mq_worker_stats* out) {
  if (!w || !out) return MQ_ERR_INVAL;
  std::lock_guard<std::mutex> g(w->stats_mu);
  *out = w->stats;
  return MQ_OK;
}
int mq_worker_get_occupancy(mq_worker* w, mq_worker_occupancy* out) {
  if (!w || !out) return MQ_ERR_INVAL;
  return run_job(w, [=] {  // on the worker thread: slot table, page pool and queues are owned by it
    out->total_pages = (uint64_t)w->n_pages - 1;  // page 0 is the scratch page
    out->free_pages = (uint64_t)w->free_pages.size();
    uint64_t act = 0;
    for (mq_req* r : w->slot_req) act += r != nullptr;
    out->active_slots = act;
    out->waiting = (uint64_t)(w->waiting.size() + w->prefilling.size());
    out->in_flight_gpu_passes = (uint64_t)w->flights.size();
    return (int)MQ_OK;
  });
}
int mq_worker_reset_stats(mq_worker* w) {
  if (!w) return MQ_ERR_INVAL;
  std::lock_guard<std::mutex> g(w->stats_mu);
  w->stats = mq_worker_stats{};
  return MQ_OK;
}
int mq_debug_trace_read(mq_worker* w, unsigned long long* out, int32_t max_slots) {
  if (!w || !out || max_slots < 1) return MQ_ERR_INVAL;
  if (!w->d_trace) {
    set_last_error("mq_debug_trace_read: the worker was opened without MQ_TRACE=1");
    return MQ_ERR_INVAL;
  }
  const int n = std::min((int)max_slots, kTraceSlots);
  const int rc = run_job(w, [=] {
    if (cudaStreamSynchronize(w->stream) != cudaSuccess) return (int)MQ_ERR_CUDA;
    if (cudaMemcpy(out, w->d_trace, (size_t)n * 4 * 8, cudaMemcpyDeviceToHost) != cudaSuccess) return (int)MQ_ERR_CUDA;
    return (int)MQ_OK;
  });
  return rc < 0 ? rc : n;
}
int mq_worker_set_timing(mq_worker* w, int32_t enable) {
  if (!w) return MQ_ERR_INVAL;
  w->timing = enable != 0;
  return MQ_OK;
}

int mq_debug_forward(mq_worker* w, const int32_t* tokens, int32_t n, int32_t all_positions, float* logits_out) {
  if (!w || !tokens || !logits_out) return MQ_ERR_INVAL;
  return run_job(w, [=] { return engine_forward_logits(w, tokens, n, all_positions, logits_out); });
}

}  // extern "C"
