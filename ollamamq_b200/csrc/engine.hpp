// GPU worker runtime: one per B200.  Owns the weights, the paged KV cache, the slot table and a host thread
// that runs continuous batching (prefill passes + CUDA-graphed decode steps) and fires the C-ABI callbacks.
// This is what stands where the reference has `reqwest -> remote Ollama` (dispatcher.rs:287-312).
#pragma once
#include "../../include/ollamamq_b200.h"
#include "framing.hpp"
#include "gemm_host.cuh"
#include "kernels.cuh"
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <deque>
#include <functional>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

namespace mq {
using Clock = std::chrono::steady_clock;

struct DevTensor {
  void* ptr = nullptr;
  size_t bytes = 0;
};

// Owner of every device and pinned host allocation of a worker or an encoder: each one is recorded when it is made and
// free_all releases them together, so a close after a partial setup frees exactly what setup got.
struct Allocations {
  std::vector<void*> dev_ptrs, host_ptrs;
  int alloc(void** p, size_t bytes, bool pinned_host);  // MQ_ERR_NOMEM (with the error text set) on failure
  template <typename T> int dev(T** p, size_t n) { return alloc(reinterpret_cast<void**>(p), n * sizeof(T), false); }
  template <typename T> int host(T** p, size_t n) { return alloc(reinterpret_cast<void**>(p), n * sizeof(T), true); }
  void free_all();
};

// Per-request sampling settings, also one entry per slot in the worker's slot table
struct SamplingParams {
  float temperature = 0.f;  // <= 0: greedy
  int top_k = 0;            // <= 0: off
  float top_p = 0.f;        // <= 0 or >= 1: off
  unsigned long long seed = 0;
  int top_logprobs = -1;  // -1: no logprobs; 0..MQ_TOP_LOGPROBS_MAX: a record per relayed token with that many alternatives
};

struct LayerWeights {
  __nv_bfloat16 *attn_norm, *wqkv, *bqkv, *wo, *mlp_norm, *w_gate_up, *w_down;
};

// All GEMM plans for one activation-row count T (decode bucket or prefill pass size).
struct PassPlans {
  int T = 0;
  bool decode = false;
  int s_qkv = 1, s_o = 1, s_down = 1;
  std::vector<GemmPlan> qkv, o, gate_up, down;  // per layer
  // decode chain (gemm_dk.cuh): O and down are cluster split-K GEMMs with the residual add / next-norm partials fused,
  // RMSNorm itself is folded into the consumers' epilogues - 6 launches per layer instead of 8, no norm kernels;
  // `qkv` (planes) and `gate_up` then carry the rstd fold
  bool chain = false;
  std::vector<DkPlan> o_dk, down_dk;
  // prefill with the same fold (all four GEMMs on the persistent 2-CTA kernel): O / down add into the residual stream and
  // emit xg + h^2 partials (EPI_RESID), QKV / gate-up scale by rstd - no add_rmsnorm launches (4 GEMMs + rope + attention)
  bool pfold = false;
};

}  // namespace mq

struct mq_req {
  std::atomic<int> refs{2};  // caller handle + engine
  mq_worker* w = nullptr;
  mq_request rq{};
  std::vector<int32_t> prompt;
  std::string body;
  std::string path;
  mq_callbacks cb{};
  void* user = nullptr;
  int slot = -1;
  int n_prefilled = 0;   // prompt tokens whose KV is (or is scheduled to be) in the cache
  int n_sched = 0;       // generated tokens scheduled on the GPU so far
  int n_emitted = 0;     // generated tokens delivered to the callback
  int max_new = 0;
  mq::SamplingParams sp;
  size_t text_len = 0;    // characters relayed so far (/v1/completions text_offset)
  std::vector<mq::TokenLogprobs> agg_lp;  // stream=0 with logprobs: every relayed token's entry
  std::atomic<bool> cancel{false};
  bool status_sent = false;
  bool finished = false;
  bool stopped = false;  // ended on the model's EOS token rather than on max_new
  bool bad_request = false;  // malformed JSON body: answered 400 on the worker thread, never scheduled
  int done_rc = 0;
  std::string agg;       // stream=0: aggregated text
  std::vector<int32_t> agg_tokens;
  std::vector<int> pages;
  mq::Clock::time_point t_submit, t_first, t_last, deadline;
  bool has_deadline = false;
};

constexpr int kTraceSlots = 512;

struct mq_worker {
  mq_model_cfg cfg{};
  int gpu = 0;
  int sm_count = 148;
  cudaStream_t stream = nullptr;
  int qkv_dim = 0, max_pages = 0, n_pages = 0, MT = 0, MB = 0;
  double p_mm_bytes = 0, kv_bytes_per_tok = 0;
  mq::Allocations allocs;  // owns every buffer below (weights included) except the stream-K workspace

  // weights
  std::map<std::string, mq::DevTensor> tensors;
  std::vector<mq::LayerWeights> layers;
  __nv_bfloat16 *embed = nullptr, *final_norm = nullptr, *lm_head = nullptr;
  __nv_bfloat16 *k_cache = nullptr, *v_cache = nullptr;  // [layers][pages][n_kv][16][128]
  size_t cache_layer_stride = 0;

  // activations
  float* h = nullptr;
  __nv_bfloat16 *x = nullptr, *q = nullptr, *attn = nullptr, *act = nullptr, *x_last = nullptr;
  void *qkv_part = nullptr, *proj_part = nullptr;
  float *logits = nullptr, *part_o = nullptr, *part_ml = nullptr, *inv_freq = nullptr;
  float2* rope_table = nullptr;  // [max_seq][head_dim / 2] (cos, sin)
  // metadata (device)
  int *d_tok = nullptr, *d_pos_tok = nullptr, *d_slot_tok = nullptr, *d_last_idx = nullptr, *d_dst_slot = nullptr;
  int4* d_tiles = nullptr;
  int *d_cur_token = nullptr, *d_identity = nullptr;
  // slot table: a pinned host mirror (h_slots) and its device copy (d_slots) with one layout, sections of MBp entries
  // pos | active | temperature | top_k | top_p | seed | top_logprobs | block_table, uploaded whole when it changed.
  // The d_* / h_* pointers below are views into the two blocks (captured graphs read the d_* views).
  uint8_t *d_slots = nullptr, *h_slots = nullptr;
  size_t slot_bytes = 0;
  int *d_pos = nullptr, *d_active = nullptr, *d_block_table = nullptr;
  int *h_pos = nullptr, *h_active = nullptr, *h_block_table = nullptr;
  float *d_temp = nullptr, *d_topp = nullptr, *h_temp = nullptr, *h_topp = nullptr;
  int *d_topk = nullptr, *h_topk = nullptr;
  unsigned long long *d_seed = nullptr, *h_seed = nullptr;
  int *d_lp_top = nullptr, *h_lp_top = nullptr;  // top_logprobs per slot, -1 = off (read by the sampler, graphs included)
  int* d_out_ring = nullptr;  // [kRing][MB]
  mq::LogprobRec* d_lp_ring = nullptr;  // [kRing][MB] records beside d_out_ring, copied out only when a slot asked
  int* d_split_counter = nullptr;  // [MB][n_kv] arrival counters of the split-KV decode attention
  // decode chain: per-weight-tile partial sums of h^2 (RMSNorm fold, gemm.cuh RstdIn), [tiles][round_up(MB, 16)]
  float *ssq_e = nullptr, *ssq_o = nullptr, *ssq_d = nullptr;
  int ssq_stride = 0;        // tokens per partial row: max(prefill pass, decode batch)
  // prefill attention on tcgen05 (attn_tc.cu): tensor maps of q and of every layer's K / V cache; 128-row query tiles
  bool attn_tc = false;      // head_dim 128 && MQ_ATTN_TC != 0
  int prefill_tile_rows = 64;
  CUtensorMap tm_q;
  std::vector<CUtensorMap> tm_k, tm_v;
  bool chain = true;         // MQ_DECODE_CHAIN=0: the round-1 plane-based decode path (A/B and parity cross-check)
  unsigned long long* d_trace = nullptr;  // MQ_TRACE=1: [kTraceSlots][4] %globaltimer stamps of the latest pass
  // pinned host staging
  int* h_stage = nullptr;     // ring of staging areas for metadata uploads
  int* h_out_ring = nullptr;  // [kRing][MB]
  mq::LogprobRec* h_lp_ring = nullptr;  // [kRing][MB]
  size_t stage_ints = 0;
  int stage_next = 0;
  std::vector<cudaEvent_t> stage_ev;

  mq::StreamKWorkspace sk_ws;
  std::map<int, mq::PassPlans> plans_decode, plans_prefill;
  std::map<long long, cudaGraphExec_t> graphs;  // key: Bcap * 1024 + n_splits
  std::map<int, mq::GemmPlan> lm_plans;          // key: rows

  // slots / pages
  std::vector<mq_req*> slot_req;
  std::vector<int> free_pages;
  bool slots_dirty = false;

  // threading
  std::thread thr;
  std::mutex mu;
  std::condition_variable cv;
  std::deque<mq_req*> inbox;
  std::deque<std::function<void()>> jobs;
  bool stop = false;
  std::atomic<bool> healthy{true};
  std::atomic<bool> probe_fail{false};  // fault injection: the health probe fails while the engine keeps serving
  std::string fatal;

  // in-flight GPU work (FIFO)
  struct Flight {
    cudaEvent_t ev;
    cudaEvent_t ev_begin;  // timing only
    bool timed = false;
    bool decode = false;
    int ring = 0;
    double bytes = 0;
    std::vector<std::pair<mq_req*, int>> emits;  // (request, index into h_out_ring row and h_lp_ring row)
  };
  std::deque<Flight> flights;
  std::vector<cudaEvent_t> ev_pool;
  int ring_next = 0;

  std::deque<mq_req*> waiting;   // admitted-pending (no slot yet)
  std::deque<mq_req*> prefilling;  // have a slot, prompt not fully prefilled

  // stats
  mq_worker_stats stats{};
  bool timing = false;
  std::mutex stats_mu;
};

namespace mq {
int engine_forward_logits(mq_worker* w, const int32_t* tokens, int n, int all_positions, float* out);
}
