// Embedding worker: a BERT-family encoder on one B200 (BASELINE.json configs[4]: bge-small behind /api/embed).
//
// Stands where the reference forwards /api/embed, /api/embeddings and /v1/embeddings to the external backend
// (route table main.rs:89-121, executor dispatcher.rs:287-312).  It is a sibling of the generation worker
// (engine.cu) on the same GPU - own stream, own host thread - so embedding batches interleave with chat decode
// steps exactly as two models share one Ollama instance.
//
// One pass = whole sequences packed back to back (<= max_tokens_per_pass tokens, <= max_seqs sequences):
//   embeddings + LayerNorm -> per layer [ QKV GEMM (tcgen05) with the bias added in the epilogue -> bidirectional flash
//   attention reading q / k / v straight out of the packed [T, 3H] activation (an encoder keeps no cache, so there is
//   no paging and no scatter kernel: r01 measured the decoder's rope/scatter kernel at 47 us per layer for what is a
//   pure copy here) -> O GEMM -> bias + residual + LayerNorm -> up GEMM with bias + erf-GELU epilogue -> down GEMM ->
//   bias + residual + LayerNorm ] -> [CLS] pooling + L2 normalisation.
#include "engine.hpp"
#include "framing.hpp"
#include <algorithm>
#include <cmath>
#include <cstring>
#include <new>

namespace mq {
void set_last_error(const char* fmt, ...);
}
using namespace mq;

#define ENC_TRY(expr)                                                                              \
  do {                                                                                             \
    cudaError_t _e = (expr);                                                                       \
    if (_e != cudaSuccess) {                                                                       \
      set_last_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return MQ_ERR_CUDA;                                                                          \
    }                                                                                              \
  } while (0)

namespace {
struct EncLayer {
  __nv_bfloat16 *wqkv, *bqkv, *wo, *bo, *attn_ln_g, *attn_ln_b, *w_up, *b_up, *w_down, *b_down, *mlp_ln_g, *mlp_ln_b;
};
struct EncJob {
  std::vector<std::vector<int32_t>> seqs;
  std::vector<float> out;  // [n_seq][H]
  // async (dispatcher) form
  mq_req* req = nullptr;
  std::string path, model;
  // blocking form
  bool done = false;
  int rc = 0;
  std::string err;
};
constexpr int kEncTileRows = kPrefillTileRows;  // query rows per attention CTA (GQA group of 1: rows = tokens)
}  // namespace

struct mq_encoder {
  mq_encoder_cfg cfg{};
  int gpu = 0;
  cudaStream_t stream = nullptr;
  Allocations allocs;  // every buffer below (weights included) is owned here
  std::map<std::string, DevTensor> tensors;
  __nv_bfloat16 *word = nullptr, *pos_emb = nullptr, *type_emb = nullptr, *emb_g = nullptr, *emb_b = nullptr;
  std::vector<EncLayer> layers;
  int MT = 0, max_seqs = 0;
  // activations
  float *h = nullptr, *d_out = nullptr;
  __nv_bfloat16 *x = nullptr, *qkv = nullptr, *attn = nullptr, *sub = nullptr, *act = nullptr;
  CUtensorMap tm_qkv{};   // tcgen05 attention: {32 d, 64 rows} boxes of the packed q | k | v activation
  bool attn_tc = false;
  bool rowln = false;      // O / down projections fused with bias + residual + LayerNorm (gemm_rowln.cuh)
  int* d_meta = nullptr;  // tok | pos | first_tok | seq_len | tiles
  int* h_meta = nullptr;                            // pinned mirror
  float* h_out = nullptr;                           // pinned [max_seqs][H]
  size_t meta_ints = 0;
  // threading
  std::thread thr;
  std::mutex mu;
  std::condition_variable cv, cv_done;
  std::deque<EncJob*> queue;
  bool stop = false;
  // replies (JSON framing + callbacks) run on their own thread: a 64 x 384 reply takes ~1 ms to format, a third of the
  // GPU time of the request it answers, and the pass thread has the next request's pass to launch
  std::thread reply_thr;
  std::mutex reply_mu;
  std::condition_variable reply_cv;
  std::deque<std::pair<EncJob*, int>> replies;
  bool reply_stop = false;
  std::atomic<bool> healthy{true};
  std::atomic<uint64_t> passes{0}, sequences{0}, tokens{0}, launches{0}, gpu_us{0};
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
};

namespace {

int enc_tensor(mq_encoder* e, const std::string& name, size_t n, __nv_bfloat16** out) {
  int rc = e->allocs.dev(out, n);
  if (rc) return rc;
  e->tensors[name] = DevTensor{*out, n * 2};
  return MQ_OK;
}

int enc_setup(mq_encoder* e) {
  const mq_encoder_cfg& c = e->cfg;
  const int H = c.hidden, I = c.ffn, L = c.n_layers;
  int rc;
#define T_(name, n, field) if ((rc = enc_tensor(e, name, (size_t)(n), &field))) return rc
  T_("word_embed", (size_t)c.vocab * H, e->word);
  T_("pos_embed", (size_t)c.max_positions * H, e->pos_emb);
  T_("type_embed", (size_t)c.type_vocab * H, e->type_emb);
  T_("emb_ln_g", H, e->emb_g);
  T_("emb_ln_b", H, e->emb_b);
  e->layers.resize(L);
  for (int l = 0; l < L; ++l) {
    const std::string p = "layers." + std::to_string(l) + ".";
    EncLayer& w = e->layers[l];
    T_(p + "wqkv", (size_t)3 * H * H, w.wqkv);
    T_(p + "bqkv", 3 * H, w.bqkv);
    T_(p + "wo", (size_t)H * H, w.wo);
    T_(p + "bo", H, w.bo);
    T_(p + "attn_ln_g", H, w.attn_ln_g);
    T_(p + "attn_ln_b", H, w.attn_ln_b);
    T_(p + "w_up", (size_t)I * H, w.w_up);
    T_(p + "b_up", I, w.b_up);
    T_(p + "w_down", (size_t)H * I, w.w_down);
    T_(p + "b_down", H, w.b_down);
    T_(p + "mlp_ln_g", H, w.mlp_ln_g);
    T_(p + "mlp_ln_b", H, w.mlp_ln_b);
  }
#undef T_
  e->MT = (std::max(c.max_tokens_per_pass, c.max_seq) + 255) / 256 * 256;
  e->max_seqs = std::max(1, std::min(1024, e->MT / 8));
  const size_t MT = e->MT;
  Allocations& m = e->allocs;
  if ((rc = m.dev(&e->h, MT * H))) return rc;
  if ((rc = m.dev(&e->x, MT * H))) return rc;
  if ((rc = m.dev(&e->qkv, MT * 3 * H))) return rc;
  // the tcgen05 attention loads whole 64-row boxes: rows past a pass's last token must hold finite values (they meet
  // probabilities of exactly 0)
  ENC_TRY(cudaMemset(e->qkv, 0, MT * 3 * H * sizeof(__nv_bfloat16)));
  const char* tc_env = getenv("MQ_ENC_ATTN_TC");
  e->attn_tc = enc_attn_tc_supported(c.head_dim, c.max_seq, H) && !(tc_env && tc_env[0] == '0') &&
               enc_attn_tc_encode(&e->tm_qkv, e->qkv, (int)MT, H);
  if (e->attn_tc) enc_attn_tc_set_attrs();
  const char* rl_env = getenv("MQ_ENC_ROWLN");
  e->rowln = rowln_supported(H, H) && rowln_supported(H, I) && !(rl_env && rl_env[0] == '0');
  if ((rc = m.dev(&e->attn, MT * H))) return rc;
  if ((rc = m.dev(&e->sub, MT * H))) return rc;
  if ((rc = m.dev(&e->act, MT * I))) return rc;
  if ((rc = m.dev(&e->d_out, (size_t)e->max_seqs * H))) return rc;
  const size_t max_tiles = MT / kEncTileRows + e->max_seqs + 1;
  e->meta_ints = 2 * MT + 2 * (size_t)e->max_seqs + 4 * max_tiles;
  if ((rc = m.dev(&e->d_meta, e->meta_ints)) || (rc = m.host(&e->h_meta, e->meta_ints)) ||
      (rc = m.host(&e->h_out, (size_t)e->max_seqs * H)))
    return rc;
  return MQ_OK;
}

// one pass over `n` whole sequences; results land in e->h_out[0 .. n*H)
int enc_pass(mq_encoder* e, const std::vector<const std::vector<int32_t>*>& seqs) {
  const mq_encoder_cfg& c = e->cfg;
  const int H = c.hidden, I = c.ffn, n = (int)seqs.size();
  const LaunchCfg lc{e->stream, c.use_pdl != 0};
  int T = 0;
  for (auto* s : seqs) T += (int)s->size();
  int *m_tok = e->h_meta, *m_pos = m_tok + e->MT, *m_first = m_pos + e->MT, *m_len = m_first + e->max_seqs,
      *m_tiles = m_len + e->max_seqs;
  int t = 0, n_tiles = 0;
  for (int s = 0; s < n; ++s) {
    const int len = (int)seqs[s]->size();
    m_first[s] = t;
    m_len[s] = len;
    for (int i = 0; i < len; ++i) {
      const int id = (*seqs[s])[i];
      m_tok[t + i] = id < 0 ? 0 : (id >= c.vocab ? c.vocab - 1 : id);
      m_pos[t + i] = i;
    }
    if (e->attn_tc) {
      for (int i = 0; i < len; i += kEncAttnItemRows) {
        int* tl = m_tiles + 4 * n_tiles++;
        tl[0] = t + i; tl[1] = std::min(kEncAttnItemRows, len - i); tl[2] = t; tl[3] = len;
      }
    } else {
      for (int i = 0; i < len; i += kEncTileRows) {
        int* tl = m_tiles + 4 * n_tiles++;
        tl[0] = t + i; tl[1] = std::min(kEncTileRows, len - i); tl[2] = s; tl[3] = i;
      }
    }
    t += len;
  }
  ENC_TRY(cudaEventRecord(e->ev0, e->stream));
  ENC_TRY(cudaMemcpyAsync(e->d_meta, e->h_meta, e->meta_ints * 4, cudaMemcpyHostToDevice, e->stream));
  const int *d_tok = e->d_meta, *d_pos = d_tok + e->MT, *d_first = d_pos + e->MT;
  const int* d_len = d_first + e->max_seqs;
  const int4* d_tiles = reinterpret_cast<const int4*>(d_len + e->max_seqs);
  static_assert(sizeof(int4) == 16, "tiles are 4 ints");
  uint64_t nl = 0;
  launch_enc_embed_ln(lc, d_tok, d_pos, e->word, e->pos_emb, e->type_emb, e->emb_g, e->emb_b, e->h, e->x, T, H, c.ln_eps);
  ++nl;
  for (int l = 0; l < c.n_layers; ++l) {
    const EncLayer& w = e->layers[l];
    GemmPlan g;
    if (!gemm_plan(&g, w.wqkv, 3 * H, 3 * H, H, e->x, e->MT, T, EPI_BIAS_BF16, e->qkv, 3 * H, 1, 0, 0)) return MQ_ERR_CUDA;
    gemm_plan_set_bias(&g, w.bqkv);
    if (gemm_launch(g, lc) != cudaSuccess) return MQ_ERR_CUDA;
    const float scale_log2 = (1.0f / sqrtf((float)c.head_dim)) * 1.4426950408889634f;
    if (e->attn_tc) {
      if (launch_enc_attn_tc(lc, e->tm_qkv, d_tiles, n_tiles, c.n_heads, H, e->attn, scale_log2) != cudaSuccess) {
        set_last_error("encoder attention launch failed: %s", cudaGetErrorString(cudaGetLastError()));
        return MQ_ERR_CUDA;
      }
    } else {
      AttnParams ap = {};
      ap.head_dim = c.head_dim; ap.bidirectional = 1; ap.seq_len = d_len;
      ap.seq_start = d_first; ap.row_stride = 3 * H;          // packed mode: q | k | v column blocks of e->qkv
      ap.q = e->qkv; ap.k_cache = e->qkv + H; ap.v_cache = e->qkv + 2 * H;
      ap.block_table = e->d_meta; ap.max_pages = 0;            // unused in packed mode
      ap.tiles = d_tiles; ap.out = e->attn; ap.n_q = c.n_heads; ap.n_kv = c.n_heads;
      ap.T = T; ap.n_splits = 1; ap.n_warps = 1;
      ap.scale_log2 = scale_log2;
      launch_attn_prefill(lc, ap, n_tiles);
    }
    const bool ln_warp = enc_add_ln_warp_supported(H);
    RowLnPlan rl;
    if (e->rowln) {  // x = LayerNorm(x + attn W_o^T + b_o): one kernel, no `sub` round trip
      if (!rowln_plan(&rl, w.wo, H, H, e->attn, e->MT, T, e->x, w.bo, w.attn_ln_g, w.attn_ln_b, c.ln_eps, nullptr) ||
          rowln_launch(rl, lc) != cudaSuccess)
        return MQ_ERR_CUDA;
    } else {
      if (!gemm_plan(&g, w.wo, H, H, H, e->attn, e->MT, T, EPI_BIAS_BF16, e->sub, H, 1, 0, 0)) return MQ_ERR_CUDA;  // (bias: in the LayerNorm kernel)
      if (gemm_launch(g, lc) != cudaSuccess) return MQ_ERR_CUDA;
      if (ln_warp) launch_enc_add_ln_warp(lc, e->x, e->sub, w.bo, w.attn_ln_g, w.attn_ln_b, nullptr, T, H, c.ln_eps);
      else launch_enc_add_ln(lc, e->h, e->sub, w.bo, w.attn_ln_g, w.attn_ln_b, e->x, T, H, c.ln_eps);
    }
    if (!gemm_plan(&g, w.w_up, I, I, H, e->x, e->MT, T, EPI_GELU_BF16, e->act, I, 1, 0, 0)) return MQ_ERR_CUDA;
    gemm_plan_set_bias(&g, w.b_up);
    if (gemm_launch(g, lc) != cudaSuccess) return MQ_ERR_CUDA;
    float* h_last = l + 1 == c.n_layers ? e->h : nullptr;  // the model's last LayerNorm also leaves an fp32 copy for the pooling kernel
    if (e->rowln) {
      if (!rowln_plan(&rl, w.w_down, H, I, e->act, e->MT, T, e->x, w.b_down, w.mlp_ln_g, w.mlp_ln_b, c.ln_eps, h_last) ||
          rowln_launch(rl, lc) != cudaSuccess)
        return MQ_ERR_CUDA;
    } else {
      if (!gemm_plan(&g, w.w_down, H, H, I, e->act, e->MT, T, EPI_BIAS_BF16, e->sub, H, 1, 0, 0)) return MQ_ERR_CUDA;
      if (gemm_launch(g, lc) != cudaSuccess) return MQ_ERR_CUDA;
      if (ln_warp) launch_enc_add_ln_warp(lc, e->x, e->sub, w.b_down, w.mlp_ln_g, w.mlp_ln_b, h_last, T, H, c.ln_eps);
      else launch_enc_add_ln(lc, e->h, e->sub, w.b_down, w.mlp_ln_g, w.mlp_ln_b, e->x, T, H, c.ln_eps);
    }
    nl += e->rowln ? 5 : 7;
  }
  launch_enc_pool(lc, e->h, d_first, e->d_out, n, H);
  ++nl;
  ENC_TRY(cudaMemcpyAsync(e->h_out, e->d_out, (size_t)n * H * 4, cudaMemcpyDeviceToHost, e->stream));
  ENC_TRY(cudaEventRecord(e->ev1, e->stream));
  ENC_TRY(cudaStreamSynchronize(e->stream));
  float pass_ms = 0.f;
  if (cudaEventElapsedTime(&pass_ms, e->ev0, e->ev1) == cudaSuccess) e->gpu_us += (uint64_t)(pass_ms * 1e3f);
  e->passes++; e->sequences += n; e->tokens += T; e->launches += nl;
  return MQ_OK;
}

int enc_run_job(mq_encoder* e, EncJob* j) {
  const mq_encoder_cfg& c = e->cfg;
  const int H = c.hidden, n = (int)j->seqs.size();
  j->out.assign((size_t)n * H, 0.f);
  for (auto& s : j->seqs) {
    if (s.empty()) s.push_back(0);
    if ((int)s.size() > c.max_seq) s.resize(c.max_seq);  // truncation, like the backend's context limit
  }
  int i = 0;
  while (i < n) {
    if (j->req && j->req->cancel.load()) return MQ_ERR_CANCELED;
    std::vector<const std::vector<int32_t>*> pass;
    int toks = 0, first = i;
    while (i < n && (int)pass.size() < e->max_seqs && toks + (int)j->seqs[i].size() <= e->MT) {
      toks += (int)j->seqs[i].size();
      pass.push_back(&j->seqs[i++]);
    }
    int rc = enc_pass(e, pass);
    if (rc) return rc;
    memcpy(j->out.data() + (size_t)first * H, e->h_out, pass.size() * (size_t)H * 4);
  }
  return MQ_OK;
}

void enc_req_unref(mq_req* r) {
  if (r->refs.fetch_sub(1) == 1) delete r;
}

// Status, one JSON chunk, Done (the relay of dispatcher.rs:294-312) for finished dispatcher-form jobs
void enc_reply_main(mq_encoder* e) {
  for (;;) {
    std::pair<EncJob*, int> it;
    {
      std::unique_lock<std::mutex> lk(e->reply_mu);
      e->reply_cv.wait(lk, [&] { return e->reply_stop || !e->replies.empty(); });
      if (e->replies.empty()) return;  // stop requested and drained
      it = e->replies.front();
      e->replies.pop_front();
    }
    EncJob* j = it.first;
    const int rc = it.second;
    mq_req* r = j->req;
    if (rc == MQ_OK) {
      int n_tok = 0;
      for (auto& s : j->seqs) n_tok += (int)s.size();
      const std::string body = frame_embeddings(j->path, j->model.c_str(), j->out.data(), (int)j->seqs.size(),
                                                e->cfg.hidden, n_tok);
      r->cb.on_status(r->user, 200, "application/json");
      r->cb.on_chunk(r->user, (const uint8_t*)body.data(), body.size());
      r->cb.on_done(r->user, 0, nullptr);
    } else {
      r->cb.on_done(r->user, rc, rc == MQ_ERR_CANCELED ? "cancelled" : "embedding pass failed");
    }
    r->finished = true;
    enc_req_unref(r);
    delete j;
  }
}

void enc_main(mq_encoder* e) {
  cudaSetDevice(e->gpu);
  for (;;) {
    EncJob* j = nullptr;
    {
      std::unique_lock<std::mutex> lk(e->mu);
      e->cv.wait(lk, [&] { return e->stop || !e->queue.empty(); });
      if (e->queue.empty()) return;  // stop requested and drained
      j = e->queue.front();
      e->queue.pop_front();
    }
    int rc = e->healthy.load() ? enc_run_job(e, j) : MQ_ERR_CUDA;
    if (rc == MQ_ERR_CUDA) e->healthy.store(false);  // sticky, like mq_worker_healthy
    if (j->req) {  // dispatcher form: answered by the reply thread, in submission order
      {
        std::lock_guard<std::mutex> g(e->reply_mu);
        e->replies.emplace_back(j, rc);
      }
      e->reply_cv.notify_one();
    } else {
      std::lock_guard<std::mutex> g(e->mu);
      j->rc = rc;
      j->done = true;
      e->cv_done.notify_all();
    }
  }
}

}  // namespace

extern "C" {

int mq_encoder_open(int32_t gpu, const mq_encoder_cfg* cfg, mq_encoder** out) {
  if (!cfg || !out) return MQ_ERR_INVAL;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || gpu < 0 || gpu >= n) {
    set_last_error("no CUDA device %d (the embedding worker has no CPU path)", gpu);
    return MQ_ERR_NODEV;
  }
  cudaDeviceProp prop;
  ENC_TRY(cudaGetDeviceProperties(&prop, gpu));
  if (prop.major != 10) {
    set_last_error("device %d is sm_%d%d; this library is built for sm_100a only", gpu, prop.major, prop.minor);
    return MQ_ERR_NODEV;
  }
  const mq_encoder_cfg& c = *cfg;
  if (c.hidden % 128 != 0 || c.hidden / 4 > 1024 || c.ffn % 64 != 0 || c.n_heads * c.head_dim != c.hidden ||
      !(c.head_dim == 32 || c.head_dim == 64 || c.head_dim == 96 || c.head_dim == 128) || c.n_layers < 1 ||
      c.vocab < 8 || c.max_positions < 1 || c.type_vocab < 1 || c.max_seq < 1 || c.max_seq > c.max_positions ||
      c.max_tokens_per_pass < 16) {
    set_last_error("unsupported encoder geometry (need hidden %% 128 == 0, heads x head_dim == hidden, head_dim in "
                   "{32, 64, 96, 128}, ffn %% 64 == 0, max_seq <= max_positions)");
    return MQ_ERR_INVAL;
  }
  ENC_TRY(cudaSetDevice(gpu));
  mq_encoder* e = new (std::nothrow) mq_encoder();
  if (!e) return MQ_ERR_NOMEM;
  e->cfg = c;
  e->cfg.model_name[sizeof(e->cfg.model_name) - 1] = 0;
  e->gpu = gpu;
  gemm_set_attrs();
  attn_set_attrs();
  if (cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking) != cudaSuccess) { delete e; return MQ_ERR_CUDA; }
  if (cudaEventCreate(&e->ev0) != cudaSuccess || cudaEventCreate(&e->ev1) != cudaSuccess) { delete e; return MQ_ERR_CUDA; }
  int rc = enc_setup(e);
  if (rc) { mq_encoder_close(e); return rc; }
  e->thr = std::thread(enc_main, e);
  e->reply_thr = std::thread(enc_reply_main, e);
  *out = e;
  return MQ_OK;
}

void mq_encoder_close(mq_encoder* e) {
  if (!e) return;
  {
    std::lock_guard<std::mutex> g(e->mu);
    e->stop = true;
  }
  e->cv.notify_all();
  if (e->thr.joinable()) e->thr.join();     // drains the pass queue: every job has been handed to the reply thread
  {
    std::lock_guard<std::mutex> g(e->reply_mu);
    e->reply_stop = true;
  }
  e->reply_cv.notify_all();
  if (e->reply_thr.joinable()) e->reply_thr.join();
  cudaSetDevice(e->gpu);
  if (e->stream) cudaStreamSynchronize(e->stream);
  e->allocs.free_all();
  if (e->ev0) cudaEventDestroy(e->ev0);
  if (e->ev1) cudaEventDestroy(e->ev1);
  if (e->stream) cudaStreamDestroy(e->stream);
  delete e;
}

static DevTensor* enc_find(mq_encoder* e, const char* name) {
  if (!e || !name) { set_last_error("null encoder / tensor name"); return nullptr; }
  auto it = e->tensors.find(name);
  if (it == e->tensors.end()) { set_last_error("encoder has no tensor '%s'", name); return nullptr; }
  return &it->second;
}
int mq_encoder_load_tensor(mq_encoder* e, const char* name, const void* src, size_t nbytes) {
  DevTensor* t = enc_find(e, name);
  if (!t) return MQ_ERR_NOENT;
  if (nbytes != t->bytes) { set_last_error("tensor '%s': got %zu bytes, expected %zu", name, nbytes, t->bytes); return MQ_ERR_INVAL; }
  cudaSetDevice(e->gpu);
  ENC_TRY(cudaMemcpy(t->ptr, src, nbytes, cudaMemcpyDefault));
  return MQ_OK;
}
int mq_encoder_read_tensor(mq_encoder* e, const char* name, void* dst, size_t nbytes) {
  DevTensor* t = enc_find(e, name);
  if (!t) return MQ_ERR_NOENT;
  if (nbytes != t->bytes) { set_last_error("tensor '%s': asked %zu bytes, tensor has %zu", name, nbytes, t->bytes); return MQ_ERR_INVAL; }
  cudaSetDevice(e->gpu);
  ENC_TRY(cudaMemcpy(dst, t->ptr, nbytes, cudaMemcpyDefault));
  return MQ_OK;
}
int mq_encoder_init_random(mq_encoder* e, uint64_t seed, float std) {
  if (!e) return MQ_ERR_INVAL;
  cudaSetDevice(e->gpu);
  uint64_t k = 0;
  for (auto& kv : e->tensors) {  // std::map: deterministic name order
    const std::string leaf = kv.first.substr(kv.first.rfind('.') + 1);
    __nv_bfloat16* p = (__nv_bfloat16*)kv.second.ptr;
    const size_t n = kv.second.bytes / 2;
    if (leaf.size() > 4 && leaf.compare(leaf.size() - 4, 4, "ln_g") == 0) launch_fill_bf16(0, p, n, 1.0f);
    else if ((leaf.size() > 4 && leaf.compare(leaf.size() - 4, 4, "ln_b") == 0) || leaf[0] == 'b') launch_fill_bf16(0, p, n, 0.0f);
    else launch_init_normal(0, p, n, seed * 0x9E3779B97F4A7C15ull + (++k) * 0xD6E8FEB86659FD93ull, std);
  }
  ENC_TRY(cudaDeviceSynchronize());
  return MQ_OK;
}
int mq_encoder_healthy(mq_encoder* e) { return e && e->healthy.load() ? 1 : 0; }

int mq_encoder_embed(mq_encoder* e, const int32_t* tokens, const int32_t* offsets, int32_t n_seq, float* out) {
  if (!e || !tokens || !offsets || !out || n_seq < 1) return MQ_ERR_INVAL;
  EncJob j;
  j.seqs.resize(n_seq);
  for (int s = 0; s < n_seq; ++s) {
    if (offsets[s + 1] < offsets[s]) { set_last_error("offsets must be non-decreasing"); return MQ_ERR_INVAL; }
    j.seqs[s].assign(tokens + offsets[s], tokens + offsets[s + 1]);
  }
  {
    std::unique_lock<std::mutex> lk(e->mu);
    if (e->stop) return MQ_ERR_BUSY;
    e->queue.push_back(&j);
    e->cv.notify_all();
    e->cv_done.wait(lk, [&] { return j.done; });
  }
  if (j.rc) { if (j.rc == MQ_ERR_CUDA) set_last_error("embedding pass failed on the GPU"); return j.rc; }
  memcpy(out, j.out.data(), j.out.size() * 4);
  return MQ_OK;
}

int mq_encoder_submit(mq_encoder* e, const mq_request* rq, const mq_callbacks* cb, void* user, mq_req** out) {
  if (!e || !rq || !cb) return MQ_ERR_INVAL;
  if (!e->healthy.load()) { set_last_error("embedding worker unhealthy"); return MQ_ERR_CUDA; }
  EncJob* j = new (std::nothrow) EncJob();
  mq_req* r = new (std::nothrow) mq_req();
  if (!j || !r) { delete j; delete r; return MQ_ERR_NOMEM; }
  j->path = rq->path ? rq->path : "/api/embed";
  j->model = e->cfg.model_name;
  if (rq->prompt_tokens && rq->n_prompt_tokens > 0) {
    j->seqs.emplace_back(rq->prompt_tokens, rq->prompt_tokens + rq->n_prompt_tokens);
  } else {
    ParsedEmbed pe;
    const std::string body = rq->body && rq->body_len ? std::string((const char*)rq->body, rq->body_len) : std::string();
    if (!parse_embed_body(body, &pe) || (pe.texts.empty() && pe.token_seqs.empty())) {
      delete j; delete r;
      set_last_error("embedding request: body is not a JSON object with \"input\" / \"prompt\"");
      return MQ_ERR_INVAL;
    }
    if (!pe.model.empty()) j->model = pe.model;
    for (auto& t : pe.texts) j->seqs.push_back(embed_tokenize(t, e->cfg.vocab, e->cfg.max_seq));
    for (auto& t : pe.token_seqs) j->seqs.push_back(t);
  }
  r->w = nullptr;
  r->rq = *rq;
  r->rq.body = nullptr; r->rq.prompt_tokens = nullptr; r->rq.path = nullptr;
  r->cb = *cb;
  r->user = user;
  r->t_submit = Clock::now();
  j->req = r;
  if (out) *out = r; else r->refs.store(1);
  {
    std::lock_guard<std::mutex> g(e->mu);
    if (e->stop) { delete j; delete r; return MQ_ERR_BUSY; }
    e->queue.push_back(j);
  }
  e->cv.notify_all();
  return MQ_OK;
}

int mq_encoder_get_stats(mq_encoder* e, mq_encoder_stats* out) {
  if (!e || !out) return MQ_ERR_INVAL;
  out->passes = e->passes.load(); out->sequences = e->sequences.load(); out->tokens = e->tokens.load();
  out->kernel_launches = e->launches.load();
  out->gpu_us = e->gpu_us.load();
  return MQ_OK;
}

}  // extern "C"
