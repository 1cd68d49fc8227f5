/* ollamamq_b200.h — C ABI of libollamamq_b200.so
 *
 * Drop-in boundary for ollamaMQ's hot path (SURVEY.md section 8b).  The reference has no FFI; the seam is
 * the reqwest call inside the executor task, /root/reference/src/dispatcher.rs:287-312, and the
 * BackendStatus slot it occupies (:41-47).  A Rust front would bind exactly these symbols (INTEGRATION.md
 * shows the `extern "C"` block); tests/ and bench.py bind them through ctypes.
 *
 * Conventions: plain pointers and sizes only; every function returns 0 on success or a negative MQ_ERR_*;
 * no C++ exception crosses this boundary; mq_last_error() is thread-local.  There is NO CPU fallback:
 * every worker entry point fails with MQ_ERR_NODEV when no sm_100 GPU is present.
 */
#ifndef OLLAMAMQ_B200_H
#define OLLAMAMQ_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MQ_OK 0
#define MQ_ERR_INVAL (-22)
#define MQ_ERR_NOMEM (-12)
#define MQ_ERR_CUDA (-5)
#define MQ_ERR_BUSY (-16)
#define MQ_ERR_NODEV (-19)
#define MQ_ERR_TIMEOUT (-110)
#define MQ_ERR_CANCELED (-125)
#define MQ_ERR_BLOCKED (-13)
#define MQ_ERR_NOENT (-2)

const char* mq_last_error(void);
const char* mq_version(void);

/* =====================================================================================================
 * 1. Fair-share scheduler — the decision the reference keeps (dispatcher.rs:195-262) plus the completion
 *    side effects that feed it (:314-341).  Pure state machine, no threads, no clock: the same object is
 *    driven by the live dispatcher (section 3) and by the simulated-clock parity tests.
 * ===================================================================================================== */
typedef struct mq_sched mq_sched;

#define MQ_USER_MAX 256

typedef struct mq_dispatch {
  uint64_t task_id;          /* id returned by mq_sched_enqueue                                        */
  uint64_t user_seq;         /* 0-based index of this task among the user's enqueued tasks (FIFO, :244) */
  int32_t backend;           /* selected backend index (:250-254)                                      */
  int32_t reserved;
  char user[MQ_USER_MAX];    /* NUL-terminated user id                                                 */
} mq_dispatch;

/* outcome codes for mq_sched_complete — the three exits of the executor task */
#define MQ_DONE_PROCESSED 0  /* stream ended, client still there:  processed_counts[u]++ (:314-316)     */
#define MQ_DONE_DROPPED 1    /* blocked / client gone / backend error: dropped_counts[u]++ (:280,:318,:326) */
#define MQ_DONE_UNCOUNTED 2  /* Status send failed: neither counter moves (:299)                         */

/* AppState::new (:67-96): all backends online, last_backend_idx = 0, global_counter = 0.
 * capacity = in-flight requests per backend; the reference hard-wires 1 (:204).                         */
mq_sched* mq_sched_new(int32_t n_backends, int32_t capacity);
void mq_sched_free(mq_sched* s);

/* proxy_handler enqueue (:397-405).  user == NULL means "anonymous" (:364-368).                         */
int mq_sched_enqueue(mq_sched* s, const char* user, uint64_t* task_id_out);
/* One iteration of the run_worker loop body (:195-262).  Returns 1 and fills *out when a task was
 * dispatched (active_requests already bumped, :254), 0 when the loop would park on select! (:344-349).   */
int mq_sched_next(mq_sched* s, mq_dispatch* out);
/* Executor epilogue (:314-341): user counters by outcome, backend.active_requests-- (saturating),
 * backend.processed_count++.                                                                            */
int mq_sched_complete(mq_sched* s, int32_t backend, const char* user, int32_t outcome);
/* executor pre-flight bookkeeping: processing_counts[u]++ (:283-284) / -- saturating (:330-333)          */
int mq_sched_processing(mq_sched* s, const char* user, int32_t delta);

/* TUI-driven flags (tui.rs:126-179): setting VIP on the Boost holder clears Boost and vice versa.
 * NULL clears.  The reference has one VIP and one Boost slot (:57-58).                                  */
int mq_sched_set_vip(mq_sched* s, const char* user);
int mq_sched_set_boost(mq_sched* s, const char* user);
/* EXTENSION (BASELINE config 3: "2 VIP + 4 Boost"; the reference has no semantics for this): flags become sets;
 * the winner is the first member in the reference sort order (:224-228).  With <= 1 member: the reference.     */
int mq_sched_add_vip(mq_sched* s, const char* user);
int mq_sched_add_boost(mq_sched* s, const char* user);
/* health prober result (:185-189) */
int mq_sched_set_online(mq_sched* s, int32_t backend, int32_t online);
/* generalisations with reference defaults: capacity 1 (:204), boost every 2nd dispatch (:233)            */
int mq_sched_set_capacity(mq_sched* s, int32_t capacity);
int mq_sched_set_boost_mod(mq_sched* s, int32_t mod);

/* counters (what the TUI snapshot reads, tui.rs:55-69) */
typedef struct mq_user_stats {
  uint64_t queued, processing, processed, dropped;
} mq_user_stats;
typedef struct mq_backend_stats {
  uint64_t active_requests, processed_count;
  int32_t is_online, reserved;
} mq_backend_stats;
int mq_sched_user_stats(mq_sched* s, const char* user, mq_user_stats* out);
int mq_sched_backend_stats(mq_sched* s, int32_t backend, mq_backend_stats* out);
int32_t mq_sched_user_count(mq_sched* s);
/* users in TUI order (queued+processing desc, processed+dropped desc, name asc; tui.rs:70-80)           */
int mq_sched_user_name(mq_sched* s, int32_t index, char* out, size_t cap);
uint64_t mq_sched_counter(mq_sched* s);
/* decision micro-benchmark (SURVEY.md 8d): U users x R requests, unit service time, same driver loop as the
 * oracle's orc_bench; reports dispatches made and the seconds they took (enqueue excluded)                 */
int mq_debug_sched_bench(int32_t n_users, int32_t reqs_per_user, int32_t n_backends, int32_t capacity,
                         uint64_t* dispatches_out, double* seconds_out);

/* =====================================================================================================
 * 2. GPU worker — replaces `client.request(method, backend_url + path).headers(h).body(b).send()` and
 *    the byte-stream relay (dispatcher.rs:287-312) with an on-box sm_100a engine, one per B200.
 * ===================================================================================================== */
typedef struct mq_worker mq_worker;
typedef struct mq_req mq_req;

typedef struct mq_model_cfg {
  int32_t vocab, hidden, ffn, n_layers, n_q_heads, n_kv_heads, head_dim;
  int32_t qkv_bias;        /* 1: Qwen2-style bias on q/k/v                                              */
  float rope_theta;
  float rms_eps;
  int32_t max_batch;       /* capacity: concurrent sequences per worker (reference semantics: 1)         */
  int32_t max_seq;         /* max prompt + generated tokens per sequence                                 */
  int32_t max_prefill_tokens; /* prompt tokens processed per prefill pass                               */
  int32_t kv_pages;        /* paged KV cache size in 16-token pages (0 = derive from max_batch*max_seq)  */
  int32_t use_graphs;      /* 1: CUDA-graph the decode step                                              */
  int32_t use_pdl;         /* 1: programmatic dependent launch between kernels                           */
  int32_t eos_token_id;    /* > 0: a request without ignore_eos ends when this token is drawn (it is not relayed;
                              done_reason / finish_reason "stop"); 0 = the model has none                 */
  char model_name[64];     /* echoed in response JSON ("model" field)                                    */
} mq_model_cfg;

/* number of usable B200 workers on this box (the reference's `--ollama-urls` list length)                */
int mq_worker_count(void);
int mq_worker_open(int32_t gpu, const mq_model_cfg* cfg, mq_worker** out);
void mq_worker_close(mq_worker* w);

/* weights: names are "embed", "final_norm", "lm_head", "layers.<i>.{attn_norm,wqkv,bqkv,wo,mlp_norm,
 * w_gate_up,w_down}" (bf16, torch Linear [out,in] layout; wqkv = [q;k;v] rows, w_gate_up = [gate;up]).
 * src/dst may be host or device memory.                                                                 */
int mq_worker_load_tensor(mq_worker* w, const char* name, const void* src, size_t nbytes);
int mq_worker_read_tensor(mq_worker* w, const char* name, void* dst, size_t nbytes);
/* random-init every tensor on the device: N(0, std^2) from a counter-based generator, norms = 1        */
int mq_worker_init_random(mq_worker* w, uint64_t seed, float std);

/* BackendStatus analogues: capacity (:204 generalised) and health (:181-189: any answer = online)        */
int mq_worker_capacity(mq_worker* w);
int mq_worker_healthy(mq_worker* w);

/* endpoints the worker terminates (routes of main.rs:92-112 that carry generation)                      */
#define MQ_EP_API_GENERATE 0   /* /api/generate            NDJSON */
#define MQ_EP_API_CHAT 1       /* /api/chat                NDJSON */
#define MQ_EP_V1_CHAT 2        /* /v1/chat/completions     SSE    */
#define MQ_EP_V1_COMPLETIONS 3 /* /v1/completions          SSE    */
#define MQ_EP_RAW_TOKENS 4     /* no framing: chunks are little-endian int32 token ids                    */
/* Raw-token record of a request with logprobs on (mq_request.logprobs != 0, N = top_logprobs): one chunk per token is
 * int32 id, float32 logprob, then N x (int32 id, float32 logprob), little-endian (8 + 8 N bytes); with logprobs off it
 * stays the 4-byte id.  stream = 0 concatenates the same records.                                                  */
#define MQ_EP_EMBED 6          /* /api/embed, /api/embeddings, /v1/embeddings: one JSON reply, served by the
                                  embedding worker attached to the backend (section 2b); `path` picks the
                                  reply shape; 501 when no encoder is attached                             */
#define MQ_EP_OTHER 5          /* any other routed path (main.rs:92-112): answered by the worker without
                                  touching the GPU (model listings, version) or with 501 (embeddings, model
                                  management); still queued and dispatched like every request               */

typedef struct mq_request {
  int32_t endpoint;          /* MQ_EP_*                                                                   */
  int32_t stream;            /* 1: one chunk per token; 0: one chunk at the end; <0: take "stream" from body  */
  const uint8_t* body;       /* request body as the client sent it (JSON) — may be NULL with raw tokens   */
  size_t body_len;
  const int32_t* prompt_tokens; /* optional pre-tokenised prompt (synthetic workloads); overrides body    */
  int32_t n_prompt_tokens;
  int32_t max_new_tokens;    /* generation length; <=0: take options.num_predict / max_tokens from body   */
  int32_t ignore_eos;        /* benchmark mode: always generate max_new_tokens                            */
  uint32_t timeout_ms;       /* whole-request timeout (reqwest Client::timeout, :165-167); 0 = none       */
  const char* path;          /* request path (uri.path(), :362); only consulted for MQ_EP_OTHER; may be NULL  */
  /* sampling (the backend's "sample" step).  All zero = greedy, which is what BASELINE measures.  A JSON body may
   * carry them too (Ollama "options": {temperature, top_k, top_p, seed}; OpenAI top-level temperature, top_p, seed)
   * and wins over these fields.                                                                          */
  float temperature;         /* <= 0: greedy argmax (lowest index wins ties)                              */
  int32_t top_k;             /* <= 0: off                                                                 */
  float top_p;               /* <= 0 or >= 1: off; applied to what top_k kept                             */
  uint64_t seed;             /* stream of the counter-based generator: same seed, same tokens             */
  int32_t body_kind;         /* MQ_BODY_JSON: `body` is the client's JSON.  MQ_BODY_TEXT: the front already parsed
                              * it (on its connection thread, never on the scheduler's) and `body` is the extracted
                              * prompt text; stream / max_new_tokens / sampling fields above carry the rest       */
  /* token log-probabilities (0 = off, so a zeroed struct asks for none).  logprobs != 0: every relayed token carries
   * its logprob and the top_logprobs (clamped to 0..MQ_TOP_LOGPROBS_MAX) most probable tokens with theirs.  Defined
   * as log-softmax of the raw logits the token was drawn from (temperature 1, before top-k / top-p), alternatives
   * ordered by logit descending then token id ascending; the EOS token that ends a generation gets no entry.  A JSON
   * body may carry them too ("logprobs": true / false and "top_logprobs": N; on /v1/completions the legacy
   * "logprobs": N) and wins over these fields.  Turning them on never changes a token.                        */
  int16_t logprobs;
  int16_t top_logprobs;
} mq_request;
#define MQ_TOP_LOGPROBS_MAX 20
#ifdef __cplusplus
static_assert(sizeof(mq_request) == 88, "mq_request layout is part of the ABI");
#else
_Static_assert(sizeof(mq_request) == 88, "mq_request layout is part of the ABI");
#endif
#define MQ_BODY_JSON 0
#define MQ_BODY_TEXT 1

typedef struct mq_callbacks {
  /* exactly once, first: ResponsePart::Status (:299).                                                    */
  void (*on_status)(void* user, int32_t http_status, const char* content_type);
  /* 0..N times in order: ResponsePart::Chunk (:305).  Buffer valid only during the call.  A non-zero
   * return means the client is gone (send().is_err(), :305-308): the worker cancels the request.          */
  int32_t (*on_chunk)(void* user, const uint8_t* data, size_t len);
  /* exactly once, last.  rc = 0: stream ended.  rc < 0 before on_status: ResponsePart::Error (:323-325). */
  void (*on_done)(void* user, int32_t rc, const char* errmsg);
} mq_callbacks;

/* Non-blocking (the scheduler loop must not stall, :270).  The body and token arrays are copied before
 * returning.  Callbacks fire on the worker's own host thread, never from inside mq_submit.               */
int mq_submit(mq_worker* w, const mq_request* r, const mq_callbacks* cb, void* user, mq_req** out);
/* client disconnect (:305-308): frees the KV pages; on_done still fires (rc = MQ_ERR_CANCELED).          */
void mq_cancel(mq_req* r);
/* release the handle after on_done has fired */
void mq_req_release(mq_req* r);

/* per-request timing, valid after on_done: microseconds from mq_submit to first token / last token       */
typedef struct mq_req_stats {
  uint64_t ttft_us, total_us;
  int32_t n_prompt, n_generated;
} mq_req_stats;
int mq_req_get_stats(mq_req* r, mq_req_stats* out);

/* worker counters for the roofline: kernels launched and CUDA-event time spent in prefill / decode      */
typedef struct mq_worker_stats {
  uint64_t kernel_launches, graph_launches, decode_steps, prefill_passes, prefill_tokens, decode_tokens;
  double decode_ms, prefill_ms;       /* CUDA-event durations, summed (only when timing is enabled)       */
  double decode_bytes;                /* algorithmic bytes moved by the timed decode steps (SURVEY 8d)    */
} mq_worker_stats;
int mq_worker_get_stats(mq_worker* w, mq_worker_stats* out);
/* what the worker holds right now (answered on the worker thread): a drained worker has every page back in
 * the pool, no slot in use and nothing waiting - the leak check of the soak test                           */
typedef struct mq_worker_occupancy {
  uint64_t total_pages, free_pages, active_slots, waiting, in_flight_gpu_passes;
} mq_worker_occupancy;
int mq_worker_get_occupancy(mq_worker* w, mq_worker_occupancy* out);
int mq_worker_reset_stats(mq_worker* w);
int mq_worker_set_timing(mq_worker* w, int32_t enable);

/* kernel-level test ABI (not on the serving path): logits of the last position of `tokens` (fp32 [vocab]),
 * or of every position when all_positions != 0 (fp32 [n][vocab]); logits_out is host memory.              */
/* Fault injection for the health path (dispatcher.rs:171-193).  probe_fail = 1: mq_worker_healthy() reports 0 while
 * the engine keeps serving what it has (a backend whose /api/tags stopped answering); 0 restores it.
 * mq_debug_worker_inject_fault: the sticky fault a CUDA error raises - every request on the worker fails with `msg`
 * and the worker stays unhealthy until it is closed.                                                          */
int mq_debug_worker_set_probe_fail(mq_worker* w, int32_t probe_fail);
int mq_debug_worker_inject_fault(mq_worker* w, const char* msg);
int mq_debug_forward(mq_worker* w, const int32_t* tokens, int32_t n, int32_t all_positions, float* logits_out);

/* =====================================================================================================
 * 2b. Embedding worker - the same seam (dispatcher.rs:287-312) for the embedding routes of main.rs:89-121
 *     (/api/embed, /api/embeddings, /v1/embeddings): a BERT-family encoder on one B200 (BASELINE configs[4]:
 *     bge-small), sibling of the generation worker on the same GPU (own stream and host thread).
 *     Tensors (bf16, torch Linear [out, in]): word_embed [vocab, H], pos_embed [max_positions, H],
 *     type_embed [type_vocab, H], emb_ln_g / emb_ln_b [H], layers.<i>.{wqkv [3H, H], bqkv [3H], wo [H, H], bo [H],
 *     attn_ln_g, attn_ln_b [H], w_up [ffn, H], b_up [ffn], w_down [H, ffn], b_down [H], mlp_ln_g, mlp_ln_b [H]}.
 * ===================================================================================================== */
typedef struct mq_encoder mq_encoder;
typedef struct mq_encoder_cfg {
  int32_t vocab, hidden, ffn, n_layers, n_heads, head_dim; /* heads x head_dim == hidden; head_dim 32/64/96/128 */
  int32_t max_positions, type_vocab;
  float ln_eps;
  int32_t max_seq;               /* inputs are truncated to this many tokens (<= max_positions)             */
  int32_t max_tokens_per_pass;   /* whole sequences are packed into passes of at most this many tokens      */
  int32_t use_pdl;
  char model_name[64];
} mq_encoder_cfg;
typedef struct mq_encoder_stats {
  uint64_t passes, sequences, tokens, kernel_launches;
  uint64_t gpu_us; /* device time of the passes (CUDA events on the worker's stream around each pass), microseconds */
} mq_encoder_stats;
int mq_encoder_open(int32_t gpu, const mq_encoder_cfg* cfg, mq_encoder** out); /* MQ_ERR_NODEV without sm_100 */
void mq_encoder_close(mq_encoder* e);
int mq_encoder_load_tensor(mq_encoder* e, const char* name, const void* src, size_t nbytes);
int mq_encoder_read_tensor(mq_encoder* e, const char* name, void* dst, size_t nbytes);
int mq_encoder_init_random(mq_encoder* e, uint64_t seed, float std); /* N(0, std^2); LayerNorm gains 1, biases 0 */
int mq_encoder_healthy(mq_encoder* e);
int mq_encoder_get_stats(mq_encoder* e, mq_encoder_stats* out);
/* Blocking compute call (tests, benchmarks, batch jobs): sequence s = tokens[offsets[s] .. offsets[s+1]);
 * out = fp32 [n_seq][hidden] in host memory, each row the L2-normalised [CLS] state.                       */
int mq_encoder_embed(mq_encoder* e, const int32_t* tokens, const int32_t* offsets, int32_t n_seq, float* out);
/* Non-blocking, same contract as mq_submit: body = {"model":..,"input": "s" | ["s",..] | [ids] | [[ids],..]}
 * (or "prompt": "s" on /api/embeddings), or one sequence in prompt_tokens; exactly one on_status(200,
 * application/json), one on_chunk with the whole reply (shape chosen by `path`), one on_done.              */
int mq_encoder_submit(mq_encoder* e, const mq_request* r, const mq_callbacks* cb, void* user, mq_req** out);

/* =====================================================================================================
 * 3. Dispatcher — AppState + run_worker + executor bookkeeping (dispatcher.rs:49-96,164-352) driving a
 *    pool of workers in-process.  This is what `main()` would own in a Rust front (main.rs:82-87).
 * ===================================================================================================== */
typedef struct mq_dispatcher mq_dispatcher;

int mq_dispatcher_new(mq_worker** workers, int32_t n_workers, int32_t capacity_override, mq_dispatcher** out);
void mq_dispatcher_free(mq_dispatcher* d);
/* proxy_handler (:354-428) minus HTTP: 403 pre-checks, enqueue, notify.  ip may be NULL.  Returns
 * MQ_ERR_BLOCKED for a blocked ip/user (:370-378).  The callbacks see Status/Chunk/Done exactly as the
 * reference's mpsc receiver would.                                                                       */
int mq_dispatcher_submit(mq_dispatcher* d, const char* user, const char* ip, const mq_request* r,
                         const mq_callbacks* cb, void* user_data, uint64_t* task_id_out);
mq_sched* mq_dispatcher_sched(mq_dispatcher* d); /* borrowed; guarded by the dispatcher's lock            */
int mq_dispatcher_set_vip(mq_dispatcher* d, const char* user);
int mq_dispatcher_set_boost(mq_dispatcher* d, const char* user);
/* EXTENSION (BASELINE config 3, "2 VIP + 4 Boost"): sets instead of the reference's single slots, see mq_sched_add_* */
int mq_dispatcher_add_vip(mq_dispatcher* d, const char* user);
int mq_dispatcher_add_boost(mq_dispatcher* d, const char* user);
int mq_dispatcher_block_user(mq_dispatcher* d, const char* user, int32_t blocked);   /* :127-153 */
int mq_dispatcher_block_ip(mq_dispatcher* d, const char* ip, int32_t blocked);       /* :117-144 */
/* dispatch log: (user, user_seq, backend) of every dispatch so far, in order — the parity observable     */
int mq_dispatcher_log(mq_dispatcher* d, mq_dispatch* out, int32_t cap, int32_t* n_out);
/* block until every submitted task has completed */
int mq_dispatcher_drain(mq_dispatcher* d, uint32_t timeout_ms);
/* health prober result for one backend (:185-189); like the reference, recovery does not wake the scheduler */
int mq_dispatcher_set_online(mq_dispatcher* d, int32_t backend, int32_t online);
/* block list persistence: load `path` now (AppState::new, :69,:98-105) and rewrite it on every block / unblock
 * (:107-115).  Format pinned by the reference: pretty JSON {"ips": [...], "users": [...]} (:21-25); the reference
 * uses "blocked_items.json" in the working directory (:19).                                                   */
/* Whole-request timeout applied to every dispatched request that does not carry its own (the reference builds its
 * HTTP client with `--timeout` seconds, dispatcher.rs:165-167, main.rs:31-33); 0 = none.                   */
int mq_dispatcher_set_timeout(mq_dispatcher* d, uint32_t timeout_ms);
/* Give backend `backend` an embedding worker: MQ_EP_EMBED requests dispatched to that backend go to it (without
 * one they are answered 501 like any unimplemented route).  The dispatcher does not own the encoder.        */
int mq_dispatcher_attach_encoder(mq_dispatcher* d, int32_t backend, mq_encoder* e);
int mq_dispatcher_set_block_file(mq_dispatcher* d, const char* path);
/* Everything the reference dashboard shows, captured under one lock (tui.rs:55-95 capture_snapshot), as one JSON
 * object: vip[], boost[], blocked_users[], blocked_ips[], counter, users[{id, ip, queued, processing, processed,
 * dropped}] in the dashboard's order (tui.rs:70-80), backends[{label, active, processed, online}].  Returns the bytes
 * needed including the terminator; nothing is written when that exceeds cap.                              */
long long mq_dispatcher_snapshot_json(mq_dispatcher* d, char* out, size_t cap);
/* The dashboard's control keys (tui.rs:126-237) as one atomic call, for front ends without a terminal (the HTTP
 * ingress exposes it as loopback-only POST /admin/{vip,boost,block,unblock}, body {"user": ..} / {"ip": ..} /
 * {"mode": "add" | "clear" | ..}, and GET /admin/state = the snapshot above).  action:
 *   "vip" | "boost"           the 'p' | 'b' key on `user`: toggle; clears the other flag when it names the same user
 *   "vip_add" | "boost_add"   EXTENSION (BASELINE config 3): add `user` to the set;  "vip_clear" | "boost_clear"
 *   "block_user"  'x';  "block_ip"  'X' (`ip`, or the address `user` was last seen from);
 *   "unblock"  'u' on the users panel (user + its address);  "unblock_user" | "unblock_ip"  'u' on the blocked panel */
int mq_dispatcher_control(mq_dispatcher* d, const char* action, const char* user, const char* ip);
/* health prober (:171-193): every period_ms (reference: 10 000) copy mq_worker_healthy() into is_online         */
int mq_dispatcher_start_health(mq_dispatcher* d, uint32_t period_ms);
/* the HTTP connection behind a queued / in-flight task closed (responder.is_closed(), :278; send error, :305) */
int mq_dispatcher_client_gone(mq_dispatcher* d, uint64_t task_id);
/* block until the run_worker thread is parked on {notify, backend_freed} with nothing pending (:344-349)   */
int mq_dispatcher_wait_parked(mq_dispatcher* d, uint32_t timeout_ms);

/* Step-driven MOCK backends (test/dev infrastructure — the fake backend the reference never shipped): a
 * submitted request stays in flight until mq_dispatcher_mock_complete() is called, so a test can impose the
 * completion order of a simulated clock on the live, threaded dispatcher.  Emits fake chunks; never used by
 * mq_dispatcher_new and never a substitute for a GPU worker.                                             */
int mq_dispatcher_new_mock(int32_t n_backends, int32_t capacity, mq_dispatcher** out);
int mq_dispatcher_mock_complete(mq_dispatcher* d, int32_t backend, int32_t rc);
int mq_dispatcher_mock_fail_next(mq_dispatcher* d, int32_t backend, int32_t n);
/* what mock backend `backend` answers to the health prober from now on (0 = GET /api/tags unreachable, :181-183)    */
int mq_dispatcher_mock_set_healthy(mq_dispatcher* d, int32_t backend, int32_t healthy);

/* =====================================================================================================
 * 3b. HTTP/1.1 ingress (SURVEY.md 8f rank 1): the route table of main.rs:89-121 and the proxy_handler
 *     semantics of dispatcher.rs:354-428 (X-User-ID, 403 / 500 bodies, streamed relay) over a dispatcher.
 * ===================================================================================================== */
typedef struct mq_http_server mq_http_server;
/* port 0 picks a free port (read it back with mq_http_server_port).  allow_all_routes = --allow-all-routes.   */
int mq_http_server_start(mq_dispatcher* d, const char* bind_addr, int32_t port, int32_t allow_all_routes,
                         mq_http_server** out);
int mq_http_server_port(mq_http_server* s);
void mq_http_server_stop(mq_http_server* s);

/* =====================================================================================================
 * 4. Kernel-level test ABI (device pointers).  See csrc/debug_api.cu.
 * ===================================================================================================== */
int mq_debug_gemm(const void* W, int w_rows, int n_out, int K, const void* X, int x_rows_alloc, int T, int epi,
                  void* out, int ldo, int splits, long long split_stride, int a2_row_off, int pdl, int reps,
                  float* ms_out);
int mq_debug_embed(const int* token_ids, const void* embed, float* h, int T, int H);
/* ---- decode chain (csrc/gemm_dk.cuh): cluster split-K GEMM + fused epilogues, RMSNorm folded into the consumer.
 * `cs` = cluster size = K splits (1..8; <= 0: the engine's own pick).  The RMSNorm fold scales token column t by
 * rstd[t] = rsqrt(sum_{i < parts} ssq[i * stride + t] * inv_h + eps); ssq == NULL: no scaling.                     */
int mq_debug_embed_chain(const int* token_ids, const void* embed, float* h, int T, int H, const void* gamma, void* xg,
                         float* ssq);
/* encoder GEMM epilogues: out[t][f] = act(sum_k X[t][k] W[f][k] + bias[f]), epi = 4 (bias) or 3 (bias + erf-GELU), bf16 out */
int mq_debug_gemm_bias(const void* W, int n_out, int K, const void* X, int x_rows_alloc, int T, int epi, const void* bias,
                       void* out, int ldo);
/* x = LayerNorm(x + X W^T + bias) * gamma + beta in one kernel: x = device bf16 [T][n_out], n_out in {256, 384} */
int mq_debug_gemm_rowln(const void* W, int n_out, int K, const void* X, int x_rows_alloc, int T, void* x, const void* bias,
                        const void* gamma, const void* beta, float eps, float* h32);
/* encoder attention on tcgen05 (head_dim 32, bidirectional): qkv = device [rows_alloc][3H] bf16, sequences packed back to
 * back (host arrays seq_first / seq_len, lengths 1..512), out = device [rows][H] bf16                                 */
int mq_debug_enc_attn(const void* qkv, int rows_alloc, int H, int n_heads, const int* seq_first, const int* seq_len, int n_seq,
                      void* out);
/* out_k[0..7] = co-resident clusters of 1..8 CTAs (occupancy query for the chain kernel's footprint)              */
int mq_debug_cluster_info(int* out8);
/* plain kernel with tile_rows (<= 128, multiple of 8; 0 = 128, < 0 = balanced over the SMs) and the rstd fold      */
int mq_debug_gemm_fold(const void* W, int w_rows, int n_out, int K, const void* X, int x_rows_alloc, int T, int epi,
                       void* out, int ldo, int a2_row_off, int tile_rows, int streamk, const float* ssq, int parts,
                       int stride, float inv_h, float eps, int reps, float* ms_out);
/* the same epilogue on the persistent 2-CTA prefill kernel (T > 128, n_out % 256 == 0); ssq_in != NULL additionally
 * scales the product by rstd[t] before it is added (not used by the engine: exercises the fold on this kernel)          */
int mq_debug_gemm_resid_prefill(const void* W, int n_out, int K, const void* X, int x_rows_alloc, int T, float* h,
                                const void* gamma_next, void* xg, float* ssq_out, int ssq_stride, const float* ssq_in, int parts,
                                int stride_in, float inv_h, float eps, int reps, float* ms_out);
/* h[t,f] += X[t,:] . W[f,:];  xg = bf16(h * gamma_next);  ssq_out[tile][t] = sum_f h^2 per 128-feature tile        */
int mq_debug_gemm_dk_resid(const void* W, int n_out, int K, const void* X, int x_rows_alloc, int T, int cs, float* h,
                           const void* gamma_next, void* xg, float* ssq_out, int ssq_stride, int reps, float* ms_out);
int mq_debug_add_rmsnorm(float* h, const void* partial, int partial_is_f32, int n_planes, long long plane_stride,
                         const void* gamma, void* x, const int* row_idx, int rows, int H, float eps);
int mq_debug_rope_kv(const void* qkv, int qkv_is_f32, int n_planes, long long plane_stride, const void* bias,
                     const int* pos, const int* slot_of_tok, const int* block_table, int max_pages,
                     const float* inv_freq, void* q_out, void* k_cache, void* v_cache, int T, int n_q, int n_kv,
                     int head_dim /* 128, 96 or 64 */);
int mq_debug_attn_prefill(const void* q, const void* k_cache, const void* v_cache, const int* block_table,
                          int max_pages, const int* tiles, int n_tiles, void* out, int n_q, int n_kv, int T,
                          float scale, int head_dim);
/* prefill attention on tcgen05 (csrc/attn_tc.cu): head_dim 128; q is [q_rows][n_q * 128], the caches hold n_pages pages */
int mq_debug_attn_prefill_tc(const void* q, int q_rows, const void* k_cache, const void* v_cache, int n_pages, const int* block_table,
                             int max_pages, const int* tiles, int n_tiles, void* out, int n_q, int n_kv, float scale);
int mq_debug_attn_decode(const void* q, const void* k_cache, const void* v_cache, const int* block_table,
                         int max_pages, const int* pos, void* out, float* part_o, float* part_ml, int* split_counter,
                         int n_q, int n_kv, int n_slots, int n_splits /* 1..8 grid-level KV splits, or -2 / -4 / -8 =
                         that many warps per CTA with the shared-memory combine */, float scale, int head_dim);
/* Timeline of the worker's most recent decode step (worker opened with MQ_TRACE=1 in the environment): for launch
 * slot i, out[4*i+0..3] = %globaltimer ns of {first CTA start, first CTA past its dependency wait, first CTA end,
 * ~(last CTA end)}; untouched slots read as all-ones.  Slots: 1 + 8*layer + {0 norm, 1 qkv, 2 rope, 3 attention,
 * 4 o-proj, 5 norm, 6 gate/up, 7 down}; 510 final norm, 511 LM head.  Returns the slot count copied (<= 512). */
int mq_debug_trace_read(mq_worker* w, unsigned long long* out, int32_t max_slots);
/* host-only test ABI of the request parsers / response framers (no GPU): each returns the bytes needed incl. the
 * terminator and writes a JSON description when it fits                                                   */
long long mq_debug_parse_body(int32_t endpoint, const uint8_t* body, size_t len, int32_t vocab, char* out, size_t cap);
long long mq_debug_parse_embed(const uint8_t* body, size_t len, int32_t vocab, int32_t max_len, char* out, size_t cap);
long long mq_debug_frame_embeddings(const char* path, const char* model, const float* emb, int32_t n, int32_t dim,
                                    int32_t n_tokens, char* out, size_t cap);
long long mq_debug_frame_final(int32_t endpoint, int32_t stream, const char* model, const char* agg, int32_t n_prompt,
                               int32_t n_gen, int32_t stopped, char* out, size_t cap);
/* the whole reply of a generation request with n tokens: ids[n], records = n x (float logprob, N x (int32 id, float
 * logprob)) (the raw-token record without its leading id); top_logprobs < 0 = logprobs off.  stream = 1: the per-token frames then
 * the final frame, concatenated; stream = 0: the final object.  MQ_EP_RAW_TOKENS: the binary records (length =
 * return value - 1)                                                                                            */
long long mq_debug_frame_logprobs(int32_t endpoint, int32_t stream, const char* model, const int32_t* ids,
                                  const float* records, int32_t n, int32_t top_logprobs, int32_t n_prompt, char* out,
                                  size_t cap);
/* the sampler kernel on given logits: per-row controls (device arrays, row == slot), counter = RNG position  */
int mq_debug_sample(const float* logits, int rows, int V, int ldl, int* out_tokens, const float* temperature,
                    const int* top_k, const float* top_p, const unsigned long long* seed, const int* counter);
/* the same with log-probability records: top_logprobs = device int[rows] (-1 = no record for that row, 0..20 = that
 * many alternatives), lp_out = device [rows] records of 164 bytes: float logprob, int32 id[20], float lp[20]
 * (entries past the row's N and the records of -1 rows are left as they were)                                  */
int mq_debug_sample_logprobs(const float* logits, int rows, int V, int ldl, int* out_tokens, const float* temperature,
                             const int* top_k, const float* top_p, const unsigned long long* seed, const int* counter,
                             const int* top_logprobs, void* lp_out);
int mq_debug_argmax(const float* logits, int rows, int V, int ldl, int* out_tokens, const int* dst_slot,
                    int* cur_token, int* pos_inc, const int* active);
int mq_debug_init_normal(void* w, unsigned long long n, unsigned long long seed, float std);

#ifdef __cplusplus
}
#endif
#endif /* OLLAMAMQ_B200_H */
