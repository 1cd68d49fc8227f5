// Dispatcher: AppState + run_worker + executor bookkeeping, driving a pool of backends in-process.
//
// Reference behaviour restated (all in /root/reference/src/dispatcher.rs):
//   :49-96    AppState (queues, counters, vip/boost, blocked sets, backends, last_backend_idx)
//   :195-262  run_worker loop body            -> mq::Scheduler::next (sched.cpp)
//   :270-342  executor task: pre-flight drop (:271-280), processing++ (:283-284), backend call (:287-292),
//             Status/Chunk relay (:294-312), processed/dropped classification (:314-327), processing--
//             (:330-333), backend release + backend_freed.notify_one() (:336-341)
//   :344-349  park on {notify, backend_freed}
//   :354-405  proxy_handler: 403 pre-checks, user_ips, enqueue, notify
// The reqwest call is replaced by Backend::submit: either a GPU worker (engine.cu) or the step-driven mock
// used by the CPU parity tests (the "fake backend the reference never had", SURVEY.md 7 step 2).
#include "../../include/ollamamq_b200.h"
#include "sched.hpp"
#include "framing.hpp"
#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstdio>
#include <cstring>
#include <deque>
#include <map>
#include <memory>
#include <mutex>
#include <set>
#include <string>
#include <thread>
#include <vector>

namespace mq {
void set_last_error(const char* fmt, ...);

struct Backend {
  virtual ~Backend() {}
  virtual int submit(const mq_request* rq, const mq_callbacks* cb, void* user, void** handle) = 0;
  virtual void cancel(void* handle) = 0;
  virtual void release(void* handle) = 0;
  virtual bool healthy() = 0;
};

struct GpuBackend : Backend {
  mq_worker* w;
  std::atomic<mq_encoder*> enc{nullptr};  // optional embedding worker on the same GPU (mq_dispatcher_attach_encoder)
  explicit GpuBackend(mq_worker* w_) : w(w_) {}
  int submit(const mq_request* rq, const mq_callbacks* cb, void* user, void** handle) override {
    mq_req* r = nullptr;
    mq_encoder* e = enc.load();
    int rc;
    if (rq->endpoint == MQ_EP_EMBED && e) {
      rc = mq_encoder_submit(e, rq, cb, user, &r);
    } else if (rq->endpoint == MQ_EP_EMBED) {  // no encoder: the route exists but nothing serves it -> 501
      mq_request other = *rq;
      other.endpoint = MQ_EP_OTHER;
      rc = mq_submit(w, &other, cb, user, &r);
    } else {
      rc = mq_submit(w, rq, cb, user, &r);
    }
    *handle = r;
    return rc;
  }
  void cancel(void* h) override { mq_cancel((mq_req*)h); }
  void release(void* h) override { mq_req_release((mq_req*)h); }
  bool healthy() override { return mq_worker_healthy(w) != 0; }
};

// Step-driven mock: a submitted request stays in flight until the test calls complete_oldest().
struct MockBackend : Backend {
  struct Pending {
    mq_callbacks cb;
    void* user;
    int n_tokens;
    bool canceled = false;
  };
  std::mutex mu;
  std::deque<std::shared_ptr<Pending>> q;
  int fail_next = 0;
  std::atomic<bool> answers_probe{true};  // what the health prober sees (GET /api/tags answered or not, :181-183)
  int submit(const mq_request* rq, const mq_callbacks* cb, void* user, void** handle) override {
    std::lock_guard<std::mutex> g(mu);
    if (fail_next > 0) {
      --fail_next;
      set_last_error("mock backend: connection refused");
      return MQ_ERR_CUDA;
    }
    auto p = std::make_shared<Pending>();
    p->cb = *cb;
    p->user = user;
    p->n_tokens = rq->max_new_tokens > 0 ? rq->max_new_tokens : 1;
    q.push_back(p);
    *handle = p.get();
    return MQ_OK;
  }
  void cancel(void* h) override {
    std::lock_guard<std::mutex> g(mu);
    for (auto& p : q) if (p.get() == h) p->canceled = true;
  }
  void release(void*) override {}
  bool healthy() override { return answers_probe.load(); }
  // returns 1 when a request was completed
  int complete_oldest(int rc) {
    std::shared_ptr<Pending> p;
    {
      std::lock_guard<std::mutex> g(mu);
      if (q.empty()) return 0;
      p = q.front();
      q.pop_front();
    }
    if (rc != 0) {
      p->cb.on_done(p->user, rc, "mock backend error");
      return 1;
    }
    p->cb.on_status(p->user, 200, "application/x-ndjson");
    bool gone = p->canceled;
    for (int i = 0; i < p->n_tokens && !gone; ++i) {
      char buf[32];
      int n = snprintf(buf, sizeof(buf), "{\"tok\":%d}\n", i);
      if (p->cb.on_chunk(p->user, (const uint8_t*)buf, (size_t)n) != 0) gone = true;
    }
    p->cb.on_done(p->user, gone ? MQ_ERR_CANCELED : 0, gone ? "client gone" : "");
    return 1;
  }
};

}  // namespace mq

using namespace mq;

struct mq_dispatcher {
  struct Task {
    uint64_t id;
    std::string user, ip;
    mq_request rq;
    std::vector<uint8_t> body;
    std::vector<int32_t> tokens;
    std::string path;
    mq_callbacks cb;
    void* user_data;
    mq_dispatcher* d;
    int backend = -1;
    void* handle = nullptr;
    bool bad_json = false;           // body failed to parse on the connection thread: answered 400 at dispatch time
    bool status_ok = false;          // Status delivered (:299)
    bool client_gone = false;        // chunk send failed (:305-308)
    std::atomic<bool> closed{false}; // responder.is_closed() (:278)
  };

  mq_sched* sched = nullptr;
  std::vector<std::unique_ptr<Backend>> backends;
  std::vector<MockBackend*> mocks;  // aliases into backends when built with mq_dispatcher_new_mock
  std::mutex mu;
  std::condition_variable cv;       // notify + backend_freed
  std::condition_variable cv_idle;
  std::map<uint64_t, std::unique_ptr<Task>> tasks;
  std::map<std::string, std::string> user_ips;
  std::set<std::string> blocked_users, blocked_ips;
  std::deque<mq_dispatch> log;      // most recent dispatch decisions (parity tests read it): bounded ring
  size_t log_cap = 1 << 16;
  std::string block_file;           // BLOCKED_FILE = "blocked_items.json" in the reference (:19); empty = no persistence
  std::thread health_thr;
  uint32_t health_period_ms = 0;
  uint32_t default_timeout_ms = 0;  // --timeout of the reference (main.rs:31-33), 0 = none
  uint64_t outstanding = 0;
  uint64_t wake_seq = 0, handled_seq = 0;
  bool parked = false;
  bool stop = false;
  std::thread thr;
};

namespace {

void executor_epilogue(mq_dispatcher* d, mq_dispatcher::Task* t, int outcome) {
  void* handle = nullptr;
  Backend* be = nullptr;
  {
    std::lock_guard<std::mutex> g(d->mu);
    handle = t->handle;  // null when submit() has not returned yet: run_worker releases it instead
    be = t->backend >= 0 ? d->backends[t->backend].get() : nullptr;
    d->sched->s.processing(t->user, -1);                 // :330-333
    d->sched->s.complete(t->backend, t->user, outcome);  // :314-327, :336-340
    d->outstanding--;
    d->wake_seq++;
    d->tasks.erase(t->id);                               // frees t
  }
  if (handle && be) be->release(handle);
  d->cv.notify_all();                                    // backend_freed.notify_one() (:341)
  d->cv_idle.notify_all();
}

// ---- callbacks handed to the backend: the relay loop of the executor (:294-312)
void cb_status(void* u, int32_t status, const char* ctype) {
  auto* t = (mq_dispatcher::Task*)u;
  if (t->closed.load()) return;  // Status send fails -> neither processed nor dropped (:299)
  t->status_ok = true;
  if (t->cb.on_status) t->cb.on_status(t->user_data, status, ctype);
}
int32_t cb_chunk(void* u, const uint8_t* data, size_t len) {
  auto* t = (mq_dispatcher::Task*)u;
  if (!t->status_ok) return 1;
  if (t->client_gone) return 1;
  if (t->closed.load() || (t->cb.on_chunk && t->cb.on_chunk(t->user_data, data, len) != 0)) {
    t->client_gone = true;  // :305-308
    return 1;
  }
  return 0;
}
void cb_done(void* u, int32_t rc, const char* msg) {
  auto* t = (mq_dispatcher::Task*)u;
  mq_dispatcher* d = t->d;
  // a disconnect reported through mq_dispatcher_client_gone cancels the backend request at once, so no further chunk
  // send gets the chance to fail: it is the same event as the failed send of :305-308
  const bool gone = t->client_gone || (t->status_ok && rc != 0 && t->closed.load());  // rc == 0: the whole body went out
  int outcome;
  if (t->status_ok) outcome = gone ? MQ_DONE_DROPPED : MQ_DONE_PROCESSED;            // mid-stream errors count processed (:310,:314)
  else if (rc != 0 && !t->closed.load()) outcome = MQ_DONE_DROPPED;                  // ResponsePart::Error (:323-327)
  else outcome = MQ_DONE_UNCOUNTED;                                                  // Status send failed (:299)
  if (t->cb.on_done) t->cb.on_done(t->user_data, t->status_ok && !gone ? 0 : (rc ? rc : MQ_ERR_CANCELED), msg);
  executor_epilogue(d, t, outcome);
}

void run_worker(mq_dispatcher* d) {
  std::unique_lock<std::mutex> lk(d->mu);
  for (;;) {
    if (d->stop) return;
    SchedDispatch sd;
    if (!d->sched->s.next(&sd)) {  // park on {notify, backend_freed} (:344-349)
      d->handled_seq = d->wake_seq;
      d->parked = true;
      d->cv_idle.notify_all();
      d->cv.wait(lk, [&] { return d->stop || d->wake_seq != d->handled_seq; });
      d->parked = false;
      continue;
    }
    mq_dispatch rec;
    memset(&rec, 0, sizeof(rec));
    rec.task_id = sd.task_id;
    rec.user_seq = sd.user_seq;
    rec.backend = sd.backend;
    strncpy(rec.user, sd.user.c_str(), MQ_USER_MAX - 1);
    d->log.push_back(rec);
    if (d->log.size() > d->log_cap) d->log.pop_front();
    auto it = d->tasks.find(sd.task_id);
    if (it == d->tasks.end()) continue;
    mq_dispatcher::Task* t = it->second.get();
    t->backend = sd.backend;
    // ---- executor pre-flight (:271-280)
    bool blocked = d->blocked_users.count(t->user) > 0;
    auto ipit = d->user_ips.find(t->user);
    if (!blocked && ipit != d->user_ips.end()) blocked = d->blocked_ips.count(ipit->second) > 0;
    if (blocked || t->closed.load()) {
      d->sched->s.complete(sd.backend, t->user, MQ_DONE_DROPPED);  // dropped++, backend released (:336-340)
      d->outstanding--;
      d->wake_seq++;
      mq_callbacks cb = t->cb;
      void* ud = t->user_data;
      d->tasks.erase(it);
      lk.unlock();
      if (cb.on_done) cb.on_done(ud, MQ_ERR_BLOCKED, "Worker failed to respond");  // proxy_handler :427
      d->cv_idle.notify_all();
      lk.lock();
      continue;
    }
    d->sched->s.processing(t->user, +1);  // :283-284
    mq_request rq = t->rq;
    if (rq.timeout_ms == 0) rq.timeout_ms = d->default_timeout_ms;  // client-wide timeout of the reference (:165-167)
    rq.body = t->body.empty() ? nullptr : t->body.data();
    rq.body_len = t->body.size();
    rq.prompt_tokens = t->tokens.empty() ? nullptr : t->tokens.data();
    rq.n_prompt_tokens = (int32_t)t->tokens.size();
    rq.path = t->path.empty() ? nullptr : t->path.c_str();
    mq_callbacks cb{cb_status, cb_chunk, cb_done};
    Backend* be = d->backends[sd.backend].get();
    lk.unlock();  // the reference spawns the executor and loops immediately (:270)
    if (t->bad_json) {
      // what a backend answers to a malformed body (the reference relays it like any response: processed, :314-316)
      static const char kMsg[] = "{\"error\":\"invalid JSON request body\"}";
      cb_status(t, 400, "application/json");
      cb_chunk(t, (const uint8_t*)kMsg, sizeof(kMsg) - 1);
      cb_done(t, 0, "");
      lk.lock();
      continue;
    }
    void* h = nullptr;
    int rc = be->submit(&rq, &cb, t, &h);
    if (rc != MQ_OK) {
      // request error before any response: ResponsePart::Error -> HTTP 500 "Backend error: ..." (:323-327)
      std::string msg = std::string("Backend error: ") + mq_last_error();
      if (t->cb.on_done) t->cb.on_done(t->user_data, rc, msg.c_str());
      executor_epilogue(d, t, MQ_DONE_DROPPED);
    } else {
      std::lock_guard<std::mutex> g(d->mu);
      auto it2 = d->tasks.find(sd.task_id);
      if (it2 != d->tasks.end()) it2->second->handle = h;  // may already have completed and been erased
      else be->release(h);
    }
    lk.lock();
  }
}

// blocked_items.json: pretty JSON {"ips": [...], "users": [...]} (BlockedConfig, :21-25; load :98-105, save :107-115)
void save_blocked(mq_dispatcher* d) {  // caller holds d->mu
  if (d->block_file.empty()) return;
  std::string o = "{\n  \"ips\": [";
  bool first = true;
  for (const auto& ip : d->blocked_ips) { o += first ? "\n    \"" : ",\n    \""; o += ip + "\""; first = false; }
  o += first ? "],\n  \"users\": [" : "\n  ],\n  \"users\": [";
  first = true;
  for (const auto& u : d->blocked_users) {
    o += first ? "\n    \"" : ",\n    \"";
    for (char c : u) { if (c == '"' || c == '\\') o.push_back('\\'); o.push_back(c); }
    o += "\"";
    first = false;
  }
  o += first ? "]\n}" : "\n  ]\n}";
  FILE* f = fopen(d->block_file.c_str(), "w");
  if (!f) return;  // the reference ignores write errors too (`let _ = fs::write`, :113)
  fwrite(o.data(), 1, o.size(), f);
  fclose(f);
}

// tolerant reader for the two string arrays
void load_blocked(mq_dispatcher* d) {  // caller holds d->mu
  FILE* f = fopen(d->block_file.c_str(), "r");
  if (!f) return;
  std::string txt;
  char buf[4096];
  size_t n;
  while ((n = fread(buf, 1, sizeof(buf), f)) > 0) txt.append(buf, n);
  fclose(f);
  auto read_array = [&](const char* key, std::set<std::string>* out) {
    size_t k = txt.find(std::string("\"") + key + "\"");
    if (k == std::string::npos) return;
    size_t b = txt.find('[', k), e = txt.find(']', k);
    if (b == std::string::npos || e == std::string::npos || e < b) return;
    size_t p = b;
    while (true) {
      size_t q1 = txt.find('"', p + 1);
      if (q1 == std::string::npos || q1 > e) break;
      std::string v;
      size_t q = q1 + 1;
      while (q < txt.size() && txt[q] != '"') {
        if (txt[q] == '\\' && q + 1 < txt.size()) ++q;
        v.push_back(txt[q++]);
      }
      out->insert(v);
      p = q;
    }
  };
  read_array("ips", &d->blocked_ips);
  read_array("users", &d->blocked_users);
}

// health prober (:171-193): periodically asks every backend whether it still answers; flipping a backend back
// online does not wake the scheduler, exactly like the reference
void health_loop(mq_dispatcher* d) {
  std::unique_lock<std::mutex> lk(d->mu);
  while (!d->stop) {
    for (size_t i = 0; i < d->backends.size(); ++i) d->sched->s.set_online((int)i, d->backends[i]->healthy());
    d->cv_idle.wait_for(lk, std::chrono::milliseconds(d->health_period_ms), [&] { return d->stop; });
  }
}

mq_dispatcher* make_dispatcher(std::vector<std::unique_ptr<Backend>> bes, int capacity) {
  auto* d = new (std::nothrow) mq_dispatcher();
  if (!d) return nullptr;
  d->sched = mq_sched_new((int32_t)bes.size(), capacity);
  if (!d->sched) { delete d; return nullptr; }
  d->backends = std::move(bes);
  d->thr = std::thread(run_worker, d);
  return d;
}

}  // namespace

extern "C" {

int mq_dispatcher_new(mq_worker** workers, int32_t n_workers, int32_t capacity_override, mq_dispatcher** out) {
  if (!workers || n_workers < 1 || !out) return MQ_ERR_INVAL;
  std::vector<std::unique_ptr<Backend>> bes;
  for (int i = 0; i < n_workers; ++i) {
    if (!workers[i]) return MQ_ERR_INVAL;
    bes.emplace_back(new GpuBackend(workers[i]));
  }
  // reference default: one in-flight request per backend (:204); >1 only when the caller asks for it
  *out = make_dispatcher(std::move(bes), capacity_override > 0 ? capacity_override : 1);
  return *out ? MQ_OK : MQ_ERR_NOMEM;
}

int mq_dispatcher_add_vip(mq_dispatcher* d, const char* user) {  // EXTENSION (BASELINE config 3): see mq_sched_add_vip
  if (!d || !user) return MQ_ERR_INVAL;
  std::lock_guard<std::mutex> g(d->mu);
  d->sched->s.add_vip(user);
  return MQ_OK;
}
int mq_dispatcher_add_boost(mq_dispatcher* d, const char* user) {
  if (!d || !user) return MQ_ERR_INVAL;
  std::lock_guard<std::mutex> g(d->mu);
  d->sched->s.add_boost(user);
  return MQ_OK;
}

int mq_dispatcher_set_timeout(mq_dispatcher* d, uint32_t timeout_ms) {
  if (!d) return MQ_ERR_INVAL;
  std::lock_guard<std::mutex> g(d->mu);
  d->default_timeout_ms = timeout_ms;
  return MQ_OK;
}

int mq_dispatcher_attach_encoder(mq_dispatcher* d, int32_t backend, mq_encoder* e) {
  if (!d || backend < 0 || backend >= (int)d->backends.size()) return MQ_ERR_INVAL;
  auto* gb = dynamic_cast<GpuBackend*>(d->backends[backend].get());
  if (!gb) {
    mq::set_last_error("backend %d is not a GPU worker", backend);
    return MQ_ERR_INVAL;
  }
  gb->enc.store(e);
  return MQ_OK;
}

int mq_dispatcher_new_mock(int32_t n_backends, int32_t capacity, mq_dispatcher** out) {
  if (n_backends < 1 || !out) return MQ_ERR_INVAL;
  std::vector<std::unique_ptr<Backend>> bes;
  std::vector<MockBackend*> mocks;
  for (int i = 0; i < n_backends; ++i) {
    auto* m = new MockBackend();
    mocks.push_back(m);
    bes.emplace_back(m);
  }
  *out = make_dispatcher(std::move(bes), capacity > 0 ? capacity : 1);
  if (!*out) return MQ_ERR_NOMEM;
  (*out)->mocks = mocks;
  return MQ_OK;
}

// complete the oldest in-flight request of mock backend `backend` (rc != 0: backend error before Status)
int mq_dispatcher_mock_complete(mq_dispatcher* d, int32_t backend, int32_t rc) {
  if (!d || backend < 0 || backend >= (int)d->mocks.size()) return MQ_ERR_INVAL;
  return d->mocks[backend]->complete_oldest(rc);
}
int mq_dispatcher_mock_fail_next(mq_dispatcher* d, int32_t backend, int32_t n) {
  if (!d || backend < 0 || backend >= (int)d->mocks.size()) return MQ_ERR_INVAL;
  std::lock_guard<std::mutex> g(d->mocks[backend]->mu);
  d->mocks[backend]->fail_next = n;
  return MQ_OK;
}
// what mock backend `backend` answers to the health probe from now on (0: like an unreachable /api/tags)
int mq_dispatcher_mock_set_healthy(mq_dispatcher* d, int32_t backend, int32_t healthy) {
  if (!d || backend < 0 || backend >= (int)d->mocks.size()) return MQ_ERR_INVAL;
  d->mocks[backend]->answers_probe.store(healthy != 0);
  return MQ_OK;
}

void mq_dispatcher_free(mq_dispatcher* d) {
  if (!d) return;
  {
    std::lock_guard<std::mutex> g(d->mu);
    d->stop = true;
    d->wake_seq++;
  }
  d->cv.notify_all();
  d->cv_idle.notify_all();
  if (d->thr.joinable()) d->thr.join();
  if (d->health_thr.joinable()) d->health_thr.join();
  // in-flight tasks belong to backends that outlive us only for GPU workers; drain what the mocks hold
  for (auto* m : d->mocks) while (m->complete_oldest(MQ_ERR_CANCELED)) {}
  mq_dispatcher_drain(d, 5000);
  mq_sched_free(d->sched);
  delete d;
}

int mq_dispatcher_submit(mq_dispatcher* d, const char* user, const char* ip, const mq_request* r,
                         const mq_callbacks* cb, void* user_data, uint64_t* task_id_out) {
  if (!d || !r || !cb) return MQ_ERR_INVAL;
  const std::string u = user ? user : "anonymous";  // :364-368
  if (u.size() >= MQ_USER_MAX) {
    set_last_error("user id too long");
    return MQ_ERR_INVAL;
  }
  auto t = std::unique_ptr<mq_dispatcher::Task>(new mq_dispatcher::Task());
  t->user = u;
  t->ip = ip ? ip : "";
  t->rq = *r;
  if (r->body && r->body_len) t->body.assign(r->body, r->body + r->body_len);
  if (r->prompt_tokens && r->n_prompt_tokens > 0) t->tokens.assign(r->prompt_tokens, r->prompt_tokens + r->n_prompt_tokens);
  if (r->path) t->path = r->path;
  t->cb = *cb;
  t->user_data = user_data;
  t->d = d;
  // The JSON body of a generation request is parsed HERE, on the caller's (HTTP connection) thread: the scheduler thread
  // only ever moves the result (advisor finding r01: a parser stall froze dispatch for every user and GPU).
  const bool gen_ep = r->endpoint == MQ_EP_API_GENERATE || r->endpoint == MQ_EP_API_CHAT || r->endpoint == MQ_EP_V1_CHAT ||
                      r->endpoint == MQ_EP_V1_COMPLETIONS || r->endpoint == MQ_EP_RAW_TOKENS;
  if (gen_ep && r->body_kind == MQ_BODY_JSON && !t->body.empty() && t->tokens.empty()) {
    ParsedBody pb;
    if (!parse_body(std::string((const char*)t->body.data(), t->body.size()), r->endpoint, &pb)) {
      t->bad_json = true;
      t->body.clear();
    } else {
      if (!pb.tokens.empty()) { t->tokens = pb.tokens; t->body.clear(); }
      else { t->body.assign(pb.text.begin(), pb.text.end()); t->rq.body_kind = MQ_BODY_TEXT; }
      apply_body(pb, &t->rq);
    }
  }
  {
    std::lock_guard<std::mutex> g(d->mu);
    if (ip && d->blocked_ips.count(t->ip)) {  // :370-373
      set_last_error("IP blocked");
      return MQ_ERR_BLOCKED;
    }
    if (d->blocked_users.count(u)) {          // :375-378
      set_last_error("User blocked");
      return MQ_ERR_BLOCKED;
    }
    if (ip) d->user_ips[u] = t->ip;           // :380-383
    uint64_t id = d->sched->s.enqueue(u);     // :397-403
    t->id = id;
    if (task_id_out) *task_id_out = id;
    d->tasks[id] = std::move(t);
    d->outstanding++;
    d->wake_seq++;
  }
  d->cv.notify_all();                          // notify.notify_one() (:405)
  return MQ_OK;
}

// the HTTP connection of a queued / in-flight task went away (responder closed)
int mq_dispatcher_client_gone(mq_dispatcher* d, uint64_t task_id) {
  if (!d) return MQ_ERR_INVAL;
  std::lock_guard<std::mutex> g(d->mu);
  auto it = d->tasks.find(task_id);
  if (it == d->tasks.end()) return MQ_ERR_NOENT;
  it->second->closed.store(true);
  if (it->second->handle && it->second->backend >= 0) d->backends[it->second->backend]->cancel(it->second->handle);
  return MQ_OK;
}

mq_sched* mq_dispatcher_sched(mq_dispatcher* d) { return d ? d->sched : nullptr; }

int mq_dispatcher_set_vip(mq_dispatcher* d, const char* user) {
  if (!d) return MQ_ERR_INVAL;
  std::lock_guard<std::mutex> g(d->mu);  // no notify: takes effect at the next natural wake-up (tui.rs:126-179)
  d->sched->s.set_vip(user);
  return MQ_OK;
}
int mq_dispatcher_set_boost(mq_dispatcher* d, const char* user) {
  if (!d) return MQ_ERR_INVAL;
  std::lock_guard<std::mutex> g(d->mu);
  d->sched->s.set_boost(user);
  return MQ_OK;
}
int mq_dispatcher_block_user(mq_dispatcher* d, const char* user, int32_t blocked) {
  if (!d || !user) return MQ_ERR_INVAL;
  std::lock_guard<std::mutex> g(d->mu);
  if (blocked) d->blocked_users.insert(user); else d->blocked_users.erase(user);
  save_blocked(d);  // rewritten on every change (:107-115)
  return MQ_OK;
}
int mq_dispatcher_block_ip(mq_dispatcher* d, const char* ip, int32_t blocked) {
  if (!d || !ip) return MQ_ERR_INVAL;
  std::lock_guard<std::mutex> g(d->mu);
  if (blocked) d->blocked_ips.insert(ip); else d->blocked_ips.erase(ip);
  save_blocked(d);
  return MQ_OK;
}
// The dashboard's control keys as ONE atomic call (tui.rs:126-237), for front ends without a terminal (HTTP /admin/*):
//   "vip" / "boost"            the 'p' / 'b' key on `user`: toggle, and clear the other flag when it names the same user
//   "vip_add" / "boost_add"    EXTENSION (BASELINE config 3): add `user` to the set; "vip_clear" / "boost_clear": empty it
//   "block_user"               'x'         "block_ip"  'X' (`ip`, or the last address `user` was seen from)
//   "unblock"                  'u' on the users panel: the user AND its last address
//   "unblock_user" / "unblock_ip"   'u' on an entry of the blocked panel
int mq_dispatcher_control(mq_dispatcher* d, const char* action, const char* user, const char* ip) {
  if (!d || !action) return MQ_ERR_INVAL;
  const std::string a = action;
  std::lock_guard<std::mutex> g(d->mu);  // no notify: takes effect at the next natural wake-up, like the reference
  auto has = [](const std::vector<std::string>& v, const char* u) { return u && std::find(v.begin(), v.end(), u) != v.end(); };
  auto need_user = [&]() { if (!user || !*user) { set_last_error("'%s' needs a user", action); return false; } return true; };
  auto last_ip = [&]() -> std::string {
    if (ip && *ip) return ip;
    auto it = user ? d->user_ips.find(user) : d->user_ips.end();
    return it == d->user_ips.end() ? std::string() : it->second;
  };
  Scheduler& s = d->sched->s;
  if (a == "vip" || a == "boost") {
    if (!need_user()) return MQ_ERR_INVAL;
    const bool is_vip = a == "vip";
    const bool on = has(is_vip ? s.vips() : s.boosts(), user);
    const bool other = has(is_vip ? s.boosts() : s.vips(), user);
    if (is_vip) { s.set_vip(on ? nullptr : user); if (other) s.set_boost(nullptr); }
    else { s.set_boost(on ? nullptr : user); if (other) s.set_vip(nullptr); }
    return MQ_OK;
  }
  if (a == "vip_add") { if (!need_user()) return MQ_ERR_INVAL; s.add_vip(user); return MQ_OK; }
  if (a == "boost_add") { if (!need_user()) return MQ_ERR_INVAL; s.add_boost(user); return MQ_OK; }
  if (a == "vip_clear") { s.set_vip(nullptr); return MQ_OK; }
  if (a == "boost_clear") { s.set_boost(nullptr); return MQ_OK; }
  if (a == "block_user") { if (!need_user()) return MQ_ERR_INVAL; d->blocked_users.insert(user); save_blocked(d); return MQ_OK; }
  if (a == "unblock_user") { if (!need_user()) return MQ_ERR_INVAL; d->blocked_users.erase(user); save_blocked(d); return MQ_OK; }
  if (a == "block_ip" || a == "unblock_ip") {
    const std::string v = last_ip();
    if (v.empty()) { set_last_error("'%s' needs an ip (or a user that has been seen)", action); return MQ_ERR_INVAL; }
    if (a == "block_ip") d->blocked_ips.insert(v); else d->blocked_ips.erase(v);
    save_blocked(d);
    return MQ_OK;
  }
  if (a == "unblock") {
    if (!need_user()) return MQ_ERR_INVAL;
    d->blocked_users.erase(user);
    const std::string v = last_ip();
    if (!v.empty()) d->blocked_ips.erase(v);
    save_blocked(d);
    return MQ_OK;
  }
  set_last_error("unknown control action '%s'", action);
  return MQ_ERR_INVAL;
}

// One consistent view of everything the reference dashboard shows (tui.rs:55-95 capture_snapshot): taken under the
// dispatcher lock, users already in the dashboard's order.  JSON so that a curses / web front end needs one call.
static void js_str(std::string& o, const std::string& v) {
  o += '"';
  for (unsigned char ch : v) {
    if (ch == '"' || ch == '\\') { o += '\\'; o += (char)ch; }
    else if (ch < 0x20) { char b[8]; snprintf(b, sizeof b, "\\u%04x", ch); o += b; }
    else o += (char)ch;
  }
  o += '"';
}
static void js_list(std::string& o, const char* key, const std::vector<std::string>& v) {
  o += '"'; o += key; o += "\":[";
  for (size_t i = 0; i < v.size(); ++i) { if (i) o += ','; js_str(o, v[i]); }
  o += ']';
}
long long mq_dispatcher_snapshot_json(mq_dispatcher* d, char* out, size_t cap) {
  if (!d) return MQ_ERR_INVAL;
  std::string o = "{";
  {
    std::lock_guard<std::mutex> g(d->mu);
    const mq::Scheduler& sc = d->sched->s;
    js_list(o, "vip", sc.vips()); o += ',';
    js_list(o, "boost", sc.boosts()); o += ',';
    js_list(o, "blocked_users", std::vector<std::string>(d->blocked_users.begin(), d->blocked_users.end())); o += ',';
    js_list(o, "blocked_ips", std::vector<std::string>(d->blocked_ips.begin(), d->blocked_ips.end()));
    o += ",\"counter\":" + std::to_string(sc.counter()) + ",\"users\":[";
    bool first = true;
    for (const mq::Scheduler::User* u : sc.users_tui_order()) {
      if (!first) o += ',';
      first = false;
      o += "{\"id\":"; js_str(o, u->name);
      auto ip = d->user_ips.find(u->name);
      o += ",\"ip\":"; js_str(o, ip == d->user_ips.end() ? std::string() : ip->second);
      o += ",\"queued\":" + std::to_string(u->queue.size()) + ",\"processing\":" + std::to_string(u->processing) +
           ",\"processed\":" + std::to_string(u->processed) + ",\"dropped\":" + std::to_string(u->dropped) + "}";
    }
    o += "],\"backends\":[";
    for (int i = 0; i < sc.n_backends(); ++i) {
      const mq::Scheduler::Backend* b = sc.backend(i);
      if (i) o += ',';
      o += "{\"label\":\"gpu" + std::to_string(i) + "\",\"active\":" + std::to_string(b->active) + ",\"processed\":" +
           std::to_string(b->processed_count) + ",\"online\":" + (b->online ? "true" : "false") + "}";
    }
    o += "]}";
  }
  if (out && cap > o.size()) memcpy(out, o.c_str(), o.size() + 1);
  return (long long)o.size() + 1;  // bytes needed incl. the terminator (call again with a larger buffer if > cap)
}
int mq_dispatcher_set_block_file(mq_dispatcher* d, const char* path) {
  if (!d || !path) return MQ_ERR_INVAL;
  std::lock_guard<std::mutex> g(d->mu);
  d->block_file = path;
  load_blocked(d);  // AppState::new -> load_blocked_items (:69, :98-105)
  return MQ_OK;
}
int mq_dispatcher_start_health(mq_dispatcher* d, uint32_t period_ms) {
  if (!d || period_ms == 0) return MQ_ERR_INVAL;
  std::lock_guard<std::mutex> g(d->mu);
  if (d->health_thr.joinable()) return MQ_ERR_BUSY;
  d->health_period_ms = period_ms;
  d->health_thr = std::thread(health_loop, d);
  return MQ_OK;
}
int mq_dispatcher_set_online(mq_dispatcher* d, int32_t backend, int32_t online) {
  if (!d) return MQ_ERR_INVAL;
  std::lock_guard<std::mutex> g(d->mu);  // a backend coming back does NOT wake the scheduler (:185-189)
  d->sched->s.set_online(backend, online != 0);
  return MQ_OK;
}

int mq_dispatcher_log(mq_dispatcher* d, mq_dispatch* out, int32_t cap, int32_t* n_out) {
  if (!d || !n_out) return MQ_ERR_INVAL;
  std::lock_guard<std::mutex> g(d->mu);
  *n_out = (int32_t)d->log.size();
  if (out)
    for (int i = 0; i < cap && i < (int)d->log.size(); ++i) out[i] = d->log[i];
  return MQ_OK;
}

// wait until the scheduler thread is parked with nothing left to look at (test harness: "runs to quiescence")
int mq_dispatcher_wait_parked(mq_dispatcher* d, uint32_t timeout_ms) {
  if (!d) return MQ_ERR_INVAL;
  std::unique_lock<std::mutex> lk(d->mu);
  bool ok = d->cv_idle.wait_for(lk, std::chrono::milliseconds(timeout_ms),
                                [&] { return d->parked && d->handled_seq == d->wake_seq; });
  return ok ? MQ_OK : MQ_ERR_TIMEOUT;
}

int mq_dispatcher_drain(mq_dispatcher* d, uint32_t timeout_ms) {
  if (!d) return MQ_ERR_INVAL;
  std::unique_lock<std::mutex> lk(d->mu);
  bool ok = d->cv_idle.wait_for(lk, std::chrono::milliseconds(timeout_ms), [&] { return d->outstanding == 0; });
  return ok ? MQ_OK : MQ_ERR_TIMEOUT;
}

}  // extern "C"
