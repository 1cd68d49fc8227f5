// Request-body parsing and response framing for the endpoints the worker terminates.
// The reference relays opaque bytes (dispatcher.rs:287-312), so these formats follow the public Ollama /
// OpenAI wire shapes seen in the reference's own client script (test_dispatcher.sh:37-39,69,93) and README.
// Parity here is UNPINNED by the reference (SURVEY.md 7 "hard parts").
#pragma once
#include "../../include/ollamamq_b200.h"
#include <cstdint>
#include <string>
#include <utility>
#include <vector>

namespace mq {

struct ParsedBody {
  std::string model;
  std::string text;             // prompt / concatenated message contents
  std::vector<int32_t> tokens;  // "context": [ids] (Ollama /api/generate) or "prompt": [ids] (OpenAI completions)
  bool has_stream = false;
  bool stream = true;
  int num_predict = 0;          // options.num_predict | max_tokens | max_completion_tokens
  // sampling: options.{temperature, top_k, top_p, seed} (Ollama) or top-level temperature / top_p / seed (OpenAI)
  bool has_temperature = false, has_top_k = false, has_top_p = false, has_seed = false;
  double temperature = 0, top_p = 0;
  long long top_k = 0;
  unsigned long long seed = 0;
  // token log-probabilities, top level only: "logprobs": true / false (/api/*, /v1/chat/completions) or N / null
  // (/v1/completions, where N also sets top_logprobs); "top_logprobs": N.  N is clamped to 0..MQ_TOP_LOGPROBS_MAX.
  bool has_logprobs = false, logprobs = false;
  bool has_top_logprobs = false;
  int top_logprobs = 0;
};

// One relayed token's log-probability entry: its own, and the top alternatives (logit descending, id ascending).
struct TokenLogprobs {
  int id = 0;
  float logprob = 0.f;
  std::vector<std::pair<int, float>> top;
};

bool parse_body(const std::string& body, int endpoint, ParsedBody* out);
// Folds a parsed body into the request: "stream" when the request left it to the body (< 0), the body's num_predict
// when max_new_tokens is unset (<= 0), and every sampling / logprobs option the body sets, over the struct's value.
void apply_body(const ParsedBody& pb, mq_request* rq);
std::vector<int32_t> byte_tokenize(const std::string& text, int vocab);
std::string token_text(int tok);
const char* content_type_for(int endpoint, int stream);
// lp: the token's logprobs entry (nullptr = off: the frame is exactly the one without); text_off = characters of the
// reply before this token (/v1/completions "text_offset")
std::string frame_token(int endpoint, const char* model, int tok, const TokenLogprobs* lp = nullptr, size_t text_off = 0);
// raw-token record (MQ_EP_RAW_TOKENS with logprobs): int32 id, float32 logprob, N x (int32 id, float32 logprob)
void append_raw_record(std::string* out, const TokenLogprobs& e);
// MQ_EP_OTHER: what the backend answers on the non-generation routes (main.rs:92-112) without touching the GPU
void other_route_response(const std::string& path, const char* model, int* status, std::string* ctype, std::string* body);
// stopped: done_reason / finish_reason "stop" (EOS) instead of "length".  lps: every token's entry, carried by the
// stream = 0 reply (nullptr = off: the reply is exactly the one without)
std::string frame_final(int endpoint, int stream, const char* model, const std::string& agg, int n_prompt, int n_gen,
                        bool stopped = false, const std::vector<TokenLogprobs>* lps = nullptr);

// ---- embeddings (/api/embed, /api/embeddings, /v1/embeddings)
struct ParsedEmbed {
  std::string model;
  std::vector<std::string> texts;              // "input": "s" | ["s", ...]   or "prompt": "s" (/api/embeddings)
  std::vector<std::vector<int32_t>> token_seqs;  // "input": [ids] | [[ids], ...] (OpenAI token inputs)
};
bool parse_embed_body(const std::string& body, ParsedEmbed* out);
// [CLS] bytes... [SEP] over a byte-level vocabulary (random-init weights have no word pieces), truncated to max_len
std::vector<int32_t> embed_tokenize(const std::string& text, int vocab, int max_len);
// emb: n rows of `dim` floats; the reply shape follows the route (Ollama /api/embed, legacy /api/embeddings, OpenAI)
std::string frame_embeddings(const std::string& path, const char* model, const float* emb, int n, int dim, int n_tokens);

}  // namespace mq
