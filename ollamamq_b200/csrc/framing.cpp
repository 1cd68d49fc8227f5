#include "framing.hpp"
#include "../../include/ollamamq_b200.h"
#include <cctype>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>

namespace mq {

// ------------------------------------------------------------------ minimal JSON walker
// Strict by construction (round-1 advisor findings): every loop consumes at least one byte per turn or fails, nesting
// is bounded (kMaxDepth) so the recursion cannot be driven into the guard page, numbers are clamped before they are
// narrowed (NaN / inf / 1e300 never reach a cast), and \u escapes are validated (surrogate pairs are combined).
namespace {
constexpr int kMaxDepth = 64;

double clamp_num(double v, double lo, double hi) { return !(v == v) ? 0.0 : (v < lo ? lo : (v > hi ? hi : v)); }

struct J {
  const char* p;
  const char* e;
  int depth = 0;
  void ws() { while (p < e && (*p == ' ' || *p == '\n' || *p == '\t' || *p == '\r')) ++p; }
  bool at(char c) { ws(); return p < e && *p == c; }
  bool lit(const char* s) {
    size_t n = strlen(s);
    if ((size_t)(e - p) >= n && memcmp(p, s, n) == 0) { p += n; return true; }
    return false;
  }
  static int hexv(char c) {
    if (c >= '0' && c <= '9') return c - '0';
    if (c >= 'a' && c <= 'f') return c - 'a' + 10;
    if (c >= 'A' && c <= 'F') return c - 'A' + 10;
    return -1;
  }
  bool hex4(unsigned* cp) {
    if (e - p < 4) return false;
    unsigned v = 0;
    for (int i = 0; i < 4; ++i) {
      const int h = hexv(p[i]);
      if (h < 0) return false;
      v = v * 16 + (unsigned)h;
    }
    p += 4;
    *cp = v;
    return true;
  }
  static void utf8(std::string* out, unsigned cp) {
    if (!out) return;
    if (cp < 0x80) out->push_back((char)cp);
    else if (cp < 0x800) { out->push_back((char)(0xC0 | (cp >> 6))); out->push_back((char)(0x80 | (cp & 0x3F))); }
    else if (cp < 0x10000) {
      out->push_back((char)(0xE0 | (cp >> 12))); out->push_back((char)(0x80 | ((cp >> 6) & 0x3F))); out->push_back((char)(0x80 | (cp & 0x3F)));
    } else {
      out->push_back((char)(0xF0 | (cp >> 18))); out->push_back((char)(0x80 | ((cp >> 12) & 0x3F)));
      out->push_back((char)(0x80 | ((cp >> 6) & 0x3F))); out->push_back((char)(0x80 | (cp & 0x3F)));
    }
  }
  bool str(std::string* out) {
    ws();
    if (p >= e || *p != '"') return false;
    ++p;
    while (p < e && *p != '"') {
      if (*p == '\\') {
        if (p + 1 >= e) return false;
        ++p;
        const char c = *p++;
        switch (c) {
          case 'n': if (out) out->push_back('\n'); break;
          case 't': if (out) out->push_back('\t'); break;
          case 'r': if (out) out->push_back('\r'); break;
          case 'b': if (out) out->push_back('\b'); break;
          case 'f': if (out) out->push_back('\f'); break;
          case '"': case '\\': case '/': if (out) out->push_back(c); break;
          case 'u': {
            unsigned cp = 0;
            if (!hex4(&cp)) return false;
            if (cp >= 0xD800 && cp <= 0xDBFF) {  // high surrogate: a low one must follow
              unsigned lo = 0;
              if (e - p >= 6 && p[0] == '\\' && p[1] == 'u') {
                p += 2;
                if (!hex4(&lo)) return false;
              }
              cp = (lo >= 0xDC00 && lo <= 0xDFFF) ? 0x10000 + ((cp - 0xD800) << 10) + (lo - 0xDC00) : 0xFFFD;
            } else if (cp >= 0xDC00 && cp <= 0xDFFF) {
              cp = 0xFFFD;  // lone low surrogate
            }
            utf8(out, cp);
            break;
          }
          default: return false;
        }
      } else {
        if (out) out->push_back(*p);
        ++p;
      }
    }
    if (p >= e) return false;
    ++p;
    return true;
  }
  // {"k": v, ...}: f(key) consumes the value.  Fails on anything but `,` or `}` after a member.
  template <class F>
  bool object(F&& f) {
    if (!at('{') || depth >= kMaxDepth) return false;
    ++p;
    ++depth;
    if (at('}')) { ++p; --depth; return true; }
    for (;;) {
      std::string k;
      if (!str(&k)) return false;
      if (!at(':')) return false;
      ++p;
      if (!f(k)) return false;
      if (at(',')) { ++p; continue; }
      if (at('}')) { ++p; --depth; return true; }
      return false;
    }
  }
  // [v, ...]: f() consumes one element
  template <class F>
  bool array(F&& f) {
    if (!at('[') || depth >= kMaxDepth) return false;
    ++p;
    ++depth;
    if (at(']')) { ++p; --depth; return true; }
    for (;;) {
      if (!f()) return false;
      if (at(',')) { ++p; continue; }
      if (at(']')) { ++p; --depth; return true; }
      return false;
    }
  }
  bool skip() {  // skip any value; recursion is bounded by kMaxDepth
    ws();
    if (p >= e) return false;
    if (*p == '"') return str(nullptr);
    if (*p == '{') return object([&](const std::string&) { return skip(); });
    if (*p == '[') return array([&] { return skip(); });
    const char* b = p;  // number / true / false / null: must consume at least one byte
    while (p < e && *p != ',' && *p != '}' && *p != ']' && *p != ' ' && *p != '\n' && *p != '\t' && *p != '\r') ++p;
    return p > b;
  }
  bool number(double* v) {
    ws();
    if (p >= e || !(*p == '-' || (*p >= '0' && *p <= '9'))) return false;  // JSON numbers only: no nan / inf / hex
    {  // plain integers of up to 15 digits (token ids, num_predict, seeds): no strtod
      const char* q = p + (*p == '-');
      double acc = 0.0;
      int nd = 0;
      while (q < e && *q >= '0' && *q <= '9' && nd < 15) { acc = acc * 10.0 + (*q - '0'); ++q; ++nd; }
      if (nd > 0 && (q >= e || (*q != '.' && *q != 'e' && *q != 'E' && !(*q >= '0' && *q <= '9')))) {
        *v = *p == '-' ? -acc : acc;
        p = q;
        return true;
      }
    }
    char* end = nullptr;
    *v = strtod(p, &end);  // the buffer is a std::string: NUL-terminated
    if (end == p || end > e) return false;
    p = end;
    return true;
  }
  bool int_array(std::vector<int32_t>* out) {
    return array([&] {
      double v;
      if (!number(&v)) return false;
      out->push_back((int32_t)clamp_num(v, -2147483647.0, 2147483647.0));
      return true;
    });
  }
  // number into *v, or skip whatever else is there (null, a string, ...): *got tells which
  bool number_or_skip(double* v, bool* got) {
    const char* save = p;
    *got = number(v);
    if (*got) return true;
    p = save;
    return skip();
  }
};

bool parse_content(J& j, std::string* text) {  // string or [{type:text,text:..},..]
  if (j.at('"')) { std::string s; if (!j.str(&s)) return false; *text += s; return true; }
  if (j.at('['))
    return j.array([&] {
      if (!j.at('{')) return j.skip();
      return j.object([&](const std::string& k) {
        if (k == "text" && j.at('"')) { std::string s; if (!j.str(&s)) return false; *text += s; return true; }
        return j.skip();
      });
    });
  return j.skip();
}

bool parse_messages(J& j, std::string* text) {
  if (!j.at('[')) return j.skip();
  return j.array([&] {
    if (!j.at('{')) return j.skip();
    return j.object([&](const std::string& k) {
      if (k == "content") { if (!parse_content(j, text)) return false; text->push_back('\n'); return true; }
      return j.skip();
    });
  });
}

bool parse_sampling(J& j, const std::string& k, ParsedBody* out, bool* used) {
  double v;
  bool got;
  *used = true;
  if (k == "num_predict" || k == "max_tokens" || k == "max_completion_tokens") {
    if (!j.number_or_skip(&v, &got)) return false;
    if (got) out->num_predict = (int)clamp_num(v, -1.0, 1073741824.0);
  } else if (k == "temperature") {
    if (!j.number_or_skip(&v, &got)) return false;
    if (got) { out->temperature = clamp_num(v, 0.0, 1e6); out->has_temperature = true; }
  } else if (k == "top_k") {
    if (!j.number_or_skip(&v, &got)) return false;
    if (got) { out->top_k = (long long)clamp_num(v, 0.0, 1073741824.0); out->has_top_k = true; }
  } else if (k == "top_p") {
    if (!j.number_or_skip(&v, &got)) return false;
    if (got) { out->top_p = clamp_num(v, 0.0, 1.0); out->has_top_p = true; }
  } else if (k == "seed") {
    if (!j.number_or_skip(&v, &got)) return false;
    if (got) { out->seed = (unsigned long long)clamp_num(v, 0.0, 9007199254740992.0); out->has_seed = true; }
  } else {
    *used = false;
  }
  return true;
}
}  // namespace

bool parse_body(const std::string& body, int endpoint, ParsedBody* out) {
  J j{body.data(), body.data() + body.size()};
  const bool legacy_lp = endpoint == MQ_EP_V1_COMPLETIONS;  // "logprobs": N | null instead of true | false
  int legacy_n = -1;
  const bool ok = j.object([&](const std::string& k) {
    bool used = false;
    if (k == "model") return j.at('"') ? j.str(&out->model) : j.skip();
    if (k == "logprobs") {
      j.ws();
      if (legacy_lp) {
        if (j.lit("null")) { out->has_logprobs = true; out->logprobs = false; legacy_n = -1; return true; }
        double v;
        bool got;
        if (!j.number_or_skip(&v, &got)) return false;
        if (got) { out->has_logprobs = out->logprobs = true; legacy_n = (int)clamp_num(v, 0.0, MQ_TOP_LOGPROBS_MAX); }
        return true;
      }
      if (j.lit("true")) { out->has_logprobs = out->logprobs = true; return true; }
      if (j.lit("false")) { out->has_logprobs = true; out->logprobs = false; return true; }
      return j.skip();
    }
    if (k == "top_logprobs") {
      double v;
      bool got;
      if (!j.number_or_skip(&v, &got)) return false;
      if (got) { out->has_top_logprobs = true; out->top_logprobs = (int)clamp_num(v, 0.0, MQ_TOP_LOGPROBS_MAX); }
      return true;
    }
    if (k == "prompt") {
      if (j.at('[')) return j.int_array(&out->tokens);
      if (j.at('"')) return j.str(&out->text);
      return j.skip();
    }
    if (k == "context") return j.at('[') ? j.int_array(&out->tokens) : j.skip();
    if (k == "messages") return parse_messages(j, &out->text);
    if (k == "stream") {
      j.ws();
      if (j.lit("true")) { out->has_stream = true; out->stream = true; return true; }
      if (j.lit("false")) { out->has_stream = true; out->stream = false; return true; }
      return j.skip();
    }
    if (k == "options") {
      if (!j.at('{')) return j.skip();
      return j.object([&](const std::string& ok2) {
        bool u2 = false;
        if (!parse_sampling(j, ok2, out, &u2)) return false;
        return u2 ? true : j.skip();
      });
    }
    if (k != "top_k") {  // OpenAI top level: temperature, top_p, seed, max_tokens (top_k lives in Ollama's options only)
      if (!parse_sampling(j, k, out, &used)) return false;
      if (used) return true;
    }
    return j.skip();
  });
  if (!ok) return false;
  if (legacy_n >= 0) { out->has_top_logprobs = true; out->top_logprobs = legacy_n; }
  j.ws();
  return j.p == j.e;  // nothing but whitespace after the object
}

void apply_body(const ParsedBody& pb, mq_request* rq) {
  if (pb.has_stream && rq->stream < 0) rq->stream = pb.stream ? 1 : 0;
  if (rq->max_new_tokens <= 0 && pb.num_predict > 0) rq->max_new_tokens = pb.num_predict;
  if (pb.has_temperature) rq->temperature = (float)pb.temperature;
  if (pb.has_top_k) rq->top_k = (int32_t)pb.top_k;  // parse_body clamped it to 0..2^30
  if (pb.has_top_p) rq->top_p = (float)pb.top_p;
  if (pb.has_seed) rq->seed = pb.seed;
  if (pb.has_logprobs) rq->logprobs = pb.logprobs ? 1 : 0;
  if (pb.has_top_logprobs) rq->top_logprobs = (int16_t)pb.top_logprobs;
}

// deterministic byte-level tokenizer: random-init weights have no vocabulary (SURVEY.md 7)
std::vector<int32_t> byte_tokenize(const std::string& text, int vocab) {
  std::vector<int32_t> t;
  t.reserve(text.size());
  for (unsigned char c : text) t.push_back((int32_t)(c % (unsigned)vocab));
  return t;
}

std::string token_text(int tok) {
  char b[24];
  snprintf(b, sizeof(b), " t%d", tok);
  return b;
}

const char* content_type_for(int endpoint, int stream) {
  if (endpoint == MQ_EP_RAW_TOKENS) return "application/octet-stream";
  if (!stream) return "application/json";
  return (endpoint == MQ_EP_V1_CHAT || endpoint == MQ_EP_V1_COMPLETIONS) ? "text/event-stream" : "application/x-ndjson";
}

static std::string json_escape(const std::string& s) {
  std::string o;
  for (unsigned char c : s) {
    if (c == '"' || c == '\\') { o.push_back('\\'); o.push_back((char)c); }
    else if (c < 0x20) { char b[8]; snprintf(b, sizeof(b), "\\u%04x", c); o += b; }
    else o.push_back((char)c);
  }
  return o;
}

static std::string now_iso() {
  char b[40];
  time_t t = time(nullptr);
  struct tm tmv;
  gmtime_r(&t, &tmv);
  strftime(b, sizeof(b), "%Y-%m-%dT%H:%M:%SZ", &tmv);
  return b;
}

// model names are client-visible strings of ours (cfg.model_name) or, for embeddings, of the client's: cap them so a
// frame stays a frame
static std::string model_field(const char* model) {
  std::string m = model ? model : "";
  if (m.size() > 256) m.resize(256);
  return json_escape(m);
}

// ---- token log-probabilities: Ollama's api.Logprob list on /api/*, OpenAI's choices[0].logprobs on /v1/*
static char* put_float(char* w, float f);
static void put_num(std::string& o, float f) {
  char b[32];
  o.append(b, (size_t)(put_float(b, f) - b));
}
static void lp_fields(std::string& o, int id, float lp) {  // "token":..,"logprob":..,"bytes":[..]
  const std::string t = token_text(id);
  o += "\"token\":\"" + json_escape(t) + "\",\"logprob\":";
  put_num(o, lp);
  o += ",\"bytes\":[";
  for (size_t i = 0; i < t.size(); ++i) {
    if (i) o += ',';
    o += std::to_string((unsigned char)t[i]);
  }
  o += ']';
}
// the "logprobs" member of a reply carrying n entries; /v1/completions counts text_offset from off0
static std::string lp_member(int endpoint, const TokenLogprobs* e, size_t n, size_t off0) {
  if (endpoint == MQ_EP_V1_COMPLETIONS) {
    std::string toks, lps, tops, offs;
    size_t off = off0;
    for (size_t i = 0; i < n; ++i) {
      const char* sep = i ? "," : "";
      const std::string t = token_text(e[i].id);
      toks += sep; toks += "\"" + json_escape(t) + "\"";
      lps += sep; put_num(lps, e[i].logprob);
      tops += sep; tops += '{';
      for (size_t j = 0; j < e[i].top.size(); ++j) {
        if (j) tops += ',';
        tops += "\"" + json_escape(token_text(e[i].top[j].first)) + "\":";
        put_num(tops, e[i].top[j].second);
      }
      tops += '}';
      offs += sep; offs += std::to_string(off);
      off += t.size();
    }
    return "\"logprobs\":{\"tokens\":[" + toks + "],\"token_logprobs\":[" + lps + "],\"top_logprobs\":[" + tops +
           "],\"text_offset\":[" + offs + "]}";
  }
  const bool chat = endpoint == MQ_EP_V1_CHAT;
  std::string o = chat ? "\"logprobs\":{\"content\":[" : "\"logprobs\":[";
  for (size_t i = 0; i < n; ++i) {
    if (i) o += ',';
    o += '{';
    lp_fields(o, e[i].id, e[i].logprob);
    o += ",\"top_logprobs\":[";
    for (size_t j = 0; j < e[i].top.size(); ++j) {
      if (j) o += ',';
      o += '{';
      lp_fields(o, e[i].top[j].first, e[i].top[j].second);
      o += '}';
    }
    o += "]}";
  }
  return o + (chat ? "]}" : "]");
}

void append_raw_record(std::string* out, const TokenLogprobs& e) {
  char b[8];
  memcpy(b, &e.id, 4); memcpy(b + 4, &e.logprob, 4);
  out->append(b, 8);
  for (auto& t : e.top) {
    memcpy(b, &t.first, 4); memcpy(b + 4, &t.second, 4);
    out->append(b, 8);
  }
}

std::string frame_token(int endpoint, const char* model, int tok, const TokenLogprobs* lp, size_t text_off) {
  const std::string m = model_field(model), txt = json_escape(token_text(tok));
  const std::string lpm = lp ? "," + lp_member(endpoint, lp, 1, text_off) : std::string();
  switch (endpoint) {
    case MQ_EP_API_GENERATE:
      return "{\"model\":\"" + m + "\",\"created_at\":\"" + now_iso() + "\",\"response\":\"" + txt + "\",\"done\":false" + lpm + "}\n";
    case MQ_EP_API_CHAT:
      return "{\"model\":\"" + m + "\",\"created_at\":\"" + now_iso() + "\",\"message\":{\"role\":\"assistant\",\"content\":\"" + txt +
             "\"},\"done\":false" + lpm + "}\n";
    case MQ_EP_V1_CHAT:
      return "data: {\"id\":\"chatcmpl-mq\",\"object\":\"chat.completion.chunk\",\"created\":" + std::to_string((long)time(nullptr)) +
             ",\"model\":\"" + m + "\",\"choices\":[{\"index\":0,\"delta\":{\"content\":\"" + txt + "\"}" + lpm +
             ",\"finish_reason\":null}]}\n\n";
    default:
      return "data: {\"id\":\"cmpl-mq\",\"object\":\"text_completion\",\"created\":" + std::to_string((long)time(nullptr)) +
             ",\"model\":\"" + m + "\",\"choices\":[{\"text\":\"" + txt + "\",\"index\":0" + lpm + ",\"finish_reason\":null}]}\n\n";
  }
}

void other_route_response(const std::string& path, const char* model, int* status, std::string* ctype, std::string* body) {
  const std::string m = model_field(model);
  *status = 200;
  *ctype = "application/json";
  if (path == "/") {
    *ctype = "text/plain; charset=utf-8";
    *body = "Ollama is running";
  } else if (path == "/api/version") {
    *body = "{\"version\":\"0.0.0-ollamamq-b200\"}";
  } else if (path == "/api/tags" || path == "/api/ps") {
    *body = "{\"models\":[{\"name\":\"" + m + "\",\"model\":\"" + m + "\",\"details\":{\"format\":\"bf16\",\"family\":\"llama\"}}]}";
  } else if (path == "/api/show") {
    *body = "{\"details\":{\"format\":\"bf16\",\"family\":\"llama\"},\"model_info\":{\"general.name\":\"" + m + "\"}}";
  } else if (path == "/v1/models") {
    *body = "{\"object\":\"list\",\"data\":[{\"id\":\"" + m + "\",\"object\":\"model\",\"owned_by\":\"ollamamq-b200\"}]}";
  } else if (path.rfind("/v1/models/", 0) == 0) {
    *body = "{\"id\":\"" + json_escape(path.substr(11)) + "\",\"object\":\"model\",\"owned_by\":\"ollamamq-b200\"}";
  } else {
    *status = 501;  // embeddings and model management are not served by this worker
    *body = "{\"error\":\"" + json_escape(path) + " is not implemented by the B200 worker\"}";
  }
}

std::string frame_final(int endpoint, int stream, const char* model, const std::string& agg, int n_prompt, int n_gen,
                        bool stopped, const std::vector<TokenLogprobs>* lps) {
  const char* why = stopped ? "stop" : "length";  // EOS reached vs generation budget spent
  if (endpoint == MQ_EP_RAW_TOKENS) return stream ? std::string() : agg;
  const std::string m = model_field(model), txt = json_escape(agg);
  const std::string lpm = lps && !stream ? "," + lp_member(endpoint, lps->data(), lps->size(), 0) : std::string();
  std::string o;
  char buf[256];  // integers and the fixed words only: cannot truncate
  if (endpoint == MQ_EP_API_GENERATE || endpoint == MQ_EP_API_CHAT) {
    o = "{\"model\":\"" + m + "\",\"created_at\":\"" + now_iso() + "\",";
    if (endpoint == MQ_EP_API_GENERATE) o += "\"response\":\"" + (stream ? std::string() : txt) + "\",";
    else o += "\"message\":{\"role\":\"assistant\",\"content\":\"" + (stream ? std::string() : txt) + "\"},";
    snprintf(buf, sizeof(buf), "\"done\":true,\"done_reason\":\"%s\",\"prompt_eval_count\":%d,\"eval_count\":%d",
             why, n_prompt, n_gen);
    return o + buf + lpm + "}\n";
  }
  const bool chat = endpoint == MQ_EP_V1_CHAT;
  if (stream) {
    const std::string head = std::string(chat ? "data: {\"id\":\"chatcmpl-mq\",\"object\":\"chat.completion.chunk\",\"created\":"
                                              : "data: {\"id\":\"cmpl-mq\",\"object\":\"text_completion\",\"created\":") +
                             std::to_string((long)time(nullptr)) + ",\"model\":\"" + m + "\",";
    return head + (chat ? "\"choices\":[{\"index\":0,\"delta\":{},\"finish_reason\":\"" : "\"choices\":[{\"text\":\"\",\"index\":0,\"finish_reason\":\"") +
           why + "\"}]}\n\ndata: [DONE]\n\n";
  }
  snprintf(buf, sizeof(buf), "\"usage\":{\"prompt_tokens\":%d,\"completion_tokens\":%d,\"total_tokens\":%d}}", n_prompt,
           n_gen, n_prompt + n_gen);
  if (chat)
    o = "{\"id\":\"chatcmpl-mq\",\"object\":\"chat.completion\",\"model\":\"" + m +
        "\",\"choices\":[{\"index\":0,\"message\":{\"role\":\"assistant\",\"content\":\"" + txt +
        "\"}" + lpm + ",\"finish_reason\":\"" + std::string(why) + "\"}],";
  else
    o = "{\"id\":\"cmpl-mq\",\"object\":\"text_completion\",\"model\":\"" + m + "\",\"choices\":[{\"text\":\"" + txt +
        "\",\"index\":0" + lpm + ",\"finish_reason\":\"" + std::string(why) + "\"}],";
  return o + buf;
}


// ------------------------------------------------------------------ embeddings
bool parse_embed_body(const std::string& body, ParsedEmbed* out) {
  J j{body.data(), body.data() + body.size()};
  const bool ok = j.object([&](const std::string& k) {
    if (k == "model") return j.at('"') ? j.str(&out->model) : j.skip();
    if (k != "input" && k != "prompt") return j.skip();
    if (j.at('"')) { std::string s; if (!j.str(&s)) return false; out->texts.push_back(s); return true; }
    if (!j.at('[')) return j.skip();
    // ["s", ...] | [[ids], ...] | [ids]: decided by the first element
    const char* save = j.p;
    ++j.p;
    j.ws();
    const char first = j.p < j.e ? *j.p : 0;
    j.p = save;
    if (first == '"') return j.array([&] { std::string s; if (!j.str(&s)) return false; out->texts.push_back(s); return true; });
    if (first == '[')
      return j.array([&] {
        std::vector<int32_t> t;
        if (!j.int_array(&t)) return false;
        out->token_seqs.push_back(t);
        return true;
      });
    if (first == ']') return j.skip();
    std::vector<int32_t> t;
    if (!j.int_array(&t)) return false;
    out->token_seqs.push_back(t);
    return true;
  });
  if (!ok) return false;
  j.ws();
  return j.p == j.e;
}

std::vector<int32_t> embed_tokenize(const std::string& text, int vocab, int max_len) {
  // BERT conventions where the vocabulary has room for them: [CLS] = 101, [SEP] = 102, bytes from 1000
  const int cls = vocab > 1300 ? 101 : 1, sep = vocab > 1300 ? 102 : 2, base = vocab > 1300 ? 1000 : 3;
  std::vector<int32_t> t;
  t.push_back(cls);
  for (unsigned char c : text) {
    if ((int)t.size() >= max_len - 1) break;
    t.push_back(base + (int)(c % (unsigned)(vocab - base)));
  }
  if ((int)t.size() < max_len) t.push_back(sep);
  return t;
}

// One float as a JSON number with 9 significant digits (enough to round-trip a float32), trailing zeros trimmed.
// Fixed notation through 64-bit integer arithmetic for 1e-5 <= |x| < 1e9 (every component of a unit-norm embedding
// that matters); snprintf for the rest.  r02: "%.8g" per component was 5.2 ms for a 64 x 384 reply - on the embedding
// worker's thread, i.e. longer than the 3.4 ms the GPU needs for the 32 768 tokens of that request.
static char* put_float(char* w, float f) {
  if (!(f == f) || f - f != 0.f) { *w++ = '0'; return w; }  // NaN / inf have no JSON spelling
  double x = f;
  if (x < 0) { *w++ = '-'; x = -x; }
  if (x == 0.0) { *w++ = '0'; return w; }
  if (x < 1e-5 || x >= 1e9) return w + snprintf(w, 24, "%.9g", x);
  static const double p10[] = {1e0, 1e1, 1e2, 1e3, 1e4, 1e5, 1e6, 1e7, 1e8, 1e9, 1e10, 1e11, 1e12, 1e13, 1e14};
  int ex = x >= 1.0 ? 0 : -1;  // decimal exponent: 10^ex <= x < 10^(ex+1)
  if (x >= 1.0) { while (ex < 8 && x >= p10[ex + 1]) ++ex; }
  else { while (ex > -5 && x < 1.0 / p10[-ex]) --ex; }
  unsigned long long d = (unsigned long long)(x * p10[8 - ex] + 0.5);  // 9 significant digits
  if (d >= 1000000000ull) { d /= 10; ++ex; }
  if (d < 100000000ull) { d *= 10; --ex; }   // (x sat just below a power of ten)
  char dig[9];
  for (int i = 8; i >= 0; --i) { dig[i] = (char)('0' + d % 10); d /= 10; }
  int last = 8;
  while (last > 0 && dig[last] == '0') --last;  // significant digits to print: dig[0 .. last]
  if (ex >= 0) {
    for (int i = 0; i <= ex; ++i) *w++ = i <= 8 ? dig[i] : '0';
    if (last > ex) {
      *w++ = '.';
      for (int i = ex + 1; i <= last; ++i) *w++ = dig[i];
    }
  } else {
    *w++ = '0'; *w++ = '.';
    for (int i = -1; i > ex; --i) *w++ = '0';
    for (int i = 0; i <= last; ++i) *w++ = dig[i];
  }
  return w;
}
static void append_vec(std::string& o, const float* v, int dim) {
  const size_t at = o.size();
  o.resize(at + (size_t)dim * 26 + 2);
  char* w = &o[at];
  *w++ = '[';
  for (int i = 0; i < dim; ++i) {
    if (i) *w++ = ',';
    w = put_float(w, v[i]);
  }
  *w++ = ']';
  o.resize((size_t)(w - o.data()));
}
std::string frame_embeddings(const std::string& path, const char* model, const float* emb, int n, int dim, int n_tokens) {
  const std::string m = model_field(model);
  std::string o;
  o.reserve((size_t)n * dim * 14 + 256);
  char b[96];  // integers only
  if (path == "/api/embeddings") {  // legacy Ollama route: one prompt, one vector
    o = "{\"embedding\":";
    append_vec(o, emb, n > 0 ? dim : 0);
    return o + "}";
  }
  if (path == "/v1/embeddings") {
    o = "{\"object\":\"list\",\"data\":[";
    for (int i = 0; i < n; ++i) {
      if (i) o += ',';
      o += "{\"object\":\"embedding\",\"embedding\":";
      append_vec(o, emb + (size_t)i * dim, dim);
      snprintf(b, sizeof b, ",\"index\":%d}", i);
      o += b;
    }
    snprintf(b, sizeof b, "\",\"usage\":{\"prompt_tokens\":%d,\"total_tokens\":%d}}", n_tokens, n_tokens);
    return o + "],\"model\":\"" + m + b;
  }
  o = "{\"model\":\"" + m + "\",\"embeddings\":[";
  for (int i = 0; i < n; ++i) {
    if (i) o += ',';
    append_vec(o, emb + (size_t)i * dim, dim);
  }
  snprintf(b, sizeof b, "],\"prompt_eval_count\":%d}", n_tokens);
  return o + b;
}

}  // namespace mq

// ------------------------------------------------------------------ host-only test ABI for the parsers / framers
extern "C" {
static long long emit_json(const std::string& o, char* out, size_t cap) {
  if (out && cap > o.size()) memcpy(out, o.c_str(), o.size() + 1);
  return (long long)o.size() + 1;
}
long long mq_debug_parse_body(int32_t endpoint, const uint8_t* body, size_t len, int32_t vocab, char* out, size_t cap) {
  using namespace mq;
  ParsedBody pb;
  const bool ok = parse_body(std::string((const char*)body, body ? len : 0), endpoint, &pb);
  std::string toks = "[";
  const std::vector<int32_t> t = !pb.tokens.empty() ? pb.tokens : byte_tokenize(pb.text, vocab > 0 ? vocab : 256);
  for (size_t i = 0; i < t.size(); ++i) toks += (i ? "," : "") + std::to_string(t[i]);
  toks += "]";
  char b[640];
  snprintf(b, sizeof b, "{\"ok\":%s,\"has_stream\":%s,\"stream\":%s,\"num_predict\":%d,\"has_temperature\":%s,\"temperature\":%.9g,"
           "\"has_top_k\":%s,\"top_k\":%lld,\"has_top_p\":%s,\"top_p\":%.9g,\"has_seed\":%s,\"seed\":%llu,\"n_text\":%zu,"
           "\"has_logprobs\":%s,\"logprobs\":%s,\"has_top_logprobs\":%s,\"top_logprobs\":%d,",
           ok ? "true" : "false", pb.has_stream ? "true" : "false", pb.stream ? "true" : "false", pb.num_predict,
           pb.has_temperature ? "true" : "false", pb.temperature, pb.has_top_k ? "true" : "false", pb.top_k,
           pb.has_top_p ? "true" : "false", pb.top_p, pb.has_seed ? "true" : "false", pb.seed, pb.text.size(),
           pb.has_logprobs ? "true" : "false", pb.logprobs ? "true" : "false", pb.has_top_logprobs ? "true" : "false",
           pb.top_logprobs);
  return emit_json(std::string(b) + "\"model\":\"" + json_escape(pb.model) + "\",\"tokens\":" + toks + "}", out, cap);
}
long long mq_debug_parse_embed(const uint8_t* body, size_t len, int32_t vocab, int32_t max_len, char* out, size_t cap) {
  using namespace mq;
  ParsedEmbed pe;
  const bool ok = parse_embed_body(std::string((const char*)body, body ? len : 0), &pe);
  std::string o = std::string("{\"ok\":") + (ok ? "true" : "false") + ",\"model\":\"" + json_escape(pe.model) + "\",\"seqs\":[";
  bool first = true;
  auto put = [&](const std::vector<int32_t>& t) {
    o += first ? "[" : ",[";
    first = false;
    for (size_t i = 0; i < t.size(); ++i) o += (i ? "," : "") + std::to_string(t[i]);
    o += "]";
  };
  for (auto& t : pe.texts) put(embed_tokenize(t, vocab, max_len));
  for (auto& t : pe.token_seqs) put(t);
  return emit_json(o + "]}", out, cap);
}
long long mq_debug_frame_embeddings(const char* path, const char* model, const float* emb, int32_t n, int32_t dim,
                                    int32_t n_tokens, char* out, size_t cap) {
  return emit_json(mq::frame_embeddings(path ? path : "/api/embed", model ? model : "", emb, n, dim, n_tokens), out, cap);
}
long long mq_debug_frame_final(int32_t endpoint, int32_t stream, const char* model, const char* agg, int32_t n_prompt,
                               int32_t n_gen, int32_t stopped, char* out, size_t cap) {
  return emit_json(mq::frame_final(endpoint, stream, model ? model : "", agg ? agg : "", n_prompt, n_gen, stopped != 0), out, cap);
}
long long mq_debug_frame_logprobs(int32_t endpoint, int32_t stream, const char* model, const int32_t* ids,
                                  const float* records, int32_t n, int32_t top_logprobs, int32_t n_prompt, char* out,
                                  size_t cap) {
  using namespace mq;
  const char* mdl = model ? model : "";
  const bool on = top_logprobs >= 0;
  std::vector<TokenLogprobs> lps;
  std::string agg, o;
  size_t text_len = 0;
  for (int i = 0; i < n; ++i) {
    TokenLogprobs e;
    e.id = ids[i];
    if (on) {
      const float* r = records + (size_t)i * (1 + 2 * top_logprobs);
      e.logprob = r[0];
      for (int j = 0; j < top_logprobs; ++j) {
        int id;
        memcpy(&id, r + 1 + 2 * j, 4);
        e.top.push_back({id, r[2 + 2 * j]});
      }
    }
    if (stream) {
      if (endpoint == MQ_EP_RAW_TOKENS) {
        if (on) append_raw_record(&o, e);
        else o.append((const char*)&e.id, 4);
      } else {
        o += frame_token(endpoint, mdl, e.id, on ? &e : nullptr, text_len);
      }
    } else if (endpoint == MQ_EP_RAW_TOKENS) {
      if (on) append_raw_record(&agg, e);
      else agg.append((const char*)&e.id, 4);
    } else {
      agg += token_text(e.id);
    }
    text_len += token_text(e.id).size();
    lps.push_back(e);
  }
  o += frame_final(endpoint, stream, mdl, agg, n_prompt, n, false, on ? &lps : nullptr);
  return emit_json(o, out, cap);  // (raw tokens: binary, the returned length minus the terminator)
}
}  // extern "C"

namespace mq {
}  // namespace mq
