"""Host-side mirror of the GPU worker / dispatcher C ABI (include/ollamamq_b200.h sections 2-3).
Marshalling only: there is no Python implementation of the forward pass."""
from __future__ import annotations

import ctypes as C
import threading
import time
from typing import Callable, Dict, List, Optional, Sequence

from . import _lib
from ._lib import lib, check, MQError

EP_API_GENERATE, EP_API_CHAT, EP_V1_CHAT, EP_V1_COMPLETIONS, EP_RAW_TOKENS = 0, 1, 2, 3, 4
ENDPOINT_OF_PATH = {"/api/generate": EP_API_GENERATE, "/api/chat": EP_API_CHAT,
                    "/v1/chat/completions": EP_V1_CHAT, "/v1/completions": EP_V1_COMPLETIONS}


def model_cfg(geom: dict, max_batch=64, max_seq=1024, max_prefill_tokens=2048, kv_pages=0, use_graphs=1,
              use_pdl=0, model_name="random-init", eos_token_id=0) -> _lib.ModelCfg:
    c = _lib.ModelCfg()
    for k in ("vocab", "hidden", "ffn", "n_layers", "n_q_heads", "n_kv_heads", "head_dim"):
        setattr(c, k, int(geom[k]))
    c.qkv_bias = int(geom.get("qkv_bias", 0))
    c.rope_theta = float(geom.get("rope_theta", 500000.0))
    c.rms_eps = float(geom.get("rms_eps", 1e-5))
    c.max_batch, c.max_seq, c.max_prefill_tokens = max_batch, max_seq, max_prefill_tokens
    c.kv_pages, c.use_graphs, c.use_pdl = kv_pages, use_graphs, use_pdl
    c.eos_token_id = int(geom.get("eos_token_id", eos_token_id))
    c.model_name = model_name.encode()[:63]
    return c


def encoder_cfg(geom: dict, max_seq=512, max_tokens_per_pass=32768, use_pdl=1, model_name="random-init-encoder"):
    c = _lib.EncoderCfg()
    for k in ("vocab", "hidden", "ffn", "n_layers", "n_heads", "head_dim", "max_positions"):
        setattr(c, k, int(geom[k]))
    c.type_vocab = int(geom.get("type_vocab", 2))
    c.ln_eps = float(geom.get("ln_eps", 1e-12))
    c.max_seq, c.max_tokens_per_pass, c.use_pdl = min(max_seq, c.max_positions), max_tokens_per_pass, use_pdl
    c.model_name = model_name.encode()[:63]
    return c


class Stream:
    """Receives the Status / Chunk / Done parts of one request (the reference's mpsc receiver)."""

    def __init__(self, on_chunk: Optional[Callable[[bytes], bool]] = None):
        self.status = None
        self.content_type = None
        self.chunks: List[bytes] = []
        self.chunk_times: List[float] = []
        self.rc = None
        self.err = ""
        self.done = threading.Event()
        self._on_chunk = on_chunk
        self.t_submit = time.perf_counter()
        self.t_done = None
        self.handle = None
        self.top_logprobs = -1   # >= 0: the request asked for logprobs (raw chunks are then records, see tokens())

        def _status(_u, code, ctype):
            self.status, self.content_type = code, (ctype or b"").decode()

        def _chunk(_u, data, n):
            b = C.string_at(data, n)
            self.chunks.append(b)
            self.chunk_times.append(time.perf_counter())
            if self._on_chunk is not None and self._on_chunk(b) is False:
                return 1
            return 0

        def _done(_u, rc, msg):
            self.rc, self.err = rc, (msg or b"").decode("utf-8", "replace")
            self.t_done = time.perf_counter()
            self.done.set()

        self._keep = (_lib.ON_STATUS(_status), _lib.ON_CHUNK(_chunk), _lib.ON_DONE(_done))
        self.cb = _lib.Callbacks(*self._keep)

    def wait(self, timeout=None) -> "Stream":
        if not self.done.wait(timeout):
            raise TimeoutError("request did not complete")
        return self

    @property
    def body(self) -> bytes:
        return b"".join(self.chunks)

    def _records(self):
        import numpy as np
        n = self.top_logprobs
        rec = np.dtype([("id", "<i4"), ("logprob", "<f4"), ("top", [("id", "<i4"), ("logprob", "<f4")], (n,))])
        return np.frombuffer(self.body, dtype=rec)

    def tokens(self) -> List[int]:
        """Token ids of a raw-token reply (4-byte ids, or the ids of the logprob records when logprobs were asked)."""
        import struct
        if self.top_logprobs >= 0:
            return [int(t) for t in self._records()["id"]]
        b = self.body
        return list(struct.unpack("<%di" % (len(b) // 4), b))

    def logprobs(self) -> List[tuple]:
        """Raw-token reply of a request with logprobs: (logprob, [(id, logprob), ...top_logprobs]) per token."""
        if self.top_logprobs < 0:
            raise ValueError("the request did not ask for logprobs")
        return [(float(r["logprob"]), [(int(t["id"]), float(t["logprob"])) for t in r["top"]]) for r in self._records()]

    @property
    def ttft(self) -> Optional[float]:
        return self.chunk_times[0] - self.t_submit if self.chunk_times else None


def make_request(endpoint=EP_RAW_TOKENS, prompt_tokens: Optional[Sequence[int]] = None, body: Optional[bytes] = None,
                 max_new_tokens=16, stream=1, timeout_ms=0, path: Optional[str] = None, temperature=0.0, top_k=0,
                 top_p=0.0, seed=0, ignore_eos=1, logprobs=False, top_logprobs=0):
    r = _lib.Request()
    if path is not None:
        r.path = path.encode()
    r.endpoint, r.stream, r.max_new_tokens, r.ignore_eos, r.timeout_ms = endpoint, stream, max_new_tokens, ignore_eos, timeout_ms
    r.temperature, r.top_k, r.top_p, r.seed = float(temperature), int(top_k), float(top_p), int(seed)
    r.logprobs = 1 if logprobs else 0
    r.top_logprobs = max(0, min(int(top_logprobs), _lib.MQ_TOP_LOGPROBS_MAX))
    keep = []
    if body is not None:
        buf = C.create_string_buffer(body, len(body))
        keep.append(buf)
        r.body, r.body_len = C.cast(buf, C.c_void_p), len(body)
    if prompt_tokens is not None:
        arr = (C.c_int32 * len(prompt_tokens))(*prompt_tokens)
        keep.append(arr)
        r.prompt_tokens, r.n_prompt_tokens = C.cast(arr, C.c_void_p), len(prompt_tokens)
    return r, keep


class Worker:
    """One B200 worker (`BackendStatus` slot of the reference, dispatcher.rs:41-47)."""

    def __init__(self, gpu: int, cfg: _lib.ModelCfg):
        self.cfg = cfg
        h = C.c_void_p()
        check(lib.mq_worker_open(gpu, C.byref(cfg), C.byref(h)))
        self._h = h
        self.gpu = gpu

    def close(self):
        if self._h:
            lib.mq_worker_close(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    @property
    def handle(self):
        return self._h

    def load_weights(self, weights: Dict[str, "object"]):
        """weights: name -> contiguous torch bf16 tensor (CPU or CUDA)."""
        for name, t in weights.items():
            t = t.contiguous()
            check(lib.mq_worker_load_tensor(self._h, name.encode(), C.c_void_p(t.data_ptr()),
                                            t.numel() * t.element_size()))

    def read_tensor(self, name: str, like):
        check(lib.mq_worker_read_tensor(self._h, name.encode(), C.c_void_p(like.data_ptr()),
                                        like.numel() * like.element_size()))
        return like

    def init_random(self, seed=0, std=0.02):
        check(lib.mq_worker_init_random(self._h, seed, std))

    def capacity(self) -> int:
        return lib.mq_worker_capacity(self._h)

    def healthy(self) -> bool:
        return bool(lib.mq_worker_healthy(self._h))

    def forward_logits(self, tokens: Sequence[int], all_positions=False):
        import numpy as np
        n = len(tokens)
        arr = (C.c_int32 * n)(*tokens)
        out = np.empty(((n if all_positions else 1), self.cfg.vocab), dtype=np.float32)
        check(lib.mq_debug_forward(self._h, arr, n, 1 if all_positions else 0, out.ctypes.data_as(C.c_void_p)))
        return out

    def submit(self, sink: Stream, **kw) -> Stream:
        """kw: endpoint, prompt_tokens, body, max_new_tokens, stream (1/0/-1), timeout_ms, sampling, logprobs /
        top_logprobs."""
        r, keep = make_request(**kw)
        h = C.c_void_p()
        sink.top_logprobs = r.top_logprobs if r.logprobs else -1
        sink.t_submit = time.perf_counter()
        check(lib.mq_submit(self._h, C.byref(r), C.byref(sink.cb), None, C.byref(h)))
        sink.handle = h
        sink._worker = self
        return sink

    def generate(self, prompt_tokens: Sequence[int], max_new_tokens: int, timeout=120, logprobs=False, top_logprobs=0):
        """Token ids; with logprobs=True, (token ids, Stream.logprobs())."""
        s = self.submit(Stream(), prompt_tokens=list(prompt_tokens), max_new_tokens=max_new_tokens, logprobs=logprobs,
                        top_logprobs=top_logprobs)
        s.wait(timeout)
        lib.mq_req_release(s.handle)
        if s.rc != 0:
            raise MQError(s.rc, s.err)
        return (s.tokens(), s.logprobs()) if logprobs else s.tokens()

    def stats(self) -> dict:
        st = _lib.WorkerStats()
        check(lib.mq_worker_get_stats(self._h, C.byref(st)))
        return {k: getattr(st, k) for k, _ in st._fields_}

    def occupancy(self) -> dict:
        oc = _lib.WorkerOccupancy()
        check(lib.mq_worker_get_occupancy(self._h, C.byref(oc)))
        return {k: getattr(oc, k) for k, _ in oc._fields_}

    def reset_stats(self):
        check(lib.mq_worker_reset_stats(self._h))

    def set_timing(self, on: bool):
        check(lib.mq_worker_set_timing(self._h, 1 if on else 0))


class Encoder:
    """Embedding worker on one B200 (BERT-family encoder; /api/embed, /api/embeddings, /v1/embeddings)."""

    EP_EMBED = 6

    def __init__(self, gpu: int, cfg: _lib.EncoderCfg):
        self.cfg = cfg
        h = C.c_void_p()
        check(lib.mq_encoder_open(gpu, C.byref(cfg), C.byref(h)))
        self._h = h

    def close(self):
        if self._h:
            lib.mq_encoder_close(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    @property
    def handle(self):
        return self._h

    def load_weights(self, weights: Dict[str, "object"]):
        for name, t in weights.items():
            t = t.contiguous()
            check(lib.mq_encoder_load_tensor(self._h, name.encode(), C.c_void_p(t.data_ptr()),
                                             t.numel() * t.element_size()))

    def read_tensor(self, name: str, like):
        check(lib.mq_encoder_read_tensor(self._h, name.encode(), C.c_void_p(like.data_ptr()),
                                         like.numel() * like.element_size()))
        return like

    def init_random(self, seed=0, std=0.05):
        check(lib.mq_encoder_init_random(self._h, seed, std))

    def healthy(self) -> bool:
        return bool(lib.mq_encoder_healthy(self._h))

    def stats(self) -> dict:
        st = _lib.EncoderStats()
        check(lib.mq_encoder_get_stats(self._h, C.byref(st)))
        return {k: getattr(st, k) for k, _ in st._fields_}

    def embed(self, sequences: Sequence[Sequence[int]]):
        """Blocking: numpy fp32 [n_seq, hidden], rows L2-normalised."""
        import numpy as np
        if isinstance(sequences, np.ndarray) and sequences.ndim == 2:   # [n_seq, seq_len] ids: no per-token python work
            toks = np.ascontiguousarray(sequences, dtype=np.int32).reshape(-1)
            off = np.arange(0, (sequences.shape[0] + 1) * sequences.shape[1], max(1, sequences.shape[1]), dtype=np.int32)
            n = sequences.shape[0]
        else:
            arrs = [np.asarray(s, dtype=np.int32).reshape(-1) for s in sequences]
            n = len(arrs)
            toks = np.concatenate(arrs) if arrs else np.zeros(0, np.int32)
            off = np.zeros(n + 1, dtype=np.int32)
            np.cumsum([len(a) for a in arrs], out=off[1:])
        if toks.size == 0:
            toks = np.zeros(1, np.int32)
        out = np.empty((n, self.cfg.hidden), dtype=np.float32)
        check(lib.mq_encoder_embed(self._h, toks.ctypes.data_as(C.c_void_p), off.ctypes.data_as(C.c_void_p), n,
                                   out.ctypes.data_as(C.c_void_p)))
        return out

    def submit(self, sink: "Stream", body: bytes, path: str = "/api/embed") -> "Stream":
        r, keep = make_request(endpoint=self.EP_EMBED, body=body, path=path)
        h = C.c_void_p()
        sink.t_submit = time.perf_counter()
        check(lib.mq_encoder_submit(self._h, C.byref(r), C.byref(sink.cb), None, C.byref(h)))
        sink.handle = h
        return sink


class Dispatcher:
    """`AppState` + `run_worker` (dispatcher.rs:49-96,164-352) over GPU workers or step-driven mock backends."""

    def __init__(self, workers: Optional[Sequence[Worker]] = None, capacity: int = 1, mock_backends: int = 0):
        h = C.c_void_p()
        if workers:
            arr = (C.c_void_p * len(workers))(*[w.handle for w in workers])
            check(lib.mq_dispatcher_new(arr, len(workers), capacity, C.byref(h)))
            self.n_backends = len(workers)
        else:
            check(lib.mq_dispatcher_new_mock(mock_backends, capacity, C.byref(h)))
            self.n_backends = mock_backends
        self._h = h
        self._streams = []

    def close(self):
        self.stop_http()
        if self._h:
            lib.mq_dispatcher_free(self._h)
            self._h = None

    def submit(self, user: Optional[str], sink: Optional[Stream] = None, ip: Optional[str] = None, **kw) -> Stream:
        sink = sink or Stream()
        r, keep = make_request(**kw)
        sink.top_logprobs = r.top_logprobs if r.logprobs else -1
        tid = C.c_uint64()
        sink.t_submit = time.perf_counter()
        check(lib.mq_dispatcher_submit(self._h, None if user is None else user.encode(),
                                       None if ip is None else ip.encode(), C.byref(r), C.byref(sink.cb), None,
                                       C.byref(tid)))
        sink.task_id = tid.value
        self._streams.append(sink)
        return sink

    def set_vip(self, user):
        check(lib.mq_dispatcher_set_vip(self._h, None if user is None else user.encode()))

    def set_boost(self, user):
        check(lib.mq_dispatcher_set_boost(self._h, None if user is None else user.encode()))

    def add_vip(self, user):      # extension: several VIPs (BASELINE config 3)
        check(lib.mq_dispatcher_add_vip(self._h, user.encode()))

    def add_boost(self, user):
        check(lib.mq_dispatcher_add_boost(self._h, user.encode()))

    def control(self, action: str, user: Optional[str] = None, ip: Optional[str] = None):
        """The dashboard's control keys as one atomic call (tui.rs:126-237): see mq_dispatcher_control."""
        check(lib.mq_dispatcher_control(self._h, action.encode(), user.encode() if user is not None else None,
                                        ip.encode() if ip is not None else None))

    def block_user(self, user, blocked=True):
        check(lib.mq_dispatcher_block_user(self._h, user.encode(), 1 if blocked else 0))

    def block_ip(self, ip, blocked=True):
        check(lib.mq_dispatcher_block_ip(self._h, ip.encode(), 1 if blocked else 0))

    def set_online(self, backend, online):
        check(lib.mq_dispatcher_set_online(self._h, backend, 1 if online else 0))

    def set_timeout(self, seconds: float):
        """`--timeout` of the reference: whole-request limit for requests without their own."""
        check(lib.mq_dispatcher_set_timeout(self._h, int(seconds * 1000)))

    def attach_encoder(self, backend: int, enc: "Encoder"):
        check(lib.mq_dispatcher_attach_encoder(self._h, backend, enc.handle))

    def set_block_file(self, path: str):
        check(lib.mq_dispatcher_set_block_file(self._h, path.encode()))

    def start_health(self, period_ms: int = 10000):
        check(lib.mq_dispatcher_start_health(self._h, period_ms))

    def client_gone(self, task_id):
        return lib.mq_dispatcher_client_gone(self._h, task_id)

    def wait_parked(self, timeout_ms=5000):
        check(lib.mq_dispatcher_wait_parked(self._h, timeout_ms))

    def mock_complete(self, backend, rc=0) -> bool:
        return check(lib.mq_dispatcher_mock_complete(self._h, backend, rc)) == 1

    def mock_set_healthy(self, backend, healthy=True):
        check(lib.mq_dispatcher_mock_set_healthy(self._h, backend, 1 if healthy else 0))

    def mock_fail_next(self, backend, n=1):
        check(lib.mq_dispatcher_mock_fail_next(self._h, backend, n))

    def drain(self, timeout_ms=600000):
        check(lib.mq_dispatcher_drain(self._h, timeout_ms))

    def serve_http(self, port: int = 0, bind: str = "127.0.0.1", allow_all_routes: bool = False) -> int:
        """Start the HTTP/1.1 ingress (route table of main.rs:89-121) on this dispatcher; returns the port."""
        h = C.c_void_p()
        check(lib.mq_http_server_start(self._h, bind.encode(), port, 1 if allow_all_routes else 0, C.byref(h)))
        self._http = h
        return lib.mq_http_server_port(h)

    def stop_http(self):
        if getattr(self, "_http", None):
            lib.mq_http_server_stop(self._http)
            self._http = None

    def log(self):
        n = C.c_int32()
        check(lib.mq_dispatcher_log(self._h, None, 0, C.byref(n)))
        arr = (_lib.Dispatch * max(1, n.value))()
        check(lib.mq_dispatcher_log(self._h, arr, n.value, C.byref(n)))
        return [(arr[i].user.decode(), arr[i].user_seq, arr[i].backend) for i in range(n.value)]

    def snapshot(self) -> dict:
        """Everything the reference dashboard shows, captured under one lock (tui.rs:55-95)."""
        import json
        need = lib.mq_dispatcher_snapshot_json(self._h, None, 0)
        while True:
            check(need)
            buf = C.create_string_buffer(int(need) + 256)
            got = lib.mq_dispatcher_snapshot_json(self._h, buf, len(buf))
            if 0 < got <= len(buf):
                return json.loads(buf.value.decode("utf-8", "replace"))
            need = got

    def user_stats(self, user: str) -> dict:
        st = _lib.UserStats()
        check(lib.mq_sched_user_stats(lib.mq_dispatcher_sched(self._h), user.encode(), C.byref(st)))
        return {k: getattr(st, k) for k, _ in st._fields_}

    def backend_stats(self, b: int) -> dict:
        st = _lib.BackendStats()
        check(lib.mq_sched_backend_stats(lib.mq_dispatcher_sched(self._h), b, C.byref(st)))
        return {"active_requests": st.active_requests, "processed_count": st.processed_count,
                "is_online": bool(st.is_online)}
