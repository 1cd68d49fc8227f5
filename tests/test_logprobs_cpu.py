"""CPU: token log-probabilities in the request parser and the response framers (csrc/framing.cpp), through the
host-only test ABI (mq_debug_parse_body, mq_debug_frame_logprobs).  The numbers themselves come from the sampler
kernel (tests/test_logprobs_gpu.py); here: which bodies turn logprobs on, and the reply shapes of every route."""
import ctypes as C
import json
import re
import struct

import numpy as np
import pytest

import ollamamq_b200 as mq

EP_GEN, EP_CHAT, EP_V1_CHAT, EP_V1_COMPL, EP_RAW = 0, 1, 2, 3, 4
ROUTES = [EP_GEN, EP_CHAT, EP_V1_CHAT, EP_V1_COMPL]


def _call(fn, *args):
    need = fn(*args, None, 0)
    buf = C.create_string_buffer(int(need) + 16)
    assert fn(*args, buf, len(buf)) == need
    return buf.raw[:int(need) - 1]


def parse(endpoint, body):
    if not isinstance(body, bytes):
        body = json.dumps(body).encode()
    return json.loads(_call(mq.lib.mq_debug_parse_body, endpoint, body, len(body), 256))


def on_n(p):
    """(logprobs on, N) the way the worker reads a parsed body that carries no struct fields."""
    on = p["has_logprobs"] and p["logprobs"]
    return on, (p["top_logprobs"] if p["has_top_logprobs"] else 0)


# ------------------------------------------------------------------------------------------------ parser
@pytest.mark.parametrize("ep", [EP_GEN, EP_CHAT, EP_V1_CHAT])
def test_boolean_spelling(ep):
    assert on_n(parse(ep, {"prompt": "x", "logprobs": True, "top_logprobs": 3})) == (True, 3)
    assert on_n(parse(ep, {"prompt": "x", "logprobs": True})) == (True, 0)
    p = parse(ep, {"prompt": "x", "logprobs": False, "top_logprobs": 3})
    assert p["ok"] and p["has_logprobs"] and on_n(p) == (False, 3)
    assert on_n(parse(ep, {"logprobs": True, "top_logprobs": 25})) == (True, 20)        # clamped to 0..20
    assert on_n(parse(ep, {"logprobs": True, "top_logprobs": -3})) == (True, 0)
    assert on_n(parse(ep, {"logprobs": True, "top_logprobs": 2.7})) == (True, 2)
    # wrong types are skipped like any other field: the body still parses
    for bad in ({"logprobs": 5}, {"logprobs": "yes"}, {"logprobs": None}, {"logprobs": [True]}):
        p = parse(ep, dict(bad, prompt="x"))
        assert p["ok"] and not p["has_logprobs"], bad
    p = parse(ep, {"logprobs": True, "top_logprobs": "4"})
    assert p["ok"] and not p["has_top_logprobs"] and on_n(p) == (True, 0)
    p = parse(ep, {"logprobs": True, "top_logprobs": None})
    assert p["ok"] and on_n(p) == (True, 0)


def test_legacy_completions_spelling():
    assert on_n(parse(EP_V1_COMPL, {"prompt": "x", "logprobs": 5})) == (True, 5)
    assert on_n(parse(EP_V1_COMPL, {"prompt": "x", "logprobs": 0})) == (True, 0)
    assert on_n(parse(EP_V1_COMPL, {"logprobs": 25})) == (True, 20)
    assert on_n(parse(EP_V1_COMPL, {"logprobs": -3})) == (True, 0)
    p = parse(EP_V1_COMPL, {"prompt": "x", "logprobs": None})
    assert p["ok"] and p["has_logprobs"] and on_n(p)[0] is False
    for bad in ({"logprobs": True}, {"logprobs": "3"}, {"logprobs": {"n": 3}}):   # boolean is not this route's spelling
        p = parse(EP_V1_COMPL, dict(bad, prompt="x"))
        assert p["ok"] and not p["has_logprobs"], bad
    # the legacy integer is the number of alternatives, whatever order the keys come in
    assert on_n(parse(EP_V1_COMPL, b'{"logprobs":2,"top_logprobs":7}')) == (True, 2)
    assert on_n(parse(EP_V1_COMPL, b'{"top_logprobs":7,"logprobs":2}')) == (True, 2)


@pytest.mark.parametrize("ep", ROUTES)
def test_bodies_without_logprobs_parse_to_off(ep):
    for body in ({"prompt": "hi", "stream": False}, {"messages": [{"role": "user", "content": "hi"}], "max_tokens": 4},
                 {"prompt": [1, 2, 3], "options": {"temperature": 0.5, "logprobs": True, "top_logprobs": 5}}):
        p = parse(ep, body)
        assert p["ok"] and not p["has_logprobs"] and not p["logprobs"] and not p["has_top_logprobs"], body
        assert on_n(p) == (False, 0)
    # keys inside "options" are not the top-level switch
    p = parse(ep, {"options": {"logprobs": 3, "top_logprobs": 5}})
    assert p["ok"] and on_n(p) == (False, 0) and not p["has_top_logprobs"]
    # a value the parser skips as it skipped every unknown key before (bare words included) still parses
    assert parse(ep, b'{"logprobs": tru, "top_logprobs": fals}')["ok"]
    assert on_n(parse(ep, b'{"logprobs" : true , "top_logprobs" : 1e0}')) == (ep != EP_V1_COMPL, 1)


# ------------------------------------------------------------------------------------------------ framing
def _records(n, N, seed):
    """n tokens: ids and records (float logprob, N x (int32 id, float logprob)) as the kernel writes them."""
    rng = np.random.default_rng(seed)
    ids = rng.integers(0, 128256, n).astype(np.int32)
    lp = np.concatenate([[-0.0, -1e-7, -80.123456, -3.3e-6], rng.standard_normal(4 * n * (N + 1)) * 5])
    lp = -np.abs(lp).astype(np.float32)
    lp[lp == 0] = 0.0          # l - lse is +0 when l is the whole mass (x - x rounds to +0); JSON has no -0 here
    recs, k = [], 0
    for i in range(n):
        top_ids = rng.choice(128256, N, replace=False).astype(np.int32)
        r = [lp[k]]
        k += 1
        tops = np.sort(lp[k:k + N])[::-1]
        k += N
        for j in range(N):
            r += [np.array(top_ids[j], np.int32).view(np.float32), tops[j]]
        recs.append(r)
    flat = np.array(recs, dtype=np.float32).reshape(-1) if N >= 0 else np.zeros(1, np.float32)
    return ids, flat


def frame(ep, stream, ids, recs, N, model=b"m", n_prompt=7):
    ids = np.ascontiguousarray(ids, np.int32)
    recs = np.ascontiguousarray(recs, np.float32)
    return _call(mq.lib.mq_debug_frame_logprobs, ep, stream, model, ids.ctypes.data_as(C.c_void_p),
                 recs.ctypes.data_as(C.c_void_p), len(ids), N, n_prompt)


def _split(ep, stream, raw):
    """The JSON objects of a reply: NDJSON lines, SSE data lines (without [DONE]), or one object."""
    txt = raw.decode()
    if not stream:
        return [json.loads(txt)]
    if ep in (EP_GEN, EP_CHAT):
        assert txt.endswith("\n")
        return [json.loads(line) for line in txt.split("\n") if line]
    events = [e for e in txt.split("\n\n") if e]
    assert all(e.startswith("data: ") for e in events) and events[-1] == "data: [DONE]"
    return [json.loads(e[6:]) for e in events[:-1]]


def _expected(ids, recs, N):
    out = []
    for i, t in enumerate(ids):
        r = recs[i * (1 + 2 * N):(i + 1) * (1 + 2 * N)]
        out.append((int(t), r[0], [(int(r[1 + 2 * j].view(np.int32)), r[2 + 2 * j]) for j in range(N)]))
    return out


def _exact(x, f32):
    assert np.float32(x).tobytes() == np.float32(f32).tobytes(), (x, f32)   # bit-exact float32 round trip


def _check_entry(e, tok, lp, tops):
    assert e["token"] == " t%d" % tok and bytes(e["bytes"]).decode() == e["token"]
    _exact(e["logprob"], lp)
    assert len(e["top_logprobs"]) == len(tops)
    for a, (tid, tlp) in zip(e["top_logprobs"], tops):
        assert set(a) == {"token", "logprob", "bytes"}
        assert a["token"] == " t%d" % tid and bytes(a["bytes"]).decode() == a["token"]
        _exact(a["logprob"], tlp)


def _entries(ep, obj):
    c = obj.get("choices", [{}])[0]
    if ep in (EP_GEN, EP_CHAT):
        return obj.get("logprobs")
    return c.get("logprobs")


@pytest.mark.parametrize("N", [0, 3, 20])
@pytest.mark.parametrize("stream", [1, 0])
@pytest.mark.parametrize("ep", ROUTES)
def test_reply_shapes(ep, stream, N):
    n = 6
    ids, recs = _records(n, N, seed=ep * 100 + N + stream)
    exp = _expected(ids, recs, N)
    objs = _split(ep, stream, frame(ep, stream, ids, recs, N))
    plain = _split(ep, stream, frame(ep, stream, ids, recs, -1))
    assert len(objs) == len(plain) == (n + 1 if stream else 1)
    # removing the logprobs member gives exactly the reply without logprobs
    for a, b in zip(objs, plain):
        a = json.loads(json.dumps(a))
        if ep in (EP_GEN, EP_CHAT):
            a.pop("logprobs", None)
            a.pop("created_at"); b.pop("created_at")
        else:
            a["choices"][0].pop("logprobs", None)
            a.pop("created", None); b.pop("created", None)
        assert a == b
    if stream:
        per_token = [_entries(ep, o) for o in objs[:-1]]
        assert _entries(ep, objs[-1]) is None              # the final frame carries none
    else:
        per_token = None
    if ep == EP_V1_COMPL:
        blocks = per_token if stream else [_entries(ep, objs[0])]
        toks, lps, tops, offs = [], [], [], []
        for b in blocks:
            assert set(b) == {"tokens", "token_logprobs", "top_logprobs", "text_offset"}
            toks += b["tokens"]; lps += b["token_logprobs"]; tops += b["top_logprobs"]; offs += b["text_offset"]
        texts = [" t%d" % t for t, _, _ in exp]
        assert toks == texts
        assert offs == list(np.cumsum([0] + [len(t) for t in texts])[:-1])   # from 0 at the first generated character
        for (t, lp, tp), got_lp, got_top in zip(exp, lps, tops):
            _exact(got_lp, lp)
            assert list(got_top) == [" t%d" % i for i, _ in tp]               # ordered as the record
            for (i, v) in tp:
                _exact(got_top[" t%d" % i], v)
        return
    if stream:
        assert all(len(e) == (1 if ep != EP_V1_CHAT else 1) for e in per_token)
        entries = [(e["content"] if ep == EP_V1_CHAT else e) for e in per_token]
        assert all(len(e) == 1 for e in entries)
        entries = [e[0] for e in entries]
    else:
        e = _entries(ep, objs[0])
        entries = e["content"] if ep == EP_V1_CHAT else e
    assert len(entries) == n
    for e, (t, lp, tp) in zip(entries, exp):
        assert set(e) == {"token", "logprob", "bytes", "top_logprobs"}
        _check_entry(e, t, lp, tp)


_TS = [(re.compile(rb'"created_at":"[^"]*"'), b'"created_at":"T"'), (re.compile(rb'"created":\d+'), b'"created":0')]


def _norm(b):
    for rx, rep in _TS:
        b = rx.sub(rep, b)
    return b


@pytest.mark.parametrize("stream", [1, 0])
@pytest.mark.parametrize("ep", ROUTES)
def test_off_is_byte_identical_to_the_existing_frames(ep, stream):
    ids = np.array([5, 42, 128255, 0], np.int32)
    got = _norm(frame(ep, stream, ids, np.zeros(1, np.float32), -1, model=b"mdl", n_prompt=3))
    text = "".join(" t%d" % t for t in ids).encode()
    final = _norm(_call(mq.lib.mq_debug_frame_final, ep, stream, b"mdl", b"" if stream else text, 3, len(ids), 0))
    if not stream:
        assert got == final
        return
    per = b""
    for t in ids:
        txt = b" t%d" % t
        per += {EP_GEN: b'{"model":"mdl","created_at":"T","response":"' + txt + b'","done":false}\n',
                EP_CHAT: b'{"model":"mdl","created_at":"T","message":{"role":"assistant","content":"' + txt +
                         b'"},"done":false}\n',
                EP_V1_CHAT: b'data: {"id":"chatcmpl-mq","object":"chat.completion.chunk","created":0,"model":"mdl",'
                            b'"choices":[{"index":0,"delta":{"content":"' + txt + b'"},"finish_reason":null}]}\n\n',
                EP_V1_COMPL: b'data: {"id":"cmpl-mq","object":"text_completion","created":0,"model":"mdl",'
                             b'"choices":[{"text":"' + txt + b'","index":0,"finish_reason":null}]}\n\n'}[ep]
    assert got == per + final


@pytest.mark.parametrize("stream", [1, 0])
def test_raw_token_records(stream):
    N = 4
    ids, recs = _records(5, N, seed=3)
    b = frame(EP_RAW, stream, ids, recs, N)
    assert len(b) == 5 * (8 + 8 * N)
    for i, (t, lp, tops) in enumerate(_expected(ids, recs, N)):
        rec = b[i * (8 + 8 * N):(i + 1) * (8 + 8 * N)]
        assert struct.unpack("<i", rec[:4])[0] == t
        assert rec[4:8] == np.float32(lp).tobytes()
        for j, (tid, tlp) in enumerate(tops):
            assert struct.unpack("<i", rec[8 + 8 * j:12 + 8 * j])[0] == tid and rec[12 + 8 * j:16 + 8 * j] == np.float32(tlp).tobytes()
    # off: 4-byte ids, as before
    assert frame(EP_RAW, stream, ids, recs, -1) == ids.astype("<i4").tobytes()
    # the Python decoder of the same bytes
    s = mq.Stream()
    s.top_logprobs = N
    s.chunks = [b]
    assert s.tokens() == ids.tolist()
    got = s.logprobs()
    for (lp, tops), (_, elp, etops) in zip(got, _expected(ids, recs, N)):
        assert np.float32(lp) == elp and [(i, np.float32(v)) for i, v in tops] == etops


def test_request_struct_keeps_its_layout():
    r = mq._lib.Request()
    assert C.sizeof(r) == 88 and mq._lib.Request.logprobs.offset == 84 and mq._lib.Request.top_logprobs.offset == 86
    req, _ = mq.worker.make_request(logprobs=True, top_logprobs=30)
    assert req.logprobs == 1 and req.top_logprobs == 20
    req, _ = mq.worker.make_request()
    assert req.logprobs == 0 and req.top_logprobs == 0
