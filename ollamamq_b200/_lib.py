"""ctypes binding of libollamamq_b200.so (signatures mirror include/ollamamq_b200.h)."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libollamamq_b200.so")

MQ_USER_MAX = 256


class MQError(RuntimeError):
    def __init__(self, rc: int, msg: str):
        super().__init__("mq error %d: %s" % (rc, msg))
        self.rc = rc


if not os.path.exists(LIB_PATH):
    raise ImportError(
        "libollamamq_b200.so is not built (expected %s). Run `python build_native.py` "
        "(nvcc, sm_100a). There is no CPU fallback." % LIB_PATH)

lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)


class Dispatch(C.Structure):
    _fields_ = [("task_id", C.c_uint64), ("user_seq", C.c_uint64), ("backend", C.c_int32),
                ("reserved", C.c_int32), ("user", C.c_char * MQ_USER_MAX)]


class UserStats(C.Structure):
    _fields_ = [("queued", C.c_uint64), ("processing", C.c_uint64), ("processed", C.c_uint64),
                ("dropped", C.c_uint64)]


class BackendStats(C.Structure):
    _fields_ = [("active_requests", C.c_uint64), ("processed_count", C.c_uint64), ("is_online", C.c_int32),
                ("reserved", C.c_int32)]


class ModelCfg(C.Structure):
    _fields_ = [("vocab", C.c_int32), ("hidden", C.c_int32), ("ffn", C.c_int32), ("n_layers", C.c_int32),
                ("n_q_heads", C.c_int32), ("n_kv_heads", C.c_int32), ("head_dim", C.c_int32),
                ("qkv_bias", C.c_int32), ("rope_theta", C.c_float), ("rms_eps", C.c_float),
                ("max_batch", C.c_int32), ("max_seq", C.c_int32), ("max_prefill_tokens", C.c_int32),
                ("kv_pages", C.c_int32), ("use_graphs", C.c_int32), ("use_pdl", C.c_int32),
                ("eos_token_id", C.c_int32), ("model_name", C.c_char * 64)]


class EncoderCfg(C.Structure):
    _fields_ = [("vocab", C.c_int32), ("hidden", C.c_int32), ("ffn", C.c_int32), ("n_layers", C.c_int32),
                ("n_heads", C.c_int32), ("head_dim", C.c_int32), ("max_positions", C.c_int32),
                ("type_vocab", C.c_int32), ("ln_eps", C.c_float), ("max_seq", C.c_int32),
                ("max_tokens_per_pass", C.c_int32), ("use_pdl", C.c_int32), ("model_name", C.c_char * 64)]


class EncoderStats(C.Structure):
    _fields_ = [("passes", C.c_uint64), ("sequences", C.c_uint64), ("tokens", C.c_uint64),
                ("kernel_launches", C.c_uint64), ("gpu_us", C.c_uint64)]


class Request(C.Structure):
    _fields_ = [("endpoint", C.c_int32), ("stream", C.c_int32), ("body", C.c_void_p), ("body_len", C.c_size_t),
                ("prompt_tokens", C.c_void_p), ("n_prompt_tokens", C.c_int32), ("max_new_tokens", C.c_int32),
                ("ignore_eos", C.c_int32), ("timeout_ms", C.c_uint32), ("path", C.c_char_p),
                ("temperature", C.c_float), ("top_k", C.c_int32), ("top_p", C.c_float), ("seed", C.c_uint64),
                ("body_kind", C.c_int32), ("logprobs", C.c_int16), ("top_logprobs", C.c_int16)]


MQ_TOP_LOGPROBS_MAX = 20


ON_STATUS = C.CFUNCTYPE(None, C.c_void_p, C.c_int32, C.c_char_p)
ON_CHUNK = C.CFUNCTYPE(C.c_int32, C.c_void_p, C.POINTER(C.c_uint8), C.c_size_t)
ON_DONE = C.CFUNCTYPE(None, C.c_void_p, C.c_int32, C.c_char_p)


class Callbacks(C.Structure):
    _fields_ = [("on_status", ON_STATUS), ("on_chunk", ON_CHUNK), ("on_done", ON_DONE)]


class ReqStats(C.Structure):
    _fields_ = [("ttft_us", C.c_uint64), ("total_us", C.c_uint64), ("n_prompt", C.c_int32),
                ("n_generated", C.c_int32)]


class WorkerOccupancy(C.Structure):
    _fields_ = [("total_pages", C.c_uint64), ("free_pages", C.c_uint64), ("active_slots", C.c_uint64),
                ("waiting", C.c_uint64), ("in_flight_gpu_passes", C.c_uint64)]


class WorkerStats(C.Structure):
    _fields_ = [("kernel_launches", C.c_uint64), ("graph_launches", C.c_uint64), ("decode_steps", C.c_uint64),
                ("prefill_passes", C.c_uint64), ("prefill_tokens", C.c_uint64), ("decode_tokens", C.c_uint64),
                ("decode_ms", C.c_double), ("prefill_ms", C.c_double), ("decode_bytes", C.c_double)]


def _sig(name, restype, argtypes):
    fn = getattr(lib, name)
    fn.restype = restype
    fn.argtypes = argtypes
    return fn


P = C.c_void_p
_sig("mq_last_error", C.c_char_p, [])
_sig("mq_version", C.c_char_p, [])
# scheduler
_sig("mq_sched_new", P, [C.c_int32, C.c_int32])
_sig("mq_sched_free", None, [P])
_sig("mq_sched_enqueue", C.c_int, [P, C.c_char_p, C.POINTER(C.c_uint64)])
_sig("mq_sched_next", C.c_int, [P, C.POINTER(Dispatch)])
_sig("mq_sched_complete", C.c_int, [P, C.c_int32, C.c_char_p, C.c_int32])
_sig("mq_sched_processing", C.c_int, [P, C.c_char_p, C.c_int32])
_sig("mq_sched_set_vip", C.c_int, [P, C.c_char_p])
_sig("mq_sched_set_boost", C.c_int, [P, C.c_char_p])
_sig("mq_sched_add_vip", C.c_int, [P, C.c_char_p])
_sig("mq_sched_add_boost", C.c_int, [P, C.c_char_p])
_sig("mq_sched_set_online", C.c_int, [P, C.c_int32, C.c_int32])
_sig("mq_sched_set_capacity", C.c_int, [P, C.c_int32])
_sig("mq_sched_set_boost_mod", C.c_int, [P, C.c_int32])
_sig("mq_sched_user_stats", C.c_int, [P, C.c_char_p, C.POINTER(UserStats)])
_sig("mq_sched_backend_stats", C.c_int, [P, C.c_int32, C.POINTER(BackendStats)])
_sig("mq_sched_user_count", C.c_int32, [P])
_sig("mq_sched_user_name", C.c_int, [P, C.c_int32, C.c_char_p, C.c_size_t])
_sig("mq_sched_counter", C.c_uint64, [P])
# worker
_sig("mq_worker_count", C.c_int, [])
_sig("mq_worker_open", C.c_int, [C.c_int32, C.POINTER(ModelCfg), C.POINTER(P)])
_sig("mq_worker_close", None, [P])
_sig("mq_worker_load_tensor", C.c_int, [P, C.c_char_p, P, C.c_size_t])
_sig("mq_worker_read_tensor", C.c_int, [P, C.c_char_p, P, C.c_size_t])
_sig("mq_worker_init_random", C.c_int, [P, C.c_uint64, C.c_float])
_sig("mq_worker_capacity", C.c_int, [P])
_sig("mq_worker_healthy", C.c_int, [P])
_sig("mq_submit", C.c_int, [P, C.POINTER(Request), C.POINTER(Callbacks), P, C.POINTER(P)])
_sig("mq_cancel", None, [P])
_sig("mq_req_release", None, [P])
_sig("mq_req_get_stats", C.c_int, [P, C.POINTER(ReqStats)])
_sig("mq_worker_get_stats", C.c_int, [P, C.POINTER(WorkerStats)])
_sig("mq_worker_reset_stats", C.c_int, [P])
_sig("mq_worker_set_timing", C.c_int, [P, C.c_int32])
_sig("mq_debug_forward", C.c_int, [P, P, C.c_int32, C.c_int32, P])
# dispatcher
_sig("mq_dispatcher_new", C.c_int, [C.POINTER(P), C.c_int32, C.c_int32, C.POINTER(P)])
_sig("mq_dispatcher_free", None, [P])
_sig("mq_dispatcher_submit", C.c_int, [P, C.c_char_p, C.c_char_p, C.POINTER(Request), C.POINTER(Callbacks), P,
                                        C.POINTER(C.c_uint64)])
_sig("mq_dispatcher_sched", P, [P])
_sig("mq_dispatcher_set_vip", C.c_int, [P, C.c_char_p])
_sig("mq_dispatcher_set_boost", C.c_int, [P, C.c_char_p])
_sig("mq_dispatcher_block_user", C.c_int, [P, C.c_char_p, C.c_int32])
_sig("mq_dispatcher_block_ip", C.c_int, [P, C.c_char_p, C.c_int32])
_sig("mq_dispatcher_log", C.c_int, [P, C.POINTER(Dispatch), C.c_int32, C.POINTER(C.c_int32)])
_sig("mq_dispatcher_drain", C.c_int, [P, C.c_uint32])
_sig("mq_dispatcher_set_online", C.c_int, [P, C.c_int32, C.c_int32])
_sig("mq_dispatcher_set_block_file", C.c_int, [P, C.c_char_p])
_sig("mq_dispatcher_start_health", C.c_int, [P, C.c_uint32])
_sig("mq_dispatcher_client_gone", C.c_int, [P, C.c_uint64])
_sig("mq_dispatcher_wait_parked", C.c_int, [P, C.c_uint32])
_sig("mq_dispatcher_new_mock", C.c_int, [C.c_int32, C.c_int32, C.POINTER(P)])
_sig("mq_dispatcher_mock_complete", C.c_int, [P, C.c_int32, C.c_int32])
_sig("mq_dispatcher_mock_fail_next", C.c_int, [P, C.c_int32, C.c_int32])
_sig("mq_dispatcher_mock_set_healthy", C.c_int, [P, C.c_int32, C.c_int32])
_sig("mq_debug_worker_set_probe_fail", C.c_int, [P, C.c_int32])
_sig("mq_debug_worker_inject_fault", C.c_int, [P, C.c_char_p])
_sig("mq_http_server_start", C.c_int, [P, C.c_char_p, C.c_int32, C.c_int32, C.POINTER(P)])
_sig("mq_http_server_port", C.c_int, [P])
_sig("mq_http_server_stop", None, [P])
# kernel-level test ABI
_sig("mq_debug_gemm", C.c_int, [P, C.c_int, C.c_int, C.c_int, P, C.c_int, C.c_int, C.c_int, P, C.c_int, C.c_int,
                                 C.c_longlong, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float)])
_sig("mq_debug_embed", C.c_int, [P, P, P, C.c_int, C.c_int])
_sig("mq_debug_embed_chain", C.c_int, [P, P, P, C.c_int, C.c_int, P, P, P])
_sig("mq_debug_cluster_info", C.c_int, [P])
_sig("mq_debug_gemm_bias", C.c_int, [P, C.c_int, C.c_int, P, C.c_int, C.c_int, C.c_int, P, P, C.c_int])
_sig("mq_debug_gemm_rowln", C.c_int, [P, C.c_int, C.c_int, P, C.c_int, C.c_int, P, P, P, P, C.c_float, P])
_sig("mq_debug_enc_attn", C.c_int, [P, C.c_int, C.c_int, C.c_int, P, P, C.c_int, P])
_sig("mq_debug_gemm_fold", C.c_int, [P, C.c_int, C.c_int, C.c_int, P, C.c_int, C.c_int, C.c_int, P, C.c_int, C.c_int, C.c_int,
                                      C.c_int, P, C.c_int, C.c_int, C.c_float, C.c_float, C.c_int, C.POINTER(C.c_float)])
_sig("mq_debug_gemm_resid_prefill", C.c_int, [P, C.c_int, C.c_int, P, C.c_int, C.c_int, P, P, P, P, C.c_int, P, C.c_int, C.c_int,
                                               C.c_float, C.c_float, C.c_int, C.POINTER(C.c_float)])
_sig("mq_debug_gemm_dk_resid", C.c_int, [P, C.c_int, C.c_int, P, C.c_int, C.c_int, C.c_int, P, P, P, P, C.c_int, C.c_int,
                                          C.POINTER(C.c_float)])
_sig("mq_debug_add_rmsnorm", C.c_int, [P, P, C.c_int, C.c_int, C.c_longlong, P, P, P, C.c_int, C.c_int, C.c_float])
_sig("mq_debug_rope_kv", C.c_int, [P, C.c_int, C.c_int, C.c_longlong, P, P, P, P, C.c_int, P, P, P, P, C.c_int,
                                    C.c_int, C.c_int, C.c_int])
_sig("mq_debug_attn_prefill", C.c_int, [P, P, P, P, C.c_int, P, C.c_int, P, C.c_int, C.c_int, C.c_int, C.c_float,
                                         C.c_int])
_sig("mq_debug_attn_prefill_tc", C.c_int, [P, C.c_int, P, P, C.c_int, P, C.c_int, P, C.c_int, P, C.c_int, C.c_int, C.c_float])
_sig("mq_debug_attn_decode", C.c_int, [P, P, P, P, C.c_int, P, P, P, P, P, C.c_int, C.c_int, C.c_int, C.c_int,
                                        C.c_float, C.c_int])
_sig("mq_worker_get_occupancy", C.c_int, [P, P])
_sig("mq_debug_sched_bench", C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, P, P])
_sig("mq_dispatcher_snapshot_json", C.c_longlong, [P, P, C.c_size_t])
_sig("mq_dispatcher_control", C.c_int, [P, C.c_char_p, C.c_char_p, C.c_char_p])
_sig("mq_dispatcher_attach_encoder", C.c_int, [P, C.c_int32, P])
_sig("mq_dispatcher_add_vip", C.c_int, [P, C.c_char_p])
_sig("mq_dispatcher_add_boost", C.c_int, [P, C.c_char_p])
_sig("mq_dispatcher_set_timeout", C.c_int, [P, C.c_uint32])
_sig("mq_encoder_open", C.c_int, [C.c_int32, P, P])
_sig("mq_encoder_close", None, [P])
_sig("mq_encoder_load_tensor", C.c_int, [P, C.c_char_p, P, C.c_size_t])
_sig("mq_encoder_read_tensor", C.c_int, [P, C.c_char_p, P, C.c_size_t])
_sig("mq_encoder_init_random", C.c_int, [P, C.c_uint64, C.c_float])
_sig("mq_encoder_healthy", C.c_int, [P])
_sig("mq_encoder_get_stats", C.c_int, [P, P])
_sig("mq_encoder_embed", C.c_int, [P, P, P, C.c_int32, P])
_sig("mq_encoder_submit", C.c_int, [P, P, P, P, P])
_sig("mq_debug_trace_read", C.c_int, [P, P, C.c_int])
_sig("mq_debug_parse_body", C.c_longlong, [C.c_int32, P, C.c_size_t, C.c_int32, P, C.c_size_t])
_sig("mq_debug_parse_embed", C.c_longlong, [P, C.c_size_t, C.c_int32, C.c_int32, P, C.c_size_t])
_sig("mq_debug_frame_embeddings", C.c_longlong, [C.c_char_p, C.c_char_p, P, C.c_int32, C.c_int32, C.c_int32, P, C.c_size_t])
_sig("mq_debug_frame_final", C.c_longlong, [C.c_int32, C.c_int32, C.c_char_p, C.c_char_p, C.c_int32, C.c_int32, C.c_int32, P,
                                              C.c_size_t])
_sig("mq_debug_sample", C.c_int, [P, C.c_int, C.c_int, C.c_int, P, P, P, P, P, P])
_sig("mq_debug_sample_logprobs", C.c_int, [P, C.c_int, C.c_int, C.c_int, P, P, P, P, P, P, P, P])
_sig("mq_debug_frame_logprobs", C.c_longlong, [C.c_int32, C.c_int32, C.c_char_p, P, P, C.c_int32, C.c_int32, C.c_int32, P,
                                                 C.c_size_t])
_sig("mq_debug_argmax", C.c_int, [P, C.c_int, C.c_int, C.c_int, P, P, P, P, P])
_sig("mq_debug_init_normal", C.c_int, [P, C.c_ulonglong, C.c_ulonglong, C.c_float])


def last_error() -> str:
    return lib.mq_last_error().decode("utf-8", "replace")


def check(rc: int) -> int:
    if rc < 0:
        raise MQError(rc, last_error())
    return rc
