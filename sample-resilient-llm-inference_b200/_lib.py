"""ctypes binding of librr_b200.so (include/rr_b200.h).

The product path has no CPU fallback: if the shared library is missing this module raises at
import time (build it with `python __graft_entry__.py` or `python -m rr_b200_build`).
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_PKG = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ.get("RR_B200_LIB", _PKG / "librr_b200.so"))


class LibraryMissing(ImportError):
    pass


def _load() -> C.CDLL:
    if not LIB_PATH.exists():
        raise LibraryMissing(
            f"{LIB_PATH} not found: the CUDA extension is required (no CPU fallback). "
            f"Build it with `python -c 'import __graft_entry__ as g; g.build()'`.")
    return C.CDLL(str(LIB_PATH), mode=C.RTLD_GLOBAL)


lib = _load()

c_i32p = C.POINTER(C.c_int32)
c_f32p = C.POINTER(C.c_float)
vp = C.c_void_p

# ---------------------------------------------------------------- structs (mirror rr_b200.h)


class DeploymentDesc(C.Structure):
    _fields_ = [("group", C.c_int32), ("rpm", C.c_int32), ("tpm", C.c_int32),
                ("weight", C.c_int32), ("replica", C.c_int32), ("reserved", C.c_int32)]


class RouterSettings(C.Structure):
    _fields_ = [("strategy", C.c_int32), ("enable_pre_call_checks", C.c_int32),
                ("allowed_fails", C.c_int32), ("cooldown_ms", C.c_int32),
                ("weight_by", C.c_int32), ("reserved", C.c_int32 * 3)]


class Event(C.Structure):
    _fields_ = [("type", C.c_int32), ("target", C.c_int32), ("tokens", C.c_int32),
                ("chain_start", C.c_int32), ("now_ms", C.c_int64)]


class Decision(C.Structure):
    _fields_ = [("status", C.c_int32), ("deployment", C.c_int32), ("served_group", C.c_int32),
                ("chain_pos", C.c_int32)]


class DeploymentState(C.Structure):
    _fields_ = [("window", C.c_int64), ("req_count", C.c_int32), ("tok_count", C.c_int32),
                ("fail_window", C.c_int64), ("fail_count", C.c_int32), ("inflight", C.c_int32),
                ("cooldown_until_ms", C.c_int64), ("total_admitted", C.c_int64)]


class ModelDesc(C.Structure):
    _fields_ = [("vocab", C.c_int32), ("hidden", C.c_int32), ("inter", C.c_int32),
                ("n_layers", C.c_int32), ("n_heads", C.c_int32), ("n_kv_heads", C.c_int32),
                ("head_dim", C.c_int32), ("rope_theta", C.c_float), ("rms_eps", C.c_float)]


class ModelWeights(C.Structure):
    _fields_ = [("embed", vp), ("lm_head", vp), ("final_norm", vp),
                ("wqkv", C.POINTER(vp)), ("wo", C.POINTER(vp)), ("wgu", C.POINTER(vp)),
                ("wdown", C.POINTER(vp)), ("norm_attn", C.POINTER(vp)),
                ("norm_mlp", C.POINTER(vp)), ("flags", C.c_int32), ("reserved", C.c_int32)]


class EngineOpts(C.Structure):
    _fields_ = [("device", C.c_int32), ("max_batch", C.c_int32), ("ctx_max", C.c_int32),
                ("max_prefill_tokens", C.c_int32), ("use_cuda_graph", C.c_int32),
                ("fail_seed", C.c_int32), ("fail_prob", C.c_float), ("reserved", C.c_int32 * 4)]


class Completion(C.Structure):
    _fields_ = [("ticket", C.c_uint64), ("status", C.c_int32), ("n_prompt", C.c_int32),
                ("n_generated", C.c_int32), ("reserved", C.c_int32),
                ("t_submit_s", C.c_double), ("t_first_token_s", C.c_double),
                ("t_done_s", C.c_double)]


class EngineStats(C.Structure):
    _fields_ = [("kernel_launches", C.c_uint64), ("decode_steps", C.c_uint64),
                ("prefill_chunks", C.c_uint64), ("prefill_tokens", C.c_uint64),
                ("generated_tokens", C.c_uint64), ("decode_ms_total", C.c_double),
                ("prefill_ms_total", C.c_double), ("active_rows", C.c_int32),
                ("queued", C.c_int32), ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64)]


class GatewayOpts(C.Structure):
    _fields_ = [("manual_clock", C.c_int32), ("record_trace", C.c_int32), ("max_batch_events", C.c_int32),
                ("reserved", C.c_int32 * 5)]


class GatewayResult(C.Structure):
    _fields_ = [("ticket", C.c_uint64), ("status", C.c_int32), ("deployment", C.c_int32), ("served_group", C.c_int32),
                ("chain_pos", C.c_int32), ("replica", C.c_int32), ("n_prompt", C.c_int32), ("n_generated", C.c_int32),
                ("attempts", C.c_int32), ("t_submit_s", C.c_double), ("t_admit_s", C.c_double),
                ("t_first_token_s", C.c_double), ("t_done_s", C.c_double)]


class GatewayStats(C.Structure):
    _fields_ = [(k, C.c_uint64) for k in ("submitted", "admitted", "completed", "rate_limited", "failed", "failed_over",
                                          "launches", "events", "max_batch", "in_flight")] + [("admit_wait_s", C.c_double)]


# ---------------------------------------------------------------- prototypes
# name -> (restype, argtypes).  tests/test_abi.py checks this table against include/rr_b200.h.
PROTOTYPES = {
    "rr_version": (C.c_char_p, []),
    "rr_strerror": (C.c_char_p, [C.c_int]),
    "rr_last_cuda_error": (C.c_char_p, []),
    "rr_set_pdl": (C.c_int, [C.c_int]),
    "rr_debug_trace_start": (C.c_int, [C.c_int]),
    "rr_debug_trace_detail": (C.c_int, [C.c_int]),
    "rr_debug_trace_stop": (C.c_int, [C.POINTER(C.c_uint64), C.c_int, c_i32p]),
    "rr_debug_mlp_schedule": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, c_i32p, C.c_int, c_i32p]),
    "rr_router_create": (C.c_int, [C.POINTER(DeploymentDesc), C.c_int, C.c_int, c_i32p, c_i32p,
                                   C.POINTER(RouterSettings), C.c_uint64, C.c_int,
                                   C.POINTER(vp)]),
    "rr_router_destroy": (None, [vp]),
    "rr_router_process": (C.c_int, [vp, C.POINTER(Event), C.c_int, C.POINTER(Decision)]),
    "rr_router_process_device": (C.c_int, [vp, vp, C.c_int, vp, vp]),
    "rr_router_snapshot": (C.c_int, [vp, C.POINTER(DeploymentState)]),
    "rr_router_seed": (C.c_int, [vp, C.c_uint64]),
    "rr_mt_seed_state": (C.c_int, [C.c_uint64, C.POINTER(C.c_uint32)]),
    "rr_count_tokens": (C.c_int, [C.c_char_p, C.c_size_t, c_i32p]),
    "rr_tokenize": (C.c_int, [C.c_char_p, C.c_size_t, C.c_int32, c_i32p, C.c_int32, c_i32p]),
    "rr_tokenize_batch": (C.c_int, [C.c_char_p, C.POINTER(C.c_int64), C.c_int, C.c_int32, c_i32p, c_i32p, C.c_int64,
                                    C.POINTER(C.c_int64)]),
    "rr_tokenize_batch_device": (C.c_int, [vp, vp, C.c_int, C.c_int64, C.c_int32, vp, vp, vp, vp]),
    "rr_gemm_bf16": (C.c_int, [vp, C.c_int, C.c_int, vp, C.c_int, C.c_int, C.c_int, vp, C.c_int,
                               C.c_int, C.c_int, C.c_int, C.c_int, vp]),
    "rr_op_embed": (C.c_int, [vp, vp, vp, C.c_int, C.c_int, vp, vp]),
    "rr_op_add_rmsnorm": (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_longlong, C.c_int, vp, vp,
                                    C.c_int, C.c_int, C.c_float, vp]),
    "rr_op_silu_mul": (C.c_int, [vp, C.c_int, C.c_int, C.c_longlong, C.c_int, vp, C.c_int,
                                 C.c_int, vp]),
    "rr_op_rope_kv": (C.c_int, [vp, C.c_int, C.c_int, C.c_longlong, C.c_int, vp, vp, vp, vp, vp,
                                C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, vp]),
    "rr_op_argmax": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp, vp]),
    "rr_op_decode_attn": (C.c_int, [vp, vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                    C.c_float, C.c_int, vp]),
    "rr_op_prefill_attn": (C.c_int, [vp, vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int,
                                     C.c_int, C.c_float, vp]),
    "rr_engine_create": (C.c_int, [C.POINTER(ModelDesc), C.POINTER(ModelWeights),
                                   C.POINTER(EngineOpts), C.POINTER(vp)]),
    "rr_engine_destroy": (None, [vp]),
    "rr_engine_prefill": (C.c_int, [vp, c_i32p, c_i32p, c_i32p, C.c_int, c_i32p, c_f32p]),
    "rr_engine_decode_step": (C.c_int, [vp, c_i32p, c_i32p, c_i32p, C.c_int, c_i32p, c_f32p]),
    "rr_engine_submit": (C.c_int, [vp, c_i32p, C.c_int, C.c_int, C.POINTER(C.c_uint64)]),
    "rr_engine_wait": (C.c_int, [vp, C.c_uint64, C.c_double, C.POINTER(Completion), c_i32p,
                                 C.c_int]),
    "rr_engine_peek": (C.c_int, [vp, C.c_uint64, C.c_int, C.c_double, c_i32p, C.c_int, c_i32p, c_i32p,
                                 C.POINTER(C.c_double)]),
    "rr_engine_run_batch": (C.c_int, [vp, c_i32p, c_i32p, C.c_int, C.c_int,
                                      C.POINTER(Completion), c_i32p]),
    "rr_engine_now": (C.c_double, [vp]),
    "rr_engine_get_stats": (C.c_int, [vp, C.POINTER(EngineStats)]),
    "rr_engine_reset_stats": (C.c_int, [vp]),
    "rr_engine_cancel": (C.c_int, [vp, C.c_uint64]),
    "rr_gateway_create": (C.c_int, [vp, C.POINTER(vp), c_i32p, C.c_int, C.POINTER(GatewayOpts), C.POINTER(vp)]),
    "rr_gateway_destroy": (None, [vp]),
    "rr_gateway_set_now": (C.c_int, [vp, C.c_int64]),
    "rr_gateway_submit": (C.c_int, [vp, C.c_int, c_i32p, C.c_int, C.c_int, C.POINTER(C.c_uint64)]),
    "rr_gateway_submit_batch": (C.c_int, [vp, C.c_int, c_i32p, c_i32p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_uint64)]),
    "rr_gateway_wait": (C.c_int, [vp, C.c_uint64, C.c_double, C.POINTER(GatewayResult), c_i32p, C.c_int]),
    "rr_gateway_peek": (C.c_int, [vp, C.c_uint64, C.c_int, C.c_double, c_i32p, C.c_int, c_i32p, c_i32p,
                                  C.POINTER(GatewayResult)]),
    "rr_gateway_cancel": (C.c_int, [vp, C.c_uint64, C.c_int]),
    "rr_gateway_quiesce": (C.c_int, [vp, C.c_double]),
    "rr_gateway_get_stats": (C.c_int, [vp, C.POINTER(GatewayStats)]),
    "rr_gateway_trace": (C.c_int, [vp, C.POINTER(Event), C.POINTER(Decision), C.c_int, c_i32p]),
}

MISSING = []
for _name, (_res, _args) in PROTOTYPES.items():
    try:
        _fn = getattr(lib, _name)
    except AttributeError:
        MISSING.append(_name)
        continue
    _fn.restype = _res
    _fn.argtypes = _args


class RRError(RuntimeError):
    def __init__(self, rc: int, where: str = ""):
        self.rc = rc
        msg = lib.rr_strerror(rc).decode()
        cuda = lib.rr_last_cuda_error().decode()
        super().__init__(f"{where}: {msg} (rc={rc})" + (f" [cuda: {cuda}]" if cuda else ""))


def check(rc: int, where: str = "") -> None:
    if rc != 0:
        raise RRError(rc, where)
