"""Python handle on one model replica (rr_engine in librr_b200.so).

Thin by design: torch provides device memory for the weights and the current device; every
computation happens in the CUDA library.  Replaces one `bedrock/...` deployment of the reference
(config/config.yaml:39-91) — the thing `litellm` would call over the network.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import List, Optional, Sequence

import numpy as np
import torch

from . import _lib
from .models import ModelSpec, Weights, make_weights


@dataclass
class CompletionRecord:
    ticket: int
    status: int
    n_prompt: int
    tokens: List[int]
    t_submit: float
    t_first_token: float
    t_done: float

    @property
    def ttft(self) -> float:
        return self.t_first_token - self.t_submit

    @property
    def latency(self) -> float:
        return self.t_done - self.t_submit


def _i32(a) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(a, dtype=np.int32))


def _p(a: np.ndarray):
    return a.ctypes.data_as(C.POINTER(C.c_int32))


class Engine:
    def __init__(self, weights: Weights, device: int = 0, max_batch: int = 64, ctx_max: int = 1024,
                 max_prefill_tokens: int = 8192, use_cuda_graph: bool = True,
                 fail_prob: float = 0.0, fail_seed: int = 0, fuse_silu: bool = True,
                 fuse_mlp: bool = True, defer_norm: bool = True):
        if not torch.cuda.is_available():
            raise RuntimeError("rr_b200.Engine needs a CUDA device (no CPU fallback)")
        self.spec: ModelSpec = weights.spec
        self.weights = weights          # keep the tensors alive
        self.device = device
        self.max_batch = max_batch
        self.ctx_max = ctx_max
        s = self.spec
        desc = _lib.ModelDesc(s.vocab, s.hidden, s.inter, s.n_layers, s.n_heads, s.n_kv_heads,
                              s.head_dim, s.rope_theta, s.rms_eps)
        L = s.n_layers

        def arr(ts):
            return (C.c_void_p * L)(*[t.data_ptr() for t in ts])

        # Engine-owned layout of the gate/up weights: rows interleaved in 64-row gate/up blocks so that the GEMM
        # epilogue can apply SiLU(gate) * up itself (csrc/rr_gemm.cu, OUT_*_SILU).  Needs one gate/up plane at this
        # batch size (no split-K for gate/up) and batch tiles >= 32 rows; otherwise the [gate; up] layout is kept.
        n_sm = torch.cuda.get_device_properties(device).multi_processor_count
        tiles, kb = (2 * s.inter + 127) // 128, (s.hidden + 63) // 64
        gu_splits = max(1, min(8, n_sm // tiles))                 # mirrors pick_splits() in csrc/rr_engine.cu
        while gu_splits > 1 and kb // gu_splits < 8:
            gu_splits -= 1
        self.fuse_silu = bool(fuse_silu and s.inter % 64 == 0 and gu_splits == 1 and max_batch > 16)
        wgu = weights.wgu
        if self.fuse_silu:
            self._wgu_il = []
            for t in weights.wgu:
                g, u = t[: s.inter].view(-1, 64, s.hidden), t[s.inter:].view(-1, 64, s.hidden)
                self._wgu_il.append(torch.stack([g, u], 1).reshape(2 * s.inter, s.hidden).contiguous())
            wgu = self._wgu_il
        self._arrs = [arr(weights.wqkv), arr(weights.wo), arr(wgu), arr(weights.wdown),
                      arr(weights.norm_attn), arr(weights.norm_mlp)]
        for t in weights.tensors():
            assert t.is_cuda and t.dtype == torch.bfloat16 and t.is_contiguous()
        mw = _lib.ModelWeights(weights.embed.data_ptr(), weights.lm_head.data_ptr(),
                               weights.final_norm.data_ptr(), *self._arrs, 1 if self.fuse_silu else 0, 0)
        opts = _lib.EngineOpts(device, max_batch, ctx_max, max_prefill_tokens,
                               1 if use_cuda_graph else 0, fail_seed, fail_prob,
                               (C.c_int32 * 4)(0, 0, 0 if fuse_mlp else 1, 0 if defer_norm else 1))
        torch.cuda.synchronize(device)   # weights were produced on torch's stream
        self._h = C.c_void_p()
        _lib.check(_lib.lib.rr_engine_create(C.byref(desc), C.byref(mw), C.byref(opts),
                                             C.byref(self._h)), "rr_engine_create")

    @classmethod
    def synthetic(cls, spec: ModelSpec, seed: int = 0, device: int = 0, **kw) -> "Engine":
        return cls(make_weights(spec, seed=seed, device=f"cuda:{device}"), device=device, **kw)

    def close(self):
        if getattr(self, "_h", None):
            _lib.lib.rr_engine_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- low-level synchronous steps (parity tests) ---------------------------------------------
    def prefill(self, prompts: Sequence[Sequence[int]], slots: Sequence[int], want_logits=False):
        ids = _i32([t for p in prompts for t in p])
        start = _i32(np.concatenate([[0], np.cumsum([len(p) for p in prompts])]))
        sl = _i32(slots)
        n = len(prompts)
        first = np.zeros(n, dtype=np.int32)
        logits = np.zeros((n, self.spec.vocab), dtype=np.float32) if want_logits else None
        lp = logits.ctypes.data_as(C.POINTER(C.c_float)) if want_logits else None
        _lib.check(_lib.lib.rr_engine_prefill(self._h, _p(ids), _p(start), _p(sl), n, _p(first), lp),
                   "rr_engine_prefill")
        return first, logits

    def decode_step(self, slots, toks, pos, want_logits=False):
        sl, tk, ps = _i32(slots), _i32(toks), _i32(pos)
        n = len(sl)
        nxt = np.zeros(n, dtype=np.int32)
        logits = np.zeros((n, self.spec.vocab), dtype=np.float32) if want_logits else None
        lp = logits.ctypes.data_as(C.POINTER(C.c_float)) if want_logits else None
        _lib.check(_lib.lib.rr_engine_decode_step(self._h, _p(sl), _p(tk), _p(ps), n, _p(nxt), lp),
                   "rr_engine_decode_step")
        return nxt, logits

    # ---- serving interface ----------------------------------------------------------------------
    def submit(self, prompt_ids: Sequence[int], max_new_tokens: int) -> int:
        ids = _i32(prompt_ids)
        t = C.c_uint64()
        _lib.check(_lib.lib.rr_engine_submit(self._h, _p(ids), len(ids), max_new_tokens, C.byref(t)),
                   "rr_engine_submit")
        return t.value

    def wait(self, ticket: int, timeout: float = 0.0, max_tokens: int = 4096) -> CompletionRecord:
        c = _lib.Completion()
        buf = np.zeros(max_tokens, dtype=np.int32)
        rc = _lib.lib.rr_engine_wait(self._h, ticket, float(timeout), C.byref(c), _p(buf), max_tokens)
        if rc not in (0, 6, 7):
            _lib.check(rc, "rr_engine_wait")
        return CompletionRecord(ticket, rc, c.n_prompt, buf[:c.n_generated].tolist(), c.t_submit_s,
                                c.t_first_token_s, c.t_done_s)

    def peek(self, ticket: int, have: int, timeout: float = 0.05, max_tokens: int = 4096):
        """Streaming: wait until more than `have` tokens exist (or done / timeout). -> (tokens so far, done, ttft_s)."""
        buf = np.zeros(max_tokens, dtype=np.int32)
        n, done, ttft = C.c_int32(), C.c_int32(), C.c_double()
        _lib.check(_lib.lib.rr_engine_peek(self._h, ticket, have, float(timeout), _p(buf), max_tokens, C.byref(n),
                                           C.byref(done), C.byref(ttft)), "rr_engine_peek")
        return buf[: n.value].tolist(), bool(done.value), ttft.value

    def run_batch(self, prompt_ids: np.ndarray, prompt_start: np.ndarray, max_new_tokens: int):
        """Closed burst: submit every prompt, wait for all.  `prompt_ids` is a host buffer; the
        H2D copies happen inside the library.  -> (completions, tokens [n, max_new])."""
        ids, start = _i32(prompt_ids), _i32(prompt_start)
        n = len(start) - 1
        comps = (_lib.Completion * n)()
        toks = np.zeros((n, max_new_tokens), dtype=np.int32)
        rc = _lib.lib.rr_engine_run_batch(self._h, _p(ids), _p(start), n, max_new_tokens, comps, _p(toks))
        if rc not in (0, 7):
            _lib.check(rc, "rr_engine_run_batch")
        recs = [CompletionRecord(c.ticket, c.status, c.n_prompt, toks[i, :c.n_generated].tolist(),
                                 c.t_submit_s, c.t_first_token_s, c.t_done_s) for i, c in enumerate(comps)]
        return recs, toks

    def now(self) -> float:
        return _lib.lib.rr_engine_now(self._h)

    def stats(self) -> dict:
        s = _lib.EngineStats()
        _lib.check(_lib.lib.rr_engine_get_stats(self._h, C.byref(s)), "stats")
        return {k: getattr(s, k) for k, _ in s._fields_}

    def reset_stats(self):
        _lib.check(_lib.lib.rr_engine_reset_stats(self._h), "reset_stats")
