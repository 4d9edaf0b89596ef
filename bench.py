#!/usr/bin/env python
"""bench.py — headline benchmark of the request-router hot path (BASELINE.json):
completions/sec and p50 TTFT, 512-in / 128-out, Llama-3-8B shape, one replica per GPU,
64 concurrent requests per replica, least-busy routing.

A "step" = one closed burst of (64 x n_gpus) chat-completion requests through the whole path:
K1 admission (rpm/tpm debit + least-busy pick) -> per-GPU engine: chunked prefill + 127 decode steps
(CUDA graph) -> DONE events.  Launch:  python bench.py --gpus N --steps K --warmup W
(N > 1: python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...).
Inputs (weights, prompts) are seeded: --dump-outputs DIR stores what the last timed burst returned (generated tokens, router
picks) as .npy, so that two builds can be compared output for output.

  value      completions/s from device time only: CUDA events on each engine's stream around every
             prefill chunk and every decode step of the timed steps (inputs resident), max over ranks.
  e2e        the same metric by host wall clock through the public API: prompts start in pinned HOST memory,
             admission events H2D, decisions D2H, prompt ids H2D, generated tokens D2H all inside the timed region.
             N = 1: Router.completion_batch (native gateway: rr_gateway_submit_batch / rr_gateway_wait);
             N > 1: rank 0 admits with rr_router_process, assignments travel by NCCL, every rank serves its share
             with rr_engine_run_batch.
  roofline   decode step (one CUDA-graph launch = the dominant unit): algorithmic bytes
             (weights streamed once + KV read) / mean CUDA-event step time, against MEASURED_PEAKS.json;
             `kernels` = per-kernel table (algorithmic bytes, in-graph critical-path us, fraction of peak) from the
             library's in-kernel timeline, taken AFTER the timed region.
  per_request / http (N = 1, after the timed region): the same burst issued by 64 concurrent Router.completion()
             callers, and by 64 OpenAI-SDK clients over HTTP against the in-process gateway (server.py).
  cpu_baseline / --impl reference: the CPU restatement (oracle/) of the same path timed on the box's host
             cores on a bounded sample (the reference's own router, litellm, cannot be installed:
             BASELINE.md §2; there is no baseline/_ref).

Other BASELINE.json configs (single process driving --gpus N devices through the native gateway, the layout of the
reference's one-process gateway):  --config quota | fallback | fleet   (see run_fleet).
"""
from __future__ import annotations

import argparse
import importlib.util
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "completions/sec (512-in/128-out, Llama-3-8B, 64 concurrent per GPU)"
CONFIGS = {"1": "headline", "headline": "headline", "2": "quota", "quota": "quota", "3": "fallback", "fallback": "fallback",
           "4": "fleet", "fleet": "fleet"}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--model", default="llama-3-8b")
    ap.add_argument("--concurrency", type=int, default=64, help="concurrent requests per GPU")
    ap.add_argument("--prompt-len", type=int, default=512)
    ap.add_argument("--max-new", type=int, default=128)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the per-request / HTTP / per-kernel legs after the timed region")
    ap.add_argument("--config", default="headline", choices=sorted(CONFIGS),
                    help="BASELINE.json config: headline (#1, default), quota (#2), fallback (#3), fleet (#4)")
    ap.add_argument("--trace-out", default=None, help="fleet configs: write the recorded admission trace here (JSON)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="headline config: after the timed steps write what the last one returned to its callers as DIR/*.npy "
                         "(float32): tokens [requests, max_new] = generated token ids, deployment [requests] = router pick")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or CONFIGS[args.config] != "headline"):
        ap.error("--dump-outputs applies to the headline config of --impl b200")
    return args


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops_sustained", 1400.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, 1400.0, "fallback (B200_PROFILING.md)"


def load_models_module():
    """models.py (specs only) WITHOUT importing the package: the package __init__ dlopens librr_b200.so, and the
    reference arm must not touch this repo's native code."""
    spec = importlib.util.spec_from_file_location(
        "_rr_models_only", os.path.join(ROOT, "sample-resilient-llm-inference_b200", "models.py"))
    mod = importlib.util.module_from_spec(spec)
    sys.modules["_rr_models_only"] = mod
    spec.loader.exec_module(mod)
    return mod


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.idx), "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------
def make_prompts(n_req: int, prompt_len: int, vocab: int, pinned: bool):
    """int32[prompt_len] ids per request, torch.Generator().manual_seed(1234 + req_id), uniform in [0, vocab)."""
    import torch
    buf = torch.empty((n_req, prompt_len), dtype=torch.int32, pin_memory=pinned)
    for r in range(n_req):
        g = torch.Generator().manual_seed(1234 + r)
        buf[r] = torch.randint(0, vocab, (prompt_len,), generator=g, dtype=torch.int32)
    return buf


def executed_prefill_flops(spec, n_prompts: int, prompt_len: int) -> int:
    """FLOPs the prefill of one burst EXECUTES (linear layers only): every layer's QKV on all tokens; O / gate-up / down
    on all tokens for layers 0..L-2; the last layer's O / MLP and the lm_head only on the last token of each prompt
    (csrc/rr_engine.cu: trimmed tail).  SURVEY 8(d)'s 15.01 GFLOP/token counts lm_head and a full last layer per token."""
    H, KV, D, hid, inter, L = spec.n_heads, spec.n_kv_heads, spec.head_dim, spec.hidden, spec.inter, spec.n_layers
    qkv = hid * (H + 2 * KV) * D
    rest = H * D * hid + 3 * hid * inter
    T = n_prompts * prompt_len
    return 2 * (T * (L * qkv + (L - 1) * rest) + n_prompts * (rest + spec.vocab * hid))


def cpu_port_sample(spec, prompt_len, max_new, concurrency, n_gpus, layers_timed=4, decode_steps_timed=2, threads=None):
    """CPU restatement of the path on a bounded sample; returns (completions/s, description, cores).

    Router: oracle admission of the full burst (all requests).  Token generation: fp32 torch CPU forward of
    ONE request at the exact Llama-3-8B layer shape; `layers_timed` of the identical layers and
    `decode_steps_timed` of the decode steps are timed and scaled to n_layers / (max_new - 1)."""
    import torch
    from oracle import router as O
    try:
        avail = len(os.sched_getaffinity(0))
    except AttributeError:
        avail = os.cpu_count() or 1
    cores = threads or min(avail, 64)          # beyond ~64 threads the fp32 GEMMs of one request stop scaling
    torch.set_num_threads(cores)
    t0 = time.perf_counter()
    deps = [O.Deployment(group=0, replica=r) for r in range(n_gpus)]
    orc = O.OracleRouter(deps, 1, {}, O.Settings(strategy=O.STRATEGY_LEAST_BUSY), seed=0)
    n_req = concurrency * n_gpus
    dec = orc.process([O.Event(O.EV_ADMIT, 0, prompt_len, 0, 0) for _ in range(n_req)])
    orc.process([O.Event(O.EV_DONE, d.deployment, max_new, 0, 1) for d in dec])
    t_router = time.perf_counter() - t0

    H, KV, D, hid, inter = spec.n_heads, spec.n_kv_heads, spec.head_dim, spec.hidden, spec.inter
    g = torch.Generator().manual_seed(0)
    mk = lambda *s: torch.empty(*s).normal_(0, 0.02, generator=g)
    layers = [dict(wqkv=mk((H + 2 * KV) * D, hid), wo=mk(hid, H * D), wgu=mk(2 * inter, hid), wdown=mk(hid, inter))
              for _ in range(layers_timed)]
    lm_head = mk(spec.vocab, hid)

    def layer_fwd(x, L, kc, vc, pos0):
        T = x.shape[0]
        h = x * torch.rsqrt(x.pow(2).mean(-1, keepdim=True) + spec.rms_eps)
        qkv = h @ L["wqkv"].t()
        q = qkv[:, : H * D].view(T, H, D)
        k = qkv[:, H * D:(H + KV) * D].view(T, KV, D)
        v = qkv[:, (H + KV) * D:].view(T, KV, D)
        kc[pos0:pos0 + T] = k; vc[pos0:pos0 + T] = v
        kk = kc[: pos0 + T].repeat_interleave(H // KV, 1); vv = vc[: pos0 + T].repeat_interleave(H // KV, 1)
        a = torch.nn.functional.scaled_dot_product_attention(q.transpose(0, 1), kk.transpose(0, 1), vv.transpose(0, 1),
                                                             is_causal=(T > 1))
        x = x + a.transpose(0, 1).reshape(T, H * D) @ L["wo"].t()
        h = x * torch.rsqrt(x.pow(2).mean(-1, keepdim=True) + spec.rms_eps)
        gu = h @ L["wgu"].t()
        return x + (torch.nn.functional.silu(gu[:, :inter]) * gu[:, inter:]) @ L["wdown"].t()

    with torch.no_grad():
        x = torch.randn(prompt_len, hid, generator=g)
        caches = [(torch.zeros(prompt_len + max_new, KV, D), torch.zeros(prompt_len + max_new, KV, D)) for _ in layers]
        t0 = time.perf_counter()
        for L, (kc, vc) in zip(layers, caches):
            x = layer_fwd(x, L, kc, vc, 0)
        (x[-1:] @ lm_head.t()).argmax()
        t_prefill_layers = time.perf_counter() - t0
        t0 = time.perf_counter()
        for s in range(decode_steps_timed):
            y = x[-1:].clone()
            for L, (kc, vc) in zip(layers, caches):
                y = layer_fwd(y, L, kc, vc, prompt_len + s)
            (y @ lm_head.t()).argmax()
        t_decode_step = (time.perf_counter() - t0) / decode_steps_timed
    scale = spec.n_layers / layers_timed
    t_completion = t_prefill_layers * scale + (max_new - 1) * t_decode_step * scale
    # one request at a time on all cores: completions/s of the whole burst
    value = n_req / (t_router + n_req * t_completion)
    sample = (f"router: oracle admission of all {n_req} requests ({t_router*1e3:.2f} ms); generation: 1 of {n_req} requests, "
              f"{layers_timed} of {spec.n_layers} identical layers and {decode_steps_timed} of {max_new - 1} decode steps timed "
              f"(fp32 torch CPU, {cores} threads) and scaled: {t_completion:.1f} s per completion")
    return value, sample, cores


# ------------------------------------------------------------------------------------------------
def run_reference_arm(args):
    """CPU restatement of the path (the reference's litellm.Router cannot be installed: BASELINE.md §2).  Pure torch-CPU +
    oracle/: nothing of this repo's package (and therefore none of its native code) is imported."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    spec = load_models_module().resolve_spec(args.model)
    vals = []
    sample, cores = "", 0
    t_all = time.perf_counter()
    for i in range(args.warmup + args.steps):
        v, sample, cores = cpu_port_sample(spec, args.prompt_len, args.max_new, args.concurrency, args.gpus,
                                           layers_timed=2, decode_steps_timed=2)
        if i >= args.warmup:
            vals.append(v)
    value = len(vals) / sum(1.0 / v for v in vals)
    n_req = args.concurrency * args.gpus
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "completions/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * n_req / value, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{args.model}: {n_req} concurrent {args.prompt_len}-in/{args.max_new}-out, least-busy "
                                   "(CPU restatement; litellm is not installable here)"},
            "cpu_baseline": {"value": value, "unit": "completions/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "completions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "wall_s": time.perf_counter() - t_all}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
def kernel_table(eng, spec, prompts_np, C, P, M, hbm_peak):
    """Per-kernel share of one decode step from the library's in-kernel timeline (CTA 0 of every kernel stamps
    %globaltimer at start / when griddepcontrol.wait returns / at exit; rr_debug_trace_*).  The critical-path time of
    kernel k inside the replayed graph = (dependency of kernel k+1 resolved) - (dependency of kernel k resolved).
    Runs one short extra burst AFTER the timed region."""
    import ctypes as Ct
    from rr_b200 import _lib
    NAMES = {1: "gemm/layer (tcgen05)", 3: "decode_attn", 5: "add_rmsnorm", 8: "embed", 9: "argmax", 10: "attn_combine"}
    ids = np.ascontiguousarray(prompts_np[:C]).reshape(-1)
    start = np.arange(0, (C + 1) * P, P, dtype=np.int32)
    N = 20000
    _lib.check(_lib.lib.rr_debug_trace_start(N), "trace_start")
    eng.run_batch(ids, start, 6)
    buf = (Ct.c_uint64 * (4 * N))(); n = Ct.c_int32()
    _lib.check(_lib.lib.rr_debug_trace_stop(buf, N, Ct.byref(n)), "trace_stop")
    a = np.frombuffer(buf, dtype=np.uint64)[: 4 * n.value].reshape(-1, 4).astype(np.int64)
    a = a[a[:, 0] < 12]                                        # kernel records only
    a = a[np.argsort(a[:, 1], kind="stable")]
    emb = np.nonzero(a[:, 0] == 8)[0]
    if len(emb) < 2:
        return None
    step = a[emb[-2]: emb[-1] + 1]                             # one whole decode step + the next step's first kernel
    L = spec.n_layers
    H, KV, D, hid, inter = spec.n_heads, spec.n_kv_heads, spec.head_dim, spec.hidden, spec.inter
    w_qkv, w_o, w_mlp, w_head = 2 * hid * (H + 2 * KV) * D, 2 * H * D * hid, 2 * 3 * hid * inter, 2 * spec.vocab * hid
    ctx = P + 3                                                # context of the traced steps (3rd..5th generated token)
    kv_layer = C * ctx * spec.kv_bytes_per_token // L
    rows = {}
    n_gemm = 0
    host_gap_us = 0.0
    gemm_total = int((step[:-1, 0] == 1).sum())
    for i in range(len(step) - 1):
        kid = int(step[i, 0])
        seg_us = (step[i + 1, 2] - step[i, 2]) / 1e3
        if i == len(step) - 2:                                 # last kernel of the step (argmax): its own dependency -> end; the
            seg_us = (step[i, 3] - step[i, 2]) / 1e3           # segment to the next step's first kernel would add the host's
            host_gap_us = (step[i + 1, 2] - step[i, 3]) / 1e3  # graph relaunch (reported separately)
        name, nbytes = NAMES.get(kid, f"kernel {kid}"), 0
        if kid == 3:
            nbytes = kv_layer
        elif kid == 1:
            if gemm_total == L + 1:                            # persistent layer kernels: QKV_0 | layer l (+ QKV_{l+1}) | last (+ lm_head)
                if n_gemm == 0:
                    name, nbytes = "decode_layer_tcgen05 [QKV of layer 0]", w_qkv
                elif n_gemm < L:
                    name, nbytes = "decode_layer_tcgen05 [O + gate/up + down + next QKV]", w_o + w_mlp + w_qkv
                else:
                    name, nbytes = "decode_layer_tcgen05 [last layer + lm_head]", w_o + w_mlp + w_head
            elif gemm_total == 3 * L + 1:                       # default path, per layer: QKV GEMM, O GEMM, fused MLP; then lm_head
                if n_gemm == 3 * L:
                    name, nbytes = "gemm_bf16_tcgen05<64,1> lm_head", w_head
                else:
                    name, nbytes = [("gemm_bf16_tcgen05<64,1> QKV projection (split-K 3)", w_qkv),
                                    ("gemm_bf16_tcgen05<64,1> O projection (split-K 4)", w_o),
                                    ("gemm_mlp_tcgen05<64> gate/up + SiLU + down", w_mlp)][n_gemm % 3]
            else:
                name = "gemm_bf16_tcgen05 (other decode configuration)"
            n_gemm += 1
        r = rows.setdefault(name, {"kernel": name, "launches": 0, "us": 0.0, "bytes": 0})
        r["launches"] += 1; r["us"] += seg_us; r["bytes"] += nbytes
    out = []
    for r in rows.values():
        gbs = r["bytes"] / (r["us"] * 1e-6) / 1e9 if r["bytes"] and r["us"] > 0 else None
        out.append({"kernel": r["kernel"], "launches": r["launches"], "us_per_launch": r["us"] / r["launches"],
                    "us_per_step": r["us"], "algorithmic_bytes_per_launch": r["bytes"] // r["launches"],
                    "achieved_gbs": gbs, "frac_of_hbm_peak": (gbs / hbm_peak) if gbs else None})
    out.sort(key=lambda x: -x["us_per_step"])
    return {"step_us_traced": float((step[-1, 2] - step[0, 2]) / 1e3), "ctx": ctx, "rows": out,
            "host_gap_between_steps_us": float(host_gap_us),
            "method": "in-kernel %globaltimer stamps of CTA 0 (rr_debug_trace_*), critical-path segments inside the replayed CUDA "
                      "graph; the stamps themselves cost ~3 us per kernel (compare step_us_traced with roofline.ms_per_launch): "
                      "read the SHARES and the per-kernel fractions as lower bounds"}


def per_request_leg(router, model, prompts_np, n_req, M, bursts=2):
    """The same closed burst issued the way the reference's demos do it: one blocking call per client thread."""
    lat, ttft, errs = [], [], []
    st0 = router.gateway_stats()
    t0 = time.perf_counter()
    for _ in range(bursts):
        out = [None] * n_req

        def work(i):
            try:
                out[i] = router.completion(model=model, prompt_ids=prompts_np[i], max_tokens=M, timeout=300)
            except Exception as e:                              # noqa: BLE001 (recorded, re-raised below)
                out[i] = e
        ths = [threading.Thread(target=work, args=(i,)) for i in range(n_req)]
        for t in ths:
            t.start()
        for t in ths:
            t.join()
        for o in out:
            if isinstance(o, Exception):
                errs.append(repr(o))
            else:
                assert len(o._token_ids) == M
                lat.append(o._latency_s); ttft.append(o._ttft_s)
    wall = time.perf_counter() - t0
    router.snapshot()
    st1 = router.gateway_stats()
    ev, la = st1["events"] - st0["events"], st1["launches"] - st0["launches"]
    return {"api": "Router.completion() from %d concurrent threads (rr_gateway_submit / rr_gateway_wait)" % n_req,
            "value": len(lat) / wall, "unit": "completions/s", "bursts": bursts, "errors": errs[:3],
            "p50_ttft_ms": float(np.percentile(ttft, 50) * 1e3), "p99_ttft_ms": float(np.percentile(ttft, 99) * 1e3),
            "p50_latency_ms": float(np.percentile(lat, 50) * 1e3),
            "k1_launches": int(la), "k1_events": int(ev), "events_per_launch": ev / max(1, la),
            "admit_wait_us_mean": 1e6 * (st1["admit_wait_s"] - st0["admit_wait_s"]) / max(1, st1["submitted"] - st0["submitted"])}


def k1_single_event_latency(router, reps=200):
    """One ADMIT + one DONE through rr_router_process (H2D + launch + D2H + sync each): the un-coalesced per-event cost."""
    now = router.now_ms()
    t0 = time.perf_counter()
    for _ in range(reps):
        (st, dep, _, _), = router.process([(0, 0, 512, 0, now)])
        router.process([(1, dep, 128, 0, now)])
    return (time.perf_counter() - t0) * 1e6 / (2 * reps)


def http_leg(router, model, prompts_np, n_req, M):
    """n_req OpenAI-SDK clients (the reference's client boundary: src/demo_load_balancing.py:24,106-110) in a SEPARATE
    process against the in-process gateway (server.py): one non-streamed burst (throughput, latency) and one streamed burst
    (TTFT = first SSE chunk).  Prompts travel as text: 505 characters -> 512 byte-level tokens."""
    try:
        import uvicorn
        from rr_b200.server import create_app
    except Exception as e:                                      # noqa: BLE001
        return {"skipped": repr(e)}
    import socket
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    server = uvicorn.Server(uvicorn.Config(create_app(router), host="127.0.0.1", port=port, log_level="error"))
    th = threading.Thread(target=server.run, daemon=True)
    th.start()
    t_wait = time.time()
    while not server.started and time.time() - t_wait < 30:
        time.sleep(0.05)
    out = {"api": "openai.OpenAI(base_url=http://127.0.0.1:<port>).chat.completions.create(...) x %d client threads in a separate "
                  "process -> server.py -> Router.completion / completion_stream" % n_req, "prompt_tokens": P_TEXT + 7}
    try:
        n_proc = 8 if n_req % 8 == 0 else 1                     # client processes: one Python GIL per 8 client threads
        per = n_req // n_proc
        for mode, key in (("0", "non_streamed"), ("1", "streamed")):
            start_at = time.time() + 4.0                        # every client process fires at this wall-clock time
            procs = [subprocess.Popen([sys.executable, os.path.join(ROOT, "tools", "http_clients.py"), str(port), model, str(per),
                                       str(M), str(P_TEXT), mode, repr(start_at), str(k * per)], stdout=subprocess.PIPE,
                                      stderr=subprocess.PIPE, text=True) for k in range(n_proc)]
            lat, ttft, errs, t_end = [], [], [], start_at
            for pr in procs:
                so, se = pr.communicate(timeout=600)
                if pr.returncode != 0:
                    errs.append(se[-300:])
                    continue
                r = json.loads(so.strip().splitlines()[-1])
                lat += r["lat"]; ttft += r["ttft"]; errs += r["errors"]; t_end = max(t_end, r["t_end"])
            wall = t_end - start_at
            d = {"value": len(lat) / wall if lat else None, "unit": "completions/s", "errors": errs[:3], "client_processes": n_proc,
                 "p50_latency_ms": float(np.percentile(lat, 50) * 1e3) if lat else None,
                 "p99_latency_ms": float(np.percentile(lat, 99) * 1e3) if lat else None}
            if ttft:
                d["p50_ttft_ms"] = float(np.percentile(ttft, 50) * 1e3)
                d["p99_ttft_ms"] = float(np.percentile(ttft, 99) * 1e3)
            out[key] = d
    finally:
        server.should_exit = True
        th.join(timeout=10)
    return out


P_TEXT = 505          # "user: " (6) + 505 characters + BOS = 512 tokens of the byte-level tokenizer


# ------------------------------------------------------------------------------------------------
def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
        return
    kind = CONFIGS[args.config]
    if kind != "headline":
        run_fleet(args, kind)
        return
    import torch
    import torch.distributed as dist
    from rr_b200.models import resolve_spec, make_weights, broadcast_weights
    from rr_b200.engine import Engine
    from rr_b200.router import Router, EngineBackend
    from rr_b200 import parallel

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    spec = resolve_spec(args.model)
    C, P, M = args.concurrency, args.prompt_len, args.max_new
    ctx_max = ((P + M + 63) // 64) * 64

    # ---- start-up: seeded weights on rank 0, NCCL broadcast to every replica (the one collective)
    t0 = time.perf_counter()
    w = make_weights(spec, seed=0, sigma=0.02, device=f"cuda:{local}", allocate_only=(rank != 0))
    bcast_s = None
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier()
        tb = time.perf_counter()
        broadcast_weights(w, src=0)
        torch.cuda.synchronize()
        bcast_s = time.perf_counter() - tb
    torch.cuda.synchronize()
    init_s = time.perf_counter() - t0
    eng = Engine(w, device=local, max_batch=C, ctx_max=ctx_max, max_prefill_tokens=8192, use_cuda_graph=True)
    backend = EngineBackend(eng)

    # ---- router (rank 0 owns the device-resident state): one model group, one deployment per GPU
    model_list = [{"model_name": args.model, "litellm_params": {"model": f"b200/{args.model}", "gpu": r},
                   "rpm": 1_000_000, "tpm": 2_000_000_000} for r in range(world)]
    router = None
    if rank == 0:
        router = Router(model_list=model_list, routing_strategy="least-busy", enable_pre_call_checks=True,
                        allowed_fails=2, cooldown_time=15, backends={0: backend}, seed=0, device=local)
    n_req = C * world
    prompts = make_prompts(n_req, P, spec.vocab, pinned=True)      # host-resident inputs (pinned)
    prompts_np = prompts.numpy()

    ttfts, lat = [], []
    token_sums = []                                                # per step: checksum of every generated token
    last = {}                                                      # what the latest burst returned (--dump-outputs)

    def one_step(collect: bool):
        """One closed burst through the public path.  Returns nothing; per-request timings collected."""
        if world == 1:
            out = router.completion_batch(args.model, [prompts_np[i] for i in range(n_req)], M)
            last["out"] = out
            chk = 0
            for i, r in enumerate(out):
                if isinstance(r, Exception):
                    raise r
                assert len(r._token_ids) == M and all(0 <= t < spec.vocab for t in r._token_ids)
                chk = (chk * 1000003 + hash(tuple(r._token_ids)) + i) & 0xFFFFFFFFFFFF
                if collect:
                    ttfts.append(r._ttft_s); lat.append(r._latency_s)
            token_sums.append(chk)
        else:
            dec = None
            if rank == 0:
                now = router.now_ms()
                dec = router.process([(0, 0, P, 0, now)] * n_req)
            mine = parallel.scatter_assignments(dec, n_req, world, rank, device=torch.device("cuda", local),
                                                replica_of=[d["litellm_params"]["gpu"] for d in model_list])
            ids = np.ascontiguousarray(prompts_np[mine]).reshape(-1)
            start = np.arange(0, (len(mine) + 1) * P, P, dtype=np.int32)
            recs, _ = eng.run_batch(ids, start, M) if len(mine) else ([], None)
            last["out"] = (mine, recs, dec)
            assert all(r.status == 0 and len(r.tokens) == M for r in recs)
            # checksum keyed by REQUEST (which rank serves a request may change from burst to burst: least-busy ties are
            # broken through the router's RNG stream), summed over the ranks
            chk = sum((hash((int(i), tuple(r.tokens))) & 0xFFFFFFFFFF) for i, r in zip(mine, recs))
            ct = torch.tensor([chk], dtype=torch.int64, device=torch.device("cuda", local))
            dist.all_reduce(ct, op=dist.ReduceOp.SUM)
            token_sums.append(int(ct.item()))
            if collect:
                ttfts.extend(r.ttft for r in recs); lat.extend(r.latency for r in recs)
            parallel.gather_done(len(mine), world, rank, device=torch.device("cuda", local))
            if rank == 0:
                now = router.now_ms()
                router.process([(1, d[1], M, 0, now) for d in dec if d[0] == 0])

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        one_step(False)
    sync_all()
    eng.reset_stats()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    sync_all()
    t_start = time.perf_counter()
    for _ in range(args.steps):
        one_step(True)
    sync_all()
    wall = time.perf_counter() - t_start
    clocks = sampler.stop() if rank == 0 else None
    st = eng.stats()
    dev_s = (st["prefill_ms_total"] + st["decode_ms_total"]) / 1e3
    # identical prompts every step and deterministic kernels: every step must have generated exactly the same tokens for
    # every request
    assert len(set(token_sums)) == 1, "generated tokens differ between bursts"
    if args.dump_outputs:
        # the last timed burst as its callers received it, by request id; token ids < 2^24 are exact in float32
        tok, dep = np.zeros((n_req, M)), np.zeros(n_req)
        if world == 1:
            for i, r in enumerate(last["out"]):
                tok[i], dep[i] = r._token_ids, r._deployment
        else:
            mine, recs, dec = last["out"]
            for i, r in zip(mine, recs):
                tok[i] = r.tokens
            if rank == 0:
                dep[:] = [d[1] for d in dec]
            both = torch.from_numpy(np.concatenate([tok.ravel(), dep])).to(f"cuda:{local}")
            dist.all_reduce(both, op=dist.ReduceOp.SUM)                # each request's row is filled on one rank only
            both = both.cpu().numpy()
            tok, dep = both[: n_req * M].reshape(n_req, M), both[n_req * M:]
        if rank == 0:
            os.makedirs(args.dump_outputs, exist_ok=True)
            np.save(os.path.join(args.dump_outputs, "tokens.npy"), tok.astype(np.float32))
            np.save(os.path.join(args.dump_outputs, "deployment.npy"), dep.astype(np.float32))

    # ---- max over ranks
    vals = torch.tensor([wall, dev_s, st["decode_ms_total"], float(st["decode_steps"]), st["prefill_ms_total"],
                         float(st["kernel_launches"]), float(st["h2d_bytes"]), float(st["d2h_bytes"])],
                        dtype=torch.float64, device="cuda")
    if world > 1:
        mx = vals.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = vals.clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        t_all = torch.tensor(sorted(ttfts) + [float("nan")] * (C * args.steps - len(ttfts)), dtype=torch.float64, device="cuda")
        gathered = [torch.empty_like(t_all) for _ in range(world)]
        dist.all_gather(gathered, t_all)
        all_ttft = torch.cat(gathered).cpu().numpy()
        all_ttft = all_ttft[~np.isnan(all_ttft)]
    else:
        mx, sm = vals, vals
        all_ttft = np.asarray(ttfts)
    wall_max, dev_max = mx[0].item(), mx[1].item()
    K = args.steps
    total_completions = n_req * K

    if rank == 0:
        hbm_peak, tf_peak, peak_src = load_peaks()
        # roofline of the dominant unit: the decode step (one CUDA-graph launch)
        steps_per_burst = M - 1
        mean_ctx = P + (1 + steps_per_burst) / 2.0                      # ctx at decode step j = P + j
        bytes_step = spec.weight_bytes_per_decode_step + C * mean_ctx * spec.kv_bytes_per_token
        dec_ms = mx[2].item() / max(1.0, mx[3].item())
        achieved = bytes_step / (dec_ms * 1e-3) / 1e9
        pf_ms = mx[4].item()
        flops_exec = executed_prefill_flops(spec, C, P) * K
        flops_survey = spec.prefill_flops_per_token * C * P * K
        pf_tflops = flops_exec / (pf_ms * 1e-3) / 1e12 if pf_ms > 0 else None
        launches_per_step = int(st["kernel_launches"] / max(1, st["decode_steps"] + st["prefill_chunks"]))
        # DRAM traffic of one decode step: from the committed ncu --set full capture of THIS code, if one exists
        traffic, traffic_src = None, "no ncu capture of the current decode step committed (profiles/r02_decode_step_traffic.json)"
        tp = os.path.join(ROOT, "profiles", "r02_decode_step_traffic.json")
        if os.path.exists(tp):
            with open(tp) as f:
                tj = json.load(f)
            if tj.get("model") == args.model and tj.get("rows") == C and tj.get("prompt_len") == P:
                traffic, traffic_src = tj.get("dram_bytes_per_step"), tj.get("source")
        line = {
            "metric": METRIC, "value": total_completions / dev_max, "unit": "completions/s", "n_gpus": world,
            "steps": K, "warmup": args.warmup, "ms_per_step": 1e3 * dev_max / K, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"{args.model} shape, seeded random weights, {C} concurrent x {world} GPU(s), "
                                   f"{P}-in/{M}-out greedy, least-busy routing over {world} replica(s)",
                       "global_batch": n_req, "prompt_len": P, "max_new": M, "parallelism": f"replicas x{world} (dp{world})",
                       "l2": "inputs larger than L2: 15 GB of weights + 4.8 GB of KV are re-read every decode step (L2 = 126 MB)",
                       "timing": "value: CUDA events on each engine stream around every prefill chunk / decode step, max over ranks"},
            "p50_ttft_ms": float(np.percentile(all_ttft, 50) * 1e3), "p99_ttft_ms": float(np.percentile(all_ttft, 99) * 1e3),
            "tokens_per_s": total_completions * M / dev_max,
            "e2e": {"value": total_completions / wall_max, "unit": "completions/s", "ms_per_step": 1e3 * wall_max / K,
                    "h2d_bytes_per_step": int(sm[6].item() / K + 24 * n_req), "d2h_bytes_per_step": int(sm[7].item() / K + 16 * n_req),
                    "api": ("Router.completion_batch -> rr_gateway_submit_batch / rr_gateway_wait (host buffers; K1 + engine hand-off "
                            "inside the library)") if world == 1 else
                           ("rank 0: Router.process (rr_router_process, host buffers) -> NCCL broadcast of the assignment vector -> "
                            "every rank: Engine.run_batch (rr_engine_run_batch, host buffers) -> NCCL all-reduce -> DONE trace")},
            "gpu_launches": int(sm[5].item() + 2 * K),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                         "traffic": traffic, "traffic_source": traffic_src,
                         "kernel": "decode step = 1 CUDA-graph launch (196 kernels, PDL edges); dominant kernels: gemm_mlp_tcgen05<64> / "
                                   "gemm_bf16_tcgen05<64,1> (weight streams) and decode_attn_mma_kernel<4> (KV stream); see `kernels`",
                         "bytes_per_launch": bytes_step, "ms_per_launch": dec_ms, "peak_source": peak_src},
            "prefill": {"tflops": pf_tflops, "peak_tflops_sustained": tf_peak, "frac": (pf_tflops / tf_peak) if pf_tflops else None,
                        "ms_per_burst": pf_ms / K, "flops_counted": "executed (last layer's O / MLP and lm_head only on each prompt's last token)",
                        "gflop_per_token_executed": flops_exec / (C * P * K) / 1e9,
                        "gflop_per_token_survey_8d": spec.prefill_flops_per_token / 1e9,
                        "frac_with_survey_8d_flops": (flops_survey / (pf_ms * 1e-3) / 1e12 / tf_peak) if pf_ms > 0 else None},
            "launches_per_decode_step_or_chunk_mean": launches_per_step,
            "clocks": clocks, "init_s": init_s, "weight_broadcast_s": bcast_s,
        }
        # K1 (router kernel) is latency-bound, not roofline-bound (SURVEY 8d): report time per event of a full trace
        try:
            line["router"] = router_kernel_timing(router)
            line["router"]["us_per_event_single_launch"] = k1_single_event_latency(router)
        except Exception as ex:                                   # never lose the headline line over the side measurement
            line["router"] = {"error": repr(ex)}
        if world == 1 and not args.no_extras:
            for key, fn in (("per_request", lambda: per_request_leg(router, args.model, prompts_np, n_req, M)),
                            ("http", lambda: http_leg(router, args.model, prompts_np, n_req, M)),
                            ("kernels", lambda: kernel_table(eng, spec, prompts_np, C, P, M, hbm_peak))):
                try:
                    line[key] = fn()
                except Exception as ex:                           # noqa: BLE001
                    line[key] = {"error": repr(ex)}
        if world == 1 and not args.no_cpu_baseline:
            router.close()
            eng.close()
            v, sample, cores = cpu_port_sample(spec, P, M, C, world)
            line["cpu_baseline"] = {"value": v, "unit": "completions/s", "cores": cores, "kind": "port", "sample": sample}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def router_kernel_timing(router, n_events: int = 2048, reps: int = 5):
    """K1 alone: one launch over a trace of ADMIT + DONE pairs on the bench router (device buffers resident,
    CUDA events on the launch stream) and the same trace through the host entry point (H2D + launch + D2H + sync)."""
    import ctypes as C
    import torch
    from rr_b200 import _lib
    n_dep = len(router.cfg.deployments)
    now = router.now_ms()
    ev = (_lib.Event * n_events)()
    for i in range(0, n_events, 2):
        ev[i] = _lib.Event(0, 0, 512, 0, now)                    # ADMIT to group 0
        ev[i + 1] = _lib.Event(1, (i // 2) % n_dep, 128, 0, now)   # DONE on some deployment (keeps in-flight bounded)
    out = (_lib.Decision * n_events)()
    host = torch.frombuffer(bytearray(bytes(ev)), dtype=torch.uint8)
    d_ev = host.cuda()
    d_out = torch.empty(n_events * C.sizeof(_lib.Decision), dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream()
    def dev_once():
        _lib.check(_lib.lib.rr_router_process_device(router._h, C.c_void_p(d_ev.data_ptr()), n_events,
                                                     C.c_void_p(d_out.data_ptr()), C.c_void_p(stream.cuda_stream)))
    for _ in range(2):
        dev_once()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(reps):
        dev_once()
    e1.record(stream)
    torch.cuda.synchronize()
    dev_ns = e0.elapsed_time(e1) * 1e6 / (reps * n_events)
    t0 = time.perf_counter()
    for _ in range(reps):
        _lib.check(_lib.lib.rr_router_process(router._h, ev, n_events, out))
    host_ns = (time.perf_counter() - t0) * 1e9 / (reps * n_events)
    return {"events_per_launch": n_events, "ns_per_event_device": dev_ns, "events_per_s_device": 1e9 / dev_ns,
            "ns_per_event_host_api": host_ns, "bound": "latency (one warp walks the trace in order; lanes = candidate deployments)"}


# ------------------------------------------------------------------------------------------------
# BASELINE.json configs #2-#4: ONE process drives all --gpus devices through the native gateway (rr_gateway.cu), one
# engine (worker thread) per GPU -- the reference's deployment shape (one gateway process, bin/start-gateway.sh:54).
def fleet_plan(kind, n_gpus, C, P, M, steps):
    """-> (model_list, router settings, engines {gpu: (spec name, fail_prob)}, workload [(group name, n requests)], notes)."""
    if kind == "quota":
        # config #2: N replicas, 64 N concurrent requests, rpm/tpm buckets + three teams with separate groups
        # (reference config/config.yaml:74-94: one model group = one rpm bucket per consumer).  Team A asks for 25 % more than
        # its rpm admits.
        share = {"a": 3, "b": 3, "c": 2}                               # of every 8 GPUs / of every 512 requests
        total = C * n_gpus
        gpus = list(range(n_gpus))
        owned = {"a": [], "b": [], "c": []}
        for i, g in enumerate(gpus):
            owned["a" if i % 8 < 3 else ("b" if i % 8 < 6 else "c")].append(g)
        for t in owned:                                                 # fewer than 8 GPUs: teams share replicas
            if not owned[t]:
                owned[t] = [gpus[hash(t) % n_gpus]] if n_gpus > 1 else [0]
        n_team = {t: total * share[t] // 8 for t in share}
        ml = []
        for t in "abc":
            # rpm window must admit `steps + warmup` bursts: the bench gives each burst its own minute (manual clock)
            per_dep = -(-n_team[t] // len(owned[t]))
            rpm = per_dep if t != "a" else int(per_dep * 0.75)
            for g in owned[t]:
                ml.append({"model_name": f"team-{t}", "litellm_params": {"model": f"b200/llama-3-8b@team-{t}", "gpu": g},
                           "rpm": rpm, "tpm": rpm * (P + M) * 2})
        eng = {g: ("llama-3-8b", 0.0) for g in gpus}
        rs = {"routing_strategy": "simple-shuffle", "enable_pre_call_checks": True, "allowed_fails": 2, "cooldown_time": 15}
        work = [(f"team-{t}", n_team[t]) for t in "abc"]
        return ml, rs, eng, work, {"expect": "about 25 % of team-a's requests answer 429; teams b and c are untouched"}
    if kind == "fallback":
        # config #3: Llama-3-8B primary with a seeded 50 % failure mask, Phi-3-mini fallback (reference config.yaml:103-108)
        g1 = 1 if n_gpus > 1 else 0
        ml = [{"model_name": "primary", "litellm_params": {"model": "b200/llama-3-8b", "gpu": 0}},
              {"model_name": "fallback", "litellm_params": {"model": "b200/phi-3-mini", "gpu": g1 if n_gpus > 1 else 1}}]
        eng = {0: ("llama-3-8b", 0.5), (g1 if n_gpus > 1 else 1): ("phi-3-mini", 0.0)}
        rs = {"routing_strategy": "simple-shuffle", "enable_pre_call_checks": True, "allowed_fails": 1_000_000,
              "cooldown_time": 15, "fallbacks": [{"primary": ["fallback"]}]}
        return ml, rs, eng, [("primary", C * max(1, n_gpus // 2))], {"fail_prob": 0.5, "fail_seed": 42}
    # config #4: mixed fleet, Llama-3-8B on 3/4 of the GPUs, Mistral-7B on the rest; weighted simple-shuffle, every
    # deployment weight 1 => 3 : 1 between the fleets; 1 000-request soak, Poisson arrivals
    n_l = max(1, (3 * n_gpus) // 4) if n_gpus > 1 else 1
    ml, eng = [], {}
    for g in range(max(2, n_gpus)):
        is_l = g < n_l
        gpu = g if n_gpus > 1 else g                                  # n_gpus == 1: two engines on device 0 (see run_fleet)
        ml.append({"model_name": "chat", "litellm_params": {"model": "b200/" + ("llama-3-8b" if is_l else "mistral-7b"),
                                                             "gpu": gpu, "weight": 1}})
        eng[gpu] = ("llama-3-8b" if is_l else "mistral-7b", 0.0)
    rs = {"routing_strategy": "simple-shuffle", "enable_pre_call_checks": False, "allowed_fails": 2, "cooldown_time": 15}
    return ml, rs, eng, [("chat", 1000)], {"arrivals": "poisson"}


def run_fleet(args, kind):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return                                                          # one process drives every GPU
    import torch
    from rr_b200.models import resolve_spec, make_weights, Weights
    from rr_b200.engine import Engine
    from rr_b200.router import Router, EngineBackend, RateLimitError, APIError

    n_gpus = min(args.gpus, torch.cuda.device_count())
    C, P, M, K, W = args.concurrency, args.prompt_len, args.max_new, args.steps, args.warmup
    ml, rs, eng_plan, work, notes = fleet_plan(kind, n_gpus, C, P, M, K)
    ctx_max = ((P + M + 63) // 64) * 64
    t0 = time.perf_counter()
    base = {}                                                           # spec name -> weights on their first device
    engines, backends = {}, {}
    for replica, (name, fail_prob) in sorted(eng_plan.items()):
        dev = replica if replica < n_gpus else 0
        if name not in base:
            base[name] = make_weights(resolve_spec(name), seed=0, sigma=0.02, device=f"cuda:{dev}")
            w = base[name]
        else:
            w = base[name].to(f"cuda:{dev}") if str(base[name].embed.device) != f"cuda:{dev}" else base[name]
        engines[replica] = Engine(w, device=dev, max_batch=C, ctx_max=ctx_max, max_prefill_tokens=8192, use_cuda_graph=True,
                                  fail_prob=fail_prob, fail_seed=42)
        backends[replica] = EngineBackend(engines[replica])
    init_s = time.perf_counter() - t0
    now = [1_000_000.0]
    router = Router(model_list=ml, routing_strategy=rs["routing_strategy"], enable_pre_call_checks=rs["enable_pre_call_checks"],
                    allowed_fails=rs["allowed_fails"], cooldown_time=rs["cooldown_time"], fallbacks=rs.get("fallbacks"),
                    backends=backends, seed=0, clock=lambda: now[0])
    router.record_trace = 1 << 16
    vocab = router._vocab()
    n_max = max(n for _, n in work)
    prompts = make_prompts(n_max, P, vocab, pinned=True).numpy()
    for e in engines.values():
        e.reset_stats()

    def burst(collect, res):
        """All groups' requests issued together by one thread per group (completion_batch = one contiguous trace block)."""
        outs = {}

        def go(gname, n):
            outs[gname] = router.completion_batch(gname, [prompts[i] for i in range(n)], M, timeout=600)
        ths = [threading.Thread(target=go, args=w_) for w_ in work]
        for t in ths:
            t.start()
        for t in ths:
            t.join()
        if collect:
            for gname, out in outs.items():
                r = res.setdefault(gname, {"ok": 0, "rate_limited": 0, "failed": 0, "fell_back": 0, "ttft": [], "lat": [], "by_model": {}})
                for o in out:
                    if isinstance(o, RateLimitError):
                        r["rate_limited"] += 1
                    elif isinstance(o, Exception):
                        r["failed"] += 1
                    else:
                        assert len(o._token_ids) == M
                        r["ok"] += 1; r["fell_back"] += int(o._fell_back)
                        r["ttft"].append(o._ttft_s); r["lat"].append(o._latency_s)
                        r["by_model"][o.model] = r["by_model"].get(o.model, 0) + 1

    def soak(collect, res, n, rate):
        """Open loop: n requests with exponential inter-arrival times at `rate` req/s, one caller thread each."""
        rng = np.random.RandomState(7)
        gaps = rng.exponential(1.0 / rate, size=n)
        out = [None] * n

        def one(i):
            try:
                out[i] = router.completion(model="chat", prompt_ids=prompts[i], max_tokens=M, timeout=600)
            except Exception as e:                                      # noqa: BLE001
                out[i] = e
        ths = []
        t_next = time.perf_counter()
        for i in range(n):
            t_next += gaps[i]
            d = t_next - time.perf_counter()
            if d > 0:
                time.sleep(d)
            th = threading.Thread(target=one, args=(i,))
            th.start(); ths.append(th)
        for th in ths:
            th.join()
        if collect:
            r = res.setdefault("chat", {"ok": 0, "rate_limited": 0, "failed": 0, "fell_back": 0, "ttft": [], "lat": [], "by_model": {}})
            for o in out:
                if isinstance(o, Exception):
                    r["failed"] += 1
                else:
                    r["ok"] += 1; r["ttft"].append(o._ttft_s); r["lat"].append(o._latency_s)
                    r["by_model"][o.model] = r["by_model"].get(o.model, 0) + 1

    res = {}
    n_rep = len(engines)
    if kind == "fleet":
        cap = 70.0 * n_rep * (64.0 / C if C else 1.0)                   # completions/s the fleet sustains (closed-burst figure)
        rate = 0.8 * cap
        soak(False, res, min(200, 64 * n_rep), rate)                    # warm-up (graph capture, first prefill plans)
        for e in engines.values():
            e.reset_stats()
        router.snapshot()
        sampler = ClockSampler(0); sampler.start()
        torch.cuda.synchronize()
        t_start = time.perf_counter()
        soak(True, res, work[0][1], rate)
        wall = time.perf_counter() - t_start
        steps_done = 1
    else:
        for _ in range(W):
            now[0] += 60.0                                              # every burst gets a fresh rpm / tpm minute
            burst(False, res)
        for e in engines.values():
            e.reset_stats()
        router.snapshot()
        sampler = ClockSampler(0); sampler.start()
        torch.cuda.synchronize()
        t_start = time.perf_counter()
        for _ in range(K):
            now[0] += 60.0
            burst(True, res)
        wall = time.perf_counter() - t_start
        steps_done = K
    clocks = sampler.stop()
    snap = router.snapshot()
    gstats = router.gateway_stats()
    trace = router.gateway_trace()
    dev_ms = max((e.stats()["prefill_ms_total"] + e.stats()["decode_ms_total"]) for e in engines.values())
    launches = sum(e.stats()["kernel_launches"] for e in engines.values()) + gstats["launches"]
    total_ok = sum(r["ok"] for r in res.values())
    all_ttft = np.asarray([t for r in res.values() for t in r["ttft"]])
    line = {"metric": f"completions/sec & TTFT, BASELINE config '{kind}' ({P}-in/{M}-out)", "value": total_ok / (dev_ms / 1e3) if dev_ms else None,
            "unit": "completions/s", "n_gpus": n_gpus, "steps": steps_done, "warmup": W, "ms_per_step": dev_ms / max(1, steps_done),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": kind, "model_list": [(d["model_name"], d["litellm_params"]["model"], d["litellm_params"]["gpu"],
                                                          d.get("rpm"), d.get("tpm")) for d in ml],
                       "router_settings": rs, "requests_per_step": {g: n for g, n in work}, "notes": notes,
                       "process_layout": f"one process, {n_rep} engines on {n_gpus} GPU(s), native gateway"},
            "e2e": {"value": total_ok / wall, "unit": "completions/s", "wall_s": wall,
                    "api": "Router.completion_batch / Router.completion -> rr_gateway_* (host buffers)",
                    "h2d_bytes_per_step": int(sum(e.stats()["h2d_bytes"] for e in engines.values()) / max(1, steps_done)),
                    "d2h_bytes_per_step": int(sum(e.stats()["d2h_bytes"] for e in engines.values()) / max(1, steps_done))},
            "p50_ttft_ms": float(np.percentile(all_ttft, 50) * 1e3) if len(all_ttft) else None,
            "p99_ttft_ms": float(np.percentile(all_ttft, 99) * 1e3) if len(all_ttft) else None,
            "groups": {g: {"ok": r["ok"], "rate_limited": r["rate_limited"], "failed": r["failed"], "fell_back": r["fell_back"],
                           "by_model": r["by_model"],
                           "p50_ttft_ms": float(np.percentile(r["ttft"], 50) * 1e3) if r["ttft"] else None,
                           "p99_ttft_ms": float(np.percentile(r["ttft"], 99) * 1e3) if r["ttft"] else None} for g, r in res.items()},
            "gateway": gstats, "gpu_launches": int(launches),
            "deployments": [{"model": d.response_model, "gpu": d.gpu, "total_admitted": s["total_admitted"], "fail_count": s["fail_count"],
                             "inflight": s["inflight"]} for d, s in zip(router.cfg.deployments, snap)],
            "decode_ms_per_step": {str(g): (e.stats()["decode_ms_total"] / max(1, e.stats()["decode_steps"])) for g, e in engines.items()},
            "clocks": clocks, "init_s": init_s}
    if args.trace_out:
        with open(args.trace_out, "w") as f:
            json.dump({"kind": kind, "seed": 0, "model_list": ml, "router_settings": rs,
                       "trace": [[list(e), list(d)] for e, d in trace]}, f)
        line["trace_file"] = args.trace_out
    router.close()
    for e in engines.values():
        e.close()
    if not args.no_cpu_baseline:
        # checker + CPU baseline of the ROUTER path on the recorded trace: the oracle replays every event; decisions must be
        # bit-exact with what K1 decided on the device
        from oracle import router as O
        from rr_b200.config import build_config
        cfg = build_config(ml, rs)
        deps = [O.Deployment(d.group, rpm=d.rpm, tpm=d.tpm, weight=d.weight) for d in cfg.deployments]
        orc = O.OracleRouter(deps, len(cfg.groups), dict(cfg.fallbacks),
                             O.Settings(strategy=cfg.strategy_id, enable_pre_call_checks=cfg.enable_pre_call_checks,
                                        allowed_fails=cfg.allowed_fails, cooldown_ms=int(round(cfg.cooldown_time * 1000))), seed=0)
        t0 = time.perf_counter()
        want = orc.process([O.Event(*e) for e, _ in trace])
        dt = time.perf_counter() - t0
        n_adm = sum(1 for e, _ in trace if e[0] == 0)
        exact = all(w_.as_tuple() == tuple(d) for w_, (e, d) in zip(want, trace) if e[0] == 0)
        line["cpu_baseline"] = {"value": n_adm / dt if dt > 0 else None, "unit": "admissions/s", "cores": 1, "kind": "port",
                                "sample": f"oracle/router.py replay of the {len(trace)} recorded events ({n_adm} admissions) of this run",
                                "decisions_bit_exact": bool(exact), "trace_complete": len(trace) == gstats["events"]}
        assert exact, "K1 decisions differ from the oracle on the recorded trace"
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
