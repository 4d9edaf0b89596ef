"""Parity of the engine (prefill + decode through the C-ABI) against the generated-token oracle.

Stated tolerance (north_star: "within a stated fp16 logit tolerance"): the engine rounds activations to
bf16 at every GEMM input and keeps an fp32 residual; the oracle is fp32 on the same bf16 weights.
Per position, with d = logit_engine - logit_oracle and s = std(oracle logits over the vocabulary):
rms(d) <= TOL_RMS * s and max|d| <= TOL_MAX * s, TOL_RMS = 0.02, TOL_MAX = 0.08 for <= 4 layers
(the 32-layer bound is stated in tests/test_full_model_gpu.py), and the engine's argmax equals the
oracle's wherever the oracle's top-2 margin exceeds 2 * TOL_MAX * s."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden", "llama_tiny_golden.pt")
TOL_RMS, TOL_MAX = 0.02, 0.08


def _cmp(got, ref, what):
    ref = ref.float().cpu()
    got = torch.as_tensor(got).float().cpu()
    std = ref.std().item()
    d = got - ref
    err, rms = d.abs().max().item(), d.pow(2).mean().sqrt().item()
    assert torch.isfinite(got).all(), what
    assert rms <= TOL_RMS * std and err <= TOL_MAX * std, (what, rms / std, err / std)
    top2 = ref.topk(2).values
    if (top2[0] - top2[1]).item() > 2 * TOL_MAX * std:
        assert int(got.argmax()) == int(ref.argmax()), what
    return rms / std


def test_engine_matches_hf_golden_tiny():
    from rr_b200.models import SPECS, make_weights
    from rr_b200.engine import Engine
    g = torch.load(GOLD)
    w = make_weights(SPECS["tiny"], seed=g["seed"], sigma=g["sigma"], device="cpu", norm_jitter=g["norm_jitter"])
    chk = float(sum(t.float().abs().sum() for t in w.tensors()))
    assert abs(chk - g["weight_checksum"]) < 1e-3 * g["weight_checksum"]
    eng = Engine(w.to("cuda"), max_batch=8, ctx_max=512, max_prefill_tokens=1024, use_cuda_graph=False)
    try:
        prompts = g["prompts"]
        slots = [3, 0, 7, 1, 5, 2]
        first, logits = eng.prefill(prompts, slots, want_logits=True)
        worst = 0.0
        for i, p in enumerate(prompts):
            worst = max(worst, _cmp(logits[i], g["logits"][i][0], f"prefill len={len(p)}"))
        # teacher-forced decode: feed the oracle's tokens, compare each step's logits
        steps = len(g["tokens"][0]) - 1
        for j in range(steps):
            toks = [g["tokens"][i][j] for i in range(len(prompts))]
            pos = [len(p) + j for p in prompts]
            nxt, lg = eng.decode_step(slots, toks, pos, want_logits=True)
            for i in range(len(prompts)):
                worst = max(worst, _cmp(lg[i], g["logits"][i][j + 1], f"decode step {j} seq {i}"))
        print(f"\n[tiny vs HF golden] worst rms(dlogit)/std = {worst:.4f}")
    finally:
        eng.close()


def test_engine_matches_hf_mistral_and_phi3_golden():
    """Engine logits against the REAL transformers MistralForCausalLM / Phi3ForCausalLM outputs committed in
    tests/golden/family_golden.pt (no oracle in between): GQA group size 2 on the tcgen05 attention path, and
    MHA with head_dim 96 on the mma.sync path with the fused-projection layout HF Phi-3 uses."""
    from test_oracle_llama import family_cases          # tests/ is on sys.path (pytest rootdir/conftest)
    from rr_b200.engine import Engine
    for fam, spec, w_cpu, prompts, logits, tokens in family_cases():
        w = w_cpu.to("cuda")
        eng = Engine(w, max_batch=8, ctx_max=256, max_prefill_tokens=512, use_cuda_graph=False)
        try:
            first, lg = eng.prefill(prompts, list(range(len(prompts))), want_logits=True)
            for i, p in enumerate(prompts):
                _cmp(lg[i], logits[i][0], f"{fam} prefill len={len(p)}")
            # one teacher-forced decode step on HF's own first token
            cur = [tk[0] for tk in tokens]
            pos = [len(p) for p in prompts]
            nxt, lg2 = eng.decode_step(list(range(len(prompts))), cur, pos, want_logits=True)
            for i in range(len(prompts)):
                _cmp(lg2[i], logits[i][1], f"{fam} decode seq {i}")
        finally:
            eng.close()


@pytest.mark.parametrize("spec_name,max_batch", [("small", 16), ("small", 64), ("llama-3-8b-2l", 64), ("tiny96", 8),
                                                 ("small96", 32), ("phi-3-mini-2l", 64), ("mistral-7b-2l", 64),
                                                 # 128 / 256 decode rows: the BN = 128 / 256 instances of the decode
                                                 # GEMMs and of the fused MLP kernel
                                                 ("small", 128), ("small", 256)])
def test_engine_matches_oracle(spec_name, max_batch):
    from oracle import llama_ref
    from rr_b200.models import SPECS, make_weights
    from rr_b200.engine import Engine
    spec = SPECS[spec_name]
    w = make_weights(spec, seed=3, sigma=0.03 if spec.hidden < 2048 else 0.02, device="cuda", norm_jitter=0.1)
    eng = Engine(w, max_batch=max_batch, ctx_max=640, max_prefill_tokens=2048, use_cuda_graph=False)
    try:
        g = torch.Generator().manual_seed(5)
        lens = [3, 64, 129, 300, 512]
        prompts = [torch.randint(0, spec.vocab, (n,), generator=g).tolist() for n in lens]
        slots = [max_batch - 1, 0, 5, 2, 3]
        first, logits = eng.prefill(prompts, slots, want_logits=True)
        refs = [llama_ref.forward_logits(w, p)[-1] for p in prompts]
        worst = max(_cmp(logits[i], refs[i], f"prefill {spec_name} len={lens[i]}") for i in range(len(lens)))
        # 3 free-running decode steps, checked teacher-forced against the oracle on the engine's own tokens
        toks = [list(p) for p in prompts]
        cur = [int(t) for t in first]
        for j in range(3):
            pos = [len(t) for t in toks]
            for t, c in zip(toks, cur):
                t.append(c)
            nxt, lg = eng.decode_step(slots, cur, pos, want_logits=True)
            for i in range(len(lens)):
                ref = llama_ref.forward_logits(w, toks[i])[-1]
                worst = max(worst, _cmp(lg[i], ref, f"decode {spec_name} step {j} seq {i}"))
            cur = [int(t) for t in nxt]
        print(f"\n[{spec_name} B={max_batch}] worst rms(dlogit)/std = {worst:.4f}")
    finally:
        eng.close()


def test_serving_loop_equals_stepwise_and_is_deterministic():
    """submit/wait (continuous batching, CUDA graph) must produce exactly the tokens of the
    synchronous prefill + decode_step path (same kernels, same order of arithmetic)."""
    from rr_b200.models import SPECS, make_weights
    from rr_b200.engine import Engine
    spec = SPECS["small"]
    w = make_weights(spec, seed=11, sigma=0.03, device="cuda", norm_jitter=0.1)
    g = torch.Generator().manual_seed(9)
    lens = [5, 40, 64, 100, 17, 256, 33, 8, 90, 300, 12, 64]
    new = [4, 9, 1, 12, 7, 5, 16, 3, 2, 8, 10, 6]
    prompts = [torch.randint(0, spec.vocab, (n,), generator=g).tolist() for n in lens]
    eng = Engine(w, max_batch=4, ctx_max=512, max_prefill_tokens=512, use_cuda_graph=True)   # forces queueing
    try:
        tickets = [eng.submit(p, m) for p, m in zip(prompts, new)]
        recs = [eng.wait(t, timeout=120) for t in tickets]
        assert all(r.status == 0 for r in recs)
        assert [len(r.tokens) for r in recs] == new
        assert all(r.t_submit <= r.t_first_token <= r.t_done for r in recs)
        # second pass: identical tokens (deterministic kernels)
        tickets = [eng.submit(p, m) for p, m in zip(prompts, new)]
        recs2 = [eng.wait(t, timeout=120) for t in tickets]
        assert [r.tokens for r in recs2] == [r.tokens for r in recs]
        st = eng.stats()
        assert st["kernel_launches"] > 0 and st["generated_tokens"] == 2 * sum(new)
        # stepwise reference on the same engine
        for i in [0, 3, 6, 9]:
            first, _ = eng.prefill([prompts[i]], [2])
            out = [int(first[0])]
            pos = lens[i]
            while len(out) < new[i]:
                nxt, _ = eng.decode_step([2], [out[-1]], [pos])
                out.append(int(nxt[0])); pos += 1
            assert out == recs[i].tokens, i
    finally:
        eng.close()


@pytest.mark.parametrize("spec_name,rows", [("small", 64), ("llama-3-8b-2l", 64), ("llama-3-8b-2l", 24)])
def test_decode_work_distribution_and_epilogue_switches_do_not_change_tokens(spec_name, rows, monkeypatch):
    """The fused decode MLP deals its down items dynamically (device counter) and the decode GEMMs store their tiles by TMA;
    which CTA computes an item, and through which store path a tile leaves, must not change a single generated token:
    same tokens as the static host schedule (RR_MLP_STATIC) and as the per-thread store epilogues (RR_NO_TMA_EPI)."""
    import numpy as np
    from rr_b200.models import SPECS, make_weights
    from rr_b200.engine import Engine
    spec = SPECS[spec_name]
    w = make_weights(spec, seed=5, sigma=0.03, device="cuda", norm_jitter=0.1)
    rng = np.random.RandomState(3)
    ids = rng.randint(0, spec.vocab, size=(rows, 96)).astype(np.int32)
    start = np.arange(0, rows * 96 + 1, 96, dtype=np.int32)

    def run(env):
        for k in ("RR_MLP_STATIC", "RR_NO_TMA_EPI"):
            monkeypatch.delenv(k, raising=False)
        for k in env:
            monkeypatch.setenv(k, "1")
        eng = Engine(w, max_batch=64, ctx_max=256, max_prefill_tokens=2048, use_cuda_graph=True)
        try:
            recs, toks = eng.run_batch(ids.reshape(-1), start, 12)
            assert all(r.status == 0 for r in recs)
            return toks.copy()
        finally:
            eng.close()

    base = run([])
    assert np.array_equal(base, run([])), "two default engines disagree (non-deterministic kernels?)"
    assert np.array_equal(base, run(["RR_MLP_STATIC"]))
    assert np.array_equal(base, run(["RR_NO_TMA_EPI"]))


def test_run_batch_and_fault_injection():
    from rr_b200.models import SPECS, make_weights
    from rr_b200.engine import Engine
    spec = SPECS["tiny"]
    w = make_weights(spec, seed=1, sigma=0.05, device="cuda")
    eng = Engine(w, max_batch=8, ctx_max=256, max_prefill_tokens=512, fail_prob=0.5, fail_seed=42)
    try:
        n = 40
        ids = np.random.RandomState(0).randint(0, spec.vocab, size=(n, 16)).astype(np.int32)
        start = np.arange(0, n * 16 + 1, 16, dtype=np.int32)
        recs, toks = eng.run_batch(ids.reshape(-1), start, 5)
        failed = [r.status == 7 for r in recs]
        assert 8 <= sum(failed) <= 32                      # Bernoulli(0.5), seeded
        assert all(len(r.tokens) == (0 if f else 5) for r, f in zip(recs, failed))
        recs2, _ = eng.run_batch(ids.reshape(-1), start, 5)
        ok1 = [r.tokens for r in recs if r.status == 0]
        assert len(ok1) > 0
    finally:
        eng.close()


def test_separate_norm_kernels_prefill_option_matches_oracle():
    """The default prefill defers RMSNorm into the GEMM epilogues (residual epilogues emit bf16(x * gamma) and sum(x^2),
    the next GEMM's epilogue applies 1 / rms; RopeEpi in csrc/rr_kernels.h) -- every other test here runs that path.
    This one covers the fallback with two norm kernels per layer (defer_norm=False).  Same tolerance."""
    from oracle import llama_ref
    from rr_b200.models import SPECS, make_weights
    from rr_b200.engine import Engine
    for name in ("small", "small96"):                     # fused-RoPE epilogue / bf16 epilogue + rope kernel
        spec = SPECS[name]
        w = make_weights(spec, seed=3, sigma=0.03, device="cuda", norm_jitter=0.1)
        eng = Engine(w, max_batch=16, ctx_max=640, max_prefill_tokens=2048, use_cuda_graph=False, defer_norm=False)
        try:
            g = torch.Generator().manual_seed(5)
            lens = [3, 64, 129, 300, 512]
            prompts = [torch.randint(0, spec.vocab, (n,), generator=g).tolist() for n in lens]
            first, logits = eng.prefill(prompts, [15, 0, 5, 2, 3], want_logits=True)
            for i, p in enumerate(prompts):
                _cmp(logits[i], llama_ref.forward_logits(w, p)[-1], f"separate-norm prefill {name} len={lens[i]}")
        finally:
            eng.close()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs in one process")
def test_two_replicas_in_one_process_agree():
    """The HTTP gateway hosts one engine per GPU inside a single process: kernel attributes (dynamic shared memory
    limits), SM counts and TMA maps must be set up per device.  Both replicas serve the same prompts concurrently
    and must emit identical tokens (same weights, deterministic kernels)."""
    from rr_b200.models import SPECS, make_weights
    from rr_b200.engine import Engine
    spec = SPECS["small"]
    g = torch.Generator().manual_seed(21)
    prompts = [torch.randint(0, spec.vocab, (n,), generator=g).tolist() for n in (300, 64, 129, 17, 512, 255)]
    engines = []
    try:
        for dev in (1, 0):           # the second device first: nothing may depend on "device 0 went first"
            w = make_weights(spec, seed=5, sigma=0.03, device=f"cuda:{dev}", norm_jitter=0.1)
            engines.append(Engine(w, device=dev, max_batch=8, ctx_max=640, max_prefill_tokens=1024))
        tickets = [[e.submit(p, 12) for p in prompts] for e in engines]
        outs = [[e.wait(t, timeout=120) for t in ts] for e, ts in zip(engines, tickets)]
        assert all(r.status == 0 and len(r.tokens) == 12 for rs in outs for r in rs)
        assert [r.tokens for r in outs[0]] == [r.tokens for r in outs[1]]
    finally:
        for e in engines:
            e.close()


def test_generation_up_to_the_last_kv_slot_and_argument_bounds():
    """Maximum sizes: prompt + max_new == ctx_max fills the KV slot to its last row (decode position ctx_max - 1);
    one token more is rejected at submit, as are empty prompts and out-of-vocabulary ids."""
    from oracle import llama_ref
    from rr_b200 import _lib
    from rr_b200.models import SPECS, make_weights
    from rr_b200.engine import Engine
    spec = SPECS["tiny"]
    w = make_weights(spec, seed=9, sigma=0.05, device="cuda", norm_jitter=0.1)
    eng = Engine(w, max_batch=4, ctx_max=128, max_prefill_tokens=256)
    try:
        g = torch.Generator().manual_seed(2)
        prompt = torch.randint(0, spec.vocab, (100,), generator=g).tolist()
        rec = eng.wait(eng.submit(prompt, 28), timeout=60)              # 100 + 28 == ctx_max
        assert rec.status == 0 and len(rec.tokens) == 28
        # teacher-forced check of the LAST step (reads all 127 earlier rows, writes row 127)
        ref = llama_ref.forward_logits(w, prompt + rec.tokens[:-1])[-1]
        std = ref.std().item()
        top2 = ref.topk(2).values
        if (top2[0] - top2[1]).item() > 2 * TOL_MAX * std:
            assert rec.tokens[-1] == int(ref.argmax())
        with pytest.raises(Exception):
            eng.submit(prompt, 29)                                       # would need row 128
        with pytest.raises(Exception):
            eng.submit([], 4)
        with pytest.raises(Exception):
            eng.submit([spec.vocab], 4)
        # a second full-length request reuses the slot: same tokens (deterministic, no stale state)
        rec2 = eng.wait(eng.submit(prompt, 28), timeout=60)
        assert rec2.tokens == rec.tokens
    finally:
        eng.close()


def test_long_prompts_match_oracle():
    """3000- and 1500-token prompts in one prefill chunk (47 / 24 key tiles per query tile in the tcgen05 attention
    kernel, deep online-softmax chains), then decode steps at context ~3000 (47 K/V tiles per row in the decode
    attention kernel)."""
    from oracle import llama_ref
    from rr_b200.models import SPECS, make_weights
    from rr_b200.engine import Engine
    spec = SPECS["small"]
    w = make_weights(spec, seed=13, sigma=0.03, device="cuda", norm_jitter=0.1)
    eng = Engine(w, max_batch=4, ctx_max=3072, max_prefill_tokens=4608, use_cuda_graph=False)
    try:
        g = torch.Generator().manual_seed(8)
        lens = [3000, 1500]
        prompts = [torch.randint(0, spec.vocab, (n,), generator=g).tolist() for n in lens]
        first, logits = eng.prefill(prompts, [1, 3], want_logits=True)
        w_cpu = w.to("cpu")
        for i, p in enumerate(prompts):
            _cmp(logits[i], llama_ref.forward_logits(w_cpu, p)[-1], f"long prefill len={lens[i]}")
        toks = [list(p) for p in prompts]
        cur = [int(t) for t in first]
        for j in range(2):
            pos = [len(t) for t in toks]
            for t, c in zip(toks, cur):
                t.append(c)
            nxt, lg = eng.decode_step([1, 3], cur, pos, want_logits=True)
            for i in range(2):
                _cmp(lg[i], llama_ref.forward_logits(w_cpu, toks[i])[-1], f"long decode step {j} seq {i}")
            cur = [int(t) for t in nxt]
    finally:
        eng.close()


def test_two_engines_on_one_device_run_concurrently():
    """Two engines that share a GPU (e.g. two model groups mapped to one device through the C-ABI) serve at the same
    time from their own worker threads.  Their persistent kernels (fused MLP: CTAs spin on sibling CTAs' tiles) must
    never be interleaved on the device -- the library alternates them per prefill chunk / decode step."""
    from rr_b200.models import SPECS, make_weights
    from rr_b200.engine import Engine
    spec = SPECS["small"]
    w = make_weights(spec, seed=17, sigma=0.03, device="cuda", norm_jitter=0.1)
    g = torch.Generator().manual_seed(3)
    prompts = [torch.randint(0, spec.vocab, (n,), generator=g).tolist() for n in (200, 64, 31, 400, 129, 257)]
    engines = [Engine(w, max_batch=32, ctx_max=640, max_prefill_tokens=1024) for _ in range(2)]
    try:
        tickets = [[e.submit(p, 24) for p in prompts] for e in engines]         # both workers busy at once
        outs = [[e.wait(t, timeout=120) for t in ts] for e, ts in zip(engines, tickets)]
        assert all(r.status == 0 and len(r.tokens) == 24 for rs in outs for r in rs)
        assert [r.tokens for r in outs[0]] == [r.tokens for r in outs[1]]
    finally:
        for e in engines:
            e.close()
