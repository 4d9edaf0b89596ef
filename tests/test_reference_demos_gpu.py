"""GPU: the request streams of the reference's three gateway demos -- recorded from the UNMODIFIED scripts by
tests/golden/make_demo_golden.py into tests/golden/reference_demo_requests.json -- replayed over HTTP with the OpenAI SDK
(the reference's client boundary, src/demo_load_balancing.py:24,106-110) against the real gateway: K1 router kernel +
config/config.yaml, with mock-completion backends and with tiny real replicas.  Outcomes are the reference README's
(README.md:167-171: 3 primary + 7 fallback; :206-213: 3 + 3 + 4; :262-264: A 3/5, B 5/5, C 5/5)."""
import json
import os
import threading
import time

import pytest

pytestmark = [pytest.mark.gpu, pytest.mark.usefixtures("rpm_window")]
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CFG = os.path.join(ROOT, "config", "config.yaml")
GOLD = os.path.join(ROOT, "tests", "golden", "reference_demo_requests.json")


def _serve(router):
    import socket
    import uvicorn
    from rr_b200.server import create_app
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    server = uvicorn.Server(uvicorn.Config(create_app(router), host="127.0.0.1", port=port, log_level="error"))
    th = threading.Thread(target=server.run, daemon=True)
    th.start()
    for _ in range(200):
        if server.started:
            break
        time.sleep(0.05)
    return server, th, port


def _replay(port, reqs, stagger, client_per_request):
    """One thread per request like the demos' dispatch loops (src/demo_fallback.py:212-220, demo_quota_isolation.py:135-139)."""
    import openai
    shared = openai.OpenAI(api_key="demo-key", base_url=f"http://127.0.0.1:{port}")
    out = [None] * len(reqs)

    def work(i, r):
        c = openai.OpenAI(api_key=f"key-{i}", base_url=f"http://127.0.0.1:{port}") if client_per_request else shared
        try:
            resp = c.chat.completions.create(model=r["model"], messages=[{"role": "user", "content": r["content"]}], timeout=30)
            out[i] = getattr(resp, "model", "unknown")
        except openai.RateLimitError:
            out[i] = 429
        except Exception as e:                                      # noqa: BLE001
            out[i] = e
    ths = []
    for i, r in enumerate(reqs):
        t = threading.Thread(target=work, args=(i, r))
        t.start(); ths.append(t)
        if stagger:
            time.sleep(stagger)
    for t in ths:
        t.join()
    return out


def _backends(real):
    from rr_b200 import StubBackend
    if not real:
        return {0: StubBackend(), 1: StubBackend()}, []
    from rr_b200 import Engine, EngineBackend, SPECS, make_weights
    w = make_weights(SPECS["tiny"], seed=2, sigma=0.05, device="cuda")
    engs = [Engine(w, max_batch=16, ctx_max=256, max_prefill_tokens=512) for _ in range(2)]   # replicas 0 and 1, one device
    return {0: EngineBackend(engs[0]), 1: EngineBackend(engs[1])}, engs


@pytest.mark.parametrize("real", [False, True], ids=["stub-backends", "tiny-replicas"])
def test_recorded_reference_demo_requests_over_http(real):
    from rr_b200 import Router, load_config
    with open(GOLD) as f:
        gold = json.load(f)
    for demo, stagger, per_req in (("demo_fallback", 0.05, False), ("demo_load_balancing", 0.1, False),
                                   ("demo_quota_isolation", 0.0, True)):
        backends, engs = _backends(real)
        r = Router(config=load_config(CFG), backends=backends, seed=0, default_max_tokens=8)
        server, th, port = _serve(r)
        try:
            got = _replay(port, gold[demo], stagger, per_req)
            assert not [g for g in got if isinstance(g, Exception)], got
            if demo == "demo_fallback":
                fb = [g for g in got if g != 429 and "3-5-sonnet" in g]
                assert len(got) == 10 and 429 not in got and len(fb) == 7 and len(got) - len(fb) == 3
            elif demo == "demo_load_balancing":
                dist = {}
                for g in got:
                    dist[g] = dist.get(g, 0) + 1
                assert 429 not in dist and sorted(dist.values()) == [3, 3, 4]
                assert dist["llama-3-8b@claude-3-5-sonnet"] == 4               # the overflow lands on the fallback group
            else:
                by = {}
                for req, g in zip(gold[demo], got):
                    ok, lim = by.get(req["model"], (0, 0))
                    by[req["model"]] = (ok + (g != 429), lim + (g == 429))
                assert by == {"consumer-a-model": (3, 2), "consumer-b-model": (5, 0), "consumer-c-model": (5, 0)}
            snap = r.snapshot()
            assert sum(s["inflight"] for s in snap) == 0
        finally:
            server.should_exit = True
            th.join(10)
            r.close()
            for e in engs:
                e.close()
