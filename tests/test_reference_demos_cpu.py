"""CPU: the traffic of the reference's three gateway demo scripts (reference src/demo_fallback.py,
src/demo_load_balancing.py, src/demo_quota_isolation.py) against this repo's HTTP gateway
(sample-resilient-llm-inference_b200/server.py), sent with the OpenAI SDK the scripts use.

The router kernel needs a GPU, so a RECORDING DOUBLE sits behind server.py (first-fit over the config's rpm limits -- a
test double, not the product and not the oracle): what this proves is the wire contract -- the scripts' OpenAI-SDK calls
are served, `.model` / HTTP 429 are understood by their exception handling, and their end-of-run tables come out with the
README's counts (reference README.md:167-171, 206-213, 262-264).

tests/golden/make_demo_golden.py ran the UNMODIFIED scripts against this gateway and stored in
tests/golden/reference_demo_wire.json every request they sent (SDK retries included), what the double answered, and the
figures the scripts printed at the end.  This test issues the same calls the way the scripts issue them (one thread per
request, their stagger and timeout, a shared client or one client per request, the SDK's default retries) and checks that
the gateway receives the same requests, answers them the same way, and that the scripts' own tallying of the responses
gives the recorded figures.  tests/test_reference_demos_gpu.py replays the distinct requests
(tests/golden/reference_demo_requests.json) against the real K1-backed gateway on the B200."""
import json
import os
import socket
import threading
import time
from collections import Counter

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CFG = os.path.join(ROOT, "config", "config.yaml")
WIRE = os.path.join(ROOT, "tests", "golden", "reference_demo_wire.json")
GOLD = os.path.join(ROOT, "tests", "golden", "reference_demo_requests.json")

# how each script issues its requests: seconds between thread starts, one OpenAI client per request, request timeout
# (src/demo_fallback.py:28,146,216; src/demo_load_balancing.py:24,109,199; src/demo_quota_isolation.py:42,55,135)
CALLS = {"demo_fallback": (0.05, False, 30), "demo_load_balancing": (0.1, False, 30), "demo_quota_isolation": (0.0, True, 10)}


class RecordingDouble:
    """First-fit admission over the YAML's rpm limits + fallbacks; records every request and its answer."""

    def __init__(self, cfg):
        from rr_b200.router import Choice, Message, ModelResponse, RateLimitError, BadRequestError, Usage
        self.cfg, self.used, self.log, self.lock = cfg, [0] * len(cfg.deployments), [], threading.Lock()
        self._t = (Choice, Message, ModelResponse, RateLimitError, BadRequestError, Usage)

    def _admit(self, model):
        g = self.cfg.group_index(model)
        if g < 0:
            return 400
        for grp in [g] + self.cfg.fallbacks.get(g, []):
            for d in self.cfg.deployments:
                if d.group == grp and (d.rpm < 0 or self.used[d.index] < d.rpm):
                    self.used[d.index] += 1
                    return d.response_model
        return 429

    def completion(self, model, messages, timeout=None, max_tokens=None):
        Choice, Message, ModelResponse, RateLimitError, BadRequestError, Usage = self._t
        with self.lock:
            outcome = self._admit(model)
            self.log.append({"model": model, "messages": messages, "outcome": outcome})
        if outcome == 400:
            raise BadRequestError(f"Invalid model name passed in model={model}")
        if outcome == 429:
            raise RateLimitError(f"No deployments available for selected model, passed model={model}")
        return ModelResponse("chatcmpl-double", outcome, [Choice(0, Message("assistant", "ok"))], Usage(8, 2, 10))

    def snapshot(self):
        return []


def serve_double(host="127.0.0.1"):
    """server.py in front of a fresh RecordingDouble on a free port -> (double, uvicorn server, thread, port)."""
    import uvicorn
    from rr_b200.config import load_config
    from rr_b200.server import create_app
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    dbl = RecordingDouble(load_config(CFG))
    server = uvicorn.Server(uvicorn.Config(create_app(dbl), host=host, port=port, log_level="error"))
    th = threading.Thread(target=server.run, daemon=True)
    th.start()
    for _ in range(200):
        if server.started:
            break
        time.sleep(0.05)
    return dbl, server, th, port


def tally(demo, calls, got):
    """The end-of-run figures of a demo script, counted its way from the responses (`.model`, or 429 / another error)."""
    ok = [g for g in got if isinstance(g, str)]
    if demo == "demo_fallback":                                     # src/demo_fallback.py:154,227-230
        fb = sum("sonnet-3-5" in g.lower() or "3-5-sonnet" in g.lower() for g in ok)
        return {"total": len(got), "successful": len(ok), "failed": len(got) - len(ok), "primary": len(ok) - fb, "fallback": fb}
    if demo == "demo_load_balancing":                               # src/demo_load_balancing.py:192,210-222
        return {"total": len(got), "successful": len(ok), "failed": len(got) - len(ok), "distribution": dict(Counter(ok))}
    rows = {}                                                       # src/demo_quota_isolation.py:241-243
    for c, g in zip(calls, got):
        r = rows.setdefault(c["model"].split("-")[1].upper(), [0, 0, 0, 0])   # consumer-a-model -> A
        r[0] += 1; r[1] += isinstance(g, str); r[2] += not isinstance(g, str); r[3] += g == 429
    return {"rows": rows}


def distinct_calls(wire):
    """The client calls behind a recorded request stream: SDK retries folded, first-arrival order."""
    seen, out = set(), []
    for r in wire:
        key = (r["model"], json.dumps(r["messages"]))
        if key not in seen:
            seen.add(key); out.append({"model": r["model"], "messages": r["messages"]})
    return out


def _replay(port, calls, stagger, per_request, timeout):
    import openai
    shared = openai.OpenAI(api_key="demo-key", base_url=f"http://127.0.0.1:{port}")
    got = [None] * len(calls)

    def work(i, c):
        client = openai.OpenAI(api_key=f"key-{i}", base_url=f"http://127.0.0.1:{port}") if per_request else shared
        try:
            got[i] = getattr(client.chat.completions.create(model=c["model"], messages=c["messages"], timeout=timeout), "model", "unknown")
        except openai.RateLimitError:
            got[i] = 429
        except Exception as e:                                      # noqa: BLE001  (a failed request, as the scripts count it)
            got[i] = repr(e)
    ths = []
    for i, c in enumerate(calls):
        t = threading.Thread(target=work, args=(i, c))
        t.start(); ths.append(t)
        if stagger:
            time.sleep(stagger)
    for t in ths:
        t.join()
    return got


def test_recorded_reference_demo_traffic_against_this_gateway():
    with open(WIRE) as f:
        rec = json.load(f)
    assert sorted(rec) == sorted(CALLS)
    # the scripts' recorded end-of-run figures are the README's
    assert rec["demo_fallback"]["printed"] == {"total": 10, "successful": 10, "failed": 0, "primary": 3, "fallback": 7}
    lb = rec["demo_load_balancing"]["printed"]
    assert lb["total"] == lb["successful"] == 10 and sorted(lb["distribution"].values()) == [3, 3, 4]
    assert rec["demo_quota_isolation"]["printed"] == {"rows": {"A": [5, 3, 2, 2], "B": [5, 5, 0, 0], "C": [5, 5, 0, 0]}}
    for demo, (stagger, per_request, timeout) in CALLS.items():
        wire = rec[demo]["wire"]
        calls = distinct_calls(wire)
        # every call has the shape SURVEY.md 8b states: model (group name), one user message
        assert all(len(c["messages"]) == 1 and c["messages"][0]["role"] == "user" for c in calls)
        dbl, server, th, port = serve_double()
        try:
            got = _replay(port, calls, stagger, per_request, timeout)
        finally:
            server.should_exit = True
            th.join(10)
        assert tally(demo, calls, got) == rec[demo]["printed"], (demo, got)
        # the same requests reached the gateway, as often per model group (SDK retries included: a 429 is retried twice,
        # so team A's two rejected requests arrive three times each; which two lose the race differs from run to run), and
        # were answered the same way
        assert sorted(map(json.dumps, distinct_calls(dbl.log))) == sorted(map(json.dumps, calls)), demo
        assert Counter(r["model"] for r in dbl.log) == Counter(r["model"] for r in wire), demo
        answers = lambda log: Counter((r["model"], r["outcome"]) for r in log)
        assert answers(dbl.log) == answers(wire), demo
    assert Counter(r["model"] for r in rec["demo_quota_isolation"]["wire"]) == {"consumer-a-model": 9, "consumer-b-model": 5,
                                                                                "consumer-c-model": 5}
    assert Counter(r["outcome"] for r in rec["demo_quota_isolation"]["wire"])[429] == 6
    # the GPU replay's fixture holds exactly the distinct requests of the recorded streams
    with open(GOLD) as f:
        gold = json.load(f)
    key = lambda lst: sorted((r["model"], r["content"]) for r in lst)
    assert {k: key(v) for k, v in gold.items()} == \
        {k: key([{"model": c["model"], "content": c["messages"][0]["content"]} for c in distinct_calls(r["wire"])])
         for k, r in rec.items()}
