"""Generate tests/golden/reference_demo_wire.json and tests/golden/reference_demo_requests.json: the reference's three
gateway demo scripts, UNMODIFIED, run as subprocesses against this repo's HTTP gateway (server.py in front of the
recording double of tests/test_reference_demos_cpu.py), from a directory holding ./config/config.yaml as the scripts
expect (reference src/demo_fallback.py:16, src/demo_load_balancing.py:20, src/demo_quota_isolation.py:19).
    python tests/golden/make_demo_golden.py <checkout of aws-samples/sample-resilient-llm-inference>
Per demo the fixture holds every request the gateway received in arrival order (model, messages, the double's answer)
and the end-of-run figures the script printed."""
import json
import os
import re
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))
import test_reference_demos_cpu as T  # noqa: E402


def _num(out, label):
    m = re.search(re.escape(label) + r"\s*:?\s*(\d+)", out)
    assert m, (label, out[-1500:])
    return int(m.group(1))


def printed(demo, out):
    """The script's end-of-run table, in the shape of tests/test_reference_demos_cpu.py:tally()."""
    if demo == "demo_fallback":
        return {"total": _num(out, "Total Requests"), "successful": _num(out, "Successful"), "failed": _num(out, "Failed"),
                "primary": _num(out, "Primary Model Used"), "fallback": _num(out, "Fallback Triggered")}
    if demo == "demo_load_balancing":
        dist = {m.group(1): int(m.group(2)) for m in re.finditer(r"^  (\S+)\s+:\s+(\d+) requests \(", out.split("Model Distribution:")[-1], re.M)}
        return {"total": _num(out, "Total Requests"), "successful": _num(out, "Successful"), "failed": _num(out, "Failed"),
                "distribution": dist}
    rows = {m.group(1): [int(x) for x in m.group(2, 3, 4, 5)]
            for m in re.finditer(r"^([ABC])\s+\|\s+\w+\s+\|\s+[\d.]+%\s+\|\s+(\d+) \|\s+(\d+) \|\s+(\d+) \|\s+(\d+) \|", out, re.M)}
    return {"rows": rows}


def run_demo(src, demo, workdir):
    import yaml
    dbl, server, th, port = T.serve_double(host="0.0.0.0")         # the scripts call http://0.0.0.0:<port>
    os.makedirs(os.path.join(workdir, "config"), exist_ok=True)
    with open(T.CFG) as f:
        raw = yaml.safe_load(f)
    raw["litellm"]["port"] = port                                   # the scripts read the port from ./config/config.yaml
    with open(os.path.join(workdir, "config", "config.yaml"), "w") as f:
        yaml.safe_dump(raw, f)
    try:
        env = dict(os.environ, PYTHONUNBUFFERED="1", NO_COLOR="1")
        p = subprocess.run([sys.executable, os.path.join(src, demo + ".py")], cwd=workdir, env=env, capture_output=True,
                           text=True, timeout=180)
    finally:
        server.should_exit = True
        th.join(10)
    out = re.sub(r"\x1b\[[0-9;]*m", "", p.stdout)
    assert p.returncode == 0, (p.returncode, out[-2000:], p.stderr[-2000:])
    return {"wire": dbl.log, "printed": printed(demo, out)}


def main():
    src = os.path.join(sys.argv[1], "src")
    rec = {}
    with tempfile.TemporaryDirectory() as tmp:
        for demo in T.CALLS:
            rec[demo] = run_demo(src, demo, os.path.join(tmp, demo))
    with open(T.WIRE, "w") as f:
        json.dump(rec, f, indent=1, sort_keys=True)
    slim = {k: [{"model": c["model"], "content": c["messages"][0]["content"]} for c in T.distinct_calls(r["wire"])]
            for k, r in rec.items()}
    with open(T.GOLD, "w") as f:
        json.dump(slim, f, indent=1, sort_keys=True)
    for k, r in rec.items():
        print(k, len(r["wire"]), "requests;", r["printed"])


if __name__ == "__main__":
    main()
