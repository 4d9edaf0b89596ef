"""Decode-step time (CUDA events around each graph launch) for 64 x 512-in / N-out on the full-size model."""
import argparse, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from rr_b200.models import SPECS, make_weights
from rr_b200.engine import Engine
ap = argparse.ArgumentParser()
ap.add_argument("--model", default="llama-3-8b"); ap.add_argument("--new", type=int, default=48)
ap.add_argument("--batch", type=int, default=64); ap.add_argument("--no-graph", action="store_true")
a = ap.parse_args()
spec = SPECS[a.model]
w = make_weights(spec, seed=0, device="cuda")
eng = Engine(w, max_batch=a.batch, ctx_max=640, max_prefill_tokens=8192, use_cuda_graph=not a.no_graph)
ids = np.random.RandomState(0).randint(0, spec.vocab, size=(a.batch, 512)).astype(np.int32)
start = np.arange(0, a.batch * 512 + 1, 512, dtype=np.int32)
for rep in range(2):
    eng.reset_stats()
    recs, _ = eng.run_batch(ids.reshape(-1), start, a.new)
    st = eng.stats()
    print(f"PDL={'off' if os.environ.get('RR_NO_PDL') else 'on'} graph={not a.no_graph} rep{rep}: decode {st['decode_ms_total']/st['decode_steps']:.3f} ms/step "
          f"({st['decode_steps']} steps), prefill {st['prefill_ms_total']:.1f} ms total, launches {st['kernel_launches']}")
eng.close()
