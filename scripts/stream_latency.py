"""Latency and capacity of streaming enhancement (nhans_stream_step): S live streams of synthetic mixtures, fed in
100 ms chunks, every stream in every step.  For each S it reports the step latency (host clock around the synchronous
step: median and p99), the audio seconds pushed per second of wall clock, and the real-time headroom (chunk duration
over p99 step latency: above 1 the GPU keeps up with S live streams).  Asserts nothing about speed.  Prints one JSON
line with the GPU name and power limit.

With --post, two sets of S streams fed the same audio take plain steps (nhans_stream_step) and post-mix steps
(nhans_stream_step_post, compensate 0.3) in turn, alternating which goes first, so that both are timed under the same
conditions; each result row names its mode.

  python scripts/stream_latency.py [--streams 1,64,1024] [--steps 50] [--warmup 10] [--chunk-ms 100] [--post]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from nhans_b200 import synth, weights as W          # noqa: E402
from nhans_b200.engine import Engine                # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--streams", default="1,64,1024")
ap.add_argument("--steps", type=int, default=50)
ap.add_argument("--warmup", type=int, default=10)
ap.add_argument("--chunk-ms", type=int, default=100)
ap.add_argument("--device", type=int, default=0)
ap.add_argument("--post", action="store_true", help="also time post-mix steps, alternating with plain steps")
a = ap.parse_args()


def gpu_info(device):
    out = subprocess.run(["nvidia-smi", "-i", str(device), "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().split(", ")
    return {"gpu": out[0], "power_limit": out[1]}


chunk = 16 * a.chunk_ms
seconds = (a.warmup + a.steps) * a.chunk_ms / 1000.0 + 0.1
n_distinct = 8
mixes = [synth.mixture(seconds, 9000 + u) for u in range(n_distinct)]
negs = [synth.noise_clip(9000 + u) for u in range(n_distinct)]
eng = Engine(a.device, W.SELECTIVE_NOISE)
eng.load_weights(W.seeded_init(W.SELECTIVE_NOISE, 0))
results = []
modes = {"plain": lambda ids, chunks: eng.stream_step(ids, chunks),
         "post": lambda ids, chunks: eng.stream_step_post(ids, chunks, 0.3)}
if not a.post:
    del modes["post"]
try:
    for S in [int(s) for s in a.streams.split(",")]:
        ids = {m: eng.stream_open(None, [negs[u % n_distinct] for u in range(S)], [32767] * S) for m in modes}
        times = {m: [] for m in modes}
        for k in range(a.warmup + a.steps):
            chunks = [mixes[u % n_distinct][k * chunk:(k + 1) * chunk] for u in range(S)]
            for m in (list(modes) if k % 2 == 0 else list(modes)[::-1]):
                t0 = time.perf_counter()
                modes[m](ids[m], chunks)
                if k >= a.warmup:
                    times[m].append(time.perf_counter() - t0)
        for m in modes:
            eng.stream_close(ids[m])
            t = np.array(times[m])
            results.append({"mode": m, "streams": S, "step_ms_median": round(1e3 * float(np.median(t)), 3),
                            "step_ms_p99": round(1e3 * float(np.percentile(t, 99)), 3),
                            "audio_s_per_s": round(S * chunk / 16000.0 * len(t) / float(t.sum()), 1),
                            "rt_headroom_p99": round(chunk / 16000.0 / float(np.percentile(t, 99)), 2)})
finally:
    eng.close()
print(json.dumps(dict(gpu_info(a.device), chunk_ms=a.chunk_ms, steps=a.steps, warmup=a.warmup, results=results)))
