"""Smoke-size invocations of the hot path for compute-sanitizer (scripts/sanitize.sh): tiny capacities so that every
kernel - STFT, towers, first convolution (per-frame table + generated operand), row-walk and shifted-row GEMM layers,
split-K head, iSTFT, post-mix - runs a handful of CTAs; `tiny` packs a batch of 2-3 frame utterances into several passes.
   python scripts/sanitize_run.py sn|ss|tiny"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from nhans_b200 import synth, weights as W      # noqa: E402
from nhans_b200.engine import Engine            # noqa: E402

mode = sys.argv[1] if len(sys.argv) > 1 else "sn"
variant = 1 if mode == "ss" else 0
eng = Engine(0, variant, win_capacity=8, row_capacity=1)
eng.load_weights(W.seeded_init(variant, 0))
if mode == "tiny":
    # utterances of 2-3 frames: more virtual frames than one pass's per-frame table holds -> several smaller passes
    base = synth.mixture(0.5, 1)
    mixes = [base[o:o + 560 + 160 * (i % 2)] for i, o in enumerate(range(0, 4000, 400))]
    res = eng.enhance(mixes, None, [synth.noise_clip(1)] * len(mixes))
elif mode == "ss":
    res = eng.enhance([synth.mixture(0.12, 2)], [synth.speaker_clip(2, "interference")], [synth.speaker_clip(2, "target")], want_mixproc=True)
else:
    res = eng.enhance([synth.mixture(0.12, 0), synth.mixture(0.05, 1)], None, [synth.noise_clip(0), synth.noise_clip(1)])
    post = eng.postmix(res["out_offs"], compensate=0.2, ac=False)
    assert np.isfinite(post["snr_est"]).all()
assert all(np.isfinite(y).all() for y in res["f32"]) and sum(len(y) for y in res["f32"]) > 0
eng.close()
print("sanitize_run %s ok: %d utterances, %d samples" % (mode, len(res["f32"]), sum(len(y) for y in res["f32"])))
