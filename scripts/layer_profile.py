"""Per-layer timing of the tensor-core layers on a GPU box (CUDA events around every launch).
   python scripts/layer_profile.py [utts] [seconds] [layers.json]   -> table (+ the per-layer records as JSON)"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from nhans_b200 import synth, weights as W  # noqa: E402
from nhans_b200.engine import Engine, pack  # noqa: E402

utts = int(sys.argv[1]) if len(sys.argv) > 1 else 64
secs = float(sys.argv[2]) if len(sys.argv) > 2 else 4.0
json_out = sys.argv[3] if len(sys.argv) > 3 else None
eng = Engine(0, 0, win_capacity=int(os.environ.get("NHANS_WIN_CAPACITY", "0")))
eng.load_weights(W.seeded_init(0, 0))
base = [synth.mixture(secs, u) for u in range(8)]
negs = [synth.noise_clip(u) for u in range(8)]
mix, mo = pack([base[u % 8] for u in range(utts)])
neg, no = pack([negs[u % 8] for u in range(utts)])
eng.upload(mix, mo, None, None, neg, no)
eng.run(); eng.sync()
eng.profile_reset(); eng.profile(True)
import subprocess, threading
_clk = []
_proc = subprocess.Popen(['nvidia-smi', '--query-gpu=clocks.sm,power.draw', '--format=csv,noheader,nounits', '-lms', '100'], stdout=subprocess.PIPE, text=True)
threading.Thread(target=lambda: [_clk.append(l) for l in _proc.stdout], daemon=True).start()
eng.event_record(0)
for _ in range(6):
    eng.run()
eng.event_record(1)
eng.sync()
ms = eng.event_elapsed_ms(0, 1) / 3
_proc.terminate()
_c = [tuple(float(x) for x in l.split(',')) for l in _clk if ',' in l]
_c = [c for c in _c if c[1] > 400]
print('clocks under load: median sm %.0f MHz, median power %.0f W (%d samples)' % (np.median([c[0] for c in _c]) if _c else 0, np.median([c[1] for c in _c]) if _c else 0, len(_c)))
layers = eng.profile_layers(0)
tot = sum(l["ms"] for l in layers)
print("%d x %.0f s: %.1f ms/run -> %.1f audio-s/s" % (utts, secs, ms / 2, utts * secs / (ms / 2e3)))
# TFLOP/s counts the algorithmic MACs (TF's, padding included); exec counts the MACs the kernels run, without the
# kernel rows that fall into vertical padding (the plan of an older library has no `exec_macs`: exec = TFLOP/s there)
for l, pg in zip(layers, eng.plan(0)["gemm"]):
    l["exec_tflops"] = l["tflops"] * pg.get("exec_macs", pg["macs"]) / pg["macs"]
    print("%-22s K=%5d N=%3d  %8.2f ms  %5.1f%%  %7.1f exec  %7.1f TFLOP/s" % (l["name"], l["K"], l["N"], l["ms"] / 6, 100 * l["ms"] / tot,
                                                                            l["exec_tflops"], l["tflops"]))
st = eng.profile_get(0)
print("all GEMM layers: %.1f ms, %.1f TFLOP/s;  direct conv %.1f ms" % (st["ms"] / 6, st["flops"] / st["ms"] / 1e9, eng.profile_get(3)["ms"] / 6))
if json_out:
    with open(json_out, "w") as f:
        json.dump(layers, f)
if os.environ.get("NHANS_DEBUG_STATS"):
    import ctypes
    print("wait cycles per layer (sum over 148 CTAs, %): tmem_empty | a_full | b_full | epi waits tmem_full | of MMA-warp total")
    for i, l in enumerate(layers):
        st = (ctypes.c_uint64 * 8)()
        eng.lib.nhans_debug_layer_stats(eng.h, 0, i, st)
        tot = max(1, st[4])
        print("%-22s %5.1f%% %5.1f%% %5.1f%%   epi %5.1f%%   total %.2e" % (l["name"], 100 * st[0] / tot, 100 * st[1] / tot, 100 * st[2] / tot, 100 * st[3] / tot, tot))
