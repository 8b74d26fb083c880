"""Energy per pass of the mask network on a GPU box: NVML's total-energy counter around N engine runs.
   python scripts/energy_probe.py [utts] [seconds] [runs]"""
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import pynvml  # noqa: E402
from nhans_b200 import synth, weights as W  # noqa: E402
from nhans_b200.engine import Engine, pack  # noqa: E402

utts = int(sys.argv[1]) if len(sys.argv) > 1 else 64
secs = float(sys.argv[2]) if len(sys.argv) > 2 else 4.0
runs = int(sys.argv[3]) if len(sys.argv) > 3 else 24
pynvml.nvmlInit()
dev = pynvml.nvmlDeviceGetHandleByIndex(0)
eng = Engine(0, 0)
eng.load_weights(W.seeded_init(0, 0))
base = [synth.mixture(secs, u) for u in range(8)]
negs = [synth.noise_clip(u) for u in range(8)]
mix, mo = pack([base[u % 8] for u in range(utts)])
neg, no = pack([negs[u % 8] for u in range(utts)])
eng.upload(mix, mo, None, None, neg, no)
for _ in range(4):
    eng.run()
eng.sync()
e0 = pynvml.nvmlDeviceGetTotalEnergyConsumption(dev)
t0 = time.perf_counter()
eng.event_record(0)
clk = []
for i in range(runs):
    eng.run()
    if i % 4 == 3:
        eng.sync()
        clk.append(pynvml.nvmlDeviceGetClockInfo(dev, pynvml.NVML_CLOCK_SM))
eng.event_record(1)
eng.sync()
t1 = time.perf_counter()
e1 = pynvml.nvmlDeviceGetTotalEnergyConsumption(dev)
ms = eng.event_elapsed_ms(0, 1) / runs
joule = (e1 - e0) / 1000.0 / runs
print("%.1f ms/run  %.1f J/run  %.0f W avg  sm clock samples %s  -> %.1f audio-s/s" % (
    ms, joule, joule / (ms / 1000.0), clk, utts * secs / (ms / 1000.0)))
