"""Extracts small excerpts of the wav sets the REFERENCE's own evaluate() wrote (N_HANS___Selective_Noise/main.py:
266-353, shipped under DEMO_N-HANS/) into tests/golden/demo_relations.npz.  They are the only reference-produced
numerical artefacts in the tree; tests/test_reference_artifacts.py uses them to pin the restatement of domixing
(SN/reader.py:131-180): the scaling quirk of target / noise signals and the SNR convention.
Needs a checkout of the reference project:  python tests/golden/make_demo_fixtures.py <reference checkout>"""
import glob
import os
import sys

import numpy as np
from scipy.io import wavfile

REF = os.path.join(sys.argv[1], "DEMO_N-HANS")
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "demo_relations.npz")
N = 4000                                                   # samples per excerpt (interior of the file)

out = {}
names = []
sets = sorted(glob.glob(REF + "/SPL_Selective_Noise_Suppression/Selective_Noise_Suppression_Samples/*_mixed.wav")) + \
    sorted(glob.glob(REF + "/denoising/example*/*_mixed.wav"))
for f in sets:
    pre = f[:-len("mixed.wav")]
    tag = os.path.basename(pre).rstrip("_")
    parts = tag.split("_")
    rec = {}
    for k in ("mixed", "target", "posNoise", "negNoise"):
        p = pre + k + ".wav"
        if not os.path.exists(p):
            continue
        rate, x = wavfile.read(p)
        assert rate == 16000 and x.dtype == np.float32
        rec[k] = x
    n = len(rec["mixed"])
    lo = max(400, n // 2 - N // 2)
    i = len(names)
    names.append(tag)
    for k, x in rec.items():
        out["%d_%s" % (i, k)] = x[lo:lo + N].copy()
    # whole-file statistics (float64): least-squares ratio of (target + negNoise) to mixed and its residual,
    # power ratios speech / noise
    m, t, ng = (rec[k].astype(np.float64) for k in ("mixed", "target", "negNoise"))
    s = t + ng
    r = float(np.dot(s, m) / np.dot(m, m))
    out["%d_ratio" % i] = np.float64(r)
    out["%d_resid" % i] = np.float64(np.linalg.norm(s - r * m) / np.linalg.norm(s))
    sig = t - rec["posNoise"].astype(np.float64) if "posNoise" in rec else t
    out["%d_snr_neg_est" % i] = np.float64(10 * np.log10(np.mean(sig ** 2) / np.mean(ng ** 2)))
    if "posNoise" in rec:
        out["%d_snr_pos_est" % i] = np.float64(10 * np.log10(np.mean(sig ** 2) / np.mean(rec["posNoise"].astype(np.float64) ** 2)))
    out["%d_snr_labels" % i] = np.array([int(parts[-2]), int(parts[-1])], np.int32)
out["names"] = np.array(names)
np.savez_compressed(OUT, **out)
print("wrote", OUT, os.path.getsize(OUT), "bytes,", len(names), "sets")
