"""Regenerates tests/golden/ckpt_index_{sn,ss}.json from the reference checkpoints' .index files:

    python tests/golden/make_ckpt_index.py <reference checkout>

The JSON holds name -> [dtype, shape, offset, size] for every entry of
N_HANS___Selective_Noise/trained_model/81448_0-1000000.index and
N_HANS___Source_Separation/trained_model/81457_2-545000.index - the only reference-produced artefacts
that pin the network architecture (SURVEY.md App. C)."""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from nhans_b200 import weights as W  # noqa: E402

REF = sys.argv[1]
for tag, prefix in (("sn", "N_HANS___Selective_Noise/trained_model/81448_0-1000000"),
                    ("ss", "N_HANS___Source_Separation/trained_model/81457_2-545000")):
    e = W.read_bundle_index(os.path.join(REF, prefix + ".index"))
    out = {k: [v["dtype"], list(v["shape"]), v["offset"], v["size"]] for k, v in e.items()}
    with open(os.path.join(HERE, "ckpt_index_%s.json" % tag), "w") as f:
        json.dump(out, f, indent=0, sort_keys=True)
    print(tag, len(out))
