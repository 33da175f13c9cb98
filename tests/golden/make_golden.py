"""Generates tests/golden/contraction_kat.json from the reference's own golden vectors.

    python tests/golden/make_golden.py <path to a qc-tum/TNC checkout>

Source: tnc/src/tensornetwork/contraction_test_data.json in that checkout, the data file of
test_tensor_contraction / test_tn_contraction (tnc/src/tensornetwork/contraction.rs:121-224).
The values are copied verbatim (repr round-trips float64 exactly); only the JSON layout is
compacted (re/im pairs -> two flat lists per tensor).  The tests read only the generated file.
"""
import json
import os
import sys

DST = os.path.join(os.path.dirname(os.path.abspath(__file__)), "contraction_kat.json")


def main(tnc_checkout):
    with open(os.path.join(tnc_checkout, "tnc", "src", "tensornetwork", "contraction_test_data.json")) as f:
        data = json.load(f)
    out = {"_source": "tnc/src/tensornetwork/contraction_test_data.json @ qc-tum/TNC 5dd62b3",
           "_epsilon": 1e-14, "tensors": {}}
    for name, t in data.items():
        out["tensors"][name] = {
            "legs": t["legs"], "shape": t["shape"],
            "re": [c[0] for c in t["data"]], "im": [c[1] for c in t["data"]],
        }
    with open(DST, "w") as f:
        json.dump(out, f, separators=(",", ":"))
    print("wrote", DST, {k: v["shape"] for k, v in out["tensors"].items()})


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(sys.argv[1])
