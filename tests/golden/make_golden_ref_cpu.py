"""What the REAL reference (oracle/_ref, built by oracle/build_ref.py) returns on the seeded synthetic corpus
of tests/test_ref_cpu.py: docfreq, and dtype, nonzero count and SHA-256 of every termfreqs / score vector
(300,000 docs each, too large to store whole), for every term, every planted phrase, and slop 2 on every
third phrase.  Writes tests/golden/ref_cpu.json.

    python oracle/build_ref.py && python tests/golden/make_golden_ref_cpu.py
"""
import hashlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import ref_runner  # noqa: E402
from searcharray_b200 import synth  # noqa: E402

SPEC = dict(n_docs=300_000, terms_per_bucket=5, n_phrases=16, n_bigrams=4)
K1, B = 1.2, 0.75


def vec_record(v):
    v = np.ascontiguousarray(v)
    return {"dtype": str(v.dtype), "nonzero": int(np.count_nonzero(v)), "sha256": hashlib.sha256(v.tobytes()).hexdigest()}


def main():
    spec = synth.SynthSpec(SPEC["n_docs"], terms_per_bucket=SPEC["terms_per_bucket"], n_phrases=SPEC["n_phrases"],
                           n_bigrams=SPEC["n_bigrams"])
    host, _, _ = synth.generate_shard(spec)
    arr = ref_runner.reference_array(host, avg_doc_length=synth.global_avg_doc_length(spec))
    sim = ref_runner.bm25(K1, B)
    out = {"spec": SPEC, "k1": K1, "b": B, "terms": {}, "phrases": [], "slop": []}
    for name, _, _ in spec.terms:
        out["terms"][name] = {"df": int(arr.docfreq(name)), "tf": vec_record(arr.termfreqs(name)),
                              "score": vec_record(arr.score(name, similarity=sim))}
    out["missing_term_score"] = vec_record(arr.score("nope"))
    for ph in spec.phrases:
        out["phrases"].append({"terms": ph["terms"], "tf": vec_record(arr.termfreqs(ph["terms"])),
                               "score": vec_record(arr.score(ph["terms"], similarity=sim))})
    for ph in spec.phrases[::3]:
        out["slop"].append({"terms": ph["terms"], "slop": 2, "tf": vec_record(arr.termfreqs(ph["terms"], slop=2))})
    path = os.path.join(HERE, "ref_cpu.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=0)
    print(len(out["terms"]), len(out["phrases"]), len(out["slop"]), os.path.getsize(path))


if __name__ == "__main__":
    main()
