"""The oracle port (oracle/search.py + oracle/sa_oracle.c) against the REAL reference on the seeded synthetic
corpus -- the same index object both arms of bench.py run on.  What the reference returned there is stored in
tests/golden/ref_cpu.json (made by tests/golden/make_golden_ref_cpu.py from the reference built into oracle/_ref):
docfreq, and dtype, nonzero count and SHA-256 of every vector, so the comparison stays bit for bit."""
import hashlib
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN

G = json.load(open(os.path.join(GOLDEN, "ref_cpu.json")))


@pytest.fixture(scope="module")
def corpus():
    from oracle import search as osearch
    from searcharray_b200 import synth
    s = G["spec"]
    spec = synth.SynthSpec(s["n_docs"], terms_per_bucket=s["terms_per_bucket"], n_phrases=s["n_phrases"],
                           n_bigrams=s["n_bigrams"])
    host, _, _ = synth.generate_shard(spec)
    avgdl = synth.global_avg_doc_length(spec)
    oidx = osearch.OracleIndex({t: host.term_words(t) for t in range(host.n_terms)}, host.doc_lens,
                               avg_doc_length=avgdl, corpus_size=host.n_docs, cache=True)
    return spec, host, oidx


def same_bits(got, rec):
    got = np.ascontiguousarray(got)
    return (str(got.dtype) == rec["dtype"] and int(np.count_nonzero(got)) == rec["nonzero"]
            and hashlib.sha256(got.tobytes()).hexdigest() == rec["sha256"])


def test_terms_match_the_reference(corpus):
    spec, host, oidx = corpus
    assert [name for name, _, _ in spec.terms] == list(G["terms"])
    for t, (name, _, _) in enumerate(spec.terms):
        want = G["terms"][name]
        assert int(oidx.docfreq(t)) == want["df"]
        assert same_bits(oidx.termfreqs(t), want["tf"]), name
        assert same_bits(oidx.score(t, k1=G["k1"], b=G["b"]), want["score"]), name
    assert same_bits(oidx.score(None), G["missing_term_score"])


def test_phrases_and_slop_match_the_reference(corpus):
    spec, host, oidx = corpus
    assert [ph["terms"] for ph in spec.phrases] == [r["terms"] for r in G["phrases"]]
    n_match = 0
    for r in G["phrases"]:
        ids = [spec.term_index[t] for t in r["terms"]]
        assert same_bits(oidx.termfreqs(ids), r["tf"]), r["terms"]
        assert same_bits(oidx.score(ids, k1=G["k1"], b=G["b"]), r["score"]), r["terms"]
        n_match += r["tf"]["nonzero"]
    assert n_match > 0
    from oracle import ops as oops
    assert [r["terms"] for r in G["slop"]] == [ph["terms"] for ph in spec.phrases[::3]]
    for r in G["slop"]:
        ids = [spec.term_index[t] for t in r["terms"]]
        got = oidx.termfreqs(ids, slop=r["slop"])
        if not oops.last_span_undefined:
            assert same_bits(got, r["tf"]), r["terms"]
