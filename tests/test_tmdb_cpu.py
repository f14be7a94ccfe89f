"""BASELINE configs[0]: the TMDB fixture (27,846 real documents) -- the host indexer and the CPU
oracle against what the REAL reference produced on it (tests/golden/tmdb.json: digests, counts and
top-10 lists; made by tests/golden/make_golden_tmdb.py).  The documents are read back, as token
sequences, from the fixture's stored index (tests/golden/tmdb_index.npz) and indexed again."""
import hashlib
import json
import os

import numpy as np
import pytest

from _tmdb_index import documents, load_fields
from conftest import GOLDEN

G = json.load(open(os.path.join(GOLDEN, "tmdb.json")))


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def fields():
    from oracle import search as osearch, solr as osolr
    from searcharray_b200.indexing import build_index
    out = {}
    for name, stored in load_fields().items():
        host = build_index(documents(stored), str.split)
        idx = osearch.OracleIndex({t: host.term_words(t) for t in range(host.n_terms)}, host.doc_lens,
                                  avg_doc_length=host.avg_doc_length)
        out[name] = (host, osolr.OracleField(idx, host.term_dict.term_to_ids))
    return out


def check_vec(got, rec, what):
    got = np.asarray(got)
    assert str(got.dtype) == rec["dtype"], what
    assert int(np.count_nonzero(got)) == rec["nonzero"], what
    order = np.lexsort((np.arange(len(got)), -got.astype(np.float64)))[:10]
    order = order[got[order] > 0]
    assert [int(i) for i in order] == rec["top_ids"], what
    assert sha(got) == rec["sha256"], what            # the whole vector, bit for bit


@pytest.mark.parametrize("field", ["title_tokens", "overview_tokens"])
def test_host_indexer_matches_reference_index(fields, field):
    """searcharray_b200.indexing.build_index on real text == the reference's index, word for word."""
    host, _ = fields[field]
    want = G["fields"][field]["index"]
    h = hashlib.sha256()
    t2i = host.term_dict.term_to_ids
    for t in sorted(t2i.keys()):
        h.update(t.encode("utf-8"))
        h.update(np.ascontiguousarray(host.term_words(t2i[t]), dtype=np.uint64).tobytes())
    assert (host.n_terms, len(host.words)) == (want["n_terms"], want["n_words"])
    assert h.hexdigest() == want["sha256"]
    assert sha(host.doc_lens.astype(np.float32)) == want["doc_lens_sha256"]
    assert float(host.avg_doc_length) == want["avg_doc_length"]
    assert host.n_docs == G["n_docs"]


@pytest.mark.parametrize("field", ["title_tokens", "overview_tokens"])
def test_oracle_terms_and_phrases_on_tmdb(fields, field):
    from oracle import ops as oops
    _, of = fields[field]
    rec = G["fields"][field]
    for term, r in rec["terms"].items():
        tid = of.term_to_id.get(term)
        assert int(of.index.docfreq(tid)) == r["df"], term
        check_vec(of.index.termfreqs(tid), r["tf"], (field, term, "tf"))
        check_vec(of.index.score(tid), r["score"], (field, term, "score"))
    for r in rec["phrases"]:
        ids = of.ids(r["phrase"])
        check_vec(of.index.termfreqs(ids), r["tf"], (field, r["phrase"], "tf"))
        check_vec(of.index.score(ids), r["score"], (field, r["phrase"], "score"))
    for r in rec["slop"]:
        got = of.index.termfreqs(of.ids(r["phrase"]), slop=r["slop"])
        if not oops.last_span_undefined:
            check_vec(got, r["tf"], (field, r["phrase"], r["slop"]))


def test_oracle_edismax_on_tmdb(fields):
    """reference test/test_tmdb.py:230-241: qf + pf + pf2 + pf3 over title and overview, mm=2, tie=0.3."""
    from oracle import solr as osolr
    ofields = {name: f for name, (_, f) in fields.items()}
    for r in G["edismax"]:
        got = osolr.edismax(ofields, r["q"], **G["edismax_kwargs"])
        check_vec(got, r["scores"], r["q"])
