"""BASELINE configs[0] through the CUDA path: the TMDB fixture's index (tests/golden/tmdb_index.npz, made
by make_golden_tmdb_index.py from the reference's fixtures/tmdb.json.gz; 27,846 real documents, title and
overview fields) uploaded to the GPU, against what the REAL reference produced on it (tests/golden/tmdb.json:
whole-vector SHA-256 digests, match counts and top-10 lists).  Queries: reference test/test_tmdb.py:167-191,
230-241, 315-321."""
import hashlib
import json
import os

import numpy as np
import pandas as pd
import pytest

from _tmdb_index import load_fields
from conftest import GOLDEN

pytestmark = pytest.mark.gpu

G = json.load(open(os.path.join(GOLDEN, "tmdb.json")))


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def frame():
    from searcharray_b200 import SearchArray
    cols = {}
    for name, host in load_fields().items():
        want = G["fields"][name]["index"]
        assert (host.n_terms, len(host.words), host.n_docs) == (want["n_terms"], want["n_words"], G["n_docs"])
        cols[name] = SearchArray.from_host_index(host)
    return pd.DataFrame(cols)


def check_vec(got, rec, what):
    got = np.asarray(got)
    assert str(got.dtype) == rec["dtype"], what
    assert int(np.count_nonzero(got)) == rec["nonzero"], what
    order = np.lexsort((np.arange(len(got)), -got.astype(np.float64)))[:10]
    order = order[got[order] > 0]
    assert [int(i) for i in order] == rec["top_ids"], what
    if sha(got) != rec["sha256"]:          # bit-exact first; 1e-5 relative is the contract for float scores
        np.testing.assert_allclose(got[order], rec["top_scores"], rtol=1e-5, atol=0, err_msg=str(what))
        assert "tf" not in what, what        # counts must be bit-exact


@pytest.mark.parametrize("field", ["title_tokens", "overview_tokens"])
def test_tmdb_terms_phrases_slop_on_gpu(frame, field):
    arr = frame[field].array
    rec = G["fields"][field]
    for term, r in rec["terms"].items():
        assert int(arr.docfreq(term)) == r["df"], term
        check_vec(arr.termfreqs(term), r["tf"], (field, term, "tf"))
        check_vec(arr.score(term), r["score"], (field, term, "score"))
    for r in rec["phrases"]:
        check_vec(arr.termfreqs(r["phrase"]), r["tf"], (field, tuple(r["phrase"]), "tf"))
        check_vec(arr.score(r["phrase"]), r["score"], (field, tuple(r["phrase"]), "score"))
    for r in rec["slop"]:
        check_vec(arr.termfreqs(r["phrase"], slop=r["slop"]), r["tf"], (field, tuple(r["phrase"]), r["slop"], "tf"))


def test_tmdb_batched_topk_on_gpu(frame):
    """the HBM-resident batched path on the real corpus: top-10 of every golden term / phrase query"""
    for field in ("title_tokens", "overview_tokens"):
        arr = frame[field].array
        rec = G["fields"][field]
        terms = [t for t in rec["terms"] if rec["terms"][t]["df"] > 0]
        docs, scores = arr.search_topk(terms, k=10)
        for i, t in enumerate(terms):
            want = rec["terms"][t]["score"]
            n = len(want["top_ids"])
            assert [int(d) for d in docs[i][:n]] == want["top_ids"], (field, t)
            np.testing.assert_allclose(scores[i][:n], want["top_scores"], rtol=1e-5, atol=0)
        phrases = [r for r in rec["phrases"]]
        docs, scores = arr.search_topk([r["phrase"] for r in phrases], k=10)
        for i, r in enumerate(phrases):
            want = r["score"]
            n = len(want["top_ids"])
            assert [int(d) for d in docs[i][:n]] == want["top_ids"], (field, r["phrase"])
            assert all(int(d) == 0xFFFFFFFF for d in docs[i][n:])


def test_tmdb_edismax_on_gpu(frame):
    """reference test/test_tmdb.py:230-241: qf + pf + pf2 + pf3 over title and overview, mm=2, tie=0.3"""
    from searcharray_b200.solr import edismax, edismax_topk
    for r in G["edismax"]:
        got, explain = edismax(frame, q=r["q"], **G["edismax_kwargs"])
        assert explain == r["explain"]
        check_vec(got, r["scores"], r["q"])
        d, s = edismax_topk(frame, r["q"], k=10, **G["edismax_kwargs"])
        n = len(r["scores"]["top_ids"])
        assert [int(x) for x in d[:n]] == r["scores"]["top_ids"], r["q"]


def test_tmdb_three_threads(frame):
    """reference test/test_tmdb.py:285-312: the same edismax / score calls from 3 threads at once."""
    from concurrent.futures import ThreadPoolExecutor
    from searcharray_b200.solr import edismax
    arr = frame["overview_tokens"].array
    want_e = {r["q"]: edismax(frame, q=r["q"], **G["edismax_kwargs"])[0] for r in G["edismax"][:4]}
    want_s = {t: arr.score(t) for t in ("Star", "the", "of")}
    want_p = arr.score(["of", "the"])

    def work(i):
        out = []
        for rep in range(3):
            for q, w in want_e.items():
                out.append(np.array_equal(edismax(frame, q=q, **G["edismax_kwargs"])[0], w))
            for t, w in want_s.items():
                out.append(np.array_equal(arr.score(t), w))
            out.append(np.array_equal(arr.score(["of", "the"]), want_p))
            out.append(np.array_equal(arr[i::3].termfreqs("the"), arr.termfreqs("the")[i::3]))
        return all(out)

    with ThreadPoolExecutor(3) as ex:
        assert all(ex.map(work, range(3)))
