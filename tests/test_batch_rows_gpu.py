"""The batched single-term path: its dense rows (exported by sa_batch_row, since the batch only returns the top-k, a
row written at a wrong offset would otherwise go unseen), its top-k, ties at the tile bound, and batches of several
chunks whose top-k selects overlap the next chunk's scan."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

K1, B = 1.2, 0.75
TILE = 8192


def bits_equal(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def oracle_dense(host, t, idf, avgdl):
    """BM25 of term t on every doc of the shard, from the oracle's sparse tf and score functions."""
    from oracle import ops as oops, search as osearch
    dense = np.zeros(host.n_docs, dtype=np.float32)
    ids, tfs = osearch.termfreqs_sparse(host.term_words(t))
    if len(ids):
        sc = tfs.copy()
        oops.bm25_score(sc, host.doc_lens[ids.astype(np.int64)], avgdl, np.float32(idf), K1, B)
        dense[ids.astype(np.int64)] = sc
    return dense


def oracle_topk(dense, k, doc_base):
    nz = np.flatnonzero(dense > 0)
    order = nz[np.lexsort((nz, -dense[nz].astype(np.float64)))][:k]
    docs = np.full(k, 0xFFFFFFFF, dtype=np.uint32)
    scores = np.zeros(k, dtype=np.float32)
    docs[:len(order)] = order + doc_base
    scores[:len(order)] = dense[order]
    return docs, scores


def _postings(docs, tfs, rng):
    from searcharray_b200.roaringish import encode_postings
    d = np.repeat(docs, tfs)
    p = np.concatenate([np.sort(rng.choice(700, size=k, replace=False)) for k in tfs]) if len(docs) else d
    return encode_postings(d, p)


def _mixed_shard(rng, n_docs, doc_base):
    """Terms that take every path: lists without a tile directory (words path, one of them dense in one tile), record
    tiles read one per thread and four per thread, long runs of words per doc, an empty list."""
    def pick(df, lo=0, hi=n_docs):
        return np.sort(rng.choice(np.arange(lo, hi), size=df, replace=False))
    lists = [
        (pick(300), np.ones(300, dtype=np.int64)),                          # no directory, sparse
        (pick(700, TILE, 2 * TILE), np.ones(700, dtype=np.int64)),          # no directory, 700 words in tile 1
        (pick(1300), np.minimum(1 + rng.geometric(0.5, 1300), 6)),          # directory, ~300 records per tile
        (pick(int(n_docs * 0.45)), np.minimum(1 + rng.geometric(0.5, int(n_docs * 0.45)), 40)),   # quads
        (pick(60), np.full(60, 40)),                                        # directory, ~15 records per tile
        (pick(0), np.zeros(0, dtype=np.int64)),                             # empty
        (pick(int(n_docs * 0.9)), np.ones(int(n_docs * 0.9), dtype=np.int64)),                    # quads, near-dense
    ]
    doc_lens = rng.integers(1, 300, n_docs).astype(np.float32)
    return lists, doc_lens


def _index(lists, doc_lens, doc_base, rng_seed):
    """The shard as the device sees it (doc ids shifted by doc_base) and as the oracle sees it (local ids)."""
    from searcharray_b200.indexing import index_from_term_postings
    names = [f"t{i}" for i in range(len(lists))]
    local = index_from_term_postings(names, [_postings(d, tf, np.random.default_rng(rng_seed + i))
                                             for i, (d, tf) in enumerate(lists)], doc_lens)
    shifted = index_from_term_postings(names, [_postings(d + doc_base, tf, np.random.default_rng(rng_seed + i))
                                               for i, (d, tf) in enumerate(lists)], doc_lens)
    return local, shifted


def _run_batch(h, tids, idf, avgdl, k, n_rows=0, n_docs=0):
    from searcharray_b200 import _lib
    L = _lib.lib()
    n = len(tids)
    starts = np.arange(n + 1, dtype=np.uint32)
    _lib.check(L.sa_batch_upload(h, _lib.p_u32(tids), _lib.p_u32(starts), _lib.p_f32(idf), n, 0, avgdl, K1, B, k))
    _lib.check(L.sa_batch_execute(h))
    rows = np.empty((n_rows, n_docs), dtype=np.float32)
    for r in range(n_rows):
        _lib.check(L.sa_batch_row(h, r, _lib.p_f32(rows[r])))
    docs = np.empty((n, k), dtype=np.uint32)
    scores = np.empty((n, k), dtype=np.float32)
    n_over = ctypes.c_uint32(99)
    _lib.check(L.sa_batch_download(h, _lib.p_u32(docs), _lib.p_f32(scores), ctypes.byref(n_over)))
    return docs, scores, rows, n_over.value


def test_mixed_batch_rows_and_topk():
    """13 queries over a shard with doc_base != 0 and a short last tile: every dense row bit for bit and the top-k
    (docs and score bits) against the oracle."""
    from searcharray_b200 import _lib
    from searcharray_b200.postings import DeviceIndex
    from searcharray_b200.similarity import compute_idf
    rng = np.random.default_rng(5)
    n_docs, doc_base = 3 * TILE + 1440, 3 * TILE * 7 + 96
    lists, doc_lens = _mixed_shard(rng, n_docs, doc_base)
    local, shifted = _index(lists, doc_lens, doc_base, 100)
    dev = DeviceIndex(shifted, 0, doc_base)
    avgdl = float(np.mean(doc_lens))
    order = [0, 1, 2, 3, 4, 5, _lib.NO_TERM, 6, 3, 2, 0, 4, 6]
    tids = np.asarray(order, dtype=np.uint32)
    df = [len(lists[t][0]) if t != _lib.NO_TERM else 0 for t in order]
    idf = np.asarray([np.ravel(compute_idf(n_docs, np.asarray([max(1, x)])))[0] for x in df], dtype=np.float32)
    want_rows = np.stack([oracle_dense(local, t, idf[i], avgdl) if t != _lib.NO_TERM else np.zeros(n_docs, np.float32)
                          for i, t in enumerate(order)])
    for k in (1, 10, 17, 32):
        docs, scores, rows, n_over = _run_batch(dev.handle, tids, idf, avgdl, k, len(order), n_docs)
        assert n_over == 0, k
        for i in range(len(order)):
            assert bits_equal(rows[i], want_rows[i]), (k, i)
            wd, ws = oracle_topk(want_rows[i], k, doc_base)
            assert np.array_equal(docs[i], wd) and bits_equal(scores[i], ws), (k, i)


def test_tied_scores_take_the_ties_retry():
    """Thousands of docs of one tile with the same length and tf 1 score the same: the candidate slots overflow at
    the bound, the tile collects again with the doc-id tie break and the result is exact without a re-run."""
    from searcharray_b200.postings import DeviceIndex
    from searcharray_b200.similarity import compute_idf
    rng = np.random.default_rng(9)
    n_docs = 3 * TILE + 1440
    dense_docs = np.sort(rng.choice(np.arange(TILE, 2 * TILE), size=5000, replace=False))
    sparse_docs = np.sort(rng.choice(n_docs, size=400, replace=False))
    lists = [(dense_docs, np.ones(len(dense_docs), dtype=np.int64)),
             (sparse_docs, np.ones(len(sparse_docs), dtype=np.int64))]
    doc_lens = np.full(n_docs, 50.0, dtype=np.float32)
    local, shifted = _index(lists, doc_lens, 0, 200)
    dev = DeviceIndex(shifted, 0, 0)
    avgdl = 50.0
    tids = np.asarray([0, 1, 0], dtype=np.uint32)
    idf = np.asarray([np.ravel(compute_idf(n_docs, np.asarray([len(lists[t][0])])))[0] for t in tids], dtype=np.float32)
    for k in (10, 32):
        docs, scores, _, n_over = _run_batch(dev.handle, tids, idf, avgdl, k)
        assert n_over == 0
        for i, t in enumerate(tids):
            wd, ws = oracle_topk(oracle_dense(local, int(t), idf[i], avgdl), k, 0)
            assert np.array_equal(docs[i], wd) and bits_equal(scores[i], ws), (k, i)


def test_three_chunks_overlap_selects():
    """2M docs: a chunk holds 2,048 dense rows, so 4,400 queries run as three chunks whose selects overlap the next
    chunk's scan and alternate between the two candidate areas."""
    from oracle import ops as oops, search as osearch
    from searcharray_b200 import SearchArray, synth
    from searcharray_b200.shard import shard_topk_keys, unpack_keys
    from searcharray_b200.similarity import compute_idf
    spec = synth.SynthSpec(2_000_000)
    host, _, _ = synth.generate_shard(spec)
    host.avg_doc_length = synth.global_avg_doc_length(spec)
    arr = SearchArray.from_host_index(host, avg_doc_length=host.avg_doc_length)
    names = [t[0] for t in spec.terms]
    names = (names * 5)[:4400]
    docs, scores = arr.search_topk(names, k=10)
    for i in range(0, len(names), 37):
        t = spec.term_index[names[i]]
        ids, tfs = osearch.termfreqs_sparse(host.term_words(t))
        idf = compute_idf(host.n_docs, np.asarray([len(ids)]))
        sc = tfs.copy()
        oops.bm25_score(sc, host.doc_lens[ids.astype(np.int64)], host.avg_doc_length, np.float32(idf), K1, B)
        wd, ws = unpack_keys(shard_topk_keys(ids, sc, 10))
        assert np.array_equal(docs[i], wd), names[i]
        assert bits_equal(scores[i], ws), names[i]
