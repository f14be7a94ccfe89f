"""The TMDB fixture's index (tests/golden/tmdb_index.npz, made by make_golden_tmdb_index.py; 27,846 documents,
title and overview fields): loading it as a HostIndex, and recovering each document's token sequence from it."""
import os

import numpy as np

from conftest import GOLDEN

FIELDS = ("title_tokens", "overview_tokens")


def load_fields():
    z = np.load(os.path.join(GOLDEN, "tmdb_index.npz"))
    return {name: load_field(z, name) for name in FIELDS}


def load_field(z, name):
    from searcharray_b200.indexing import HostIndex, TermDict
    lengths, offsets = z[name + ".lengths"], z[name + ".offsets"]
    words = z[name + ".delta"].copy()
    # undo the per-term delta coding: cumulative sum inside each term's slice
    starts = offsets[lengths > 0].astype(np.int64)
    csum = np.cumsum(words, dtype=np.uint64)
    order = np.argsort(starts)
    s_sorted = starts[order]
    before = np.where(s_sorted > 0, csum[np.maximum(s_sorted, 1) - 1], np.uint64(0))
    seg_len = np.diff(np.concatenate((s_sorted, [len(words)])))
    base = np.repeat(before, seg_len)
    words = csum - base
    td = TermDict()
    for t in bytes(z[name + ".terms"]).decode("utf-8").split("\n"):
        td.add_term(t)
    return HostIndex(words, offsets, lengths, z[name + ".doc_lens"], td,
                     avg_doc_length=z[name + ".avg_doc_length"][()])


def documents(host):
    """The documents as whitespace-joined token strings: every set position bit of every term's words puts
    the term at (doc, position).  The whitespace tokenizer reads back the token sequence the index was built
    from; the original spacing is not recoverable and does not matter to that tokenizer."""
    terms, docs, posns = [], [], []
    bit = np.arange(18, dtype=np.uint64)
    for t in range(host.n_terms):
        w = host.term_words(t)
        hit = ((w[:, None] >> bit) & np.uint64(1)).astype(bool)        # word x bit
        wi, bi = np.nonzero(hit)
        terms.append(np.full(len(wi), t, dtype=np.int64))
        docs.append((w[wi] >> np.uint64(36)).astype(np.int64))
        posns.append(((w[wi] >> np.uint64(18)) & np.uint64(0x3FFFF)).astype(np.int64) * 18 + bi)
    terms, docs, posns = np.concatenate(terms), np.concatenate(docs), np.concatenate(posns)
    order = np.lexsort((posns, docs))
    terms, docs, posns = terms[order], docs[order], posns[order]
    lens = np.bincount(docs, minlength=host.n_docs)
    assert np.array_equal(lens, host.doc_lens.astype(np.int64)), "every position of every document holds one term"
    assert np.array_equal(posns, np.arange(len(posns)) - np.repeat(np.cumsum(lens) - lens, lens))
    names = np.asarray([host.term_dict.get_term(t) for t in range(host.n_terms)], dtype=object)
    toks = np.split(names[terms], np.cumsum(lens)[:-1])
    return [" ".join(x) for x in toks]
