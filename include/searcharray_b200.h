/*
 * searcharray_b200.h -- C ABI of libsearcharray_b200.so (sm_100a CUDA kernels).
 *
 * Drop-in boundary for SearchArray's scoring hot path (SURVEY.md section 8b).  The
 * reference (softwaredoug/searcharray, paths below relative to its repo root) has no C
 * ABI of its own: its "operator interface" is a set of Cython `def`s taking host numpy
 * arrays.  Replacing those one-for-one would bounce every intermediate over PCIe, so
 * the boundary sits one level up, at what SearchArray.score / .termfreqs call on
 * `self.posns` and `similarity` (searcharray/postings.py:607-708).
 *
 * Conventions: every function returns 0 on success, non-zero on error (text via
 * sa_last_error(), thread-local).  Host pointers are borrowed for the duration of the
 * call only.  Plain pointers and sizes -- no torch / numpy types.  A handle may be used
 * from several host threads (calls on one handle serialise on an internal mutex, the
 * reference's tests fire .score from 3 threads: test/test_tmdb.py:285-312).
 *
 * Posting word layout (searcharray/roaringish/roaringish.py:30-35):
 *     bits 63..36 doc id (28 b) | 35..18 block = posn / 18 (18 b) | 17..0 bitmap of posn % 18
 * Words of one term are sorted ascending and header-unique (header = bits 63..18).
 */
#ifndef SEARCHARRAY_B200_H
#define SEARCHARRAY_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct sa_index sa_index;

#define SA_OK 0
#define SA_ERR_CUDA 1
#define SA_ERR_ARG 2
#define SA_ERR_NOMEM 3
#define SA_ERR_NCCL 4

#define SA_NO_TERM 0xFFFFFFFFu      /* "token not in the term dictionary" (TermMissingError) */
#define SA_NO_DOC 0xFFFFFFFFu       /* empty top-k slot */
#define SA_MAX_PHRASE_TERMS 16
#define SA_ALL_BITS 0xFFFFFFFFFFFFFFFFull

/* ----------------------------------------------------------------------- misc */
const char *sa_last_error(void);
int sa_device_count(int *n_out);
/* Pinned host memory for result vectors (D2H of a dense float32[N] at full PCIe rate). */
int sa_host_alloc(void **ptr_out, uint64_t bytes);
int sa_host_free(void *ptr);

/* ---------------------------------------------------------------------- index
 * Uploads one shard of the inverted index into HBM.  Replaces the host-side state the
 * hot path reads: ArrayDict.data / .metadata (searcharray/phrase/memmap_arrays.py:15-53),
 * SearchArray.doc_lens (postings.py:293-299) and the docfreq cache
 * (searcharray/phrase/middle_out.py:511-528, warm() :337-342: per-term df is computed on
 * the device at upload).
 *   words        all terms' posting words, concatenated          [n_words]
 *   term_offsets / term_lengths   slice of `words` per term id    [n_terms]
 *   doc_lens     float32 length of every doc in the shard         [n_docs]
 *   doc_base     global id of the shard's first doc; the shard owns [doc_base, doc_base+n_docs)
 *                and every word's doc id must lie in that range (doc-range sharding, sec. 8e)
 */
int sa_index_create(const uint64_t *words, uint64_t n_words,
                    const uint64_t *term_offsets, const uint64_t *term_lengths, uint32_t n_terms,
                    const float *doc_lens, uint64_t n_docs, uint64_t doc_base,
                    int device, sa_index **index_out);
int sa_index_destroy(sa_index *index);
/* How sa_index_create moved the posting words to HBM (SURVEY 8f-2): 0 = plain copy (small indexes), 1 = the host
 * range -- e.g. the np.memmap of the reference's MemoryMappedArrays .dat file (phrase/memmap_arrays.py:145-208) --
 * was page-locked in place with cudaHostRegister and DMA'd at PCIe rate, 2 = pipelined through pinned bounce
 * buffers because the range could not be registered. */
int sa_index_upload_mode(const sa_index *index, int *mode_out);
int sa_index_info(const sa_index *index, uint64_t *n_docs, uint64_t *n_words,
                  uint32_t *n_terms, uint64_t *device_bytes);

/* PosnBitArray.docfreq (middle_out.py:521-528): distinct docs of the term in this shard. */
int sa_docfreq(sa_index *index, uint32_t term_id, uint64_t *df_out);

/* Restricts subsequent queries to a subset of the shard's docs -- the sliced-array
 * semantics of SearchArray.__getitem__ / FilteredPosns (postings.py:344-358,
 * middle_out.py:291-317).  `rows` = sorted local doc indices (0-based in the shard);
 * results then have n_rows entries, in `rows` order.  rows == NULL clears the filter. */
int sa_index_set_rows(sa_index *index, const uint64_t *rows, uint64_t n_rows);
/* docfreq on the filtered postings (reference quirk iii: df is taken on the slice). */
int sa_docfreq_rows(sa_index *index, uint32_t term_id, uint64_t *df_out);

/* ------------------------------------------------------------------ term path
 * SearchArray.termfreqs(token) (postings.py:607-638): popcount64_reduce + as_dense fused;
 * out = float32[n_docs] on the host (or [n_rows] when a row filter is set).
 * min_payload/max_payload: RoaringishEncoder.slice's block filter exactly as the reference
 * applies it (roaringish.py:267-282 + roaringish_ops.pyx:46-68: compares the UNSHIFTED
 * masked word with min_posn/18 and max_posn/18); pass 0 and SA_ALL_BITS for "no filter". */
int sa_termfreqs(sa_index *index, uint32_t term_id,
                 uint64_t min_payload, uint64_t max_payload, float *out_host);

/* SearchArray.score(token, similarity=bm25_similarity(k1, b)) (postings.py:652-680 +
 * similarity.py:24-38 + bm25/bm25.pyx:11-41): termfreqs + BM25 fused in one kernel.
 * idf is computed by the host exactly as compute_idf does (similarity.py:19-21, float64 ->
 * C float); avg_doc_len, k1, b as the reference passes them to bm25_score. */
int sa_score_term(sa_index *index, uint32_t term_id, float idf, float avg_doc_len,
                  float k1, float b, uint64_t min_payload, uint64_t max_payload,
                  float *out_host);

/* ---------------------------------------------------------------- phrase path
 * SearchArray._phrase_freq / PosnBitArray.phrase_freqs (postings.py:689-708,
 * middle_out.py:418-446): slop == 0 -> compute_phrase_freqs (middle-out bigram chain,
 * phrase/bigram_freqs.py); slop > 0 -> span_search (phrase/spans.py, roaringish/spans.pyx).
 * Any term id == SA_NO_TERM -> zeros.  n_terms >= 2. */
int sa_phrase_freqs(sa_index *index, const uint32_t *term_ids, uint32_t n_terms, uint32_t slop,
                    uint64_t min_payload, uint64_t max_payload, float *out_host);
int sa_score_phrase(sa_index *index, const uint32_t *term_ids, uint32_t n_terms, uint32_t slop,
                    float idf, float avg_doc_len, float k1, float b,
                    uint64_t min_payload, uint64_t max_payload, float *out_host);

/* ------------------------------------------------------- batched, HBM-resident
 * The queries/sec path: scores stay in HBM, only the top-k leaves the device.
 * Query q = terms[term_starts[q] .. term_starts[q+1]) (1 term = BM25 term query, >= 2 =
 * phrase with `slop`), idf[q] as above.  For every query the dense float32[n_docs] score
 * vector is produced in HBM exactly as sa_score_term / sa_score_phrase would, then reduced
 * to the k best (score desc, doc id asc; only score > 0; empty slots = SA_NO_DOC / 0).
 * out_docs[q*k + i] are GLOBAL doc ids (doc_base added).  The reference idiom this
 * replaces is np.argpartition(scores, -N) (searcharray/utils/sort.py:24). */
int sa_score_batch_topk(sa_index *index, const uint32_t *terms, const uint32_t *term_starts,
                        const float *idf, uint32_t n_queries, uint32_t slop,
                        float avg_doc_len, float k1, float b, uint32_t k,
                        uint32_t *out_docs, float *out_scores);

/* The same batch in three stages, so a serving loop (or the benchmark) can keep the query
 * descriptors resident and time the device work alone: upload (H2D of descriptors), execute
 * (enqueue kernels only, asynchronous), download (sync, overflow repair, D2H of the top-k;
 * *n_overflow = queries whose candidate list overflowed and were re-run exactly). */
int sa_batch_upload(sa_index *index, const uint32_t *terms, const uint32_t *term_starts,
                    const float *idf, uint32_t n_queries, uint32_t slop,
                    float avg_doc_len, float k1, float b, uint32_t k);
int sa_batch_execute(sa_index *index);
int sa_batch_download(sa_index *index, uint32_t *out_docs, float *out_scores, uint32_t *n_overflow);
/* Diagnostic export: copies dense score row `row` (n_docs floats) of the last chunk that
 * sa_batch_execute ran into out_host.  A chunk's rows are its single-term queries in query order,
 * then its phrase queries.  Valid until the next upload or execute, or a download that re-runs a
 * query exactly (the re-run reuses the rows). */
int sa_batch_row(sa_index *index, uint32_t row, float *out_host);
/* CUDA-event timer on the library's own stream (the stream the kernels are launched on). */
int sa_timer_start(sa_index *index);
int sa_timer_stop(sa_index *index, double *ms_out);

/* Kernel-time accounting for roofline reporting (CUDA events on the library's stream):
 * milliseconds spent in, and launches of, the dominant kernels since the last reset. */
typedef struct {
    double term_kernel_ms;
    uint64_t term_kernel_launches;
    uint64_t term_kernel_queries;     /* queries covered by those launches */
    double topk_kernel_ms;
    uint64_t topk_kernel_launches;
    double phrase_kernel_ms;
    uint64_t phrase_kernel_launches;
    uint64_t total_launches;          /* every kernel launched by the library */
    /* phrase (slop 0) batches, summed over the queries of every sa_batch_download since the reset:
     * continuation words written (sum of C_s) and docs with a non-zero phrase count (M) -- the
     * data-dependent terms of SURVEY 8d's B_phrase = 8*sum(W) + 16*sum(C_s) + 4*N + 4*M */
    uint64_t phrase_cont_words;
    uint64_t phrase_matched_docs;
} sa_stats;
int sa_stats_reset(sa_index *index);
int sa_stats_get(sa_index *index, sa_stats *out);
int sa_set_profiling(sa_index *index, int enabled);   /* per-kernel CUDA events on/off */

/* -------------------------------------------------------------- multi-GPU (8e)
 * One process per GPU, each owning a contiguous doc-id range.  The only exchange on the
 * scoring path is one all-gather of per-shard top-k per query batch.
 * sa_comm_unique_id fills a 128-byte NCCL unique id on rank 0 (the caller broadcasts it
 * with whatever bootstrap it has); sa_comm_init joins the clique. */
int sa_comm_unique_id(void *id128_out);
int sa_comm_init(sa_index *index, const void *id128, int rank, int world_size);
int sa_comm_destroy(sa_index *index);
/* Harness plumbing over the same communicator: barrier, and max-over-ranks of a double
 * (bench.py uses these for the barrier + max-over-ranks timing rule). */
int sa_comm_barrier(sa_index *index);
int sa_comm_allreduce_max(sa_index *index, double *inout);
int sa_comm_allreduce_sum_u64(sa_index *index, uint64_t *inout, uint64_t n);
int sa_batch_execute_allgather(sa_index *index);
int sa_batch_download_allgather(sa_index *index, uint32_t *out_docs, float *out_scores,
                                uint32_t *n_overflow);
/* Like sa_score_batch_topk on every rank's shard, then ncclAllGather of the per-shard
 * (doc, score) lists and a k-way merge on the device; every rank receives the global top-k. */
int sa_score_batch_topk_allgather(sa_index *index, const uint32_t *terms, const uint32_t *term_starts,
                                  const float *idf, uint32_t n_queries, uint32_t slop,
                                  float avg_doc_len, float k1, float b, uint32_t k,
                                  uint32_t *out_docs, float *out_scores);

/* ------------------------------------------------------ multi-field edismax (8f-1)
 * Replaces the numpy half of searcharray/solr.py:117-355 (edismax): the per-(term, field) BM25
 * vectors, the phrase-phase vectors and the combined score vector stay in HBM.  The host mirror
 * (searcharray_b200/solr.py) parses the query like solr.py:77-114, computes idf like
 * similarity.py:19-21 and drives these calls.  All fields index the same documents.
 *   sa_multi_qf       solr.py:117-178.  field f has n_terms[f] query terms; term_ids / idf are the
 *                     per-field lists concatenated.  has_boost[f] == 0 <=> "field" without ^boost.
 *                     mm[f]: clauses that must score > 0 (term-centric: mm[0] over term positions;
 *                     field-centric: per field, already clamped to its term count).  The combined
 *                     vector is float64 (term-centric) or float32 (field-centric), as in numpy.
 *   sa_multi_filter   solr.py:326-330: restrict field `field`'s posting lists of `term_ids` to the docs
 *                     with qf > 0 (FilteredPosns, middle_out.py:291-317); df_out = doc frequencies of
 *                     the filtered lists (what SearchArray.docfreq reports on the sliced array).
 *   sa_multi_phrases  phrase i = filtered lists term_slots[phrase_starts[i] .. phrase_starts[i+1])
 *                     (slots index the last sa_multi_filter's term list; term_ids: the same terms' ids);
 *                     BM25 with idf[i].  Row i of the field holds the result (solr.py:181-244).
 *   sa_multi_add_phase  float32 sum, in order, of rows (entry_field[i], entry_row[i]) * entry_boost[i],
 *                     added to the combined vector where it is non-zero (solr.py:335-353).
 *   sa_multi_download / sa_multi_topk   the dense vector (float64, or float32 when as_float32), or its
 *                     exact top-k (score desc, doc asc; absolute doc ids; empty slots SA_NO_DOC / 0). */
typedef struct sa_multi sa_multi;
int sa_multi_create(sa_index *const *fields, uint32_t n_fields, sa_multi **multi_out);
int sa_multi_destroy(sa_multi *multi);
int sa_multi_qf(sa_multi *multi, int field_centric, const uint32_t *n_terms, const uint32_t *term_ids,
                const float *idf, const float *boost, const uint32_t *has_boost,
                const float *avg_doc_len, const float *k1, const float *b, const uint32_t *mm,
                double tie, uint64_t *n_matches);
int sa_multi_filter(sa_multi *multi, uint32_t field, const uint32_t *term_ids, uint32_t n_terms,
                    uint64_t *df_out);
int sa_multi_phrases(sa_multi *multi, uint32_t field, uint32_t n_phrases, const uint32_t *phrase_starts,
                     const uint32_t *term_slots, const uint32_t *term_ids, const float *idf,
                     float avg_doc_len, float k1, float b);
int sa_multi_add_phase(sa_multi *multi, uint32_t n_entries, const uint32_t *entry_field,
                       const uint32_t *entry_row, const float *entry_boost, const uint32_t *entry_has_boost);
int sa_multi_download(sa_multi *multi, void *out, int as_float32);
int sa_multi_is_float32(sa_multi *multi, int *out);
int sa_multi_topk(sa_multi *multi, uint32_t k, uint32_t *out_docs, double *out_scores);

/* ------------------------------------------------- per-op exports (parity tests)
 * Device implementations of the reference's native ops on raw arrays (host in, host out),
 * for kernel-level parity tests against the Cython originals (SURVEY.md section 8b). */
/* popcount64_reduce (roaringish/popcount.pyx:212-237): returns groups in *n_out */
int sa_op_popcount64_reduce(const uint64_t *words, uint64_t n, int device,
                            uint64_t *keys_out, float *counts_out, uint64_t *n_out);
/* bm25_score (bm25/bm25.pyx:28-41): in place over all n */
int sa_op_bm25_score(float *tf_inout, const float *doc_lens, uint64_t n, float avg_doc_len,
                     float idf, float k1, float b, int device);
/* The reference's other similarities (searcharray/similarity.py:41-89) evaluated on the device:
 * SA_SIM_BM25_IMPACT -> float32[n] `tf / (tf + k1 * (1 - b + b * dl / avgdl))` (bm25_impact, :41-54; idf unused);
 * SA_SIM_BM25_LEGACY -> float64[n] `idf * (tf * (k1 + 1)) / (...)` (bm25_legacy_similarity, :57-72);
 * SA_SIM_CLASSIC     -> float64[n] `idf * sqrt(tf) * (1 / sqrt(dl))` (classic_similarity, :75-89; k1, b, avgdl unused).
 * idf is the float64 scalar the caller computed the way the reference does; numpy's dtype promotion is reproduced. */
#define SA_SIM_BM25_IMPACT 0
#define SA_SIM_BM25_LEGACY 1
#define SA_SIM_CLASSIC 2
int sa_op_similarity(int kind, const float *term_freqs, const float *doc_lens, uint64_t n,
                     double avg_doc_len, double idf, double k1, double b, int device, void *out);
/* bigram_freqs (phrase/bigram_freqs.py:213-307): cont_rhs=1 -> Continuation.RHS else LHS.
 * ids/counts: per-doc matches (zero-count docs kept, quirk iv); next: continuation words.
 * Capacities: ids/counts >= min(n_lhs,n_rhs)*2, next >= 2*min(n_lhs, n_rhs)+2. */
int sa_op_bigram_freqs(const uint64_t *lhs, uint64_t n_lhs, const uint64_t *rhs, uint64_t n_rhs,
                       int cont_rhs, int device,
                       uint64_t *ids_out, float *counts_out, uint64_t *n_ids_out,
                       uint64_t *next_out, uint64_t *n_next_out);

/* The reference's sorted-set ops on raw arrays (sa_setops.cu), one export per Cython op, returning what the
 * op returns (index arrays, not values, for the intersect family).  Inputs sorted by (x & mask) as every
 * reference caller passes them; output capacities: intersect family min(n_lhs, n_rhs) per array (keep mode:
 * n_lhs / n_rhs), merge n_lhs + n_rhs, the grouped ops and unique / payload_slice n.
 *   sa_op_intersect                searcharray/roaringish/intersect.pyx:278-320 (drop_duplicates as there;
 *                                  mask == 0 -> SA_ERR_ARG, the reference raises ValueError)
 *   sa_op_adjacent                 :323-343   pairs with (lhs & mask) + lowbit(mask) == (rhs & mask)
 *   sa_op_intersect_with_adjacents :346-390   both in one call
 *   sa_op_merge                    searcharray/roaringish/merge.pyx:137-158
 *   sa_op_sort_merge_counts        merge.pyx:211-232
 *   sa_op_unique                   searcharray/roaringish/unique.pyx:139-145
 *   sa_op_popcount64 / sa_op_popcount_reduce_at / sa_op_key_sum_over   popcount.pyx:120-122, 150-165, 195-204
 *   sa_op_payload_slice / sa_op_as_dense   roaringish_ops.pyx:46-68, 84-98
 * sa_op_last_staged_ctas: how many CTAs of the calling thread's last intersect-family call took the
 * TMA-staged shared-memory path (the rest searched global memory): a test hook. */
int sa_op_intersect(const uint64_t *lhs, uint64_t n_lhs, const uint64_t *rhs, uint64_t n_rhs,
                    uint64_t mask, int drop_duplicates, int device,
                    uint64_t *lhs_idx_out, uint64_t *rhs_idx_out, uint64_t *n_lhs_out, uint64_t *n_rhs_out);
int sa_op_adjacent(const uint64_t *lhs, uint64_t n_lhs, const uint64_t *rhs, uint64_t n_rhs,
                   uint64_t mask, int device, uint64_t *lhs_idx_out, uint64_t *rhs_idx_out, uint64_t *n_out);
int sa_op_intersect_with_adjacents(const uint64_t *lhs, uint64_t n_lhs, const uint64_t *rhs, uint64_t n_rhs,
                                   uint64_t mask, int device,
                                   uint64_t *lhs_idx_out, uint64_t *rhs_idx_out, uint64_t *n_out,
                                   uint64_t *adj_lhs_idx_out, uint64_t *adj_rhs_idx_out, uint64_t *n_adj_out);
int sa_op_merge(const uint64_t *lhs, uint64_t n_lhs, const uint64_t *rhs, uint64_t n_rhs,
                int drop_duplicates, int device, uint64_t *out, uint64_t *n_out);
int sa_op_sort_merge_counts(const uint64_t *lhs_ids, const float *lhs_counts, uint64_t n_lhs,
                            const uint64_t *rhs_ids, const float *rhs_counts, uint64_t n_rhs,
                            int device, uint64_t *ids_out, float *counts_out, uint64_t *n_out);
int sa_op_unique(const uint64_t *arr, uint64_t n, uint64_t rshift, int device, uint64_t *out, uint64_t *n_out);
int sa_op_popcount64(const uint64_t *arr, uint64_t n, int device, uint64_t *out);
int sa_op_popcount_reduce_at(const uint64_t *ids, const uint64_t *payload, uint64_t n, int device,
                             uint64_t *ids_out, float *counts_out, uint64_t *n_out);
int sa_op_key_sum_over(const uint64_t *ids, const uint64_t *counts, uint64_t n, int device,
                       uint64_t *ids_out, float *counts_out, uint64_t *n_out);
int sa_op_payload_slice(const uint64_t *arr, uint64_t n, uint64_t msb_mask, uint64_t min_payload,
                        uint64_t max_payload, int device, uint64_t *out, uint64_t *n_out);
int sa_op_as_dense(const uint64_t *indices, const float *values, uint64_t n, uint64_t size, int device, float *out);
uint64_t sa_op_last_staged_ctas(void);

/* ------------------------------------------------------------ index build (8f-4)
 * The numpy half of the reference's index build after tokenisation (searcharray/indexing.py:101-145:
 * stable sort of the (term, doc, posn) triples by term; searcharray/roaringish/roaringish.py:93-142: encode) on
 * the device.  Triples in document order as _gather_tokens emits them (indexing.py:64-98); term ids < n_terms.
 * words_out: room for n_triples words; term_off_out / term_len_out: every term's slice of words_out. */
int sa_op_build_index(const uint32_t *term_ids, const uint32_t *doc_ids, const uint32_t *posns, uint64_t n_triples,
                      uint32_t n_terms, int device, uint64_t *words_out, uint64_t *n_words_out,
                      uint64_t *term_off_out, uint64_t *term_len_out);

#ifdef __cplusplus
}
#endif
#endif /* SEARCHARRAY_B200_H */
