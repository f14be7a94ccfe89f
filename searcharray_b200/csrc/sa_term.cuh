// sa_term.cuh -- kernel-side declarations shared by the term-path translation units.
#pragma once
#include "sa_common.cuh"

#define SA_TILE_DOCS 8192          // docs per CTA tile (32 KB of float32 scores)
#define SA_TERM_UNROLL 4           // 30-word windows loaded per warp before processing
#define SA_TERM_THREADS 256
#define SA_STAGED_NORM_MIN_WORDS 1024   // tiles with at least this many posting words stage the tile's norms (sa_term.cu)
#define SA_STAGED_NORM_MIN_RECS 96      // ... or this many (doc, tf) records on the tf-table path
#define SA_TERM_PREFETCH_TILES 8         // L2 prefetch distance of the tf-table path, in tiles (sa_term.cu)
#define SA_TERM_QUAD_MIN_RECS 512       // four records per thread from this many records per tile on (and >= 16 * k, sa_term.cu)
#define SA_TOPK_MAX 32             // warp-level threshold estimation handles k <= 32

enum TermMode { TERM_MODE_TF = 0, TERM_MODE_SCORE = 1 };

// Per-query top-k collection state in HBM (see sa_topk.cu).  No global atomics: every
// (query, tile) CTA owns `slots` candidate slots.
struct TopkCtx {
    u32 *tile_cnt;     // [Q][n_tiles] candidates written by the tile's CTA (<= slots)
    u32 *tile_max;     // [Q][n_tiles] score bits of the tile's best candidate (0 = none)
    u64 *tile_cand;    // [Q][n_tiles][slots] key = score_bits << 32 | (0xFFFFFFFF - local_doc)
    u32 *overflow;     // [Q] set when some tile had more than `slots` candidates
    u32 n_tiles;
    u32 slots;
    u32 k;             // 0 => no top-k collection
};

struct TermBatchArgs {
    const u64 *words;
    const float *doc_lens;
    const float *norm;          // per-doc BM25 length norm (padded to a tile multiple), SCORE mode
    const u32 *tile_dir;        // tile directories (see sa_index::d_tile_dir)
    const u32 *recs;            // per-term (doc, tf) records (sa_index::d_recs) or NULL
    const u32 *rec_dir;         // record directories, same offsets as tile_dir
    u64 n_docs;
    u64 doc_base;
    const TermQuery *queries;   // [Q]
    float *out;                 // [Q][out_stride]
    u64 out_stride;             // multiple of SA_TILE_DOCS
    Bm25Params bm25;            // idf field unused (per query)
    u64 min_payload, max_payload;
    int filter;                 // apply the payload_slice filter
    int mode;
    u32 staged_norm_min_words;  // set by launch_term_batch
    u32 staged_norm_min_recs, quad_min_recs;   // set by launch_term_batch
    u32 prefetch_tiles;         // L2 prefetch distance in tiles on the tf-table path (0 = off); set by launch_term_batch
    u32 query_major;            // grid layout (set by launch_term_batch): 1 = (tiles, queries), 0 = (queries, tiles)
    TopkCtx topk;
};

int launch_term_batch(sa_index *ix, const TermBatchArgs &a, u32 n_queries);
int sa_ensure_norm(sa_index *ix, float k1, float b, float avg_doc_len);
int launch_topk_select(sa_index *ix, const TopkCtx &t, u32 n_queries, u64 doc_base, u64 *d_out_keys,
                       const u32 *d_out_index, cudaStream_t stream = nullptr);   // nullptr: ix->stream
u32 sa_topk_slots(u32 k);
Bm25Params sa_make_bm25(const sa_index *ix, float idf, float avg_doc_len, float k1, float b);
TermQuery sa_make_term_query(const sa_index *ix, u32 term_id, float idf);
// d_row_idf != NULL: the rows hold raw match counts; BM25 (norm table of the last sa_ensure_norm) is applied in
// place on the way (row_idf[i] = idf of row row0 + i)
int launch_dense_topk_tiles(sa_index *ix, float *dense, u64 stride, u32 row0, u32 n_rows, const TopkCtx &t,
                            const float *d_row_idf);
int launch_topk_merge(sa_index *ix, const u64 *d_in, u64 rank_stride, u32 world, u32 n_queries, u32 k, u64 *d_out);
// A batch's result block in HBM: nq * k keys followed by SA_BATCH_TAIL summary words written by the batch's last
// kernel -- [0] queries that need the exact host-side re-run (candidate overflow, wrong same-term guess, scratch
// exhausted), [1] continuation words and [2] matched docs of the phrase queries (roofline accounting).  The tail
// travels with the keys (one D2H; one all-gather when sharded), so a clean batch costs ONE stream synchronise.
#define SA_BATCH_TAIL 4
int sa_batch_download_locked(sa_index *ix, uint32_t *out_docs, float *out_scores, uint32_t *n_overflow);
// batch plumbing shared by sa_index.cu / sa_comm.cu (callers hold ix->mu)
int sa_batch_upload_locked(sa_index *ix, const uint32_t *terms, const uint32_t *term_starts,
                           const float *idf, uint32_t n_queries, uint32_t slop,
                           float avg_doc_len, float k1, float b, uint32_t k);
int sa_batch_execute_locked(sa_index *ix);
int sa_batch_fix_overflow_locked(sa_index *ix, u32 *n_redone);
void sa_batch_dims(sa_index *ix, u32 *nq, u32 *k);
void sa_unpack_keys(const u64 *keys, u64 n, uint32_t *out_docs, float *out_scores);

#ifdef __CUDACC__
// The j-th round of "take the warp maximum, then clear it" (REDUX.MAX: one instruction per round on sm_80+).
// Exactly ONE lane gives up its value per round, so equal values are counted with their multiplicity: BM25
// scores are a function of (tf, doc length) only and repeat a lot -- collapsing duplicates used to leave fewer
// than k published values on tiles whose top scores tie, which degenerates the bound to "keep everything".
__device__ __forceinline__ u32 warp_pop_max(u32 &v) {
    const u32 m = __reduce_max_sync(0xffffffffu, v);
    const unsigned holders = __ballot_sync(0xffffffffu, v == m);
    if ((threadIdx.x & 31) == (unsigned)(__ffs(holders) - 1)) v = 0;
    return m;
}

// k-th largest (k <= 32), with multiplicity, of the CTA's thread maxima, from the per-warp top-M lists in shared
// memory (M = 4 or 8, tile_bound_width; exact unless one warp holds more than M of the CTA's top k, in which case
// the result is smaller -- still a valid lower bound of the tile's k-th best score, because thread maxima belong to
// distinct docs).  Every warp computes it redundantly, no extra barrier.
__device__ __forceinline__ u32 cta_kth_bound(const u32 *s_top /*[8][8]*/, u32 k, bool wide = false) {
    const unsigned lane = threadIdx.x & 31;
    u32 v0, v1 = 0;
    if (k <= 10 && !wide) {
        v0 = s_top[(lane >> 2) * 8 + (lane & 3)];
    } else {
        v0 = s_top[lane];
        v1 = s_top[32 + lane];
    }
    u32 kth = 0;
    for (u32 r = 0; r < k; r++) {
        const u32 m0 = __reduce_max_sync(0xffffffffu, max(v0, v1));
        kth = m0;
        if (m0 == 0) break;
        const unsigned holders = __ballot_sync(0xffffffffu, v0 == m0 || v1 == m0);
        if (lane == (unsigned)(__ffs(holders) - 1)) {        // one holder gives up ONE copy
            if (v0 == m0) v0 = 0; else v1 = 0;
        }
    }
    return kth;
}

// Candidate-slot overflow caused by TIES at the tile bound (BM25 scores are a function of (tf, doc_len) only, so
// exact ties among thousands of docs are normal): the tile is still in shared memory, so the CTA collects
// again, now breaking ties the way the final ranking does -- lower doc id first.  Scores above the bound are
// all kept; of the docs AT the bound only those with a local index <= the k-th smallest such index (a bound
// derived from the threads' smallest tied docs, which are distinct docs) are kept: a superset of what the
// top-k can take from this tile.  `negated`: the tile holds -score for scored docs and a positive leftover
// norm elsewhere (term kernel, staged norms).  All SA_TERM_THREADS threads call; returns with the slots,
// *s_ncand and *s_tile_max rewritten (the caller publishes them).  Still more than `slots` -> the caller
// flags the query for the exact host-side re-run, as before.
__device__ __forceinline__ void tile_collect_ties_retry(const float *s_out, bool negated, u32 thr_bits, const TopkCtx &t,
                                                        u64 *__restrict__ my_cand, u32 tile_doc0, u32 *s_top,
                                                        u32 *s_ncand, u32 *s_tile_max) {
    const unsigned tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const float thr_f = __uint_as_float(thr_bits);
    u32 best = 0;                                   // 0xFFFFFFFF - smallest tied local doc of this thread (0 = none)
#pragma unroll
    for (int jj = 0; jj < SA_TILE_DOCS / SA_TERM_THREADS / 4; jj++) {
        const unsigned g = tid + jj * SA_TERM_THREADS;
        const float4 raw = reinterpret_cast<const float4 *>(s_out)[g];
        const float vs[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
        for (int e = 0; e < 4; e++) {
            const float v = negated ? (__float_as_int(vs[e]) < 0 ? -vs[e] : 0.0f) : vs[e];
            if (v == thr_f) best = max(best, 0xFFFFFFFFu - (g * 4 + e));
        }
    }
    const u32 M = 8u;
    __syncthreads();                                // s_top may still be read by a slow warp of the first pass
    {
        u32 v = best;
        for (u32 r = 0; r < M; r++) {
            u32 m = warp_pop_max(v);
            if (lane == r) s_top[warp * 8 + r] = m;
        }
    }
    if (tid == 0) { *s_ncand = 0; *s_tile_max = 0; }
    __syncthreads();
    const u32 kth = cta_kth_bound(s_top, t.k, true);   // 0: fewer than k threads hold a tie -> keep every tie
    const u32 doc_bound = kth ? 0xFFFFFFFFu - kth : 0xFFFFFFFFu;
    u32 cand_max = 0;
#pragma unroll
    for (int jj = 0; jj < SA_TILE_DOCS / SA_TERM_THREADS / 4; jj++) {
        const unsigned g = tid + jj * SA_TERM_THREADS;
        const float4 raw = reinterpret_cast<const float4 *>(s_out)[g];
        const float vs[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
        for (int e = 0; e < 4; e++) {
            const float v = negated ? (__float_as_int(vs[e]) < 0 ? -vs[e] : 0.0f) : vs[e];
            if (v > thr_f || (v == thr_f && g * 4 + e <= doc_bound)) {
                u32 slot = atomicAdd(s_ncand, 1u);
                if (slot < t.slots)
                    my_cand[slot] = ((u64)__float_as_uint(v) << 32) | (u64)(0xFFFFFFFFu - (tile_doc0 + g * 4 + e));
                cand_max = max(cand_max, __float_as_uint(v));
            }
        }
    }
    if (cand_max) atomicMax(s_tile_max, cand_max);
    __syncthreads();
}

// How many of its largest thread maxima every warp publishes for the tile bound.  4 per warp are enough for k <= 10
// when all eight warps hold scores; a tile whose scores sit in two or three warps (a few dozen docs) must publish 8 per
// warp, or fewer than k values exist, the bound degenerates to "keep everything" and 65+ docs overflow the 64 slots.
// `n_holders`: how many threads can hold a score (not how many scores there are).
__device__ __forceinline__ u32 tile_bound_width(u32 k, u32 n_holders) { return (k <= 10 && n_holders >= SA_TERM_THREADS) ? 4u : 8u; }

// Flush one shared-memory score tile to its dense row with 16-byte streaming stores and, on the way,
// collect the tile's top-k candidates (private slots, count, maximum): the same step the term kernel
// ends with, shared with the phrase kernel.  `my_max` = largest score bits this thread put into the
// tile, `n_items` = number of scores in the tile, `n_holders` = how many threads can hold one of them.  All SA_TERM_THREADS threads must call.
__device__ __forceinline__ void flush_tile_collect(const float *s_out, float *__restrict__ out_tile, const TopkCtx &t,
                                                   u32 row, u32 tile, u32 my_max, u32 n_items, u32 n_holders, u32 *s_top,
                                                   u32 *s_ncand, u32 *s_tile_max) {
    const unsigned tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const u32 k = t.k;
    const u32 tile_doc0 = tile * SA_TILE_DOCS;
    const bool need_bound = k && n_items > k;                        // CTA-uniform
    const u32 M = tile_bound_width(k, n_holders);
    if (need_bound) {
        u32 v = my_max;
        for (u32 r = 0; r < M; r++) {
            u32 m = warp_pop_max(v);
            if (lane == r) s_top[warp * 8 + r] = m;
        }
    }
    if (k && tid == 0) { *s_ncand = 0; *s_tile_max = 0; }
    __syncthreads();
    float thr_f = 0.0f;
    if (k) {
        u32 thr = 1u;
        if (need_bound) thr = max(cta_kth_bound(s_top, k, M == 8u), 1u);
        thr_f = __uint_as_float(thr);
    }
    u64 *__restrict__ my_cand = k ? t.tile_cand + ((u64)row * t.n_tiles + tile) * t.slots : nullptr;
    float4 *__restrict__ out4 = reinterpret_cast<float4 *>(out_tile);
    u32 cand_max = 0;
#pragma unroll
    for (int jj = 0; jj < SA_TILE_DOCS / SA_TERM_THREADS / 4; jj++) {
        const unsigned g = tid + jj * SA_TERM_THREADS;
        const float4 v = reinterpret_cast<const float4 *>(s_out)[g];
        __stcs(out4 + g, v);
        if (k && ((v.x >= thr_f) | (v.y >= thr_f) | (v.z >= thr_f) | (v.w >= thr_f))) {
            const float vs[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int e = 0; e < 4; e++) {
                if (vs[e] >= thr_f) {
                    u32 slot = atomicAdd(s_ncand, 1u);
                    if (slot < t.slots)
                        my_cand[slot] = ((u64)__float_as_uint(vs[e]) << 32) | (u64)(0xFFFFFFFFu - (tile_doc0 + g * 4 + e));
                    cand_max = max(cand_max, __float_as_uint(vs[e]));
                }
            }
        }
    }
    if (k) {
        if (cand_max) atomicMax(s_tile_max, cand_max);
        __syncthreads();
        if (*s_ncand > t.slots)                                      // CTA-uniform: ties at the bound (see above)
            tile_collect_ties_retry(s_out, false, __float_as_uint(thr_f), t, my_cand, tile_doc0, s_top, s_ncand, s_tile_max);
        if (tid == 0) {
            const u32 n = *s_ncand;
            const u64 t_idx = (u64)row * t.n_tiles + tile;
            t.tile_cnt[t_idx] = min(n, t.slots);
            t.tile_max[t_idx] = *s_tile_max;
            if (n > t.slots) t.overflow[row] = 1u;
        }
    }
    __syncthreads();
}
#endif
