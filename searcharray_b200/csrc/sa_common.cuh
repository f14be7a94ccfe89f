// sa_common.cuh -- shared definitions for libsearcharray_b200 (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <algorithm>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/searcharray_b200.h"

typedef uint64_t u64;
typedef uint32_t u32;
typedef int64_t i64;

// ---- roaringish bit layout (reference searcharray/roaringish/roaringish.py:30-35) ----
#define SA_KEY_SHIFT 36
#define SA_LSB_BITS 18
#define SA_LSB_MASK 0x3FFFFull
#define SA_HDR_MASK 0xFFFFFFFFFFFC0000ull
#define SA_MSB_MASK 0x0000000FFFFC0000ull
#define SA_BIT17 (1ull << 17)
#define SA_ONE_BLOCK (1ull << SA_LSB_BITS)

#define SA_NUM_SMS_FALLBACK 148

// ---- error plumbing -------------------------------------------------------------
void sa_set_error(const char *fmt, ...);

#define SA_CUDA(call)                                                                  \
    do {                                                                               \
        cudaError_t e_ = (call);                                                       \
        if (e_ != cudaSuccess) {                                                       \
            sa_set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
            return SA_ERR_CUDA;                                                        \
        }                                                                              \
    } while (0)

#define SA_CHECK(cond, ...)                                                            \
    do {                                                                               \
        if (!(cond)) {                                                                 \
            sa_set_error(__VA_ARGS__);                                                 \
            return SA_ERR_ARG;                                                         \
        }                                                                              \
    } while (0)

// ---- a growable device buffer -----------------------------------------------------
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes) {
        if (bytes <= cap) return SA_OK;
        // grow geometrically: cudaFree + cudaMalloc synchronise the device, so a buffer that creeps up
        // query by query must not be reallocated on every new maximum
        const size_t want = std::max(bytes + (bytes >> 3), cap + (cap >> 1)) + 256;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) {
            sa_set_error("cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
            p = nullptr;
            return SA_ERR_NOMEM;
        }
        cap = want;
        return SA_OK;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <typename T> T *as() const { return (T *)p; }
};

// ---- BM25 parameters as the reference passes them to bm25_score ---------------------
struct Bm25Params {
    float idf, avg_doc_len, k1, b, one_minus_b;
    // 1 when a doc with tf == 0 provably scores +0.0f (k1>0, 0<=b<1, finite idf>=+0,
    // doc_lens >= 0, avgdl > 0): the kernel then only touches doc_lens of matching docs.
    // 0 -> the formula is evaluated for every doc like bm25.pyx:20-25 does (NaN/inf/-0.0
    // cases included).
    int sparse_ok;
};

// A query against one shard, as the kernels see it.
#define SA_NO_DIR 0xFFFFFFFFFFFFFFFFull
struct TermQuery {
    u64 word_off;      // offset of the term's first word in d_words
    u64 n_words;       // 0 => unknown term (zeros)
    u64 dir_off;       // offset of the term's tile directory in d_tile_dir (and d_rec_dir), or SA_NO_DIR
    u64 rec_off;       // offset of the term's (doc, tf) records in d_recs, or SA_NO_DIR
    float idf;
    u32 pad;
};

// (doc, tf) record of the per-term tf table: doc index RELATIVE to its 8192-doc tile in the high 13 bits,
// term frequency (sum of the doc's payload popcounts, < 2^18 + 1) in the low 19
#define SA_REC_TF_BITS 19
#define SA_REC_TF_MASK 0x7FFFFu

// ---- the index handle ---------------------------------------------------------------
struct TimedLaunch;
struct BatchState;
struct sa_index {
    int device = 0;
    int num_sms = SA_NUM_SMS_FALLBACK;
    u64 n_docs = 0, n_words = 0, doc_base = 0;
    u32 n_terms = 0;
    bool doc_lens_nonneg = true;
    int upload_mode = 0;             // how the posting words reached HBM (sa_index_upload_mode)

    // HBM-resident index
    u64 *d_words = nullptr;          // [n_words + 1] (one readable pad word)
    float *d_doc_lens = nullptr;     // [n_docs]
    u32 *d_df = nullptr;             // [n_terms] distinct docs per term (this shard)
    // tile directory of long posting lists: for term t with h_dir_off[t] != SA_NO_DIR,
    // d_tile_dir[h_dir_off[t] + j] = index (within the term's list) of the first word whose
    // doc lies in tile >= j, j = 0..n_tiles  (tile = 4096 docs).  Built on the device at upload.
    u32 *d_tile_dir = nullptr;
    std::vector<u64> h_dir_off;
    // per-term tf table (the analogue of the reference's termfreq_cache, middle_out.py:501-509, built on the
    // device at upload): for every term WITH a tile directory, one u32 record per (term, doc) in doc order,
    // (doc - tile_doc0) << 19 | tf; d_rec_dir mirrors d_tile_dir (same offsets) with indices into the records.
    u32 *d_recs = nullptr;
    u32 *d_rec_dir = nullptr;
    std::vector<u64> h_rec_off;
    std::vector<u32> h_max_tile_words;   // per term: the longest per-tile slice of its list (its length without a directory)
    // per-doc BM25 length norm k1*((1-b)+b*dl/avgdl) for the last used (k1, b, avgdl)
    float *d_norm = nullptr;         // [padded n_docs]
    float norm_k1 = 0, norm_b = 0, norm_avgdl = 0;
    bool norm_valid = false;
    // host mirrors for query set-up
    std::vector<u64> h_off, h_len;
    std::vector<u32> h_df;
    std::vector<unsigned char> h_first0;   // 1 = the term's first word sits at (doc 0, block 0): span-search corner

    // sliced-array filter (FilteredPosns semantics)
    u64 n_rows = 0;                  // number of selected rows
    bool rows_active = false;        // a row filter is installed (n_rows may be 0)
    u64 *d_rows = nullptr;           // sorted local doc indices
    unsigned char *d_row_mask = nullptr;  // [n_docs] 1 if doc selected

    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;   // sa_timer_start / sa_timer_stop
    // a batch's top-k selects run here, each overlapping the next chunk's scan (sa_batch_execute_locked); every
    // batch joins back into `stream` before its last kernel
    cudaStream_t select_stream = nullptr;
    cudaEvent_t ev_scan = nullptr, ev_select[2] = {nullptr, nullptr};
    bool profiling = false;
    std::vector<struct TimedLaunch> *pending_timers = nullptr;
    std::vector<cudaEvent_t> *free_events = nullptr;
    struct BatchState *batch = nullptr;
    sa_stats stats;
    std::mutex mu;

    // scratch
    DevBuf dense;        // float [chunk][n_docs_padded]
    DevBuf queries;      // TermQuery[] / phrase descriptors
    DevBuf cand;         // top-k candidates
    DevBuf cand_meta;    // per-query counters / thresholds
    DevBuf topk_out;     // per-query (doc, score) results
    DevBuf phrase_scratch;
    DevBuf phrase_slabs;  // per-CTA scratch of the persistent phrase kernel (merge regime)
    DevBuf filt;         // filtered (sliced / position-filtered) copies of posting lists
    DevBuf misc;
    void *h_pinned = nullptr;   // pinned staging
    size_t h_pinned_cap = 0;

    // NCCL
    void *nccl_comm = nullptr;
    int rank = 0, world = 1;
    DevBuf gather;

    size_t device_bytes = 0;
};

int sa_pinned_reserve(sa_index *ix, size_t bytes);

// Kernel timing without serialising the stream: when profiling is on every timed launch gets
// an event pair from a pool; elapsed times are resolved lazily (sa_stats_get syncs once).
struct TimedLaunch { cudaEvent_t e0, e1; int kind; };   // kind: 0 term, 1 topk, 2 phrase
struct KernelTimer {
    sa_index *ix;
    int kind;
    bool on;
    cudaStream_t stream;             // the launch's stream (ix->stream unless given)
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    KernelTimer(sa_index *ix_, int kind_, cudaStream_t stream_ = nullptr);
    void stop();
};
int sa_resolve_timers(sa_index *ix);

// ---- device helpers -------------------------------------------------------------------
#ifdef __CUDACC__
__device__ __forceinline__ u64 ld_stream_u64(const u64 *p) {
    u64 v;
    asm volatile("ld.global.nc.L1::no_allocate.u64 %0, [%1];" : "=l"(v) : "l"(p));
    return v;
}

// BM25 exactly as bm25.pyx:20-25 evaluates it on x86-64 without FMA contraction:
// every operation individually rounded to nearest-even float32.
__device__ __forceinline__ float bm25_one(float tf, float dl, const Bm25Params &p) {
    float ratio = __fdiv_rn(dl, p.avg_doc_len);
    float norm = __fmul_rn(p.k1, __fadd_rn(p.one_minus_b, __fmul_rn(p.b, ratio)));
    return __fmul_rn(__fdiv_rn(tf, __fadd_rn(tf, norm)), p.idf);
}

// Warp-cooperative lower bound: first index i in [lo, hi) with (a[i] >> shift) >= key,
// 32-ary search (each round probes 32 evenly spaced elements, ballot picks the bucket).
// All lanes must call; all lanes get the result.
__device__ __forceinline__ u64 warp_lower_bound_shifted(const u64 *__restrict__ a, u64 lo, u64 hi,
                                                        u64 key, int shift) {
    const unsigned lane = threadIdx.x & 31;
    while (hi - lo > 32) {
        u64 step = (hi - lo + 31) >> 5;          // ceil(len/32) >= 2
        u64 probe = lo + (u64)(lane + 1) * step - 1;   // last element of bucket `lane`
        bool below = (probe < hi) && ((__ldg(a + probe) >> shift) < key);
        unsigned m = __ballot_sync(0xffffffffu, below);
        int c = __popc(m);                        // buckets entirely below key (monotone)
        lo = lo + (u64)c * step;
        u64 nhi = lo + step;
        hi = nhi < hi ? nhi : hi;
        if (lo > hi) lo = hi;
    }
    u64 idx = lo + lane;
    bool below = (idx < hi) && ((__ldg(a + idx) >> shift) < key);
    unsigned m = __ballot_sync(0xffffffffu, below);
    return lo + (u64)__popc(m);
}
#endif
