// sa_index.cu -- index upload into HBM, per-term document frequencies, and the C-ABI entry
// points of the term path (see include/searcharray_b200.h for the reference mapping).
#include <stdarg.h>
#include <algorithm>
#include <cmath>

#include "sa_term.cuh"
#include "sa_phrase.cuh"
#include "sa_span.cuh"

// ------------------------------------------------------------------ error text
static thread_local char g_err[1024] = "";

void sa_set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

extern "C" const char *sa_last_error(void) { return g_err; }

extern "C" int sa_device_count(int *n_out) {
    SA_CHECK(n_out, "n_out is NULL");
    int n = 0;
    SA_CUDA(cudaGetDeviceCount(&n));
    *n_out = n;
    return SA_OK;
}

extern "C" int sa_host_alloc(void **ptr_out, uint64_t bytes) {
    SA_CHECK(ptr_out, "ptr_out is NULL");
    SA_CUDA(cudaHostAlloc(ptr_out, bytes ? bytes : 1, cudaHostAllocDefault));
    return SA_OK;
}

extern "C" int sa_host_free(void *ptr) {
    if (ptr) SA_CUDA(cudaFreeHost(ptr));
    return SA_OK;
}

int sa_pinned_reserve(sa_index *ix, size_t bytes) {
    if (bytes <= ix->h_pinned_cap) return SA_OK;
    if (ix->h_pinned) cudaFreeHost(ix->h_pinned);
    ix->h_pinned = nullptr;
    ix->h_pinned_cap = 0;
    SA_CUDA(cudaHostAlloc(&ix->h_pinned, bytes, cudaHostAllocDefault));
    ix->h_pinned_cap = bytes;
    return SA_OK;
}

// --------------------------------------------------------------- bulk upload
// SURVEY 8f-2: the posting words usually sit in pageable memory -- a numpy array, or the np.memmap of the
// reference's MemoryMappedArrays `.dat` file (phrase/memmap_arrays.py:145-208).  A plain cudaMemcpy from pageable
// memory crawls through the driver's small staging buffers; instead the source range is page-locked IN PLACE
// (cudaHostRegister, read-only: works on a read-only file mapping too) and copied by DMA at PCIe rate straight from
// the page cache / the array.  If the range cannot be registered (old kernels, exotic mappings) the copy is pipelined
// through two pinned bounce buffers.  mode_out: 0 plain copy (small), 1 registered in place, 2 pinned bounce.
static int upload_bulk(void *dst, const void *src, size_t bytes, cudaStream_t stream, int *mode_out) {
    *mode_out = 0;
    if (bytes == 0) return SA_OK;
    static const bool no_register = getenv("SA_NO_HOST_REGISTER") && atoi(getenv("SA_NO_HOST_REGISTER")) != 0;
    if (bytes >= (32u << 20)) {
        if (!no_register && cudaHostRegister((void *)src, bytes, cudaHostRegisterReadOnly) == cudaSuccess) {
            cudaError_t e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
            cudaHostUnregister((void *)src);
            if (e != cudaSuccess) { sa_set_error("registered upload failed: %s", cudaGetErrorString(e)); return SA_ERR_CUDA; }
            *mode_out = 1;
            return SA_OK;
        }
        cudaGetLastError();                                   // registration refused: clear the error, bounce instead
        const size_t CH = 32u << 20;
        void *pin[2] = {nullptr, nullptr};
        cudaEvent_t ev[2] = {nullptr, nullptr};
        bool ok = cudaHostAlloc(&pin[0], CH, cudaHostAllocDefault) == cudaSuccess &&
                  cudaHostAlloc(&pin[1], CH, cudaHostAllocDefault) == cudaSuccess &&
                  cudaEventCreate(&ev[0]) == cudaSuccess && cudaEventCreate(&ev[1]) == cudaSuccess;
        if (ok) {
            size_t at = 0;
            int b = 0;
            cudaError_t e = cudaSuccess;
            while (at < bytes && e == cudaSuccess) {
                const size_t n = std::min(CH, bytes - at);
                e = cudaEventSynchronize(ev[b]);              // the previous copy out of this buffer is done
                if (e != cudaSuccess) break;
                memcpy(pin[b], (const char *)src + at, n);
                e = cudaMemcpyAsync((char *)dst + at, pin[b], n, cudaMemcpyHostToDevice, stream);
                if (e == cudaSuccess) e = cudaEventRecord(ev[b], stream);
                at += n;
                b ^= 1;
            }
            if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
            for (int i = 0; i < 2; i++) { cudaFreeHost(pin[i]); cudaEventDestroy(ev[i]); }
            if (e != cudaSuccess) { sa_set_error("bounce upload failed: %s", cudaGetErrorString(e)); return SA_ERR_CUDA; }
            *mode_out = 2;
            return SA_OK;
        }
        for (int i = 0; i < 2; i++) { if (pin[i]) cudaFreeHost(pin[i]); if (ev[i]) cudaEventDestroy(ev[i]); }
        cudaGetLastError();
    }
    SA_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, stream));
    return SA_OK;
}

// --------------------------------------------------------------- df at upload
// docfreq = number of distinct doc ids among a term's words (reference: unique(words >> 36)
// .size, roaringish/unique.pyx:87-104 via middle_out.py:521-528).  One thread per word; a word
// is a "doc head" when it starts its term or its doc id differs from its predecessor's.
__global__ void df_kernel(const u64 *__restrict__ words, u64 n_words,
                          const u64 *__restrict__ term_off_sorted, const u32 *__restrict__ term_of_slot,
                          u32 n_slots, u32 *__restrict__ df) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = i < n_words;
    // slot = last j with term_off_sorted[j] <= i   (slots cover [off, off+len) disjointly)
    u32 lo = 0, hi = n_slots;
    bool head = false;
    if (live) {
        while (hi - lo > 1) {
            u32 mid = (lo + hi) >> 1;
            if (term_off_sorted[mid] <= i) lo = mid; else hi = mid;
        }
        const u64 start = term_off_sorted[lo];
        head = (i == start) || ((words[i] >> SA_KEY_SHIFT) != (words[i - 1] >> SA_KEY_SHIFT));
    }
    // a warp's 32 consecutive words almost always belong to one term: one atomic per (warp, term) instead of one
    // per doc head (a billion same-address atomics on a 10M-doc index)
    const unsigned heads = __ballot_sync(0xffffffffu, head);
    if (heads == 0) return;
    const unsigned peers = __match_any_sync(0xffffffffu, live ? lo : 0xFFFFFFFFu);
    const unsigned mine = heads & peers;
    if (live && mine && (threadIdx.x & 31) == (unsigned)(__ffs(peers) - 1)) atomicAdd(&df[term_of_slot[lo]], (u32)__popc(mine));
}

// Tile directory of a long posting list: dir[j] = index (within the list) of the first word whose
// doc falls in tile >= j, for j = 0..n_tiles.  One thread per word fills the entries it starts.
__global__ void tile_dir_kernel(const u64 *__restrict__ words, u64 n_words,
                                const u64 *__restrict__ term_off_sorted, const u64 *__restrict__ slot_len,
                                const u64 *__restrict__ slot_dir_off, u32 n_slots,
                                u32 *__restrict__ dir, u64 doc_base, u32 n_tiles) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_words) return;
    u32 lo = 0, hi = n_slots;
    while (hi - lo > 1) {
        u32 mid = (lo + hi) >> 1;
        if (term_off_sorted[mid] <= i) lo = mid; else hi = mid;
    }
    const u64 doff = slot_dir_off[lo];
    if (doff == SA_NO_DIR) return;
    const u64 start = term_off_sorted[lo], len = slot_len[lo];
    const u32 local = (u32)(i - start);
    u32 *d = dir + doff;
    const u32 t_i = (u32)(((words[i] >> SA_KEY_SHIFT) - doc_base) / SA_TILE_DOCS);
    if (local == 0) {
        for (u32 t = 0; t <= t_i && t <= n_tiles; t++) d[t] = 0;
    } else {
        const u32 t_p = (u32)(((words[i - 1] >> SA_KEY_SHIFT) - doc_base) / SA_TILE_DOCS);
        for (u32 t = t_p + 1; t <= t_i && t <= n_tiles; t++) d[t] = local;
    }
    if (local == len - 1)
        for (u32 t = t_i + 1; t <= n_tiles; t++) d[t] = (u32)len;
}

// longest per-tile slice of every list that has a directory (sizes the merge regime's per-CTA scratch)
__global__ void dir_max_kernel(const u32 *__restrict__ dir, const u64 *__restrict__ slot_dir_off, u32 n_slots, u32 n_tiles,
                               u32 *__restrict__ slot_max) {
    const u32 slot = blockIdx.x;                 // (terms can outnumber the 65,535 limit of grid.y)
    if (slot >= n_slots || slot_dir_off[slot] == SA_NO_DIR) return;
    const u32 *d = dir + slot_dir_off[slot];
    u32 m = 0;
    for (u32 t = blockIdx.y * blockDim.x + threadIdx.x; t < n_tiles; t += gridDim.y * blockDim.x) m = max(m, d[t + 1] - d[t]);
    m = __reduce_max_sync(0xffffffffu, m);
    if ((threadIdx.x & 31) == 0 && m) atomicMax(&slot_max[slot], m);
}

// ---- tf table (see sa_index::d_recs).  Pass 1 counts the doc heads of every 1024-word block, a one-CTA scan
// turns the counts into ranks, pass 2 writes each head's record at (term's record offset + rank within the
// term) and fills the term's record directory like tile_dir_kernel fills the word directory.
#define REC_BLOCK 1024
__device__ __forceinline__ u32 slot_of_word(const u64 *__restrict__ term_off_sorted, u32 n_slots, u64 i) {
    u32 lo = 0, hi = n_slots;
    while (hi - lo > 1) {
        u32 mid = (lo + hi) >> 1;
        if (term_off_sorted[mid] <= i) lo = mid; else hi = mid;
    }
    return lo;
}

__global__ void __launch_bounds__(256)
rec_count_kernel(const u64 *__restrict__ words, u64 n_words, const u64 *__restrict__ term_off_sorted, u32 n_slots,
                 u32 *__restrict__ bcount) {
    __shared__ u32 s_cnt;
    if (threadIdx.x == 0) s_cnt = 0;
    __syncthreads();
    u32 mine = 0;
    for (int e = 0; e < REC_BLOCK / 256; e++) {
        const u64 i = (u64)blockIdx.x * REC_BLOCK + e * 256 + threadIdx.x;
        if (i >= n_words) break;
        const u64 start = term_off_sorted[slot_of_word(term_off_sorted, n_slots, i)];
        if (i == start || (words[i] >> SA_KEY_SHIFT) != (words[i - 1] >> SA_KEY_SHIFT)) mine++;
    }
    mine = __reduce_add_sync(0xffffffffu, mine);
    if ((threadIdx.x & 31) == 0 && mine) atomicAdd(&s_cnt, mine);
    __syncthreads();
    if (threadIdx.x == 0) bcount[blockIdx.x] = s_cnt;
}

// exclusive scan of u64-accumulated u32 counts by ONE CTA (n ~ 1e6 entries: a few hundred microseconds)
__global__ void __launch_bounds__(1024)
rec_scan_kernel(const u32 *__restrict__ bcount, u64 *__restrict__ bbase, u32 n) {
    __shared__ u64 warp_sums[32];
    __shared__ u64 carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (u32 b0 = 0; b0 < n; b0 += 1024) {
        const u32 i = b0 + threadIdx.x;
        const u64 v = i < n ? bcount[i] : 0;
        const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        u64 incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            u64 t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) warp_sums[warp] = incl;
        __syncthreads();
        u64 wbase = 0, tot = 0;
        for (int w = 0; w < 32; w++) {
            if (w < (int)warp) wbase += warp_sums[w];
            tot += warp_sums[w];
        }
        const u64 c = carry;
        if (i < n) bbase[i] = c + wbase + incl - v;
        __syncthreads();
        if (threadIdx.x == 0) carry = c + tot;
        __syncthreads();
    }
}

__global__ void __launch_bounds__(256)
rec_write_kernel(const u64 *__restrict__ words, u64 n_words, const u64 *__restrict__ term_off_sorted,
                 const u64 *__restrict__ slot_len, const u64 *__restrict__ slot_dir_off,
                 const u64 *__restrict__ slot_rec_off, const u64 *__restrict__ slot_head_base,
                 const u32 *__restrict__ slot_df, u32 n_slots, const u64 *__restrict__ bbase,
                 u32 *__restrict__ recs, u32 *__restrict__ rec_dir, u64 doc_base, u32 n_tiles) {
    __shared__ u32 s_warp[8];
    __shared__ u32 s_run;
    if (threadIdx.x == 0) s_run = 0;
    __syncthreads();
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int e = 0; e < REC_BLOCK / 256; e++) {
        const u64 i = (u64)blockIdx.x * REC_BLOCK + e * 256 + threadIdx.x;
        bool head = false;
        u32 slot = 0;
        u64 start = 0, w = 0;
        if (i < n_words) {
            slot = slot_of_word(term_off_sorted, n_slots, i);
            start = term_off_sorted[slot];
            w = words[i];
            head = (i == start) || ((w >> SA_KEY_SHIFT) != (words[i - 1] >> SA_KEY_SHIFT));
        }
        // rank of this head among the block's heads (block-wide exclusive scan of the head flags)
        const unsigned m = __ballot_sync(0xffffffffu, head);
        if (lane == 0) s_warp[warp] = __popc(m);
        __syncthreads();
        u32 before = s_run;
        for (unsigned x = 0; x < warp; x++) before += s_warp[x];
        u32 round_total = 0;
        for (unsigned x = 0; x < 8; x++) round_total += s_warp[x];
        const u64 g = bbase[blockIdx.x] + before + __popc(m & ((1u << lane) - 1u));   // global head rank
        __syncthreads();
        if (threadIdx.x == 0) s_run += round_total;
        if (i < n_words && slot_dir_off[slot] != SA_NO_DIR) {
            const u64 len = slot_len[slot];
            const u64 doc = (w >> SA_KEY_SHIFT) - doc_base;
            const u32 t_i = (u32)(doc / SA_TILE_DOCS);
            u32 *d = rec_dir + slot_dir_off[slot];
            if (head) {
                const u32 rank = (u32)(g - slot_head_base[slot]);                     // within the term
                u32 tf = 0;
                for (u64 j = i; j < start + len; j++) {                                // the doc's run of words
                    const u64 w2 = words[j];
                    if ((w2 >> SA_KEY_SHIFT) != (w >> SA_KEY_SHIFT)) break;
                    tf += (u32)__popcll(w2 & SA_LSB_MASK);
                }
                recs[slot_rec_off[slot] + rank] = ((u32)(doc % SA_TILE_DOCS) << SA_REC_TF_BITS) | (tf & SA_REC_TF_MASK);
                if (i == start) {
                    for (u32 t = 0; t <= t_i && t <= n_tiles; t++) d[t] = 0;
                } else {
                    const u32 t_p = (u32)(((words[i - 1] >> SA_KEY_SHIFT) - doc_base) / SA_TILE_DOCS);
                    for (u32 t = t_p + 1; t <= t_i && t <= n_tiles; t++) d[t] = rank;
                }
            }
            if (i == start + len - 1)
                for (u32 t = t_i + 1; t <= n_tiles; t++) d[t] = slot_df[slot];
        }
    }
}

extern "C" int sa_index_create(const uint64_t *words, uint64_t n_words,
                               const uint64_t *term_offsets, const uint64_t *term_lengths, uint32_t n_terms,
                               const float *doc_lens, uint64_t n_docs, uint64_t doc_base,
                               int device, sa_index **index_out) {
    SA_CHECK(index_out, "index_out is NULL");
    SA_CHECK(n_words == 0 || words, "words is NULL");
    SA_CHECK(n_terms == 0 || (term_offsets && term_lengths), "term tables are NULL");
    SA_CHECK(n_docs == 0 || doc_lens, "doc_lens is NULL");
    SA_CHECK(doc_base + n_docs <= (1ull << 28), "doc ids exceed the 28-bit key space");
    for (u32 t = 0; t < n_terms; t++)
        SA_CHECK(term_offsets[t] + term_lengths[t] <= n_words, "term %u slice out of range", t);
    SA_CUDA(cudaSetDevice(device));

    sa_index *ix = new sa_index();
    ix->device = device;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) ix->num_sms = prop.multiProcessorCount;
    ix->n_docs = n_docs;
    ix->n_words = n_words;
    ix->n_terms = n_terms;
    ix->doc_base = doc_base;
    memset(&ix->stats, 0, sizeof(ix->stats));
    ix->h_off.assign(term_offsets, term_offsets + n_terms);
    ix->h_len.assign(term_lengths, term_lengths + n_terms);
    ix->h_df.assign(n_terms, 0);
    ix->h_dir_off.assign(n_terms, SA_NO_DIR);
    ix->h_first0.assign(n_terms, 0);
    ix->h_max_tile_words.assign(n_terms, 0);
    ix->h_rec_off.assign(n_terms, SA_NO_DIR);
    for (u32 t = 0; t < n_terms; t++)
        if (term_lengths[t] && (words[term_offsets[t]] & SA_HDR_MASK) == 0) ix->h_first0[t] = 1;

#define CREATE_CUDA(call)                                                              \
    do {                                                                               \
        cudaError_t e_ = (call);                                                       \
        if (e_ != cudaSuccess) {                                                       \
            sa_set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
            sa_index_destroy(ix);                                                      \
            return SA_ERR_CUDA;                                                        \
        }                                                                              \
    } while (0)

    CREATE_CUDA(cudaStreamCreateWithFlags(&ix->stream, cudaStreamNonBlocking));
    CREATE_CUDA(cudaEventCreate(&ix->ev0));
    CREATE_CUDA(cudaEventCreate(&ix->ev1));
    CREATE_CUDA(cudaMalloc(&ix->d_words, (n_words + 4) * sizeof(u64)));
    CREATE_CUDA(cudaMemsetAsync(ix->d_words + n_words, 0, 4 * sizeof(u64), ix->stream));
    if (n_words && upload_bulk(ix->d_words, words, n_words * sizeof(u64), ix->stream, &ix->upload_mode) != SA_OK) {
        sa_index_destroy(ix);
        return SA_ERR_CUDA;
    }
    CREATE_CUDA(cudaMalloc(&ix->d_doc_lens, (n_docs + 1) * sizeof(float)));
    if (n_docs)
        CREATE_CUDA(cudaMemcpyAsync(ix->d_doc_lens, doc_lens, n_docs * sizeof(float), cudaMemcpyHostToDevice, ix->stream));
    CREATE_CUDA(cudaMalloc(&ix->d_df, (size_t)(n_terms + 1) * sizeof(u32)));
    CREATE_CUDA(cudaMemsetAsync(ix->d_df, 0, (size_t)(n_terms + 1) * sizeof(u32), ix->stream));
    ix->device_bytes = (n_words + 1) * sizeof(u64) + (n_docs + 1) * sizeof(float) + (size_t)(n_terms + 1) * 4;

    ix->doc_lens_nonneg = true;
    for (u64 i = 0; i < n_docs; i++)
        if (!(doc_lens[i] >= 0.0f)) { ix->doc_lens_nonneg = false; break; }

    // df per term on the device
    if (n_words && n_terms) {
        std::vector<u32> order;
        order.reserve(n_terms);
        for (u32 t = 0; t < n_terms; t++) if (term_lengths[t]) order.push_back(t);
        std::sort(order.begin(), order.end(), [&](u32 a, u32 b) { return term_offsets[a] < term_offsets[b]; });
        // slices must be disjoint for the head test to be per-term; also cover gaps
        std::vector<u64> off_sorted;
        std::vector<u32> term_of_slot;
        u64 covered = 0;
        bool full_cover = true;
        for (u32 t : order) {
            if (term_offsets[t] != covered) { full_cover = false; break; }
            off_sorted.push_back(term_offsets[t]);
            term_of_slot.push_back(t);
            covered += term_lengths[t];
        }
        if (!full_cover || covered != n_words) {
            sa_set_error("term slices must tile `words` exactly (ArrayDict.compact layout)");
            sa_index_destroy(ix);
            return SA_ERR_ARG;
        }
        u64 *d_off = nullptr;
        u32 *d_slot = nullptr;
        u32 n_slots = (u32)off_sorted.size();
        // tile directories for long lists (short ones are searched: they stay cache resident)
        const u32 n_tiles = (u32)((n_docs + SA_TILE_DOCS - 1) / SA_TILE_DOCS);
        const u64 dir_min_words = std::max<u64>(1024, n_tiles / 2);
        std::vector<u64> slot_len(n_slots), slot_dir(n_slots, SA_NO_DIR);
        u64 dir_words = 0;
        for (u32 sI = 0; sI < n_slots; sI++) {
            u32 t = term_of_slot[sI];
            slot_len[sI] = term_lengths[t];
            if (term_lengths[t] >= dir_min_words && term_lengths[t] < 0xFFFFFFFFull) {
                slot_dir[sI] = dir_words;
                ix->h_dir_off[t] = dir_words;
                dir_words += (u64)n_tiles + 1;
            }
        }
        CREATE_CUDA(cudaMalloc(&d_off, n_slots * sizeof(u64)));
        CREATE_CUDA(cudaMalloc(&d_slot, n_slots * sizeof(u32)));
        CREATE_CUDA(cudaMemcpyAsync(d_off, off_sorted.data(), n_slots * sizeof(u64), cudaMemcpyHostToDevice, ix->stream));
        CREATE_CUDA(cudaMemcpyAsync(d_slot, term_of_slot.data(), n_slots * sizeof(u32), cudaMemcpyHostToDevice, ix->stream));
        unsigned blocks = (unsigned)((n_words + 255) / 256);
        df_kernel<<<blocks, 256, 0, ix->stream>>>(ix->d_words, n_words, d_off, d_slot, n_slots, ix->d_df);
        CREATE_CUDA(cudaGetLastError());
        ix->stats.total_launches++;
        CREATE_CUDA(cudaMemcpyAsync(ix->h_df.data(), ix->d_df, n_terms * sizeof(u32), cudaMemcpyDeviceToHost, ix->stream));
        u64 *d_slot_len = nullptr, *d_slot_dir = nullptr;
        if (dir_words) {
            CREATE_CUDA(cudaMalloc(&ix->d_tile_dir, dir_words * sizeof(u32)));
            ix->device_bytes += dir_words * sizeof(u32);
            CREATE_CUDA(cudaMalloc(&d_slot_len, n_slots * sizeof(u64)));
            CREATE_CUDA(cudaMalloc(&d_slot_dir, n_slots * sizeof(u64)));
            CREATE_CUDA(cudaMemcpyAsync(d_slot_len, slot_len.data(), n_slots * sizeof(u64), cudaMemcpyHostToDevice, ix->stream));
            CREATE_CUDA(cudaMemcpyAsync(d_slot_dir, slot_dir.data(), n_slots * sizeof(u64), cudaMemcpyHostToDevice, ix->stream));
            tile_dir_kernel<<<blocks, 256, 0, ix->stream>>>(ix->d_words, n_words, d_off, d_slot_len, d_slot_dir, n_slots,
                                                           ix->d_tile_dir, doc_base, n_tiles);
            CREATE_CUDA(cudaGetLastError());
            ix->stats.total_launches++;
        }
        ix->h_max_tile_words.assign(n_terms, 0);
        for (u32 t = 0; t < n_terms; t++) ix->h_max_tile_words[t] = (u32)std::min<u64>(term_lengths[t], 0xFFFFFFFFull);
        std::vector<u32> slot_max(n_slots, 0);
        u32 *d_slot_max = nullptr;
        if (dir_words) {
            CREATE_CUDA(cudaMalloc(&d_slot_max, n_slots * sizeof(u32)));
            CREATE_CUDA(cudaMemsetAsync(d_slot_max, 0, n_slots * sizeof(u32), ix->stream));
            dir_max_kernel<<<dim3(n_slots, std::min<u32>(32, (n_tiles + 255) / 256)), 256, 0, ix->stream>>>(
                ix->d_tile_dir, d_slot_dir, n_slots, n_tiles, d_slot_max);
            CREATE_CUDA(cudaGetLastError());
            ix->stats.total_launches++;
            CREATE_CUDA(cudaMemcpyAsync(slot_max.data(), d_slot_max, n_slots * sizeof(u32), cudaMemcpyDeviceToHost, ix->stream));
        }
        CREATE_CUDA(cudaStreamSynchronize(ix->stream));         // h_df is final from here on
        if (dir_words) {
            for (u32 sI = 0; sI < n_slots; sI++)
                if (slot_dir[sI] != SA_NO_DIR) ix->h_max_tile_words[term_of_slot[sI]] = slot_max[sI];
            cudaFree(d_slot_max);
        }
        // tf table for the terms that have a directory (the long lists: that is where the scan's time goes)
        static const bool no_tf_table = getenv("SA_NO_TF_TABLE") && atoi(getenv("SA_NO_TF_TABLE")) != 0;
        ix->h_rec_off.assign(n_terms, SA_NO_DIR);
        if (dir_words && !no_tf_table) {
            std::vector<u64> slot_rec(n_slots, SA_NO_DIR), slot_head_base(n_slots, 0);
            std::vector<u32> slot_df(n_slots, 0);
            u64 total_recs = 0, heads = 0;
            for (u32 sI = 0; sI < n_slots; sI++) {
                const u32 t = term_of_slot[sI];
                slot_head_base[sI] = heads;
                slot_df[sI] = ix->h_df[t];
                heads += ix->h_df[t];
                if (slot_dir[sI] != SA_NO_DIR) {
                    slot_rec[sI] = total_recs;
                    ix->h_rec_off[t] = total_recs;
                    total_recs += ((u64)ix->h_df[t] + 3) / 4 * 4;          // 16-byte aligned record runs
                }
            }
            const u32 n_rblocks = (u32)((n_words + REC_BLOCK - 1) / REC_BLOCK);
            u32 *d_bcount = nullptr, *d_slot_df = nullptr;
            u64 *d_bbase = nullptr, *d_slot_rec = nullptr, *d_slot_hb = nullptr;
            CREATE_CUDA(cudaMalloc(&ix->d_recs, (total_recs + 8) * sizeof(u32)));
            CREATE_CUDA(cudaMemsetAsync(ix->d_recs, 0, (total_recs + 8) * sizeof(u32), ix->stream));
            CREATE_CUDA(cudaMalloc(&ix->d_rec_dir, dir_words * sizeof(u32)));
            ix->device_bytes += (total_recs + 8) * sizeof(u32) + dir_words * sizeof(u32);
            CREATE_CUDA(cudaMalloc(&d_bcount, (size_t)n_rblocks * sizeof(u32)));
            CREATE_CUDA(cudaMalloc(&d_bbase, (size_t)n_rblocks * sizeof(u64)));
            CREATE_CUDA(cudaMalloc(&d_slot_rec, n_slots * sizeof(u64)));
            CREATE_CUDA(cudaMalloc(&d_slot_hb, n_slots * sizeof(u64)));
            CREATE_CUDA(cudaMalloc(&d_slot_df, n_slots * sizeof(u32)));
            CREATE_CUDA(cudaMemcpyAsync(d_slot_rec, slot_rec.data(), n_slots * sizeof(u64), cudaMemcpyHostToDevice, ix->stream));
            CREATE_CUDA(cudaMemcpyAsync(d_slot_hb, slot_head_base.data(), n_slots * sizeof(u64), cudaMemcpyHostToDevice, ix->stream));
            CREATE_CUDA(cudaMemcpyAsync(d_slot_df, slot_df.data(), n_slots * sizeof(u32), cudaMemcpyHostToDevice, ix->stream));
            rec_count_kernel<<<n_rblocks, 256, 0, ix->stream>>>(ix->d_words, n_words, d_off, n_slots, d_bcount);
            rec_scan_kernel<<<1, 1024, 0, ix->stream>>>(d_bcount, d_bbase, n_rblocks);
            rec_write_kernel<<<n_rblocks, 256, 0, ix->stream>>>(ix->d_words, n_words, d_off, d_slot_len, d_slot_dir, d_slot_rec,
                                                                d_slot_hb, d_slot_df, n_slots, d_bbase, ix->d_recs, ix->d_rec_dir,
                                                                doc_base, n_tiles);
            CREATE_CUDA(cudaGetLastError());
            ix->stats.total_launches += 3;
            CREATE_CUDA(cudaStreamSynchronize(ix->stream));
            cudaFree(d_bcount); cudaFree(d_bbase); cudaFree(d_slot_rec); cudaFree(d_slot_hb); cudaFree(d_slot_df);
        }
        cudaFree(d_off);
        cudaFree(d_slot);
        cudaFree(d_slot_len);
        cudaFree(d_slot_dir);
    } else {
        CREATE_CUDA(cudaStreamSynchronize(ix->stream));
    }
#undef CREATE_CUDA
    *index_out = ix;
    return SA_OK;
}

void sa_free_batch(sa_index *ix);

extern "C" int sa_index_destroy(sa_index *ix) {
    if (!ix) return SA_OK;
    cudaSetDevice(ix->device);
    if (ix->stream) cudaStreamSynchronize(ix->stream);
    sa_comm_destroy(ix);
    cudaFree(ix->d_words);
    cudaFree(ix->d_doc_lens);
    cudaFree(ix->d_df);
    cudaFree(ix->d_tile_dir);
    cudaFree(ix->d_recs);
    cudaFree(ix->d_rec_dir);
    cudaFree(ix->d_norm);
    cudaFree(ix->d_rows);
    cudaFree(ix->d_row_mask);
    ix->dense.release();
    ix->queries.release();
    ix->cand.release();
    ix->cand_meta.release();
    ix->topk_out.release();
    ix->phrase_scratch.release();
    ix->phrase_slabs.release();
    ix->filt.release();
    ix->misc.release();
    ix->gather.release();
    sa_free_batch(ix);
    if (ix->pending_timers) {
        for (auto &t : *ix->pending_timers) { cudaEventDestroy(t.e0); cudaEventDestroy(t.e1); }
        delete ix->pending_timers;
    }
    if (ix->free_events) {
        for (auto e : *ix->free_events) cudaEventDestroy(e);
        delete ix->free_events;
    }
    if (ix->h_pinned) cudaFreeHost(ix->h_pinned);
    if (ix->ev0) cudaEventDestroy(ix->ev0);
    if (ix->ev1) cudaEventDestroy(ix->ev1);
    if (ix->ev_scan) cudaEventDestroy(ix->ev_scan);
    for (cudaEvent_t e : ix->ev_select) if (e) cudaEventDestroy(e);
    if (ix->select_stream) cudaStreamDestroy(ix->select_stream);
    if (ix->stream) cudaStreamDestroy(ix->stream);
    delete ix;
    return SA_OK;
}

extern "C" int sa_index_info(const sa_index *ix, uint64_t *n_docs, uint64_t *n_words,
                             uint32_t *n_terms, uint64_t *device_bytes) {
    SA_CHECK(ix, "index is NULL");
    if (n_docs) *n_docs = ix->n_docs;
    if (n_words) *n_words = ix->n_words;
    if (n_terms) *n_terms = ix->n_terms;
    if (device_bytes) *device_bytes = ix->device_bytes;
    return SA_OK;
}

extern "C" int sa_index_upload_mode(const sa_index *ix, int *mode_out) {
    SA_CHECK(ix && mode_out, "NULL argument");
    *mode_out = ix->upload_mode;
    return SA_OK;
}

extern "C" int sa_docfreq(sa_index *ix, uint32_t term_id, uint64_t *df_out) {
    SA_CHECK(ix && df_out, "NULL argument");
    if (term_id == SA_NO_TERM) { *df_out = 0; return SA_OK; }
    SA_CHECK(term_id < ix->n_terms, "term id %u out of range", term_id);
    *df_out = ix->h_df[term_id];
    return SA_OK;
}

extern "C" int sa_stats_reset(sa_index *ix) {
    SA_CHECK(ix, "index is NULL");
    std::lock_guard<std::mutex> g(ix->mu);
    sa_resolve_timers(ix);
    memset(&ix->stats, 0, sizeof(ix->stats));
    return SA_OK;
}

extern "C" int sa_stats_get(sa_index *ix, sa_stats *out) {
    SA_CHECK(ix && out, "NULL argument");
    std::lock_guard<std::mutex> g(ix->mu);
    int rc = sa_resolve_timers(ix);
    if (rc) return rc;
    *out = ix->stats;
    return SA_OK;
}

extern "C" int sa_set_profiling(sa_index *ix, int enabled) {
    SA_CHECK(ix, "index is NULL");
    std::lock_guard<std::mutex> g(ix->mu);
    ix->profiling = enabled != 0;
    return SA_OK;
}

// ----------------------------------------------------------------- term path
static Bm25Params make_bm25(const sa_index *ix, float idf, float avg_doc_len, float k1, float b) {
    Bm25Params p;
    p.idf = idf;
    p.avg_doc_len = avg_doc_len;
    p.k1 = k1;
    p.b = b;
    p.one_minus_b = 1 - b;       // float arithmetic, as `cdef float one_minus_b = 1 - b` (bm25.pyx:19)
    p.sparse_ok = (ix->doc_lens_nonneg && k1 > 0.0f && std::isfinite(k1) && b >= 0.0f && b < 1.0f &&
                   avg_doc_len > 0.0f && std::isfinite(avg_doc_len) && std::isfinite(idf) &&
                   idf >= 0.0f && !std::signbit(idf)) ? 1 : 0;
    return p;
}

static u64 padded_docs(u64 n_docs) { return (n_docs + SA_TILE_DOCS - 1) / SA_TILE_DOCS * SA_TILE_DOCS; }

int sa_filter_terms(sa_index *ix, const uint32_t *term_ids, uint32_t n_terms, bool use_rows,
                    u64 pay_lo, u64 pay_hi, bool use_payload, std::vector<u64> &offs, std::vector<u64> &lens);
int sa_gather_rows(sa_index *ix, const float *d_dense, float *out_host);

static int single_term(sa_index *ix, uint32_t term_id, int mode, const Bm25Params &p,
                       u64 min_payload, u64 max_payload, float *out_host) {
    SA_CHECK(ix && out_host, "NULL argument");
    SA_CHECK(term_id == SA_NO_TERM || term_id < ix->n_terms, "term id %u out of range", term_id);
    std::lock_guard<std::mutex> g(ix->mu);
    SA_CUDA(cudaSetDevice(ix->device));
    if (ix->n_docs == 0) return SA_OK;
    const bool rows = ix->rows_active;
    SA_CHECK(!(rows && mode == TERM_MODE_SCORE), "score on a sliced array: call termfreqs + bm25 (the Python layer does)");
    const u64 stride = padded_docs(ix->n_docs);
    int rc = ix->dense.reserve(stride * sizeof(float));
    if (rc) return rc;
    rc = ix->queries.reserve(sizeof(TermQuery));
    if (rc) return rc;
    TermQuery tq;
    memset(&tq, 0, sizeof(tq));
    tq.word_off = term_id == SA_NO_TERM ? 0 : ix->h_off[term_id];
    tq.n_words = term_id == SA_NO_TERM ? 0 : ix->h_len[term_id];
    tq.dir_off = term_id == SA_NO_TERM ? SA_NO_DIR : ix->h_dir_off[term_id];
    tq.rec_off = (term_id == SA_NO_TERM || ix->h_rec_off.empty()) ? SA_NO_DIR : ix->h_rec_off[term_id];
    tq.idf = p.idf;
    const u64 *words = ix->d_words;
    bool filter = !(min_payload == 0 && max_payload == SA_ALL_BITS);
    if (rows && term_id != SA_NO_TERM) {
        // sliced array: run on the materialised FilteredPosns list (rows and block filter applied)
        std::vector<u64> offs, lens;
        if ((rc = sa_filter_terms(ix, &term_id, 1, true, min_payload, max_payload, filter, offs, lens))) return rc;
        words = ix->filt.as<u64>();
        tq.word_off = offs[0];
        tq.n_words = lens[0];
        tq.dir_off = SA_NO_DIR;
        tq.rec_off = SA_NO_DIR;
        filter = false;
    }
    SA_CUDA(cudaMemcpyAsync(ix->queries.p, &tq, sizeof(tq), cudaMemcpyHostToDevice, ix->stream));
    TermBatchArgs a;
    memset(&a, 0, sizeof(a));
    a.words = words;
    a.doc_lens = ix->d_doc_lens;
    a.n_docs = ix->n_docs;
    a.doc_base = ix->doc_base;
    a.queries = ix->queries.as<TermQuery>();
    a.out = ix->dense.as<float>();
    a.out_stride = stride;
    a.bm25 = p;
    a.min_payload = min_payload;
    a.max_payload = max_payload;
    a.filter = filter;
    a.mode = mode;
    a.topk.k = 0;
    rc = launch_term_batch(ix, a, 1);
    if (rc) return rc;
    if (rows) return sa_gather_rows(ix, ix->dense.as<float>(), out_host);
    SA_CUDA(cudaMemcpyAsync(out_host, ix->dense.p, ix->n_docs * sizeof(float), cudaMemcpyDeviceToHost, ix->stream));
    SA_CUDA(cudaStreamSynchronize(ix->stream));
    return SA_OK;
}

extern "C" int sa_termfreqs(sa_index *ix, uint32_t term_id, uint64_t min_payload, uint64_t max_payload,
                            float *out_host) {
    SA_CHECK(ix, "index is NULL");
    Bm25Params p = make_bm25(ix, 0, 1, 1, 0);
    return single_term(ix, term_id, TERM_MODE_TF, p, min_payload, max_payload, out_host);
}

extern "C" int sa_score_term(sa_index *ix, uint32_t term_id, float idf, float avg_doc_len,
                             float k1, float b, uint64_t min_payload, uint64_t max_payload,
                             float *out_host) {
    SA_CHECK(ix, "index is NULL");
    if (avg_doc_len == 0.0f) {   // similarity.py:31-32: zeros_like(term_freqs)
        SA_CHECK(out_host, "out is NULL");
        memset(out_host, 0, ix->n_docs * sizeof(float));
        return SA_OK;
    }
    Bm25Params p = make_bm25(ix, idf, avg_doc_len, k1, b);
    return single_term(ix, term_id, TERM_MODE_SCORE, p, min_payload, max_payload, out_host);
}

// ------------------------------------------------ batched, HBM-resident top-k
// A prepared batch: query descriptors live in HBM; sa_batch_execute only enqueues kernels.
// Queries are processed in chunks (bounded dense-vector memory).  Inside a chunk the term queries
// take dense rows [0, nT) (one fused launch) and the phrase queries rows [nT, nT + nP) (phrase
// kernel + tile scan); one select launch covers the chunk and writes each result at its
// original query index.
struct BatchChunk {
    u32 row0 = 0;          // first row (in the permuted "row space") of this chunk
    u32 n_term = 0, n_phrase = 0;
    u32 term0 = 0, phrase0 = 0;     // offsets into the batch-wide TermQuery / PhraseQuery arrays
    Bm25Params params;
    u32 phrase_chunks = 1;          // doc-range chunks per phrase query
    u64 arena_words = 64;
    // phrase queries by regime (indices relative to phrase0, stored at B.d_sel + sel0: search first, then staged)
    u32 sel0 = 0, n_search = 0, n_staged = 0, staged_chunks = 1;
    u64 slab_cap = 0;
};

struct BatchState {
    u32 nq = 0, k = 0, slots = 0, chunk = 0, slop = 0;
    float avg_doc_len = 0, k1 = 0, b = 0;
    bool ready = false;
    bool executed = false;                    // the dense rows hold the last chunk (sa_batch_row)
    std::vector<TermQuery> tqs;               // all term queries, chunk by chunk
    std::vector<PhraseQuery> pqs;             // all phrase queries, chunk by chunk
    std::vector<u32> row_query;               // row -> original query index
    std::vector<u32> term_query, phrase_query;  // index in tqs / pqs -> original query index
    std::vector<u32> phrase_missing;          // 1 = a term is unknown: result stays empty
    std::vector<BatchChunk> chunks;
    // slop > 0: the multi-term queries are span queries (one plan per chunk, descriptors concatenated)
    std::vector<SpanPlan> span_plans;
    std::vector<float> span_idf;
    DevBuf d_sq, d_scounts, d_sidf;
    DevBuf d_tq, d_pq, d_row_query;
    DevBuf d_meta;                            // u32 overflow[nq] (row space)
    DevBuf d_pstats;                          // PhraseStats[#phrase queries]
    std::vector<u32> sel;                     // per chunk: search-regime then merge-regime phrase indices
    DevBuf d_sel;
    DevBuf d_missing;                         // phrase_missing on the device (batch_summary_kernel)
};

static TermQuery make_term_query(const sa_index *ix, u32 t, float idf) {
    TermQuery tq;
    memset(&tq, 0, sizeof(tq));
    tq.word_off = t == SA_NO_TERM ? 0 : ix->h_off[t];
    tq.n_words = t == SA_NO_TERM ? 0 : ix->h_len[t];
    tq.dir_off = t == SA_NO_TERM ? SA_NO_DIR : ix->h_dir_off[t];
    tq.rec_off = (t == SA_NO_TERM || ix->h_rec_off.empty()) ? SA_NO_DIR : ix->h_rec_off[t];
    tq.idf = idf;
    return tq;
}

Bm25Params sa_make_bm25(const sa_index *ix, float idf, float avg_doc_len, float k1, float b) { return make_bm25(ix, idf, avg_doc_len, k1, b); }
TermQuery sa_make_term_query(const sa_index *ix, u32 term_id, float idf) { return make_term_query(ix, term_id, idf); }

static u32 n_tiles_of(const sa_index *ix) { return (u32)((ix->n_docs + SA_TILE_DOCS - 1) / SA_TILE_DOCS); }

static size_t cand_bytes(const sa_index *ix, u32 Q, u32 slots) {
    return ((size_t)Q * n_tiles_of(ix) * ((size_t)slots * sizeof(u64) + 2 * sizeof(u32)) + 255) / 256 * 256;
}

// A batch alternates between two candidate areas, chunk by chunk: chunk c's select reads area c % 2 while the scan of
// chunk c + 1 fills the other one.
static size_t batch_cand_bytes(const sa_index *ix, const BatchState &B) { return 2 * cand_bytes(ix, B.chunk, B.slots); }

// `area`: the candidate area (0 or 1, each cand_bytes(ix, Q, slots) long)
static TopkCtx make_topk_ctx(sa_index *ix, u32 Q, u32 slots, u32 k, u32 *d_overflow, u32 area = 0) {
    const u32 T = n_tiles_of(ix);
    TopkCtx t;
    t.tile_cand = (u64 *)((char *)ix->cand.p + area * cand_bytes(ix, Q, slots));
    t.tile_cnt = (u32 *)(t.tile_cand + (u64)Q * T * slots);
    t.tile_max = t.tile_cnt + (u64)Q * T;
    t.overflow = d_overflow;
    t.n_tiles = T;
    t.slots = slots;
    t.k = k;
    return t;
}

static TermBatchArgs make_term_args(sa_index *ix, const TermQuery *d_queries, const Bm25Params &p, const TopkCtx &t) {
    TermBatchArgs a;
    memset(&a, 0, sizeof(a));
    a.words = ix->d_words;
    a.doc_lens = ix->d_doc_lens;
    a.n_docs = ix->n_docs;
    a.doc_base = ix->doc_base;
    a.queries = d_queries;
    a.out = ix->dense.as<float>();
    a.out_stride = padded_docs(ix->n_docs);
    a.bm25 = p;
    a.min_payload = 0;
    a.max_payload = SA_ALL_BITS;
    a.filter = 0;
    a.mode = TERM_MODE_SCORE;
    a.topk = t;
    return a;
}

int sa_batch_upload_locked(sa_index *ix, const uint32_t *terms, const uint32_t *term_starts,
                           const float *idf, uint32_t n_queries, uint32_t slop,
                           float avg_doc_len, float k1, float b, uint32_t k) {
    SA_CHECK(ix && (n_queries == 0 || (terms && term_starts && idf)), "NULL argument");
    SA_CHECK(k >= 1 && k <= SA_TOPK_MAX, "k must be in [1, %d]", SA_TOPK_MAX);
    SA_CUDA(cudaSetDevice(ix->device));
    if (!ix->batch) ix->batch = new BatchState();
    if (!ix->select_stream) {
        int least = 0, greatest = 0;        // the selects' few CTAs go ahead of the waiting CTAs of the next scan
        SA_CUDA(cudaDeviceGetStreamPriorityRange(&least, &greatest));
        SA_CUDA(cudaStreamCreateWithPriority(&ix->select_stream, cudaStreamNonBlocking, greatest));
        SA_CUDA(cudaEventCreateWithFlags(&ix->ev_scan, cudaEventDisableTiming));
        for (cudaEvent_t &e : ix->ev_select) SA_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    BatchState &B = *ix->batch;
    B.ready = false;
    B.executed = false;
    B.nq = n_queries;
    B.k = k;
    B.slots = sa_topk_slots(k);
    B.avg_doc_len = avg_doc_len;
    B.k1 = k1;
    B.b = b;
    B.slop = slop;
    B.span_plans.clear(); B.span_idf.clear();
    B.tqs.clear(); B.pqs.clear(); B.row_query.clear(); B.term_query.clear(); B.phrase_query.clear();
    B.phrase_missing.clear(); B.chunks.clear(); B.sel.clear();
    int rc;
    if ((rc = ix->topk_out.reserve(std::max<size_t>(((size_t)n_queries * k + SA_BATCH_TAIL) * sizeof(u64), 256)))) return rc;
    if (n_queries == 0) { B.ready = true; return SA_OK; }
    const u64 stride = padded_docs(std::max<u64>(ix->n_docs, 1));
    // chunk so the dense score vectors of one chunk stay within ~16 GB of HBM: at 10M docs 1,024 queries run as 3 scans
    // of up to 429 queries instead of 10 of 107 (fewer launch tails; 2 % on the bench's mix, profiles/README.md)
    u32 chunk = (u32)std::max<u64>(1, std::min<u64>(n_queries, (16ull << 30) / (stride * sizeof(float))));
    B.chunk = std::min<u32>(chunk, 65535);
    u64 max_arena = 64;
    size_t max_span_scratch = 0;
    u32 n_span = 0;
    for (u32 q0 = 0; q0 < n_queries; q0 += B.chunk) {
        const u32 q1 = std::min(n_queries, q0 + B.chunk);
        BatchChunk C;
        C.row0 = (u32)B.row_query.size();
        C.term0 = (u32)B.tqs.size();
        C.phrase0 = (u32)B.pqs.size();
        C.params = make_bm25(ix, 1.0f, avg_doc_len, k1, b);
        SpanPlan plan;
        for (int pass = 0; pass < 2; pass++) {               // term queries first, then phrases
            for (u32 q = q0; q < q1; q++) {
                const u32 nt = term_starts[q + 1] - term_starts[q];
                SA_CHECK(nt >= 1 && nt <= SA_MAX_PHRASE_TERMS, "query %u: bad number of terms", q);
                const u32 *tids = terms + term_starts[q];
                for (u32 i = 0; i < nt; i++)
                    SA_CHECK(tids[i] == SA_NO_TERM || tids[i] < ix->n_terms, "term id %u out of range", tids[i]);
                if ((nt == 1) != (pass == 0)) continue;
                if (!make_bm25(ix, idf[q], avg_doc_len, k1, b).sparse_ok) C.params.sparse_ok = 0;
                B.row_query.push_back(q);
                if (nt == 1) {
                    B.tqs.push_back(make_term_query(ix, tids[0], idf[q]));
                    B.term_query.push_back(q);
                } else if (slop > 0) {
                    // phrase with slop: span search (spans.py:171-187) on the index's own lists
                    u64 offs[SA_MAX_PHRASE_TERMS], lens[SA_MAX_PHRASE_TERMS], dirs[SA_MAX_PHRASE_TERMS];
                    bool missing = false, literal = true;
                    for (u32 i = 0; i < nt; i++)
                        if (tids[i] == SA_NO_TERM || ix->h_len[tids[i]] == 0) missing = true;
                    for (u32 i = 0; i < nt; i++) {
                        offs[i] = missing ? 0 : ix->h_off[tids[i]];
                        lens[i] = missing ? 0 : ix->h_len[tids[i]];
                        dirs[i] = missing ? SA_NO_DIR : ix->h_dir_off[tids[i]];
                        literal = literal && !missing && ix->h_first0[tids[i]];
                    }
                    sa_span_plan_add(plan, offs, lens, dirs, nt, slop, idf[q], literal, missing ? 0 : ix->n_docs);
                    B.span_idf.push_back(idf[q]);
                    B.phrase_query.push_back(q);
                } else {
                    PhraseQuery pq;
                    memset(&pq, 0, sizeof(pq));
                    pq.n_terms = nt;
                    pq.idf = idf[q];
                    u32 missing = 0;
                    for (u32 i = 0; i < nt; i++) {
                        if (tids[i] == SA_NO_TERM || ix->h_len[tids[i]] == 0) { missing = 1; continue; }
                        pq.off[i] = ix->h_off[tids[i]];
                        pq.len[i] = ix->h_len[tids[i]];
                    }
                    if (missing) for (u32 i = 0; i < nt; i++) pq.len[i] = 0;     // no pairs -> zeros
                    else for (u32 i = 0; i < nt; i++)
                        if (ix->h_dir_off[tids[i]] != SA_NO_DIR) pq.dir_plus1[i] = ix->h_dir_off[tids[i]] + 1;
                    sa_phrase_plan(pq, tids);
                    if (!missing && sa_phrase_is_staged(pq, ix->n_docs)) {
                        pq.pad = 1;                                               // merge regime (see below)
                        C.slab_cap = std::max(C.slab_cap, sa_phrase_slab_cap(ix, tids, nt));
                    }
                    B.pqs.push_back(pq);
                    B.phrase_query.push_back(q);
                    B.phrase_missing.push_back(missing);
                }
            }
        }
        C.n_term = (u32)B.tqs.size() - C.term0;
        if (slop > 0) {
            C.phrase0 = n_span;
            C.n_phrase = (u32)plan.qs.size();
            n_span += C.n_phrase;
            max_span_scratch = std::max(max_span_scratch, sa_span_scratch_bytes(plan));
            B.span_plans.push_back(std::move(plan));
            B.chunks.push_back(C);
            continue;
        }
        C.n_phrase = (u32)B.pqs.size() - C.phrase0;
        if (C.n_phrase) {
            C.sel0 = (u32)B.sel.size();
            for (u32 i = 0; i < C.n_phrase; i++) if (!B.pqs[C.phrase0 + i].pad) B.sel.push_back(i);
            C.n_search = (u32)B.sel.size() - C.sel0;
            for (u32 i = 0; i < C.n_phrase; i++) if (B.pqs[C.phrase0 + i].pad) B.sel.push_back(i);
            C.n_staged = C.n_phrase - C.n_search;
            C.staged_chunks = sa_phrase_staged_chunks(ix);
            u64 want = std::max<u64>(1, (u64)ix->num_sms * 16 / std::max<u32>(C.n_search, 1));
            C.phrase_chunks = sa_phrase_chunks(ix, (u32)std::max<u64>(1, std::min<u64>(want, std::max<u64>(1, ix->n_docs / 512))));
            for (u32 i = 0; i < C.n_phrase; i++)                     // only the search regime bump-allocates
                if (!B.pqs[C.phrase0 + i].pad) C.arena_words += sa_phrase_arena_words(B.pqs[C.phrase0 + i], C.phrase_chunks);
            max_arena = std::max(max_arena, C.arena_words);
        }
        B.chunks.push_back(C);
    }
    SA_CHECK(B.chunks.empty() || B.chunks[0].params.sparse_ok || (B.pqs.empty() && n_span == 0),
             "phrase queries in a batch need ordinary BM25 parameters (k1 > 0, 0 <= b < 1, finite idf)");
    if ((rc = ix->dense.reserve((size_t)B.chunk * stride * sizeof(float)))) return rc;
    if ((rc = ix->cand.reserve(batch_cand_bytes(ix, B)))) return rc;
    if ((rc = B.d_tq.reserve(std::max<size_t>(B.tqs.size() * sizeof(TermQuery), 64)))) return rc;
    if ((rc = B.d_pq.reserve(std::max<size_t>(B.pqs.size() * sizeof(PhraseQuery), 64)))) return rc;
    if ((rc = B.d_row_query.reserve((size_t)n_queries * sizeof(u32)))) return rc;
    if ((rc = B.d_meta.reserve((size_t)n_queries * sizeof(u32)))) return rc;
    if ((rc = B.d_pstats.reserve(std::max<size_t>(B.pqs.size() * sizeof(PhraseStats), 64)))) return rc;
    if ((rc = B.d_sel.reserve(std::max<size_t>(B.sel.size() * sizeof(u32), 64)))) return rc;
    if ((rc = B.d_missing.reserve(std::max<size_t>(B.phrase_missing.size() * sizeof(u32), 64)))) return rc;
    if (!B.pqs.empty() && (rc = ix->phrase_scratch.reserve(max_arena * sizeof(u64) + 64))) return rc;
    if (n_span) {
        if ((rc = ix->phrase_scratch.reserve(max_span_scratch))) return rc;
        if ((rc = B.d_sq.reserve((size_t)n_span * sizeof(SpanQuery)))) return rc;
        if ((rc = B.d_scounts.reserve((size_t)n_span * sizeof(SpanCounts)))) return rc;
        if ((rc = B.d_sidf.reserve((size_t)n_span * sizeof(float)))) return rc;
        u32 at = 0;
        for (const SpanPlan &pl : B.span_plans) {
            if (pl.qs.empty()) continue;
            SA_CUDA(cudaMemcpyAsync(B.d_sq.as<SpanQuery>() + at, pl.qs.data(), pl.qs.size() * sizeof(SpanQuery),
                                    cudaMemcpyHostToDevice, ix->stream));
            at += (u32)pl.qs.size();
        }
        SA_CUDA(cudaMemcpyAsync(B.d_sidf.p, B.span_idf.data(), (size_t)n_span * sizeof(float), cudaMemcpyHostToDevice, ix->stream));
        SA_CUDA(cudaStreamSynchronize(ix->stream));      // the plans' host vectors may be reallocated later
    }
    if (!B.tqs.empty())
        SA_CUDA(cudaMemcpyAsync(B.d_tq.p, B.tqs.data(), B.tqs.size() * sizeof(TermQuery), cudaMemcpyHostToDevice, ix->stream));
    if (!B.pqs.empty()) {
        SA_CUDA(cudaMemcpyAsync(B.d_pq.p, B.pqs.data(), B.pqs.size() * sizeof(PhraseQuery), cudaMemcpyHostToDevice, ix->stream));
        SA_CUDA(cudaMemcpyAsync(B.d_sel.p, B.sel.data(), B.sel.size() * sizeof(u32), cudaMemcpyHostToDevice, ix->stream));
        SA_CUDA(cudaMemcpyAsync(B.d_missing.p, B.phrase_missing.data(), B.phrase_missing.size() * sizeof(u32),
                                cudaMemcpyHostToDevice, ix->stream));
    }
    SA_CUDA(cudaMemcpyAsync(B.d_row_query.p, B.row_query.data(), (size_t)n_queries * sizeof(u32), cudaMemcpyHostToDevice, ix->stream));
    B.ready = true;
    return SA_OK;
}

// Last kernel of a batch: how many queries need the exact re-run, and the phrase roofline counters.  The same-term
// speculation of every phrase query is verified here exactly as sa_phrase_guess_ok does on the host.
__global__ void __launch_bounds__(256)
batch_summary_kernel(const u32 *__restrict__ ovf, u32 nq, const PhraseQuery *__restrict__ pqs,
                     const PhraseStats *__restrict__ st, const u32 *__restrict__ missing, u32 n_phrase,
                     u64 *__restrict__ tail) {
    __shared__ unsigned long long s_acc[3];
    if (threadIdx.x < 3) s_acc[threadIdx.x] = 0;
    __syncthreads();
    unsigned long long redo = 0, cont = 0, match = 0;
    for (u32 i = threadIdx.x; i < nq; i += blockDim.x) redo += ovf[i] ? 1 : 0;
    for (u32 i = threadIdx.x; i < n_phrase; i += blockDim.x) {
        const PhraseQuery &pq = pqs[i];
        const PhraseStats &s = st[i];
        cont += s.n_cont;
        match += s.n_match;
        bool bad = s.overflow != 0;
        if (!bad && !missing[i]) {
            const u32 n = pq.n_terms;
            // every step the plan runs (sa_phrase.cu step_order): LR 1..n-1, RL 0..n-2, middle-out 1..split-1 and split..n-2
            u32 s0 = 1, s1 = n;
            if (pq.mode == SA_PHRASE_MODE_RL) { s0 = 0; s1 = n - 1; }
            else if (pq.mode == SA_PHRASE_MODE_MID) { s0 = 1; s1 = n - 1; }
            for (u32 step = s0; step < s1 && !bad; step++) {
                const bool actual = s.n_inner[step] > 0 && s.n_diff[step] == 0;
                const bool guess = (pq.same_guess >> step) & 1u;
                if (actual != guess) bad = true;
            }
        }
        // a wrong guess also sets the query's overflow flag?  No: the host re-derives which queries to redo; here
        // only the COUNT matters (non-zero -> the host takes the slow path)
        if (bad) redo++;
    }
    if (redo) atomicAdd(&s_acc[0], redo);
    if (cont) atomicAdd(&s_acc[1], cont);
    if (match) atomicAdd(&s_acc[2], match);
    __syncthreads();
    if (threadIdx.x < 3) tail[threadIdx.x] = s_acc[threadIdx.x];
    if (threadIdx.x == 3) tail[3] = 0;
}

int sa_batch_execute_locked(sa_index *ix) {
    SA_CHECK(ix && ix->batch && ix->batch->ready, "no batch uploaded (sa_batch_upload)");
    BatchState &B = *ix->batch;
    SA_CUDA(cudaSetDevice(ix->device));
    u64 *d_keys = ix->topk_out.as<u64>();
    if (B.nq == 0) {
        SA_CUDA(cudaMemsetAsync(d_keys, 0, SA_BATCH_TAIL * sizeof(u64), ix->stream));
        return SA_OK;
    }
    if (ix->n_docs == 0 || B.avg_doc_len == 0.0f) {
        SA_CUDA(cudaMemsetAsync(d_keys, 0, ((size_t)B.nq * B.k + SA_BATCH_TAIL) * sizeof(u64), ix->stream));
        return SA_OK;
    }
    const u64 stride = padded_docs(ix->n_docs);
    u32 *d_ovf = B.d_meta.as<u32>();
    SA_CUDA(cudaMemsetAsync(d_ovf, 0, (size_t)B.nq * sizeof(u32), ix->stream));
    if (!B.pqs.empty())
        SA_CUDA(cudaMemsetAsync(B.d_pstats.p, 0, B.pqs.size() * sizeof(PhraseStats), ix->stream));
    int rc;
    size_t chunk_i = 0;
    for (size_t c = 0; c < B.chunks.size(); c++) {
        const BatchChunk &C = B.chunks[c];
        const u32 Q = C.n_term + C.n_phrase;
        const u32 area = (u32)(c & 1);
        // chunk c's scan rewrites the candidate area that chunk c - 2's select reads
        if (c >= 2) SA_CUDA(cudaStreamWaitEvent(ix->stream, ix->ev_select[area], 0));
        TopkCtx t = make_topk_ctx(ix, B.chunk, B.slots, B.k, d_ovf + C.row0, area);
        if (C.n_term) {
            TermBatchArgs a = make_term_args(ix, B.d_tq.as<TermQuery>() + C.term0, C.params, t);
            if ((rc = launch_term_batch(ix, a, C.n_term))) return rc;
        }
        if (B.slop > 0) {
            const SpanPlan &plan = B.span_plans[chunk_i++];
            if (C.n_phrase) {
                // span matches become records; one tile pass writes the rows (zeros + BM25) and collects top-k
                float *rows = ix->dense.as<float>() + (u64)C.n_term * stride;
                if ((rc = sa_ensure_norm(ix, B.k1, B.b, B.avg_doc_len))) return rc;
                if ((rc = sa_span_enqueue(ix, ix->d_words, plan, B.d_sq.as<SpanQuery>() + C.phrase0,
                                          B.d_scounts.as<SpanCounts>() + C.phrase0, ix->phrase_scratch.p, rows, stride,
                                          &t, C.n_term))) return rc;
            }
        } else if (C.n_phrase) {
            float *rows = ix->dense.as<float>() + (u64)C.n_term * stride;
            unsigned long long *d_used = (unsigned long long *)ix->phrase_scratch.p;
            SA_CUDA(cudaMemsetAsync(d_used, 0, 64, ix->stream));
            // the phrase kernel materialises its dense rows (zeros + matches) and their top-k candidates
            PhraseSplit sp;
            sp.d_search = B.d_sel.as<u32>() + C.sel0;
            sp.n_search = C.n_search;
            sp.d_staged = sp.d_search + C.n_search;
            sp.n_staged = C.n_staged;
            sp.staged_chunks = C.staged_chunks;
            sp.slab_cap = C.slab_cap;
            if ((rc = sa_phrase_enqueue(ix, B.d_pq.as<PhraseQuery>() + C.phrase0, B.d_pstats.as<PhraseStats>() + C.phrase0,
                                        C.n_phrase, rows, stride, C.phrase_chunks, (u64 *)ix->phrase_scratch.p + 8,
                                        d_used, C.arena_words, 1, C.params, &t, C.n_term, &sp))) return rc;
        }
        // the select runs on the side stream, overlapping the next chunk's scan
        SA_CUDA(cudaEventRecord(ix->ev_scan, ix->stream));
        SA_CUDA(cudaStreamWaitEvent(ix->select_stream, ix->ev_scan, 0));
        if ((rc = launch_topk_select(ix, t, Q, ix->doc_base, d_keys, B.d_row_query.as<u32>() + C.row0, ix->select_stream)))
            return rc;
        SA_CUDA(cudaEventRecord(ix->ev_select[area], ix->select_stream));
    }
    B.executed = true;
    // join: the summary and everything after it on ix->stream (downloads, timers, the all-gather) follow the selects
    SA_CUDA(cudaStreamWaitEvent(ix->stream, ix->ev_select[(B.chunks.size() - 1) & 1], 0));
    const u32 n_phr = B.slop > 0 ? 0u : (u32)B.pqs.size();
    batch_summary_kernel<<<1, 256, 0, ix->stream>>>(d_ovf, B.nq, B.d_pq.as<PhraseQuery>(), B.d_pstats.as<PhraseStats>(),
                                                   B.d_missing.as<u32>(), n_phr, d_keys + (size_t)B.nq * B.k);
    SA_CUDA(cudaGetLastError());
    ix->stats.total_launches++;
    return SA_OK;
}

// Re-run one query exactly (synchronously): a tile overflowed its candidate slots, or a phrase's
// same-term speculation was wrong.  Uses a slot per doc of the tile -- cannot overflow.
static int redo_query(sa_index *ix, BatchState &B, bool is_phrase, u32 idx, u32 q, const SpanQuery *sq = nullptr) {
    int rc;
    const u64 stride = padded_docs(ix->n_docs);
    if ((rc = ix->cand.reserve(cand_bytes(ix, 1, SA_TILE_DOCS)))) return rc;
    SA_CUDA(cudaMemsetAsync(B.d_meta.p, 0, sizeof(u32), ix->stream));
    TopkCtx t = make_topk_ctx(ix, 1, SA_TILE_DOCS, B.k, B.d_meta.as<u32>());
    if (!is_phrase) {
        Bm25Params p = make_bm25(ix, B.tqs[idx].idf, B.avg_doc_len, B.k1, B.b);
        TermBatchArgs a = make_term_args(ix, B.d_tq.as<TermQuery>() + idx, p, t);
        if ((rc = launch_term_batch(ix, a, 1))) return rc;
    } else if (sq) {
        if ((rc = sa_ensure_norm(ix, B.k1, B.b, B.avg_doc_len))) return rc;
        if ((rc = sa_span_run(ix, ix->d_words, sq->off, sq->len, sq->dir_off, sq->n_terms, sq->slop, sq->literal != 0, nullptr))) return rc;
        SA_CUDA(cudaMemcpyAsync(B.d_sidf.p, &sq->idf, sizeof(float), cudaMemcpyHostToDevice, ix->stream));
        if ((rc = launch_dense_topk_tiles(ix, ix->dense.as<float>(), stride, 0, 1, t, B.d_sidf.as<float>()))) return rc;
    } else {
        Bm25Params p = make_bm25(ix, B.pqs[idx].idf, B.avg_doc_len, B.k1, B.b);
        std::vector<PhraseQuery> one(1, B.pqs[idx]);
        PhraseDump nodump;
        memset(&nodump, 0, sizeof(nodump));
        if ((rc = sa_phrase_run_sync(ix, one, ix->d_words, 1, p, 0, nodump, 0))) return rc;   // loops until the guess holds
        B.pqs[idx] = one[0];
        if ((rc = launch_dense_topk_tiles(ix, ix->dense.as<float>(), stride, 0, 1, t, nullptr))) return rc;
    }
    SA_CUDA(cudaMemcpyAsync(B.d_row_query.p, &q, sizeof(u32), cudaMemcpyHostToDevice, ix->stream));
    if ((rc = launch_topk_select(ix, t, 1, ix->doc_base, ix->topk_out.as<u64>(), B.d_row_query.as<u32>()))) return rc;
    SA_CUDA(cudaStreamSynchronize(ix->stream));
    return SA_OK;
}

// After execute: repair (synchronously) the queries that need it.
int sa_batch_fix_overflow_locked(sa_index *ix, u32 *n_redone) {
    BatchState &B = *ix->batch;
    if (n_redone) *n_redone = 0;
    if (B.nq == 0 || ix->n_docs == 0 || B.avg_doc_len == 0.0f) return SA_OK;
    int rc;
    const size_t ovf_bytes = (size_t)B.nq * sizeof(u32), st_bytes = B.pqs.size() * sizeof(PhraseStats);
    if ((rc = sa_pinned_reserve(ix, std::max<size_t>(ovf_bytes + st_bytes, 4096)))) return rc;
    SA_CUDA(cudaMemcpyAsync(ix->h_pinned, B.d_meta.p, ovf_bytes, cudaMemcpyDeviceToHost, ix->stream));
    if (st_bytes)
        SA_CUDA(cudaMemcpyAsync((char *)ix->h_pinned + ovf_bytes, B.d_pstats.p, st_bytes, cudaMemcpyDeviceToHost, ix->stream));
    SA_CUDA(cudaStreamSynchronize(ix->stream));
    std::vector<u32> ovf((const u32 *)ix->h_pinned, (const u32 *)ix->h_pinned + B.nq);       // row space
    std::vector<PhraseStats> st(B.pqs.size());
    if (st_bytes) memcpy(st.data(), (char *)ix->h_pinned + ovf_bytes, st_bytes);

    struct Redo { bool phrase; u32 idx, q; const SpanQuery *sq; };
    std::vector<Redo> redo;
    size_t chunk_i = 0;
    for (const BatchChunk &C : B.chunks) {
        for (u32 i = 0; i < C.n_term; i++)
            if (ovf[C.row0 + i]) redo.push_back({false, C.term0 + i, B.term_query[C.term0 + i], nullptr});
        if (B.slop > 0) {
            const SpanPlan &plan = B.span_plans[chunk_i++];
            for (u32 i = 0; i < C.n_phrase; i++)
                if (ovf[C.row0 + C.n_term + i])
                    redo.push_back({true, C.phrase0 + i, B.phrase_query[C.phrase0 + i], &plan.qs[i]});
            continue;
        }
        for (u32 i = 0; i < C.n_phrase; i++) {
            const u32 pi = C.phrase0 + i;
            SA_CHECK(st[pi].overflow != 1, "phrase scratch arena exhausted (internal sizing error)");
            PhraseQuery trial = B.pqs[pi];
            bool ok = st[pi].overflow == 0 && (B.phrase_missing[pi] || sa_phrase_guess_ok(trial, st[pi]));
            if (!ok || ovf[C.row0 + C.n_term + i]) redo.push_back({true, pi, B.phrase_query[pi], nullptr});
        }
    }
    if (redo.empty()) return SA_OK;
    B.executed = false;                          // the re-runs reuse the dense rows
    for (const Redo &r : redo)
        if ((rc = redo_query(ix, B, r.phrase, r.idx, r.q, r.sq))) return rc;
    // the repair buffers are larger than the batch's: restore the normal ones and descriptors
    if ((rc = ix->cand.reserve(batch_cand_bytes(ix, B)))) return rc;
    SA_CUDA(cudaMemcpyAsync(B.d_row_query.p, B.row_query.data(), (size_t)B.nq * sizeof(u32), cudaMemcpyHostToDevice, ix->stream));
    if (!B.pqs.empty())
        SA_CUDA(cudaMemcpyAsync(B.d_pq.p, B.pqs.data(), B.pqs.size() * sizeof(PhraseQuery), cudaMemcpyHostToDevice, ix->stream));
    if (!B.span_idf.empty()) {
        size_t need = 0;
        for (const SpanPlan &pl : B.span_plans) need = std::max(need, sa_span_scratch_bytes(pl));
        if ((rc = ix->phrase_scratch.reserve(need))) return rc;
        SA_CUDA(cudaMemcpyAsync(B.d_sidf.p, B.span_idf.data(), B.span_idf.size() * sizeof(float), cudaMemcpyHostToDevice, ix->stream));
    }
    SA_CUDA(cudaStreamSynchronize(ix->stream));
    if (n_redone) *n_redone = (u32)redo.size();
    return SA_OK;
}

void sa_unpack_keys(const u64 *keys, u64 n, uint32_t *out_docs, float *out_scores) {
    for (u64 i = 0; i < n; i++) {
        u64 key = keys[i];
        if (key == 0) { out_docs[i] = SA_NO_DOC; out_scores[i] = 0.0f; continue; }
        out_docs[i] = 0xFFFFFFFFu - (u32)(key & 0xFFFFFFFFull);
        u32 bits = (u32)(key >> 32);
        memcpy(&out_scores[i], &bits, 4);
    }
}

// keys + the batch's summary tail in ONE device-to-host copy and ONE synchronise
static int download_keys(sa_index *ix, const u64 *d_keys, size_t nk, uint32_t *out_docs, float *out_scores, u64 *tail) {
    int rc;
    if ((rc = sa_pinned_reserve(ix, (nk + SA_BATCH_TAIL) * sizeof(u64)))) return rc;
    SA_CUDA(cudaMemcpyAsync(ix->h_pinned, d_keys, (nk + SA_BATCH_TAIL) * sizeof(u64), cudaMemcpyDeviceToHost, ix->stream));
    SA_CUDA(cudaStreamSynchronize(ix->stream));
    sa_unpack_keys((const u64 *)ix->h_pinned, nk, out_docs, out_scores);
    if (tail) memcpy(tail, (const u64 *)ix->h_pinned + nk, SA_BATCH_TAIL * sizeof(u64));
    return SA_OK;
}

int sa_batch_download_locked(sa_index *ix, uint32_t *out_docs, float *out_scores, uint32_t *n_overflow) {
    BatchState &B = *ix->batch;
    const size_t nk = (size_t)B.nq * B.k;
    u64 tail[SA_BATCH_TAIL] = {0, 0, 0, 0};
    if (n_overflow) *n_overflow = 0;
    int rc = download_keys(ix, ix->topk_out.as<u64>(), nk, out_docs, out_scores, tail);
    if (rc) return rc;
    ix->stats.phrase_cont_words += tail[1];
    ix->stats.phrase_matched_docs += tail[2];
    if (tail[0] == 0) return SA_OK;              // the common case: nothing to repair
    if ((rc = sa_batch_fix_overflow_locked(ix, n_overflow))) return rc;
    return download_keys(ix, ix->topk_out.as<u64>(), nk, out_docs, out_scores, nullptr);
}

extern "C" int sa_batch_upload(sa_index *ix, const uint32_t *terms, const uint32_t *term_starts,
                               const float *idf, uint32_t n_queries, uint32_t slop,
                               float avg_doc_len, float k1, float b, uint32_t k) {
    SA_CHECK(ix, "index is NULL");
    std::lock_guard<std::mutex> g(ix->mu);
    return sa_batch_upload_locked(ix, terms, term_starts, idf, n_queries, slop, avg_doc_len, k1, b, k);
}

extern "C" int sa_batch_execute(sa_index *ix) {
    SA_CHECK(ix, "index is NULL");
    std::lock_guard<std::mutex> g(ix->mu);
    return sa_batch_execute_locked(ix);
}

extern "C" int sa_batch_download(sa_index *ix, uint32_t *out_docs, float *out_scores, uint32_t *n_overflow) {
    SA_CHECK(ix && ix->batch && ix->batch->ready, "no batch uploaded");
    SA_CHECK(out_docs && out_scores, "NULL argument");
    std::lock_guard<std::mutex> g(ix->mu);
    return sa_batch_download_locked(ix, out_docs, out_scores, n_overflow);
}

extern "C" int sa_batch_row(sa_index *ix, uint32_t row, float *out_host) {
    SA_CHECK(ix && out_host, "NULL argument");
    std::lock_guard<std::mutex> g(ix->mu);
    SA_CHECK(ix->batch && ix->batch->executed, "no executed batch holds its dense rows");
    const BatchChunk &C = ix->batch->chunks.back();
    SA_CHECK(row < C.n_term + C.n_phrase, "row %u out of range (the last chunk has %u)", row, C.n_term + C.n_phrase);
    SA_CUDA(cudaSetDevice(ix->device));
    SA_CUDA(cudaMemcpyAsync(out_host, ix->dense.as<float>() + (u64)row * padded_docs(ix->n_docs), ix->n_docs * sizeof(float),
                            cudaMemcpyDeviceToHost, ix->stream));
    SA_CUDA(cudaStreamSynchronize(ix->stream));
    return SA_OK;
}

extern "C" int sa_score_batch_topk(sa_index *ix, const uint32_t *terms, const uint32_t *term_starts,
                                   const float *idf, uint32_t n_queries, uint32_t slop,
                                   float avg_doc_len, float k1, float b, uint32_t k,
                                   uint32_t *out_docs, float *out_scores) {
    SA_CHECK(ix && out_docs && out_scores, "NULL argument");
    std::lock_guard<std::mutex> g(ix->mu);
    int rc = sa_batch_upload_locked(ix, terms, term_starts, idf, n_queries, slop, avg_doc_len, k1, b, k);
    if (rc) return rc;
    if ((rc = sa_batch_execute_locked(ix))) return rc;
    return sa_batch_download_locked(ix, out_docs, out_scores, nullptr);
}

// ------------------------------------------------------------------- timers
KernelTimer::KernelTimer(sa_index *ix_, int kind_, cudaStream_t stream_)
    : ix(ix_), kind(kind_), on(ix_->profiling), stream(stream_ ? stream_ : ix_->stream) {
    if (!on) return;
    if (!ix->pending_timers) ix->pending_timers = new std::vector<TimedLaunch>();
    if (!ix->free_events) ix->free_events = new std::vector<cudaEvent_t>();
    auto get = [&]() {
        cudaEvent_t e = nullptr;
        if (!ix->free_events->empty()) { e = ix->free_events->back(); ix->free_events->pop_back(); }
        else cudaEventCreate(&e);
        return e;
    };
    e0 = get();
    e1 = get();
    cudaEventRecord(e0, stream);
}

void KernelTimer::stop() {
    if (!on) return;
    cudaEventRecord(e1, stream);
    ix->pending_timers->push_back(TimedLaunch{e0, e1, kind});
    on = false;
}

int sa_resolve_timers(sa_index *ix) {
    if (!ix->pending_timers || ix->pending_timers->empty()) return SA_OK;
    SA_CUDA(cudaStreamSynchronize(ix->stream));
    for (auto &t : *ix->pending_timers) {
        float ms = 0;
        cudaEventElapsedTime(&ms, t.e0, t.e1);
        if (t.kind == 0) ix->stats.term_kernel_ms += ms;
        else if (t.kind == 1) ix->stats.topk_kernel_ms += ms;
        else ix->stats.phrase_kernel_ms += ms;
        ix->free_events->push_back(t.e0);
        ix->free_events->push_back(t.e1);
    }
    ix->pending_timers->clear();
    return SA_OK;
}

extern "C" int sa_timer_start(sa_index *ix) {
    SA_CHECK(ix, "index is NULL");
    std::lock_guard<std::mutex> g(ix->mu);
    SA_CUDA(cudaSetDevice(ix->device));
    SA_CUDA(cudaStreamSynchronize(ix->stream));
    SA_CUDA(cudaEventRecord(ix->ev0, ix->stream));
    return SA_OK;
}

extern "C" int sa_timer_stop(sa_index *ix, double *ms_out) {
    SA_CHECK(ix && ms_out, "NULL argument");
    std::lock_guard<std::mutex> g(ix->mu);
    SA_CUDA(cudaSetDevice(ix->device));
    SA_CUDA(cudaEventRecord(ix->ev1, ix->stream));
    SA_CUDA(cudaEventSynchronize(ix->ev1));
    float ms = 0;
    SA_CUDA(cudaEventElapsedTime(&ms, ix->ev0, ix->ev1));
    *ms_out = ms;
    return SA_OK;
}

void sa_free_batch(sa_index *ix) {
    if (!ix->batch) return;
    ix->batch->d_tq.release();
    ix->batch->d_pq.release();
    ix->batch->d_row_query.release();
    ix->batch->d_meta.release();
    ix->batch->d_pstats.release();
    ix->batch->d_sel.release();
    ix->batch->d_missing.release();
    ix->batch->d_sq.release();
    ix->batch->d_scounts.release();
    ix->batch->d_sidf.release();
    delete ix->batch;
    ix->batch = nullptr;
}

void sa_batch_dims(sa_index *ix, u32 *nq, u32 *k) {
    *nq = ix->batch ? ix->batch->nq : 0;
    *k = ix->batch ? ix->batch->k : 0;
}
