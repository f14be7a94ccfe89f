// sa_topk.cu -- exact top-k over the candidates the scoring kernels collected.
//
// Replaces the reference idiom np.argpartition(scores, -N)[-N:] (searcharray/utils/sort.py:24)
// for the HBM-resident batched path.  The scoring kernels append every score that is >= a
// running, provably-valid lower bound of the k-th best score (sa_term.cu step 4), so the
// candidate list is a superset of the true top-k and is normally a few hundred entries.
// Here one CTA per query selects the exact k best by (score desc, doc id asc): a tight threshold
// (k-th largest of the per-tile maxima) prefilters the per-tile candidate slots to ~k survivors,
// which are sorted in shared memory (bitonic); a radix select handles massive ties.
#include "sa_term.cuh"

#define SEL_THREADS 512
#define SEL_SMEM_KEYS 4096

__device__ void bitonic_sort_desc_smem(u64 *s, u32 n_pow2) {
    for (u32 k = 2; k <= n_pow2; k <<= 1) {
        for (u32 j = k >> 1; j > 0; j >>= 1) {
            for (u32 i = threadIdx.x; i < n_pow2; i += blockDim.x) {
                u32 ixj = i ^ j;
                if (ixj > i) {
                    u64 a = s[i], b = s[ixj];
                    bool desc = ((i & k) == 0);
                    if ((a < b) == desc) { s[i] = b; s[ixj] = a; }
                }
            }
            __syncthreads();
        }
    }
}

// visit every candidate key of query q whose tile can hold a key with score bits >= min_score
template <typename F>
__device__ __forceinline__ void for_each_candidate(const TopkCtx &t, u32 q, u32 min_score, F f) {
    const u32 *cnt = t.tile_cnt + (u64)q * t.n_tiles;
    const u32 *tmax = t.tile_max + (u64)q * t.n_tiles;
    const u64 *cand = t.tile_cand + (u64)q * t.n_tiles * t.slots;
    for (u32 tile = threadIdx.x; tile < t.n_tiles; tile += blockDim.x) {
        if (tmax[tile] < min_score) continue;
        const u32 n = cnt[tile];
        const u64 *c = cand + (u64)tile * t.slots;
        for (u32 j = 0; j < n; j++) f(c[j]);
    }
}

// thread 0: walk the 256-bin histogram from the top until `rem` keys are covered
__device__ __forceinline__ void radix_pick(const u32 *hist, u32 &rem, int &bin) {
    u32 acc = 0;
    int b = 255;
    for (; b > 0; b--) {
        if (acc + hist[b] >= rem) break;
        acc += hist[b];
    }
    rem -= acc;
    bin = b;
}

__global__ void __launch_bounds__(SEL_THREADS)
topk_select_kernel(TopkCtx t, u64 doc_base, u64 *__restrict__ out_keys, const u32 *__restrict__ out_index) {
    __shared__ u64 s_keys[SEL_SMEM_KEYS];
    __shared__ u32 s_hist[256];
    __shared__ u64 s_prefix;
    __shared__ u32 s_krem, s_n;

    const u32 q = blockIdx.x;
    const u32 k = t.k;
    const u32 T = t.n_tiles;

    // A. a tight valid threshold: the k-th largest of the per-tile(-group) best scores (they
    //    belong to distinct docs).  The tile maxima were written by the scoring kernel, so this
    //    is one coalesced read of 4*T bytes; 4-pass 8-bit radix select in shared memory.
    u32 *s_max = reinterpret_cast<u32 *>(s_keys);                   // [G] reuse (2 * SEL_SMEM_KEYS u32)
    const u32 GMAX = 2 * SEL_SMEM_KEYS;
    const u32 gs = (T + GMAX - 1) / GMAX;                            // tiles per group
    const u32 G = (T + gs - 1) / gs;
    {
        const u32 *tmax = t.tile_max + (u64)q * T;
        for (u32 g = threadIdx.x; g < G; g += blockDim.x) {
            u32 m = 0;
            for (u32 tile = g * gs; tile < min(T, (g + 1) * gs); tile++) m = max(m, tmax[tile]);
            s_max[g] = m;
        }
    }
    if (threadIdx.x == 0) { s_prefix = 0; s_krem = k; }
    __syncthreads();
    for (int shift = 24; shift >= 0; shift -= 8) {
        for (u32 i = threadIdx.x; i < 256; i += blockDim.x) s_hist[i] = 0;
        __syncthreads();
        const u32 prefix = (u32)s_prefix;
        for (u32 g = threadIdx.x; g < G; g += blockDim.x) {
            u32 key = s_max[g];
            bool match = (shift == 24) || ((key >> (shift + 8)) == (prefix >> (shift + 8)));
            if (match) atomicAdd(&s_hist[(key >> shift) & 255], 1u);
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            u32 rem = s_krem;
            int b;
            radix_pick(s_hist, rem, b);
            s_krem = rem;
            s_prefix = (u64)(prefix | ((u32)b << shift));
        }
        __syncthreads();
    }
    u32 thr_score = (u32)s_prefix;      // 0 when fewer than k tile groups hold a candidate
    if (thr_score == 0) thr_score = 1;
    __syncthreads();

    // B. survivors with score >= thr_score (a superset of the true top-k, normally ~k of them);
    //    tiles whose best score is below the threshold are skipped without touching their slots
    if (threadIdx.x == 0) s_n = 0;
    __syncthreads();
    for_each_candidate(t, q, thr_score, [&](u64 key) {
        if ((u32)(key >> 32) >= thr_score) {
            u32 slot = atomicAdd(&s_n, 1u);
            if (slot < SEL_SMEM_KEYS) s_keys[slot] = key;
        }
    });
    __syncthreads();
    u32 M = s_n;
    u32 n_valid;
    if (M <= SEL_SMEM_KEYS) {
        u32 n2 = 2;
        while (n2 < M) n2 <<= 1;
        for (u32 i = M + threadIdx.x; i < n2; i += blockDim.x) s_keys[i] = 0ull;
        __syncthreads();
        bitonic_sort_desc_smem(s_keys, n2);
        n_valid = M;
    } else {
        // massive ties around the threshold: radix-select the exact k-th key over all survivors
        if (threadIdx.x == 0) { s_prefix = 0; s_krem = k; }
        __syncthreads();
        for (int shift = 56; shift >= 0; shift -= 8) {
            for (u32 i = threadIdx.x; i < 256; i += blockDim.x) s_hist[i] = 0;
            __syncthreads();
            const u64 prefix = s_prefix;
            for_each_candidate(t, q, thr_score, [&](u64 key) {
                if ((u32)(key >> 32) < thr_score) return;
                bool match = (shift == 56) || ((key >> (shift + 8)) == (prefix >> (shift + 8)));
                if (match) atomicAdd(&s_hist[(key >> shift) & 255], 1u);
            });
            __syncthreads();
            if (threadIdx.x == 0) {
                u32 rem = s_krem;
                int b;
                radix_pick(s_hist, rem, b);
                s_krem = rem;
                s_prefix = prefix | ((u64)b << shift);
            }
            __syncthreads();
        }
        const u64 kth = s_prefix;
        if (threadIdx.x == 0) s_n = 0;
        __syncthreads();
        for_each_candidate(t, q, thr_score, [&](u64 key) {
            if (key >= kth) {
                u32 slot = atomicAdd(&s_n, 1u);
                if (slot < SEL_SMEM_KEYS) s_keys[slot] = key;
            }
        });
        __syncthreads();
        n_valid = min(s_n, (u32)SEL_SMEM_KEYS);
        u32 n2 = 2;
        while (n2 < n_valid) n2 <<= 1;
        for (u32 i = n_valid + threadIdx.x; i < n2; i += blockDim.x) s_keys[i] = 0ull;
        __syncthreads();
        bitonic_sort_desc_smem(s_keys, n2);
    }

    // result keys carry GLOBAL doc ids: score_bits << 32 | (0xFFFFFFFF - global_doc); 0 = empty
    for (u32 i = threadIdx.x; i < k; i += blockDim.x) {
        u64 key = (i < n_valid) ? s_keys[i] : 0ull;
        if (key != 0ull) key -= doc_base;      // (~local) - base == ~(local + base)
        out_keys[(u64)(out_index ? out_index[q] : q) * k + i] = key;
    }
}

// Merge per-shard top-k lists after the all-gather: in[r][q][k] -> out[q][k].
__global__ void __launch_bounds__(SEL_THREADS)
topk_merge_kernel(const u64 *__restrict__ in, u64 rank_stride, u32 world, u32 n_queries, u32 k, u64 *__restrict__ out) {
    __shared__ u64 s_keys[SEL_SMEM_KEYS];
    const u32 q = blockIdx.x;
    const u32 n = world * k;
    u32 n2 = 2;
    while (n2 < n) n2 <<= 1;
    for (u32 i = threadIdx.x; i < n2; i += blockDim.x) {
        u64 v = 0ull;
        if (i < n) {
            u32 r = i / k, j = i % k;
            v = in[(u64)r * rank_stride + (u64)q * k + j];
        }
        s_keys[i] = v;
    }
    __syncthreads();
    bitonic_sort_desc_smem(s_keys, n2);
    for (u32 i = threadIdx.x; i < k; i += blockDim.x) out[(u64)q * k + i] = s_keys[i];
}

int launch_topk_select(sa_index *ix, const TopkCtx &t, u32 n_queries, u64 doc_base, u64 *d_out_keys,
                       const u32 *d_out_index, cudaStream_t stream) {
    if (n_queries == 0) return SA_OK;
    if (!stream) stream = ix->stream;
    KernelTimer tm(ix, 1, stream);
    topk_select_kernel<<<n_queries, SEL_THREADS, 0, stream>>>(t, doc_base, d_out_keys, d_out_index);
    SA_CUDA(cudaGetLastError());
    tm.stop();
    ix->stats.topk_kernel_launches++;
    ix->stats.total_launches++;
    return SA_OK;
}

int launch_topk_merge(sa_index *ix, const u64 *d_in, u64 rank_stride, u32 world, u32 n_queries, u32 k, u64 *d_out) {
    if (n_queries == 0) return SA_OK;
    SA_CHECK((u64)world * k <= SEL_SMEM_KEYS, "world*k too large for the merge kernel");
    KernelTimer tm(ix, 1);
    topk_merge_kernel<<<n_queries, SEL_THREADS, 0, ix->stream>>>(d_in, rank_stride, world, n_queries, k, d_out);
    SA_CUDA(cudaGetLastError());
    tm.stop();
    ix->stats.topk_kernel_launches++;
    ix->stats.total_launches++;
    return SA_OK;
}

// a tile keeps up to 4 * k docs at or above its bound (four docs per thread on the dense tf-table path) plus ties
u32 sa_topk_slots(u32 k) { return k <= 16 ? 128u : 256u; }
