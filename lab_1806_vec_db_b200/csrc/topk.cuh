// topk.cuh — CTA-level bounded top-k over sortable u64 keys (see make_key in common.cuh).
//
// This is the GPU counterpart of ResultSet (reference src/index_algorithm/candidate_pair.rs:43-82)
// for scans whose visiting order is ascending id: the k smallest keys by (distance, id).
//
// Layout per query segment in shared memory: P = 2^p u64 slots.
//   [0, K)        current best, ascending (KEY_NONE padded)
//   [K, K+ncand)  unsorted candidates that beat the current threshold tau = slot[K-1]
//   rest          KEY_NONE
// Threads append candidates with one shared-memory atomic; when a segment may overflow within the
// next `period` appends the CTA sorts all segments (bitonic, all segments per barrier) and the
// first K slots become the new best. Because tau only ever decreases, filtering against a stale
// tau is always safe (it only admits extra candidates).
#pragma once
#include "common.cuh"

namespace vdb {

struct TopkSmem {
    uint64_t* keys;    // [nseg][P]
    uint32_t* ncand;   // [nseg]
    uint32_t K, P, nseg;
    uint32_t limit;    // flush when ncand > limit  (limit = P - K - period)

    __device__ __forceinline__ uint64_t* seg(uint32_t s) const { return keys + (size_t)s * P; }
    __device__ __forceinline__ uint64_t tau(uint32_t s) const { return seg(s)[K - 1]; }

    // all threads
    __device__ __forceinline__ void init() {
        for (uint32_t i = threadIdx.x; i < nseg * P; i += blockDim.x) keys[i] = KEY_NONE;
        for (uint32_t i = threadIdx.x; i < nseg; i += blockDim.x) ncand[i] = 0;
        __syncthreads();
    }
    // any thread; returns true if the segment is now past its flush limit.
    // The caller guarantees at most `period` appends per segment between two maybe_flush() calls.
    __device__ __forceinline__ bool push(uint32_t s, uint64_t key) {
        const uint32_t pos = atomicAdd(&ncand[s], 1u);
        seg(s)[K + pos] = key;
        return pos + 1 > limit;
    }
    // all threads (contains barriers). `want` = this thread saw push() return true.
    __device__ __forceinline__ void maybe_flush(bool want) {
        if (__syncthreads_or(want)) flush_nosync_entry();
    }
    // all threads; must be preceded by a barrier that orders all pushes
    __device__ __forceinline__ void flush_nosync_entry() {
        cta_bitonic_sort(keys, P, nseg, P);  // ends with __syncthreads()
        for (uint32_t i = threadIdx.x; i < nseg * (P - K); i += blockDim.x) {
            const uint32_t s = i / (P - K), j = i - s * (P - K);
            seg(s)[K + j] = KEY_NONE;
        }
        for (uint32_t i = threadIdx.x; i < nseg; i += blockDim.x) ncand[i] = 0;
        __syncthreads();
    }
    // Everything past slot K + ncand is KEY_NONE (the maximum), so sorting the smallest power-of-two prefix that holds the
    // best and the pending candidates of every segment equals sorting the whole segment - at a fraction of the
    // log^2(P) barrier stages when few candidates are pending (the usual state at the end of a scan or a merge).
    __device__ __forceinline__ void final_flush() {
        __syncthreads();
        uint32_t m = 0;
        for (uint32_t s = 0; s < nseg; ++s) m = max(m, ncand[s]);   // CTA-uniform
        const uint32_t need = K + m;
        const uint32_t n = need <= 2 ? 2u : min(P, 1u << (32 - __clz(need - 1)));
        cta_bitonic_sort(keys, n, nseg, P);  // ends with __syncthreads()
        for (uint32_t i = threadIdx.x; i < nseg * (n - min(n, K)); i += blockDim.x) {
            const uint32_t w = n - K, s = i / w, j = i - s * w;
            seg(s)[K + j] = KEY_NONE;
        }
        for (uint32_t i = threadIdx.x; i < nseg; i += blockDim.x) ncand[i] = 0;
        __syncthreads();
    }
    static __host__ __device__ size_t bytes(uint32_t nseg, uint32_t P) {
        return (size_t)nseg * P * 8 + (size_t)nseg * 4;
    }
};

// Smallest power-of-two segment that holds K best + two periods of candidates.
inline uint32_t topk_segment_size(uint32_t K, uint32_t period) { return next_pow2(K + 2 * period); }

// merges `nlists` ascending (or unsorted) key lists of length `len` per query into the k best.
// in: keys[list][query][len] when list_major, else keys[query][list][len].
void launch_merge_sorted(const uint64_t* d_keys, uint32_t nlists, uint32_t nq, uint32_t len, uint32_t k, uint64_t* d_out_keys,
                         uint64_t* d_ids, float* d_dist, uint32_t* d_counts, cudaStream_t stream);
// Optional tail of launch_merge_keys for the tensor path's final merge (one CTA per query is already there): the list's
// overflow flag, the instrumentation count and the completeness check of the merged result - four launches folded into
// the merge. cnt_raw == nullptr: off.
struct MergeFinish {
    const uint32_t* cnt_raw = nullptr;   // [nq] candidates the filter produced (before pruning): > cap = overflowed list
    const uint32_t* qbad = nullptr;      // [nq] non-finite queries (always redone)
    uint32_t cap = 0;
    uint32_t* overflow = nullptr;        // [nq] out, optional
    unsigned long long* cand_total = nullptr;   // += min(list length, cap); zeroed by the caller
    // completeness check (redo == nullptr: off): the result of q is exact iff d_need - shift < tau_q - slack
    const float* tau = nullptr;
    const float* qsq = nullptr;          // nullptr: cosine
    uint64_t n_total = 0;
    uint32_t force_mod = 0;
    uint32_t* redo = nullptr;
    uint32_t* nredo = nullptr;           // zeroed by the caller
};
// true when launch_merge_keys holds k in shared memory (k <= 15 872); above, launch_merge_sorted uses large_k_select
bool merge_keys_fits(uint32_t k);
// topk_large.cu: the k smallest of the nlists * len keys per query of list-major lists [nlists][nq][len] (any order,
// KEY_NONE entries ignored), ascending and KEY_NONE padded to k, by select + sort in global memory; any k
void large_k_select(const uint64_t* d_keys, uint32_t nlists, uint32_t nq, uint64_t len, uint32_t k, uint64_t* d_out_keys,
                    uint64_t* d_ids, float* d_dist, uint32_t* d_counts, cudaStream_t st);
void launch_merge_keys(const uint64_t* d_keys, uint32_t nlists, uint32_t nq, uint32_t len, bool list_major,
                       uint32_t k, uint64_t* d_out_keys, uint64_t* d_ids, float* d_dist,
                       uint32_t* d_counts, cudaStream_t stream, const uint64_t* d_seg_off = nullptr,
                       const uint32_t* d_seg_cnt = nullptr, const MergeFinish* finish = nullptr);

}  // namespace vdb
