// topk_large.cu — exact top-k for any k, in global memory: the large-k path of the Flat search and of the key merges.
//
// The fused top-k (topk.cuh) keeps K best + candidates of every query in one shared-memory segment, which caps k at about
// 15 900. Above that, the keys of a query (every row's key from the scan's emit pass, or the concatenated per-shard lists
// of a merge) are reduced here:
//   1. select: the k-th smallest u64 key T by eight 8-bit digit rounds from the top. Each round is one launch of several
//      CTAs per query with a shared-memory histogram of the keys that match the prefix found so far; the CTAs add it to
//      the query's global histogram and the last one to arrive picks the digit. Keys are unique (the id is the low word),
//      so "key <= T" holds for exactly k keys and ties in distance fall to the lower id. Skipped when k >= the key count.
//   2. compaction of the keys <= T (KEY_NONE excluded) into a k-slot list per query, in arrival order.
//   3. sort of each list: 4096-key tiles bitonic-sorted in shared memory, then merge passes that double the run length;
//      every key finds its output slot by a binary search in the partner run (ties, i.e. KEY_NONE padding only, go to
//      the left run), so a pass is one launch with no shared state.
// A 16-bit digit would take four rounds instead of eight, but its 65 536 32-bit bins are 256 KB, more than a CTA's shared
// memory; with 8-bit digits a round's histogram is 1 KB per warp.
#include <algorithm>

#include "topk.cuh"

namespace vdb {

constexpr int SEL_THREADS = 256;
constexpr int SEL_WARPS = SEL_THREADS / 32;
constexpr int SEL_BITS = 8;
constexpr int SEL_BINS = 1 << SEL_BITS;
constexpr uint32_t SORT_TILE = 4096;   // keys per shared-memory sort (32 KB)

struct SelState {                 // per query, zeroed before the first round
    unsigned long long prefix;    // digits of T found so far
    uint32_t krem;                // rank of T among the keys that match the prefix (1-based); 0 before round 0
    uint32_t arrived;             // CTAs of the current round done
    uint32_t hist[SEL_BINS];
};

// element i of query q: keys[((i / len) * nq + q) * len + i % len] (list-major lists; one list: keys[q * len + i])
struct KeySrc {
    const uint64_t* keys;
    uint32_t nlists, nq;
    uint64_t len;
    __device__ __forceinline__ uint64_t at(uint32_t q, uint64_t i) const {
        if (nlists == 1) return keys[(uint64_t)q * len + i];
        const uint64_t l = i / len;
        return keys[(l * nq + q) * len + (i - l * len)];
    }
};

__global__ void __launch_bounds__(SEL_THREADS) select_round_kernel(const KeySrc src, uint32_t k, int round,
                                                                   SelState* __restrict__ state) {
    __shared__ uint32_t h[SEL_WARPS][SEL_BINS];
    __shared__ uint32_t s_last;
    const uint32_t q = blockIdx.y, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    SelState& S = state[q];
    for (uint32_t i = threadIdx.x; i < SEL_WARPS * SEL_BINS; i += blockDim.x) (&h[0][0])[i] = 0;
    __syncthreads();
    const int shift = 64 - SEL_BITS * (round + 1);
    const uint64_t hi_mask = round == 0 ? 0ull : ~0ull << (shift + SEL_BITS);
    const uint64_t prefix = S.prefix;
    const uint64_t total = (uint64_t)src.nlists * src.len;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i0 = (uint64_t)blockIdx.x * blockDim.x; i0 < total; i0 += stride) {
        const uint64_t i = i0 + threadIdx.x;
        bool in = false;
        uint32_t d = 0;
        if (i < total) {
            const uint64_t key = src.at(q, i);
            in = (key & hi_mask) == prefix;
            d = (uint32_t)(key >> shift) & (SEL_BINS - 1);
        }
        // lanes with the same digit add once (the top digits of a query's keys are few: distances share an exponent)
        const uint32_t peers = __match_any_sync(0xffffffffu, in ? d : 0xffffffffu);
        if (in && lane == (uint32_t)(__ffs(peers) - 1)) atomicAdd(&h[warp][d], (uint32_t)__popc(peers));
    }
    __syncthreads();
    for (uint32_t b = threadIdx.x; b < SEL_BINS; b += blockDim.x) {
        uint32_t c = 0;
#pragma unroll
        for (int w = 0; w < SEL_WARPS; ++w) c += h[w][b];
        if (c) atomicAdd(&S.hist[b], c);
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(&S.arrived, 1u) == gridDim.x - 1 ? 1u : 0u;
    __syncthreads();
    if (!s_last) return;
    // last CTA of this query: the digit of T is the bin in which the running count reaches krem
    __threadfence();
    if (threadIdx.x == 0) {
        uint32_t krem = round == 0 ? k : S.krem, cum = 0, b = 0;
        for (; b < SEL_BINS - 1; ++b) {
            const uint32_t c = __ldcg(&S.hist[b]);
            if (cum + c >= krem) break;
            cum += c;
        }
        S.krem = krem - cum;
        S.prefix = prefix | ((uint64_t)b << shift);
        S.arrived = 0;
    }
    __syncthreads();
    for (uint32_t b = threadIdx.x; b < SEL_BINS; b += blockDim.x) S.hist[b] = 0;
}

// the keys <= T of query q (all keys when state == nullptr), KEY_NONE excluded, into out[q * kp ..) in arrival order
__global__ void __launch_bounds__(SEL_THREADS) select_compact_kernel(const KeySrc src, const SelState* __restrict__ state,
                                                                     uint32_t* __restrict__ cnt, uint64_t kp,
                                                                     uint64_t* __restrict__ out) {
    const uint32_t q = blockIdx.y, lane = threadIdx.x & 31;
    const uint64_t T = state ? state[q].prefix : KEY_NONE;
    const uint64_t total = (uint64_t)src.nlists * src.len;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i0 = (uint64_t)blockIdx.x * blockDim.x; i0 < total; i0 += stride) {
        const uint64_t i = i0 + threadIdx.x;
        uint64_t key = KEY_NONE;
        if (i < total) key = src.at(q, i);
        const bool take = key != KEY_NONE && key <= T;
        const uint32_t m = __ballot_sync(0xffffffffu, take);
        if (!m) continue;
        uint32_t base = 0;
        if (lane == 0) base = atomicAdd(&cnt[q], (uint32_t)__popc(m));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (take) out[(uint64_t)q * kp + base + __popc(m & ((1u << lane) - 1))] = key;
    }
}

__global__ void __launch_bounds__(512) sort_tiles_kernel(uint64_t* __restrict__ keys, uint64_t kp) {
    __shared__ uint64_t s[SORT_TILE];
    uint64_t* g = keys + (uint64_t)blockIdx.y * kp + (uint64_t)blockIdx.x * SORT_TILE;
    for (uint32_t i = threadIdx.x; i < SORT_TILE; i += blockDim.x) s[i] = g[i];
    __syncthreads();
    cta_bitonic_sort(s, SORT_TILE, 1, SORT_TILE);
    for (uint32_t i = threadIdx.x; i < SORT_TILE; i += blockDim.x) g[i] = s[i];
}

// runs of `run` keys, pairwise merged: out slot = own offset + rank in the partner run
__global__ void __launch_bounds__(256) merge_runs_kernel(const uint64_t* __restrict__ in, uint64_t* __restrict__ out,
                                                         uint64_t kp, uint64_t run) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= kp) return;
    const uint64_t* a = in + (uint64_t)blockIdx.y * kp;
    const uint64_t x = a[i];
    const uint64_t r = i / run, base = (r & ~1ull) * run;
    const bool left = (r & 1) == 0;
    const uint64_t p0 = left ? base + run : base;
    const uint64_t p1 = left ? std::min(base + 2 * run, kp) : base + run;
    uint64_t lo = std::min(p0, kp), hi = p1;
    while (lo < hi) {   // left: partner keys < x; right: partner keys <= x
        const uint64_t mid = (lo + hi) >> 1;
        const uint64_t y = a[mid];
        if (left ? y < x : y <= x) lo = mid + 1;
        else hi = mid;
    }
    const uint64_t own = left ? i - base : i - (base + run);
    out[(uint64_t)blockIdx.y * kp + base + own + (lo - std::min(p0, kp))] = x;
}

__global__ void __launch_bounds__(256) emit_sorted_kernel(const uint64_t* __restrict__ sorted, uint64_t kp, uint32_t k,
                                                          const uint32_t* __restrict__ cnt, uint64_t* __restrict__ out_keys,
                                                          uint64_t* __restrict__ ids, float* __restrict__ dist,
                                                          uint32_t* __restrict__ counts) {
    const uint32_t q = blockIdx.y;
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (blockIdx.x == 0 && threadIdx.x == 0 && counts) counts[q] = cnt[q];
    if (j >= k) return;
    const uint64_t key = j < kp ? sorted[(uint64_t)q * kp + j] : KEY_NONE;
    const uint64_t o = (uint64_t)q * k + j;
    if (out_keys) out_keys[o] = key;
    if (ids) {
        const bool ok = key != KEY_NONE;
        ids[o] = ok ? (uint64_t)key_id(key) : KEY_NONE;
        dist[o] = ok ? key_dist(key) : __uint_as_float(0x7fc00000u);
    }
}

// Queries per select + sort chunk: two kp-key buffers per query within 512 MiB.
static uint32_t select_chunk(uint32_t nq, uint64_t kp) {
    const uint64_t per = 2 * kp * 8;
    return (uint32_t)std::min<uint64_t>({nq, 65535, std::max<uint64_t>(1, (512ull << 20) / per)});
}

void large_k_select(const uint64_t* d_keys, uint32_t nlists, uint32_t nq, uint64_t len, uint32_t k, uint64_t* d_out_keys,
                    uint64_t* d_ids, float* d_dist, uint32_t* d_counts, cudaStream_t st) {
    if (nq == 0 || k == 0) return;
    const uint64_t total = (uint64_t)nlists * len;
    const uint64_t kp = round_up<uint64_t>(std::min<uint64_t>(k, total), SORT_TILE);   // at most `total` keys are kept
    const uint32_t chunk = select_chunk(nq, kp);
    const bool select = (uint64_t)k < total;
    // several CTAs per query, about four waves of the machine in all
    const uint32_t ctas = (uint32_t)std::max<uint64_t>(
        1, std::min<uint64_t>(ceil_div<uint64_t>(total, 16 * SEL_THREADS), ceil_div<uint64_t>(8ull * sm_count(), chunk)));
    DevBuf state(select ? (size_t)chunk * sizeof(SelState) : 0, st), cnt((size_t)chunk * 4, st);
    DevBuf buf0((size_t)chunk * kp * 8, st), buf1((size_t)chunk * kp * 8, st);
    ProfScope prof("large_k_select", st);
    for (uint32_t q0 = 0; q0 < nq; q0 += chunk) {
        const uint32_t qn = std::min(chunk, nq - q0);
        // the chunk's queries: list-major input, the same offset into every list
        const KeySrc src{d_keys + (uint64_t)q0 * len, nlists, nq, len};
        if (select) {
            VDB_CUDA(cudaMemsetAsync(state.p, 0, (size_t)qn * sizeof(SelState), st));
            for (int r = 0; r < 64 / SEL_BITS; ++r) {
                select_round_kernel<<<dim3(ctas, qn), SEL_THREADS, 0, st>>>(src, k, r, state.as<SelState>());
                VDB_LAUNCHED();
            }
        }
        VDB_CUDA(cudaMemsetAsync(cnt.p, 0, (size_t)qn * 4, st));
        VDB_CUDA(cudaMemsetAsync(buf0.p, 0xff, (size_t)qn * kp * 8, st));
        select_compact_kernel<<<dim3(ctas, qn), SEL_THREADS, 0, st>>>(src, select ? state.as<SelState>() : nullptr,
                                                                       cnt.as<uint32_t>(), kp, buf0.as<uint64_t>());
        VDB_LAUNCHED();
        sort_tiles_kernel<<<dim3((uint32_t)(kp / SORT_TILE), qn), 512, 0, st>>>(buf0.as<uint64_t>(), kp);
        VDB_LAUNCHED();
        uint64_t* cur = buf0.as<uint64_t>();
        uint64_t* nxt = buf1.as<uint64_t>();
        for (uint64_t run = SORT_TILE; run < kp; run *= 2) {
            merge_runs_kernel<<<dim3((uint32_t)ceil_div<uint64_t>(kp, 256), qn), 256, 0, st>>>(cur, nxt, kp, run);
            VDB_LAUNCHED();
            std::swap(cur, nxt);
        }
        const uint64_t o = (uint64_t)q0 * k;
        emit_sorted_kernel<<<dim3(ceil_div(k, 256u), qn), 256, 0, st>>>(
            cur, kp, k, cnt.as<uint32_t>(), d_out_keys ? d_out_keys + o : nullptr, d_ids ? d_ids + o : nullptr,
            d_dist ? d_dist + o : nullptr, d_counts ? d_counts + q0 : nullptr);
        VDB_LAUNCHED();
    }
}

}  // namespace vdb
