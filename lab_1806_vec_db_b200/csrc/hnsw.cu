// hnsw.cu — K10: HNSW build and search with the graph resident in HBM.
//
// Mirrors HNSWIndex<T> (reference src/index_algorithm/hnsw_index.rs): level-0 links [n][2M] + per-node upper-level
// links, cached-form distances (dist_with_cache :351-355, inner_dist_fn :356-358), search_on_level_fn :258-291,
// greedy_search_on_level_fn :306-330, connect_new_links :226-239, arrange_links :204-224, ResultSet::heuristic
// (candidate_pair.rs:85-99), batch insertion add_parallel :399-457 (read-only candidate search for every new node of
// the batch + brute force among the batch :431-437, then the links are connected in batch order).
//
// The reference parallelises a batch over rayon threads; here a batch is a grid:
//   hnsw_search_kernel   one CTA per query / new node: greedy descent, then search_on_level with the result set
//                        (sorted keys, an "expanded" bit per entry = the BTreeSet queue restricted to the ef best,
//                        which is all the reference's loop can ever pop), a visited hash set in shared memory, and
//                        the <= 2M neighbour rows of every expansion evaluated by the CTA's four warps
//   hnsw_select_kernel   heuristic(M) over a new node's candidates -> its links (connect_new_links)
//   hnsw_arrange_kernel  one CTA per touched (neighbour, level): appends the new back-links in batch order and
//                        re-selects with the heuristic when the list is full (arrange_links)
// Connecting all new nodes first and applying the back-links grouped by target afterwards gives the same graph as
// the reference's sequential loop over the batch: connect_new_links reads only the candidates computed in the
// read-only phase, and the back-links of one target are applied in batch order.
// The graph itself is unpinned in the reference (RNG levels, thread count dependent batches), so parity is by
// recall; the distances returned by a search are re-evaluated by the cached-form pair kernel (pairs.cu, K10).
#include <algorithm>
#include <cstdlib>
#include <utility>
#include <vector>

#include "index.cuh"
#include "topk.cuh"

namespace vdb {

constexpr int HN_THREADS = 256;
constexpr uint32_t HN_EMPTY = 0xFFFFFFFFu;
constexpr uint32_t HN_MAX_M0 = 64;  // M <= 32

struct HnswGraph {
    uint32_t* links0;   // [n][M0]
    uint32_t* len0;     // [n]
    uint32_t* ulinks;   // [(slots)][M]   slot = uoff[node] + (level - 1)
    uint32_t* ulen;     // [(slots)]
    const uint64_t* uoff;  // [n+1]
    uint32_t M, M0;
};

__device__ __forceinline__ const uint32_t* hn_links(const HnswGraph& g, uint32_t node, uint32_t level, uint32_t& len) {
    if (level == 0) {
        len = g.len0[node];
        return g.links0 + (size_t)node * g.M0;
    }
    const uint64_t slot = g.uoff[node] + (level - 1);
    len = g.ulen[slot];
    return g.ulinks + slot * g.M;
}

// dot product of a row in global memory with a vector held as zero-padded f32 in shared memory; every lane gets it
template <typename T>
__device__ __forceinline__ float warp_dot_row(const T* __restrict__ row, const float* __restrict__ qs, uint32_t pitch, int lane);
// Every lane issues ALL its loads of a 1024-element chunk (8 x 16 bytes) before the first FMA: a walk is a chain of
// dependent row gathers, and with the loads inside the FMA loop a 960-d row cost four HBM round trips instead of one
// (ncu, round 2: the FFMAs of this function held most of the long-scoreboard stalls). The two accumulation chains and
// their order (rounds 0, 2, 4, ... in s0, rounds 1, 3, 5, ... in s1) are unchanged, so the distances are bit-identical.
template <>
__device__ __forceinline__ float warp_dot_row<float>(const float* __restrict__ row, const float* __restrict__ qs, uint32_t pitch,
                                                     int lane) {
    const float4* r4 = reinterpret_cast<const float4*>(row);
    const float4* q4 = reinterpret_cast<const float4*>(qs);
    float s0 = 0.f, s1 = 0.f;
    const uint32_t n4 = pitch >> 2;
    for (uint32_t base = lane; base < n4; base += 256) {
        float4 a[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const uint32_t e = base + 32 * u;
            // UNCONDITIONAL loads (index clamped into the row; the FMAs below skip the rounds past its end): ptxas hoists
            // straight-line loads ahead of the arithmetic but keeps predicated ones next to their consumers
            a[u] = __ldg(r4 + min(e, n4 - 1));
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const uint32_t e = base + 32 * u;
            if (e < n4) {
                const float4 b = q4[e];
                if (u & 1) s1 = fmaf(a[u].x, b.x, fmaf(a[u].y, b.y, fmaf(a[u].z, b.z, fmaf(a[u].w, b.w, s1))));
                else s0 = fmaf(a[u].x, b.x, fmaf(a[u].y, b.y, fmaf(a[u].z, b.z, fmaf(a[u].w, b.w, s0))));
            }
        }
    }
    float s = s0 + s1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    return s;
}
template <>
__device__ __forceinline__ float warp_dot_row<uint8_t>(const uint8_t* __restrict__ row, const float* __restrict__ qs, uint32_t pitch,
                                                       int lane) {
    const uint32_t* r4 = reinterpret_cast<const uint32_t*>(row);
    const float4* q4 = reinterpret_cast<const float4*>(qs);
    float s = 0.f;
    const uint32_t n4 = pitch >> 2;
    for (uint32_t base = lane; base < n4; base += 256) {
        uint32_t v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const uint32_t e = base + 32 * u;
            v[u] = __ldg(r4 + min(e, n4 - 1));
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const uint32_t e = base + 32 * u;
            if (e < n4) {
                const float4 b = q4[e];
                s = fmaf((float)(v[u] & 0xffu), b.x, fmaf((float)((v[u] >> 8) & 0xffu), b.y,
                                                          fmaf((float)((v[u] >> 16) & 0xffu), b.z, fmaf((float)(v[u] >> 24), b.w, s))));
            }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    return s;
}
// L2 prefetch of a whole row by one warp (lane = 128-byte line): the rows a warp evaluates AFTER its first one of an expansion
// are then L2 hits, and so are the link lists of the entries most likely to be expanded next
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
__device__ __forceinline__ void warp_prefetch_bytes(const void* base, uint32_t bytes, int lane) {
    const char* c = reinterpret_cast<const char*>(base);
    for (uint32_t off = (uint32_t)lane * 128; off < bytes; off += 32 * 128) prefetch_l2(c + off);
}
// row -> zero-padded f32 vector in shared memory (all threads of the CTA)
template <typename T>
__device__ __forceinline__ void stage_row(const T* __restrict__ row, uint32_t dim, uint32_t dimpad, float* dst) {
    for (uint32_t e = threadIdx.x; e < dimpad; e += blockDim.x) dst[e] = e < dim ? (float)row[e] : 0.f;
}
// cached-form distance (distance/mod.rs:54-57, 67-69) from the dot product and the two caches
template <int METRIC> __device__ __forceinline__ float cached_dist(float dot, float ca, float cb) {
    if (METRIC == VDB_L2SQR) return __fsub_rn(__fadd_rn(ca, cb), __fmul_rn(2.0f, dot));
    return __fsub_rn(1.0f, __fdiv_rn(dot, fmaxf(__fmul_rn(ca, cb), 1e-10f)));
}

// visited set: open addressing in shared memory. Returns true when `id` was not present (and is now).
__device__ __forceinline__ bool hash_insert(uint32_t* hash, uint32_t mask, uint32_t id) {
    uint32_t slot = (id * 2654435761u) & mask;
    for (uint32_t probe = 0; probe <= mask; ++probe) {
        const uint32_t prev = atomicCAS(&hash[slot], HN_EMPTY, id);
        if (prev == HN_EMPTY) return true;
        if (prev == id) return false;
        slot = (slot + 1) & mask;
    }
    return false;
}

// Result-set keys: order_bits(dist) << 32 | id << 1 | expanded. Merges the m (<= 32) keys of nk[] into the sorted
// res[0..rn) keeping the `ef` smallest; the merged array lands in res2. Returns the new length. Block-wide.
__device__ __forceinline__ uint32_t merge_new(const uint64_t* res, uint64_t* res2, uint32_t rn, uint32_t ef, const uint64_t* nk,
                                              uint32_t m) {
    for (uint32_t i = threadIdx.x; i < rn; i += blockDim.x) {
        const uint64_t key = res[i];
        uint32_t cnt = 0;
        for (uint32_t j = 0; j < m; ++j) cnt += nk[j] < key;
        const uint32_t pos = i + cnt;
        if (pos < ef) res2[pos] = key;
    }
    if (threadIdx.x < m) {
        const uint64_t key = nk[threadIdx.x];
        uint32_t rank = 0;
        for (uint32_t j = 0; j < m; ++j) rank += nk[j] < key;
        uint32_t lo = 0, hi = rn;  // lower bound in res
        while (lo < hi) {
            const uint32_t mid = (lo + hi) >> 1;
            if (res[mid] < key) lo = mid + 1;
            else hi = mid;
        }
        const uint32_t pos = rank + lo;
        if (pos < ef) res2[pos] = key;
    }
    __syncthreads();
    return min(ef, rn + m);
}

struct HnswSearchParams {
    HnswGraph g;
    const void* rows;
    uint32_t pitch, dim, dimpad;
    const float* rcache;       // dist_cache of every row
    const void* queries;       // [nq][dim] (search) or nullptr
    const float* qcache;       // [nq] (search)
    uint32_t qrow_base;        // build: query i is row qrow_base + i
    const uint32_t* level;     // build: level of every row
    uint32_t nq, ef, hash_mask;
    uint32_t* ghash;           // visited sets in GLOBAL memory, one of hash_mask + 1 slots per CTA (large ef); nullptr: shared memory
    uint32_t* overflow;        // counts neighbours that could not be recorded because a visited set was 7/8 full
    unsigned long long* evals; // distance evaluations of the search_on_level loops (instrumentation: bytes gathered)
    uint32_t* next_q;          // work queue: next query index to hand out (starts at gridDim.x); nullptr: static stride
    uint32_t enter_point, enter_level;
    int build;
    const uint64_t* out_off;   // build: first list of query i; its list of level l is out_off[i] + l
    uint64_t* out_keys;        // [lists][ef] ascending, KEY_NONE padded; ids plain
    // PQ mode (knn_pq :672-697): distances are ADC sums over the 4-bit codes instead of row dot products
    const uint8_t* codes;      // [n][enc]
    uint32_t enc, m;
    const float* lut;          // [nq][m*16]
    const float* dcache;       // [m*16] (cosine: ||c||^2 per centroid)
};

template <typename T, int METRIC, bool PQ>
__global__ void __launch_bounds__(HN_THREADS, 4) hnsw_search_kernel(const HnswSearchParams p) {
    extern __shared__ __align__(16) uint8_t smem[];
    float* qs = reinterpret_cast<float*>(smem);                                  // [dimpad]: query, or LUT (+ dist_cache) in PQ mode
    uint64_t* resA = reinterpret_cast<uint64_t*>(qs + p.dimpad);                 // [ef]
    uint64_t* resB = resA + p.ef;                                                // [ef]
    uint64_t* nk = resB + p.ef;                                                  // [32]
    uint32_t* nb = reinterpret_cast<uint32_t*>(nk + 32);                         // [64]
    uint32_t* hash = p.ghash ? p.ghash + (size_t)blockIdx.x * (p.hash_mask + 1) : nb + 64;   // [hash_mask + 1]
    __shared__ int s_best;
    __shared__ uint32_t s_m, s_hcount, s_cur;
    __shared__ float s_curd;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const T* rows = reinterpret_cast<const T*>(p.rows);
    const uint32_t hcap = p.hash_mask + 1, hlimit = hcap - (hcap >> 3);

    // Queries are handed out dynamically: walks differ in length, and with a static stride a 1000-query batch on ~600
    // resident CTAs takes two full rounds whatever the second round holds
    __shared__ uint32_t s_next;
    for (uint32_t q = blockIdx.x; q < p.nq;) {
        const uint32_t qrow = p.qrow_base + q;
        __syncthreads();
        if (PQ) {
            const uint32_t tab = p.m * 16;
            for (uint32_t e = threadIdx.x; e < tab; e += blockDim.x) {
                qs[e] = p.lut[(size_t)q * tab + e];
                if (METRIC == VDB_COSINE) qs[tab + e] = p.dcache[e];
            }
        } else {
            const T* qsrc = p.build ? rows + (size_t)qrow * p.pitch : reinterpret_cast<const T*>(p.queries) + (size_t)q * p.dim;
            stage_row<T>(qsrc, p.dim, p.dimpad, qs);
        }
        const float qc = p.build ? p.rcache[qrow] : p.qcache[q];
        const uint32_t target = p.build ? p.level[qrow] : 0u;
        __syncthreads();
        auto dist_to = [&](uint32_t id) -> float {  // warp-wide
            if (PQ) {  // ADC (pq_table.rs:239-301): lanes take the groups round-robin
                const uint8_t* code = p.codes + (size_t)id * p.enc;
                const uint32_t tab = p.m * 16;
                float sv = 0.f, cv = 0.f;
                for (uint32_t g = lane; g < p.m; g += 32) {
                    const uint32_t byte = code[g >> 1];
                    const uint32_t e = g * 16 + ((g & 1) ? (byte >> 4) : (byte & 0xfu));
                    sv += qs[e];
                    if (METRIC == VDB_COSINE) cv += qs[tab + e];
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    sv += __shfl_xor_sync(0xffffffffu, sv, o);
                    if (METRIC == VDB_COSINE) cv += __shfl_xor_sync(0xffffffffu, cv, o);
                }
                if (METRIC == VDB_L2SQR) return sv;
                return 1.0f - sv / fmaxf(sqrtf(cv) * qc, 1e-10f);
            }
            const float dot = warp_dot_row<T>(rows + (size_t)id * p.pitch, qs, p.pitch, lane);
            return cached_dist<METRIC>(dot, p.rcache[id], qc);
        };
        // ---- greedy descent (greedy_search_until_level_fn): levels enter_level .. target + 1 ----
        uint32_t cur = p.enter_point;
        if (target < p.enter_level) {
            float cur_d = dist_to(cur);
            for (uint32_t lvl = p.enter_level; lvl > target; --lvl) {
                for (;;) {
                    uint32_t len;
                    const uint32_t* lk = hn_links(p.g, cur, lvl, len);
                    if (threadIdx.x == 0) {
                        s_cur = cur;
                        s_curd = cur_d;
                    }
                    __syncthreads();
                    // every warp evaluates its share; the best (distance, list position) improvement wins
                    for (uint32_t j = warp; j < len; j += HN_THREADS / 32) {
                        const uint32_t id = lk[j];
                        const float d = dist_to(id);
                        if (lane == 0) nk[j] = ((uint64_t)f32_order_bits(d) << 32) | j;
                    }
                    __syncthreads();
                    if (threadIdx.x == 0) {
                        uint64_t bestk = ~0ull;
                        for (uint32_t j = 0; j < len; ++j) bestk = nk[j] < bestk ? nk[j] : bestk;
                        if (len && key_dist(bestk) < s_curd) {
                            s_cur = lk[(uint32_t)bestk];
                            s_curd = key_dist(bestk);
                            s_m = 1;
                        } else {
                            s_m = 0;
                        }
                    }
                    __syncthreads();
                    cur = s_cur;
                    cur_d = s_curd;
                    const bool moved = s_m != 0;
                    __syncthreads();
                    if (!moved) break;
                }
            }
        }
        // ---- search_on_level for the levels the node lives on (build) or level 0 (search) ----
        const uint32_t top = min(target, p.enter_level);
        for (int lvl = (int)top; lvl >= 0; --lvl) {
            for (uint32_t e = threadIdx.x; e < hcap; e += blockDim.x) hash[e] = HN_EMPTY;
            uint64_t* res = resA;
            uint64_t* res2 = resB;
            uint32_t rn = 1;
            __syncthreads();
            {
                const float d = dist_to(cur);
                if (threadIdx.x == 0) {
                    hash_insert(hash, p.hash_mask, cur);
                    res[0] = ((uint64_t)f32_order_bits(d) << 32) | ((uint64_t)cur << 1);
                    s_hcount = 1;
                }
            }
            __syncthreads();
            for (;;) {
                if (threadIdx.x == 0) s_best = 0x7fffffff;
                __syncthreads();
                for (uint32_t i = threadIdx.x; i < rn; i += blockDim.x)
                    if (!(res[i] & 1ull)) {
                        atomicMin(&s_best, (int)i);
                        break;
                    }
                __syncthreads();
                const int best = s_best;
                // queue empty, or check_candidate fails (the best unexpanded entry is the full set's last one)
                if (best == 0x7fffffff || (rn == p.ef && (uint32_t)best == rn - 1)) break;
                const uint32_t c = (uint32_t)(res[best] & 0xffffffffull) >> 1;
                __syncthreads();
                if (threadIdx.x == 0) res[best] |= 1ull;
                if (warp == 0) {
                    uint32_t len;
                    const uint32_t* lk = hn_links(p.g, c, (uint32_t)lvl, len);
                    uint32_t base = 0;
                    for (uint32_t j0 = 0; j0 < len; j0 += 32) {
                        const uint32_t j = j0 + lane;
                        bool fresh = false;
                        uint32_t id = 0;
                        if (j < len) {
                            // at most one insertion per lane of this round: the set never holds more than hlimit ids,
                            // so hash_insert always finds a free slot, whatever the set's size
                            if (s_hcount + base + (uint32_t)lane < hlimit) {
                                id = lk[j];
                                fresh = hash_insert(hash, p.hash_mask, id);
                            } else {
                                atomicAdd(p.overflow, 1u);   // never silent: the host turns this into an error
                            }
                        }
                        const uint32_t bal = __ballot_sync(0xffffffffu, fresh);
                        if (fresh) nb[base + __popc(bal & ((1u << lane) - 1))] = id;
                        base += __popc(bal);
                    }
                    if (lane == 0) {
                        s_m = base;
                        s_hcount += base;
                    }
                }
                __syncthreads();
                const uint32_t m_all = s_m;
                // rows this warp evaluates after its first one: on their way to L2 while the first is being read
                for (uint32_t j = warp + HN_THREADS / 32; j < m_all; j += HN_THREADS / 32) {
                    if (PQ) prefetch_l2(p.codes + (size_t)nb[j] * p.enc);
                    else warp_prefetch_bytes(rows + (size_t)nb[j] * p.pitch, p.dim * (uint32_t)sizeof(T), lane);
                }
                for (uint32_t m0 = 0; m0 < m_all; m0 += 32) {  // M0 <= 64: at most two rounds
                    const uint32_t m = min(32u, m_all - m0);
                    for (uint32_t j = warp; j < m; j += HN_THREADS / 32) {
                        const uint32_t id = nb[m0 + j];
                        const float d = dist_to(id);
                        if (lane == 0) nk[j] = ((uint64_t)f32_order_bits(d) << 32) | ((uint64_t)id << 1);
                    }
                    __syncthreads();
                    rn = merge_new(res, res2, rn, p.ef, nk, m);
                    uint64_t* t = res;
                    res = res2;
                    res2 = t;
                }
                // the next expansion takes the best unexpanded entry, almost always one of the first few: its link list
                // (one dependent read at the head of every expansion) is sent to L2 now
                if (lvl == 0 && threadIdx.x < 16 && threadIdx.x < rn && !(res[threadIdx.x] & 1ull)) {
                    const uint32_t node = (uint32_t)(res[threadIdx.x] & 0xffffffffull) >> 1;
                    prefetch_l2(p.g.links0 + (size_t)node * p.g.M0);
                    prefetch_l2(p.g.len0 + node);
                }
            }
            if (threadIdx.x == 0 && p.evals) atomicAdd(p.evals, (unsigned long long)s_hcount);   // rows evaluated on this level
            cur = (uint32_t)(res[0] & 0xffffffffull) >> 1;  // nearest graph result = entry of the next level
            if (p.build) {
                // brute force among the earlier nodes of the batch that live on this level (:431-437)
                for (uint32_t j0 = 0; j0 < q; j0 += 32) {
                    if (warp == 0) {
                        const uint32_t j = j0 + lane;
                        const bool ok = j < q && p.level[p.qrow_base + j] >= (uint32_t)lvl;
                        const uint32_t bal = __ballot_sync(0xffffffffu, ok);
                        if (ok) nb[__popc(bal & ((1u << lane) - 1))] = p.qrow_base + j;
                        if (lane == 0) s_m = __popc(bal);
                    }
                    __syncthreads();
                    const uint32_t m = s_m;
                    if (m) {
                        for (uint32_t j = warp; j < m; j += HN_THREADS / 32) {
                            const uint32_t id = nb[j];
                            const float d = dist_to(id);
                            if (lane == 0) nk[j] = ((uint64_t)f32_order_bits(d) << 32) | ((uint64_t)id << 1);
                        }
                        __syncthreads();
                        rn = merge_new(res, res2, rn, p.ef, nk, m);
                        uint64_t* t = res;
                        res = res2;
                        res2 = t;
                    }
                    __syncthreads();
                }
            }
            uint64_t* out = p.out_keys + ((p.build ? p.out_off[q] + (uint64_t)lvl : (uint64_t)q) * p.ef);
            for (uint32_t i = threadIdx.x; i < p.ef; i += blockDim.x)
                out[i] = i < rn ? ((res[i] & 0xffffffff00000000ull) | ((res[i] & 0xffffffffull) >> 1)) : KEY_NONE;
            __syncthreads();
        }
        if (p.next_q) {
            if (threadIdx.x == 0) s_next = atomicAdd(p.next_q, 1u);
            __syncthreads();
            q = s_next;
        } else {
            q += gridDim.x;
        }
    }
}

// ---- connect_new_links: heuristic(M) over the candidates of one (new node, level) ---------------------------------
struct HnswSelectParams {
    HnswGraph g;
    const void* rows;
    uint32_t pitch, dim, dimpad;
    const float* rcache;
    const uint64_t* cand;      // [tasks][ef]
    uint32_t ef, ntasks;
    const uint32_t* task_node; // [tasks]
    const uint32_t* task_lvl;  // [tasks]
    uint32_t* sel;             // [tasks][M] chosen neighbours
    uint32_t* selcnt;          // [tasks]
};

// heuristic over a sorted (distance, id) list: keep x when every kept y has d(x, y) >= d(x, base). Block-wide.
// The candidates are tested a WINDOW at a time, one per warp, against the members kept so far (a candidate that fails
// against them fails in the sequential loop too, because the kept set only grows); the survivors of a window are then
// admitted in order, each later survivor re-tested against the member just admitted. The result is exactly the
// sequential heuristic's. `xs` holds one dimpad-float staging buffer per warp. Returns the number kept (ids in kept[]).
constexpr int HN_WARPS = HN_THREADS / 32;
template <typename T, int METRIC>
__device__ uint32_t heuristic_select(const T* rows, uint32_t pitch, uint32_t dim, uint32_t dimpad, const float* rcache,
                                     const uint64_t* sorted, uint32_t count, uint32_t limit, float* xs, uint32_t* kept) {
    __shared__ int s_pass[HN_WARPS];
    __shared__ uint32_t s_id[HN_WARPS];
    __shared__ float s_dx[HN_WARPS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* xw = xs + (size_t)warp * dimpad;
    uint32_t nk = 0;
    for (uint32_t i = 0; i < count && nk < limit; i += HN_WARPS) {
        if (sorted[i] == KEY_NONE) break;
        __syncthreads();
        const uint32_t idx = i + warp;
        const uint64_t key = idx < count ? sorted[idx] : KEY_NONE;
        bool pass = key != KEY_NONE;
        const uint32_t x = key_id(key);
        const float dx = key_dist(key);
        float cx = 0.f;
        if (pass) {
            const T* xr = rows + (size_t)x * pitch;
            for (uint32_t e = lane; e < dimpad; e += 32) xw[e] = e < dim ? (float)xr[e] : 0.f;
            __syncwarp();
            cx = rcache[x];
            for (uint32_t j = 0; j < nk; ++j) {
                const uint32_t y = kept[j];
                const float dot = warp_dot_row<T>(rows + (size_t)y * pitch, xw, pitch, lane);
                if (!(cached_dist<METRIC>(dot, cx, rcache[y]) >= dx)) {
                    pass = false;
                    break;
                }
            }
        }
        if (lane == 0) {
            s_pass[warp] = pass;
            s_id[warp] = x;
            s_dx[warp] = dx;
        }
        __syncthreads();
        for (int u = 0; u < HN_WARPS && nk < limit; ++u) {
            if (!s_pass[u]) continue;  // uniform: read after a barrier
            if (threadIdx.x == 0) kept[nk] = s_id[u];
            ++nk;
            if (warp > u && s_pass[warp]) {  // later survivors must also clear the member just admitted
                const uint32_t y = s_id[u];
                const float dot = warp_dot_row<T>(rows + (size_t)y * pitch, xw, pitch, lane);
                if (!(cached_dist<METRIC>(dot, cx, rcache[y]) >= dx) && lane == 0) s_pass[warp] = 0;
            }
            __syncthreads();
        }
    }
    __syncthreads();
    return nk;
}

template <typename T, int METRIC>
__global__ void __launch_bounds__(HN_THREADS, 4) hnsw_select_kernel(const HnswSelectParams p) {
    extern __shared__ __align__(16) uint8_t smem[];
    float* xs = reinterpret_cast<float*>(smem);
    __shared__ uint32_t kept[HN_MAX_M0 + 1];
    const uint32_t t = blockIdx.x;
    if (t >= p.ntasks) return;
    const T* rows = reinterpret_cast<const T*>(p.rows);
    const uint32_t node = p.task_node[t], lvl = p.task_lvl[t];
    // the initial number of neighbours is limited to M even on level 0 (:231-235)
    const uint32_t nk = heuristic_select<T, METRIC>(rows, p.pitch, p.dim, p.dimpad, p.rcache, p.cand + (size_t)t * p.ef, p.ef, p.g.M, xs,
                                                    kept);
    uint32_t* dst = lvl == 0 ? p.g.links0 + (size_t)node * p.g.M0 : p.g.ulinks + (p.g.uoff[node] + (lvl - 1)) * p.g.M;
    for (uint32_t j = threadIdx.x; j < nk; j += blockDim.x) {
        dst[j] = kept[j];
        p.sel[(size_t)t * p.g.M + j] = kept[j];
    }
    if (threadIdx.x == 0) {
        if (lvl == 0) p.g.len0[node] = nk;
        else p.g.ulen[p.g.uoff[node] + (lvl - 1)] = nk;
        p.selcnt[t] = nk;
    }
}

// ---- arrange_links: back-links of one (target, level), applied in batch order -------------------------------------
struct HnswArrangeParams {
    HnswGraph g;
    const void* rows;
    uint32_t pitch, dim, dimpad;
    const float* rcache;
    uint32_t ngroups;
    const uint32_t* grp_node;  // [groups]
    const uint32_t* grp_lvl;   // [groups]
    const uint32_t* grp_off;   // [groups + 1] into inc
    const uint32_t* inc;       // new nodes linking to the target, batch order
};

template <typename T, int METRIC>
__global__ void __launch_bounds__(HN_THREADS, 4) hnsw_arrange_kernel(const HnswArrangeParams p) {
    extern __shared__ __align__(16) uint8_t smem[];
    float* rs = reinterpret_cast<float*>(smem);  // row of the target
    float* xs = rs + p.dimpad;                   // one staging row per warp for the candidates under test
    __shared__ uint32_t lk[HN_MAX_M0 + 1], kept[HN_MAX_M0 + 1];
    __shared__ uint64_t keys[HN_MAX_M0 + 1], sorted[HN_MAX_M0 + 1];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t g = blockIdx.x;
    if (g >= p.ngroups) return;
    const T* rows = reinterpret_cast<const T*>(p.rows);
    const uint32_t r = p.grp_node[g], lvl = p.grp_lvl[g];
    const uint32_t limit = lvl == 0 ? p.g.M0 : p.g.M;
    uint32_t* dst = lvl == 0 ? p.g.links0 + (size_t)r * p.g.M0 : p.g.ulinks + (p.g.uoff[r] + (lvl - 1)) * p.g.M;
    uint32_t* dlen = lvl == 0 ? p.g.len0 + r : p.g.ulen + (p.g.uoff[r] + (lvl - 1));
    uint32_t len = *dlen;
    for (uint32_t j = threadIdx.x; j < len; j += blockDim.x) lk[j] = dst[j];
    stage_row<T>(rows + (size_t)r * p.pitch, p.dim, p.dimpad, rs);
    const float cr = p.rcache[r];
    __syncthreads();
    for (uint32_t e = p.grp_off[g]; e < p.grp_off[g + 1]; ++e) {
        if (threadIdx.x == 0) lk[len] = p.inc[e];
        __syncthreads();
        if (len + 1 <= limit) {
            ++len;
            continue;
        }
        const uint32_t cnt = len + 1;
        // ResultSet(limit + 1) of (d(target, x), x)
        for (uint32_t j = warp; j < cnt; j += HN_THREADS / 32) {
            const uint32_t x = lk[j];
            const float dot = warp_dot_row<T>(rows + (size_t)x * p.pitch, rs, p.pitch, lane);
            if (lane == 0) keys[j] = make_key(cached_dist<METRIC>(dot, cr, p.rcache[x]), x);
        }
        __syncthreads();
        if (threadIdx.x < cnt) {  // rank sort (ids are distinct)
            const uint64_t k = keys[threadIdx.x];
            uint32_t rank = 0;
            for (uint32_t j = 0; j < cnt; ++j) rank += keys[j] < k;
            sorted[rank] = k;
        }
        __syncthreads();
        len = heuristic_select<T, METRIC>(rows, p.pitch, p.dim, p.dimpad, p.rcache, sorted, cnt, limit, xs, kept);
        for (uint32_t j = threadIdx.x; j < len; j += blockDim.x) lk[j] = kept[j];
        __syncthreads();
    }
    for (uint32_t j = threadIdx.x; j < len; j += blockDim.x) dst[j] = lk[j];
    if (threadIdx.x == 0) *dlen = len;
}

__global__ void iota_pairs_kernel(const uint64_t* __restrict__ keys, uint32_t nq, uint32_t ef, uint32_t k, uint32_t* __restrict__ qidx,
                                  uint32_t* __restrict__ rid, uint8_t* __restrict__ valid) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (uint64_t)nq * k) return;
    const uint32_t q = (uint32_t)(i / k), j = (uint32_t)(i - (uint64_t)q * k);
    const uint64_t key = keys[(size_t)q * ef + j];
    qidx[i] = q;
    rid[i] = key == KEY_NONE ? 0u : key_id(key);
    valid[i] = key != KEY_NONE;
}

// ---- host side -----------------------------------------------------------------------------------------------------
// Visited-set capacity. The reference's visited set is unbounded (hnsw_index.rs:258-291); here a search records at
// most 2M nodes per expansion and typically 10-15. Up to ef = 896 the set lives in shared memory (8192 / 16384 / 32768
// slots); beyond it lives in global memory with 4 ef 2M slots per CTA. A neighbour that cannot be recorded because the
// set is 7/8 full is counted (HnswSearchParams::overflow). Long walks on large hard sets do fill the smaller tiers
// (50 000 uniform 64-d rows at M = 32 evaluate more than 7168 distinct rows at ef 200), so the host calls and every
// build batch re-run a search that overflowed with a set that cannot fill (never_full_slots); the set's size never
// changes a result, only whether the walk could finish. The `_dev` searches leave the count to the caller
// (vdb_hnsw_overflow).
constexpr uint32_t HN_SMEM_HASH_MAX_EF = 896;
static uint32_t hash_cap_for(uint32_t ef, uint32_t M0) {
    static const uint32_t small_to = getenv("VDB_HNSW_SMALL_HASH_EF") ? (uint32_t)atoi(getenv("VDB_HNSW_SMALL_HASH_EF")) : 448u;
    static const uint32_t force = getenv("VDB_HNSW_HASH_SLOTS") ? (uint32_t)atoi(getenv("VDB_HNSW_HASH_SLOTS")) : 0u;   // tests
    if (force) return next_pow2(force);
    if (ef <= small_to) return 8192u;
    if (ef <= 640) return 16384u;
    if (ef <= HN_SMEM_HASH_MAX_EF) return 32768u;
    return next_pow2(4u * ef * std::max(M0, 1u));
}
// slots of a visited set that one walk over n rows can never fill to 7/8: at least 8/7 (n + 1)
static uint32_t never_full_slots(uint64_t n) {
    const uint64_t need = (8 * (n + 1) + 6) / 7;
    uint64_t s = 1;
    while (s < need) s <<= 1;
    return (uint32_t)std::min<uint64_t>(s, 1ull << 31);
}

template <typename KernT, typename ParamT>
static void launch_dyn(KernT kern, uint32_t grid, size_t smem, const ParamT& p, cudaStream_t st) {
    if (smem > 48 * 1024) VDB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, HN_THREADS, smem, st>>>(p);
    VDB_LAUNCHED();
}

// `overflow` = the handle's device counter (vdb_hnsw::d_overflow)
static void launch_search(const vdb_dataset* ds, const HnswSearchParams& p, uint32_t* overflow, cudaStream_t st) {
    const bool pq = p.codes != nullptr;
    const size_t vec_floats = pq ? (size_t)p.m * 16 * (ds->metric == VDB_COSINE ? 2 : 1) : (size_t)p.dimpad;
    const uint32_t slots = p.hash_mask + 1;
    const bool global_hash = slots > 32768u;
    const size_t smem = round_up(vec_floats, (size_t)4) * 4 + (size_t)p.ef * 16 + 32 * 8 + 64 * 4 + (global_hash ? 0 : (size_t)slots * 4);
    VDB_REQUIRE(smem <= 200 * 1024, "HNSW search: ef=%u / dim=%u do not fit in shared memory", p.ef, p.dim);
    const uint32_t per_sm = (uint32_t)std::max<size_t>(1, std::min<size_t>(8, (220 * 1024) / smem));
    uint32_t grid = std::min<uint32_t>(p.nq, (uint32_t)sm_count() * per_sm);
    DevBuf ghash;
    if (global_hash) {   // bound the tables to 1 GiB
        grid = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(grid, (1ull << 30) / ((uint64_t)slots * 4)));
        ghash = DevBuf((size_t)grid * slots * 4, st);
    }
    DevBuf next_q(4, st);
    VDB_CUDA(cudaMemcpyAsync(next_q.p, &grid, 4, cudaMemcpyHostToDevice, st));   // the first `grid` queries are the CTAs' own
    ProfScope prof("hnsw_search", st);
    const bool l2 = ds->metric == VDB_L2SQR;
    HnswSearchParams q = p;
    q.ghash = ghash.as<uint32_t>();
    q.next_q = next_q.as<uint32_t>();
    q.overflow = overflow;
    q.evals = overflow ? reinterpret_cast<unsigned long long*>(overflow + 2) : nullptr;   // same 16-byte allocation
    if (pq) q.dimpad = (uint32_t)round_up(vec_floats, (size_t)4);  // the kernel's vector area holds the tables
    if (pq) {
        if (l2) launch_dyn(hnsw_search_kernel<uint8_t, VDB_L2SQR, true>, grid, smem, q, st);
        else launch_dyn(hnsw_search_kernel<uint8_t, VDB_COSINE, true>, grid, smem, q, st);
    } else if (ds->dtype == VDB_F32) {
        if (l2) launch_dyn(hnsw_search_kernel<float, VDB_L2SQR, false>, grid, smem, q, st);
        else launch_dyn(hnsw_search_kernel<float, VDB_COSINE, false>, grid, smem, q, st);
    } else {
        if (l2) launch_dyn(hnsw_search_kernel<uint8_t, VDB_L2SQR, false>, grid, smem, q, st);
        else launch_dyn(hnsw_search_kernel<uint8_t, VDB_COSINE, false>, grid, smem, q, st);
    }
}

// Reads and clears the handle's overflow counter (the stream is synchronised): true when a search since the last read
// could not record a neighbour in its visited set, i.e. its results may have lost recall
bool hnsw_take_overflow(const vdb_hnsw* h, cudaStream_t st) {
    if (!h->d_overflow) return false;
    uint32_t v = 0;
    VDB_CUDA(cudaMemcpyAsync(&v, h->d_overflow, 4, cudaMemcpyDeviceToHost, st));
    VDB_CUDA(cudaStreamSynchronize(st));
    if (v) VDB_CUDA(cudaMemsetAsync(h->d_overflow, 0, 4, st));
    return v != 0;
}
// a search that overflowed even a never_full_slots set (only possible past 1.8e9 rows) fails loudly
void hnsw_check_overflow(const vdb_hnsw* h, cudaStream_t st) {
    if (hnsw_take_overflow(h, st))
        fail(VDB_EUNSUPPORTED, "HNSW: the visited set of a search overflowed; results would lose recall, so the call fails");
}

static HnswGraph graph_of(const vdb_hnsw* h) {
    HnswGraph g{};
    g.links0 = h->d_links0;
    g.len0 = h->d_len0;
    g.ulinks = h->d_ulinks;
    g.ulen = h->d_ulen;
    g.uoff = h->d_uoff;
    g.M = h->M;
    g.M0 = h->M0;
    return g;
}

void hnsw_destroy(vdb_hnsw* h) {
    if (!h) return;
    cudaFree(h->d_links0);
    cudaFree(h->d_len0);
    cudaFree(h->d_ulinks);
    cudaFree(h->d_ulen);
    cudaFree(h->d_uoff);
    cudaFree(h->d_level);
    cudaFree(h->d_cache);
    cudaFree(h->d_overflow);
    delete h;
}

// allocation + level tables shared by build and load
static void hnsw_alloc(vdb_hnsw* h, const vdb_dataset* ds, uint32_t M, uint32_t ef_construction, const uint32_t* h_levels,
                       cudaStream_t st) {
    VDB_REQUIRE(M >= 2 && M <= HN_MAX_M0 / 2, "HNSW: M must be in [2, %u]", HN_MAX_M0 / 2);
    VDB_REQUIRE(ds->n < (1ull << 31), "HNSW: at most 2^31 rows");
    VDB_REQUIRE(((uintptr_t)ds->d_rows & 15) == 0 && ds->pitch % 4 == 0, "HNSW: rows must be 16-byte aligned");
    const uint64_t n = ds->n;
    h->device = ds->device;
    h->n = n;
    h->dim = ds->dim;
    h->dtype = ds->dtype;
    h->metric = ds->metric;
    h->M = M;
    h->M0 = 2 * M;
    h->ef_construction = std::max(ef_construction, 2 * M);  // :504
    h->h_level.assign(h_levels, h_levels + n);
    std::vector<uint64_t> uoff(n + 1, 0);
    for (uint64_t i = 0; i < n; ++i) {
        VDB_REQUIRE(h_levels[i] < 64, "HNSW: level %u of row %llu is out of range", h_levels[i], (unsigned long long)i);
        uoff[i + 1] = uoff[i] + h_levels[i];
    }
    h->slots = uoff[n];
    const uint64_t slots = std::max<uint64_t>(uoff[n], 1);
    VDB_CUDA(cudaMalloc(&h->d_links0, std::max<uint64_t>(n, 1) * h->M0 * 4));
    VDB_CUDA(cudaMalloc(&h->d_len0, std::max<uint64_t>(n, 1) * 4));
    VDB_CUDA(cudaMalloc(&h->d_ulinks, slots * M * 4));
    VDB_CUDA(cudaMalloc(&h->d_ulen, slots * 4));
    VDB_CUDA(cudaMalloc(&h->d_uoff, (n + 1) * 8));
    VDB_CUDA(cudaMalloc(&h->d_level, std::max<uint64_t>(n, 1) * 4));
    VDB_CUDA(cudaMalloc(&h->d_cache, std::max<uint64_t>(n, 1) * 4));
    VDB_CUDA(cudaMalloc(&h->d_overflow, 16));   // [0] overflow count, [2..3] u64 evaluation count
    VDB_CUDA(cudaMemsetAsync(h->d_overflow, 0, 16, st));
    VDB_CUDA(cudaMemsetAsync(h->d_links0, 0, std::max<uint64_t>(n, 1) * h->M0 * 4, st));
    VDB_CUDA(cudaMemsetAsync(h->d_ulinks, 0, slots * M * 4, st));
    VDB_CUDA(cudaMemsetAsync(h->d_len0, 0, std::max<uint64_t>(n, 1) * 4, st));
    VDB_CUDA(cudaMemsetAsync(h->d_ulen, 0, slots * 4, st));
    VDB_CUDA(cudaMemcpyAsync(h->d_uoff, uoff.data(), (n + 1) * 8, cudaMemcpyHostToDevice, st));
    if (n) {
        VDB_CUDA(cudaMemcpyAsync(h->d_level, h_levels, n * 4, cudaMemcpyHostToDevice, st));
        row_cache(ds, h->d_cache, st);  // push_init :251-254 / init_dist_cache_after_load :371-379
    }
    VDB_CUDA(cudaStreamSynchronize(st));
}

// an index built elsewhere (e.g. a bincode file of the reference, formats.py): links in the reference's layout —
// links0 [n][2M] + len0 [n]; upper levels concatenated per node ([level_i][M] links, [level_i] lengths)
vdb_hnsw* hnsw_from_graph(const vdb_dataset* ds, uint32_t M, uint32_t ef_construction, const uint32_t* h_levels,
                          const uint32_t* links0, const uint32_t* len0, const uint32_t* ulinks, const uint32_t* ulen,
                          int64_t enter_point, int32_t enter_level) {
    auto h = new vdb_hnsw();
    cudaStream_t st = nullptr;
    try {
        VDB_CUDA(cudaSetDevice(ds->device));
        VDB_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
        hnsw_alloc(h, ds, M, ef_construction, h_levels, st);
        const uint64_t n = ds->n;
        if (n) {
            VDB_REQUIRE(enter_point >= 0 && (uint64_t)enter_point < n && enter_level >= 0 &&
                            (uint32_t)enter_level == h_levels[enter_point],
                        "HNSW: enter point %lld / level %d do not match the level table", (long long)enter_point, enter_level);
            for (uint64_t i = 0; i < n; ++i) {
                VDB_REQUIRE(len0[i] <= h->M0, "HNSW: links_len[%llu][0] exceeds 2M", (unsigned long long)i);
                for (uint32_t j = 0; j < len0[i]; ++j)
                    VDB_REQUIRE(links0[i * h->M0 + j] < n, "HNSW: link of row %llu out of range", (unsigned long long)i);
            }
            for (uint64_t s = 0; s < h->slots; ++s) {
                VDB_REQUIRE(ulen[s] <= M, "HNSW: an upper-level list exceeds M");
                for (uint32_t j = 0; j < ulen[s]; ++j) VDB_REQUIRE(ulinks[s * M + j] < n, "HNSW: upper link out of range");
            }
            VDB_CUDA(cudaMemcpyAsync(h->d_links0, links0, n * h->M0 * 4, cudaMemcpyHostToDevice, st));
            VDB_CUDA(cudaMemcpyAsync(h->d_len0, len0, n * 4, cudaMemcpyHostToDevice, st));
            if (h->slots) {
                VDB_CUDA(cudaMemcpyAsync(h->d_ulinks, ulinks, h->slots * M * 4, cudaMemcpyHostToDevice, st));
                VDB_CUDA(cudaMemcpyAsync(h->d_ulen, ulen, h->slots * 4, cudaMemcpyHostToDevice, st));
            }
            h->enter_point = enter_point;
            h->enter_level = enter_level;
        }
        VDB_CUDA(cudaStreamSynchronize(st));
        cudaStreamDestroy(st);
    } catch (...) {
        if (st) cudaStreamDestroy(st);
        hnsw_destroy(h);
        throw;
    }
    return h;
}

// inserts rows [first, n) of `ds` into the graph, batch by batch (inner_batch_add :459-476 / add_parallel :399-457)
static void hnsw_insert_range(vdb_hnsw* h, const vdb_dataset* ds, uint64_t first, uint32_t max_batch, cudaStream_t st) {
    const uint64_t n = ds->n;
    const uint32_t M = h->M;
    const uint32_t* h_levels = h->h_level.data();
    if (n == 0) return;
    {
        uint64_t done = first;
        if (done == 0) {  // the first vector becomes the enter point (:543-551)
            h->enter_point = 0;
            h->enter_level = (int)h_levels[0];
            done = 1;
        }
        const uint32_t ef = h->ef_construction;
        const uint32_t dimpad = round_up(ds->pitch, 4u);
        const bool l2 = ds->metric == VDB_L2SQR;
        std::vector<uint32_t> task_node, task_lvl, h_sel, h_selcnt, grp_node, grp_lvl, grp_off, inc;
        std::vector<uint64_t> out_off;
        std::vector<std::pair<uint64_t, uint32_t>> back;
        while (done < n) {
            // batch size: the reference's min(threads * 4, n / M) with the thread term replaced by the grid capacity
            uint32_t b = (uint32_t)std::min<uint64_t>(std::max<uint64_t>(1, done / M), max_batch);
            b = (uint32_t)std::min<uint64_t>(b, n - done);
            const uint32_t base = (uint32_t)done;
            out_off.assign(b + 1, 0);
            task_node.clear();
            task_lvl.clear();
            for (uint32_t i = 0; i < b; ++i) {
                const uint32_t top = std::min<uint32_t>(h_levels[base + i], (uint32_t)h->enter_level);
                out_off[i + 1] = out_off[i] + top + 1;
                for (uint32_t l = 0; l <= top; ++l) {
                    task_node.push_back(base + i);
                    task_lvl.push_back(l);
                }
            }
            const uint32_t ntasks = (uint32_t)task_node.size();
            DevBuf d_out_off((size_t)(b + 1) * 8, st), d_cand((size_t)ntasks * ef * 8, st), d_tnode((size_t)ntasks * 4, st),
                d_tlvl((size_t)ntasks * 4, st), d_sel((size_t)ntasks * M * 4, st), d_selcnt((size_t)ntasks * 4, st);
            VDB_CUDA(cudaMemcpyAsync(d_out_off.p, out_off.data(), (size_t)(b + 1) * 8, cudaMemcpyHostToDevice, st));
            VDB_CUDA(cudaMemcpyAsync(d_tnode.p, task_node.data(), (size_t)ntasks * 4, cudaMemcpyHostToDevice, st));
            VDB_CUDA(cudaMemcpyAsync(d_tlvl.p, task_lvl.data(), (size_t)ntasks * 4, cudaMemcpyHostToDevice, st));
            // 1. candidates of every new node on every level it joins (read-only on the graph)
            HnswSearchParams sp{};
            sp.g = graph_of(h);
            sp.rows = ds->d_rows;
            sp.pitch = ds->pitch;
            sp.dim = ds->dim;
            sp.dimpad = dimpad;
            sp.rcache = h->d_cache;
            sp.qrow_base = base;
            sp.level = h->d_level;
            sp.nq = b;
            sp.ef = ef;
            sp.hash_mask = hash_cap_for(ef, h->M0) - 1;
            sp.enter_point = (uint32_t)h->enter_point;
            sp.enter_level = (uint32_t)h->enter_level;
            sp.build = 1;
            sp.out_off = d_out_off.as<uint64_t>();
            sp.out_keys = d_cand.as<uint64_t>();
            launch_search(ds, sp, h->d_overflow, st);
            // 2. connect_new_links: heuristic(M) -> links of the new nodes
            HnswSelectParams sl{};
            sl.g = graph_of(h);
            sl.rows = ds->d_rows;
            sl.pitch = ds->pitch;
            sl.dim = ds->dim;
            sl.dimpad = dimpad;
            sl.rcache = h->d_cache;
            sl.cand = d_cand.as<uint64_t>();
            sl.ef = ef;
            sl.ntasks = ntasks;
            sl.task_node = d_tnode.as<uint32_t>();
            sl.task_lvl = d_tlvl.as<uint32_t>();
            sl.sel = d_sel.as<uint32_t>();
            sl.selcnt = d_selcnt.as<uint32_t>();
            auto select = [&] {
                ProfScope prof("hnsw_select", st);
                const size_t smem = (size_t)HN_WARPS * dimpad * 4;  // one staging row per warp
                if (ds->dtype == VDB_F32) {
                    if (l2) launch_dyn(hnsw_select_kernel<float, VDB_L2SQR>, ntasks, smem, sl, st);
                    else launch_dyn(hnsw_select_kernel<float, VDB_COSINE>, ntasks, smem, sl, st);
                } else {
                    if (l2) launch_dyn(hnsw_select_kernel<uint8_t, VDB_L2SQR>, ntasks, smem, sl, st);
                    else launch_dyn(hnsw_select_kernel<uint8_t, VDB_COSINE>, ntasks, smem, sl, st);
                }
            };
            select();
            // 3. arrange_links: group the back-links by (level, target), targets keep the batch order of their sources
            h_sel.resize((size_t)ntasks * M);
            h_selcnt.resize(ntasks);
            uint32_t overflowed = 0;
            VDB_CUDA(cudaMemcpyAsync(&overflowed, h->d_overflow, 4, cudaMemcpyDeviceToHost, st));
            VDB_CUDA(cudaMemcpyAsync(h_sel.data(), d_sel.p, (size_t)ntasks * M * 4, cudaMemcpyDeviceToHost, st));
            VDB_CUDA(cudaMemcpyAsync(h_selcnt.data(), d_selcnt.p, (size_t)ntasks * 4, cudaMemcpyDeviceToHost, st));
            VDB_CUDA(cudaStreamSynchronize(st));
            if (overflowed) {
                // a visited set of this batch filled up: search again with sets that cannot, and select again. The graph
                // the search reads is unchanged: the select only wrote the lists of the batch's own nodes, which no
                // older node links to yet
                VDB_CUDA(cudaMemsetAsync(h->d_overflow, 0, 4, st));
                sp.hash_mask = never_full_slots(n) - 1;
                launch_search(ds, sp, h->d_overflow, st);
                select();
                VDB_CUDA(cudaMemcpyAsync(h_sel.data(), d_sel.p, (size_t)ntasks * M * 4, cudaMemcpyDeviceToHost, st));
                VDB_CUDA(cudaMemcpyAsync(h_selcnt.data(), d_selcnt.p, (size_t)ntasks * 4, cudaMemcpyDeviceToHost, st));
                hnsw_check_overflow(h, st);
            }
            // (level << 32 | target, source): a stable sort by key keeps the sources of a target in batch order
            back.clear();
            for (uint32_t t = 0; t < ntasks; ++t)
                for (uint32_t j = 0; j < h_selcnt[t]; ++j)
                    back.emplace_back(((uint64_t)task_lvl[t] << 32) | h_sel[(size_t)t * M + j], task_node[t]);
            std::stable_sort(back.begin(), back.end(),
                             [](const std::pair<uint64_t, uint32_t>& a, const std::pair<uint64_t, uint32_t>& b) { return a.first < b.first; });
            if (!back.empty()) {
                grp_node.clear();
                grp_lvl.clear();
                grp_off.clear();
                inc.clear();
                for (size_t e = 0; e < back.size(); ++e) {
                    if (e == 0 || back[e].first != back[e - 1].first) {
                        grp_node.push_back((uint32_t)back[e].first);
                        grp_lvl.push_back((uint32_t)(back[e].first >> 32));
                        grp_off.push_back((uint32_t)e);
                    }
                    inc.push_back(back[e].second);
                }
                grp_off.push_back((uint32_t)back.size());
                const uint32_t ng = (uint32_t)grp_node.size();
                DevBuf d_gn((size_t)ng * 4, st), d_gl((size_t)ng * 4, st), d_go((size_t)(ng + 1) * 4, st), d_inc(inc.size() * 4, st);
                VDB_CUDA(cudaMemcpyAsync(d_gn.p, grp_node.data(), (size_t)ng * 4, cudaMemcpyHostToDevice, st));
                VDB_CUDA(cudaMemcpyAsync(d_gl.p, grp_lvl.data(), (size_t)ng * 4, cudaMemcpyHostToDevice, st));
                VDB_CUDA(cudaMemcpyAsync(d_go.p, grp_off.data(), (size_t)(ng + 1) * 4, cudaMemcpyHostToDevice, st));
                VDB_CUDA(cudaMemcpyAsync(d_inc.p, inc.data(), inc.size() * 4, cudaMemcpyHostToDevice, st));
                HnswArrangeParams ap{};
                ap.g = graph_of(h);
                ap.rows = ds->d_rows;
                ap.pitch = ds->pitch;
                ap.dim = ds->dim;
                ap.dimpad = dimpad;
                ap.rcache = h->d_cache;
                ap.ngroups = ng;
                ap.grp_node = d_gn.as<uint32_t>();
                ap.grp_lvl = d_gl.as<uint32_t>();
                ap.grp_off = d_go.as<uint32_t>();
                ap.inc = d_inc.as<uint32_t>();
                ProfScope prof("hnsw_arrange", st);
                const size_t smem = (size_t)(1 + HN_WARPS) * dimpad * 4;
                if (ds->dtype == VDB_F32) {
                    if (l2) launch_dyn(hnsw_arrange_kernel<float, VDB_L2SQR>, ng, smem, ap, st);
                    else launch_dyn(hnsw_arrange_kernel<float, VDB_COSINE>, ng, smem, ap, st);
                } else {
                    if (l2) launch_dyn(hnsw_arrange_kernel<uint8_t, VDB_L2SQR>, ng, smem, ap, st);
                    else launch_dyn(hnsw_arrange_kernel<uint8_t, VDB_COSINE>, ng, smem, ap, st);
                }
                VDB_CUDA(cudaStreamSynchronize(st));
            }
            // 4. the enter point moves to the first new node that is higher than every older one (:447-454)
            for (uint32_t i = 0; i < b; ++i)
                if ((int)h_levels[base + i] > h->enter_level) {
                    h->enter_level = (int)h_levels[base + i];
                    h->enter_point = base + i;
                }
            done += b;
        }
        VDB_CUDA(cudaStreamSynchronize(st));
    }
}

// HNSWIndex::build_on_vec_set (:585-600) over the rows of `ds` in row order. `h_levels[i]` is rand_level (:145-149)
// of row i, drawn by the caller's RNG in row order like the reference does.
vdb_hnsw* hnsw_build(const vdb_dataset* ds, uint32_t M, uint32_t ef_construction, const uint32_t* h_levels, uint32_t max_batch) {
    auto h = new vdb_hnsw();
    cudaStream_t st = nullptr;
    try {
        VDB_CUDA(cudaSetDevice(ds->device));
        VDB_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
        hnsw_alloc(h, ds, M, ef_construction, h_levels, st);
        hnsw_insert_range(h, ds, 0, max_batch, st);
        cudaStreamDestroy(st);
    } catch (...) {
        if (st) cudaStreamDestroy(st);
        hnsw_destroy(h);
        throw;
    }
    return h;
}

// IndexBuilder::batch_add on an existing index (:573-575; DynamicIndex::HNSW add, dynamic_index.rs:44-55): the rows
// appended to `ds` since the index was built (rows [h->n, ds->n)) are inserted with the levels given for them.
void hnsw_append(vdb_hnsw* h, const vdb_dataset* ds, const uint32_t* new_levels, uint32_t max_batch) {
    VDB_REQUIRE(ds->n >= h->n && ds->dim == h->dim && ds->dtype == h->dtype && ds->metric == h->metric,
                "HNSW index was built for a different vector set");
    if (ds->n == h->n) return;
    cudaStream_t st = nullptr;
    VDB_CUDA(cudaSetDevice(ds->device));
    VDB_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    // The grown graph is assembled in a TEMPORARY handle and swapped into *h only once every allocation and copy has
    // succeeded: on failure (growing a large graph while the old one is resident makes out-of-memory plausible) the
    // caller's handle still describes the old, intact graph and nothing leaks.
    auto free_arrays = [](vdb_hnsw& g) {
        cudaFree(g.d_links0);
        cudaFree(g.d_len0);
        cudaFree(g.d_ulinks);
        cudaFree(g.d_ulen);
        cudaFree(g.d_uoff);
        cudaFree(g.d_level);
        cudaFree(g.d_cache);
        cudaFree(g.d_overflow);
        g.d_links0 = g.d_len0 = g.d_ulinks = g.d_ulen = g.d_level = g.d_overflow = nullptr;
        g.d_uoff = nullptr;
        g.d_cache = nullptr;
    };
    vdb_hnsw grown = *h;   // scalars (enter point, M, ...) carried over; the array pointers are replaced by hnsw_alloc
    grown.d_links0 = grown.d_len0 = grown.d_ulinks = grown.d_ulen = grown.d_level = grown.d_overflow = nullptr;
    grown.d_uoff = nullptr;
    grown.d_cache = nullptr;
    try {
        const uint64_t n0 = h->n, n = ds->n;
        std::vector<uint32_t> levels = h->h_level;
        levels.insert(levels.end(), new_levels, new_levels + (n - n0));
        const uint64_t old_slots = h->slots;
        hnsw_alloc(&grown, ds, h->M, h->ef_construction, levels.data(), st);
        // nodes keep their ids and the upper-level slots of old nodes keep their positions (prefix sums only grow)
        if (n0) {
            VDB_CUDA(cudaMemcpyAsync(grown.d_links0, h->d_links0, n0 * h->M0 * 4, cudaMemcpyDeviceToDevice, st));
            VDB_CUDA(cudaMemcpyAsync(grown.d_len0, h->d_len0, n0 * 4, cudaMemcpyDeviceToDevice, st));
            if (old_slots) {
                VDB_CUDA(cudaMemcpyAsync(grown.d_ulinks, h->d_ulinks, old_slots * h->M * 4, cudaMemcpyDeviceToDevice, st));
                VDB_CUDA(cudaMemcpyAsync(grown.d_ulen, h->d_ulen, old_slots * 4, cudaMemcpyDeviceToDevice, st));
            }
        }
        VDB_CUDA(cudaStreamSynchronize(st));
        hnsw_insert_range(&grown, ds, n0, max_batch, st);
        VDB_CUDA(cudaStreamSynchronize(st));
    } catch (...) {
        cudaStreamSynchronize(st);
        free_arrays(grown);
        cudaStreamDestroy(st);
        throw;
    }
    vdb_hnsw old = *h;
    *h = grown;            // commit
    free_arrays(old);
    cudaStreamDestroy(st);
}

// the k best by (cached-form distance, id) of the first `take` entries of every [ef] candidate list
static void exact_topk_of(const vdb_dataset* ds, const vdb_hnsw* h, const void* d_queries, const float* d_qcache,
                          const uint64_t* d_cand, uint32_t nq, uint32_t ef, uint32_t k, uint64_t* d_keys, cudaStream_t st,
                          uint32_t take = 0) {
    if (take == 0) take = ef;
    const uint64_t cnt = (uint64_t)nq * take;
    DevBuf qidx(cnt * 4, st), rid(cnt * 4, st), valid(cnt, st), dist(cnt * 4, st), keys2(cnt * 8, st);
    iota_pairs_kernel<<<(uint32_t)ceil_div<uint64_t>(cnt, 256), 256, 0, st>>>(d_cand, nq, ef, take, qidx.as<uint32_t>(),
                                                                            rid.as<uint32_t>(), valid.as<uint8_t>());
    VDB_LAUNCHED();
    cached_pair_distances(ds, d_queries, d_qcache, h->d_cache, qidx.as<uint32_t>(), rid.as<uint32_t>(), cnt, dist.as<float>(), st);
    rekey_based(dist.as<float>(), rid.as<uint32_t>(), (uint32_t)ds->id_base, valid.as<uint8_t>(), cnt, keys2.as<uint64_t>(), st);
    launch_merge_keys(keys2.as<uint64_t>(), 1, nq, take, false, k, d_keys, nullptr, nullptr, nullptr, st);
}

// knn_with_ef (:616-625) for a batch: [nq][k] keys ascending by (distance, id); distances are the cached form,
// re-evaluated by the pair kernel that also serves vdb_gather_dist
void hnsw_knn_keys(const vdb_dataset* ds, const vdb_hnsw* h, const void* d_queries, uint32_t nq, uint32_t k, uint32_t ef_in,
                   uint64_t* d_keys, cudaStream_t st, bool never_full) {
    // an index of a row-sharded set has no arrays of its own (its replicas do)
    VDB_REQUIRE(!h->rep && ds->n == h->n && ds->dim == h->dim && ds->dtype == h->dtype && ds->metric == h->metric,
                "HNSW index was built for a different vector set");
    if (nq == 0 || k == 0) return;
    if (h->n == 0) {
        VDB_CUDA(cudaMemsetAsync(d_keys, 0xff, (size_t)nq * k * 8, st));
        return;
    }
    const uint32_t ef = std::max(ef_in, k);  // :620
    VDB_REQUIRE(ef <= 4096, "HNSW search: ef=%u is too large (max 4096)", ef);
    DevBuf qcache((size_t)nq * 4, st), cand((size_t)nq * ef * 8, st);
    {
        vdb_dataset qd = *ds;
        qd.d_rows = const_cast<void*>(d_queries);
        qd.n = nq;
        qd.pitch = ds->dim;
        row_cache(&qd, qcache.as<float>(), st);
    }
    HnswSearchParams sp{};
    sp.g = graph_of(h);
    sp.rows = ds->d_rows;
    sp.pitch = ds->pitch;
    sp.dim = ds->dim;
    sp.dimpad = round_up(ds->pitch, 4u);
    sp.rcache = h->d_cache;
    sp.queries = d_queries;
    sp.qcache = qcache.as<float>();
    sp.nq = nq;
    sp.ef = ef;
    sp.hash_mask = (never_full ? never_full_slots(h->n) : hash_cap_for(ef, h->M0)) - 1;
    sp.enter_point = (uint32_t)h->enter_point;
    sp.enter_level = (uint32_t)h->enter_level;
    sp.build = 0;
    sp.out_keys = cand.as<uint64_t>();
    launch_search(ds, sp, h->d_overflow, st);
    // into_sorted_vec_limit(k): the k best of the ef results
    exact_topk_of(ds, h, d_queries, qcache.as<float>(), cand.as<uint64_t>(), nq, ef, k, d_keys, st, k);
}

// HNSWIndex::knn_pq (:672-697): the graph is walked with ADC distances, then ALL max(ef, k) results are re-scored
// with the exact cached form and the k best by (distance, id) returned (ResultSet::pq_resort, candidate_pair.rs:102-108)
void hnsw_knn_pq_keys(const vdb_dataset* ds, const vdb_hnsw* h, const vdb_pq* pq, const void* d_queries, uint32_t nq, uint32_t k,
                      uint32_t ef_in, uint64_t* d_keys, cudaStream_t st, bool never_full) {
    VDB_REQUIRE(!h->rep && ds->n == h->n && ds->dim == h->dim && ds->dtype == h->dtype && ds->metric == h->metric,
                "HNSW index was built for a different vector set");
    VDB_REQUIRE(pq->metric == ds->metric, "Distance algorithm mismatch.");
    VDB_REQUIRE(pq->shards.empty() && pq->n == ds->n && pq->dim == ds->dim, "PQ table was built for a different vector set");
    VDB_REQUIRE(pq->n_bits == 4, "HNSW + PQ search supports 4-bit codes");
    if (nq == 0 || k == 0) return;
    if (h->n == 0) {
        VDB_CUDA(cudaMemsetAsync(d_keys, 0xff, (size_t)nq * k * 8, st));
        return;
    }
    const uint32_t ef = std::max(ef_in, k);
    VDB_REQUIRE(ef <= 4096, "HNSW search: ef=%u is too large (max 4096)", ef);
    const uint32_t tab = pq->m * 16;
    DevBuf lut((size_t)nq * tab * 4, st), qn((size_t)nq * 4, st), qcache((size_t)nq * 4, st), cand((size_t)nq * ef * 8, st);
    pq_lut(pq, d_queries, nq, lut.as<float>(), qn.as<float>(), st);
    {
        vdb_dataset qd = *ds;
        qd.d_rows = const_cast<void*>(d_queries);
        qd.n = nq;
        qd.pitch = ds->dim;
        row_cache(&qd, qcache.as<float>(), st);
    }
    HnswSearchParams sp{};
    sp.g = graph_of(h);
    sp.dim = ds->dim;
    sp.rcache = h->d_cache;
    sp.qcache = qn.as<float>();  // cosine: ||q|| of the lookup table (pq_table.rs:215-221)
    sp.nq = nq;
    sp.ef = ef;
    sp.hash_mask = (never_full ? never_full_slots(h->n) : hash_cap_for(ef, h->M0)) - 1;
    sp.enter_point = (uint32_t)h->enter_point;
    sp.enter_level = (uint32_t)h->enter_level;
    sp.build = 0;
    sp.out_keys = cand.as<uint64_t>();
    sp.codes = pq->d_codes;
    sp.enc = pq->enc;
    sp.m = pq->m;
    sp.lut = lut.as<float>();
    sp.dcache = pq->d_dist_cache;
    launch_search(ds, sp, h->d_overflow, st);
    exact_topk_of(ds, h, d_queries, qcache.as<float>(), cand.as<uint64_t>(), nq, ef, k, d_keys, st);
}

}  // namespace vdb
