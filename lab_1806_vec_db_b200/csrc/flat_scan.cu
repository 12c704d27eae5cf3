// flat_scan.cu — K1: exact Flat kNN as one streaming pass over the row shard.
//
// Replaces FlatIndex::knn (reference src/index_algorithm/flat_index.rs:48-57): for every row the
// difference-form L2 sum((q-x)^2) (src/distance/mod.rs:75-77) or the 3-dot cosine
// (src/distance/mod.rs:60-69), then the k smallest by (distance, id)
// (src/index_algorithm/candidate_pair.rs:36-40, 61-74).
//
// HBM-bound design: each warp streams R consecutive rows with 128-bit L1-bypassing loads
// (double-buffered in registers), up to NQ=8 queries are resident in shared memory and share every
// row byte, partial sums are reduced with a V-1 shuffle reduce-scatter, and candidates that beat the
// CTA's current k-th best go to a shared-memory buffer that is bitonic-sorted only when it fills.
// Algorithmic bytes per pass: n * pitch * sizeof(T) (+ the query tile and G*k keys).
#include <cstdlib>

#include "dataset.cuh"
#include "scanmath.cuh"
#include "topk.cuh"

namespace vdb {

std::atomic<uint64_t> g_launches{0};
std::atomic<int> g_flat_path{0};

constexpr int SCAN_THREADS = 256;
constexpr int SCAN_WARPS = SCAN_THREADS / 32;

struct ScanParams {
    const uint8_t* rows;
    uint64_t n;
    uint64_t pitch_bytes;
    uint32_t nvec, nit;
    const float* q;        // query tile (see prepare_queries), first query of this pass
    const uint8_t* raw_q;  // u8 rows, L2Sqr, one launch: the caller's query bytes (dim per query); the CTA pads them itself
    uint32_t raw_dim;
    uint32_t qstride;      // floats per query
    const float* qcache;   // per query ||q|| (cosine)
    uint32_t nq_valid;
    uint32_t K, P, limit, sync_every;
    uint32_t id_base;
    uint32_t iters;        // row-group iterations per warp
    uint64_t* partial;     // [NQ][gridDim.x][K]
    // fused tail (single-launch batches): the last CTA to finish merges the partial lists of every query
    uint32_t* done;        // nullptr: off. Arrival counter, zero at launch (cleared by the query-tile kernel)
    uint64_t* out_keys;    // [NQ][K]
    uint64_t* out_ids;     // optional decoded results
    float* out_dist;
    uint32_t* out_counts;
    uint64_t* emit;        // emit instantiation only: [nq_valid][n] the key of every (query, row), see flat_large_k_keys
};

// Tail of a single-launch batch, run by the last CTA to finish: merge of the gridDim.x per-CTA lists of every query + decode.
// Kept out of line: inlined into the scan kernel it perturbed the register allocation of the main loop (the 4-query f32
// variant, 128 registers with three load buffers, went from 0.75 to 0.85 ms per pass).
struct ScanTailArgs {   // by value: a reference to the kernel's parameter block would force a copy of it onto the stack
    const uint64_t* partial;
    uint32_t nq_valid, K, P, limit;
    uint64_t* out_keys;
    uint64_t* out_ids;
    float* out_dist;
    uint32_t* out_counts;
};
static __device__ __noinline__ void scan_tail(const ScanTailArgs p, TopkSmem topk, uint32_t* s_valid) {
    __threadfence();
    topk.init();
    // Every per-CTA list is ascending, so the smallest of their K-th keys bounds the K-th key of the union: only keys up
    // to it are pushed (a few more than K instead of gridDim.x * K), and the keys of a batch are loaded before any of them
    // is tested - the L2 round trips of the tail overlap instead of lining up one per round.
    __shared__ unsigned long long s_bound[8];
    if (threadIdx.x < 8) s_bound[threadIdx.x] = KEY_NONE;
    __syncthreads();
    const uint32_t total = gridDim.x * p.K;
    for (uint32_t qi = 0; qi < p.nq_valid; ++qi) {
        unsigned long long b = KEY_NONE;
        for (uint32_t l = threadIdx.x; l < gridDim.x; l += blockDim.x)
            b = min(b, (unsigned long long)__ldcg(p.partial + (size_t)qi * total + (size_t)l * p.K + (p.K - 1)));   // other SMs wrote it: bypass L1
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) b = min(b, __shfl_xor_sync(0xffffffffu, b, d));
        if ((threadIdx.x & 31) == 0 && b != KEY_NONE) atomicMin(&s_bound[qi], b);   // 64-bit shared atomics are CAS loops: one per warp
    }
    __syncthreads();
    // at most `period` appends per segment between two flush tests (the contract of TopkSmem::push)
    const uint32_t period = min((uint32_t)blockDim.x, p.P - p.K - p.limit);
    constexpr int TAIL_U = 8;
    for (uint32_t base = 0; base < total; base += TAIL_U * period) {
        for (uint32_t qi = 0; qi < p.nq_valid; ++qi) {
            const uint64_t bound = s_bound[qi];
            uint64_t kk[TAIL_U];
#pragma unroll
            for (int u = 0; u < TAIL_U; ++u) {
                const uint32_t i = base + u * period + threadIdx.x;
                kk[u] = (threadIdx.x < period && i < total) ? __ldcg(p.partial + (size_t)qi * total + i) : KEY_NONE;
            }
#pragma unroll
            for (int u = 0; u < TAIL_U; ++u) {
                if (base + u * period >= total) break;   // CTA-uniform
                bool want = false;
                if (kk[u] <= bound && kk[u] < topk.tau(qi)) want = topk.push(qi, kk[u]);
                topk.maybe_flush(want);
            }
        }
    }
    topk.final_flush();
    for (uint32_t i = threadIdx.x; i < p.nq_valid * p.K; i += blockDim.x) {
        const uint32_t qi = i / p.K;
        const uint64_t key = topk.seg(qi)[i - qi * p.K];
        const bool ok = key != KEY_NONE;
        p.out_keys[i] = key;
        if (p.out_ids) {
            p.out_ids[i] = ok ? (uint64_t)key_id(key) : KEY_NONE;
            p.out_dist[i] = ok ? key_dist(key) : __uint_as_float(0x7fc00000u);
        }
        if (ok) atomicAdd(&s_valid[qi], 1u);
    }
    __syncthreads();
    if (p.out_counts && threadIdx.x < p.nq_valid) p.out_counts[threadIdx.x] = s_valid[threadIdx.x];
}

// PL = 1: f32 rows (4 elements per 16-byte load); PL = 4: u8 rows (16 elements per load).
// EMIT: the large-k path's instantiation - every key goes to p.emit instead of the shared-memory top-k (a compile-time
// switch: the distance code is the same, and the top-k instantiations keep their register allocation).
template <int NQ, int R, int METRIC, int PL, bool EMIT = false>
__global__ void __launch_bounds__(SCAN_THREADS, 2) flat_scan_kernel(const ScanParams p) {
    extern __shared__ __align__(16) uint8_t smem[];
    constexpr int V = NQ * R;
    constexpr int SH = 5 - Log2<V>::value;
    constexpr int SHR = 5 - Log2<R>::value;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t qs4 = p.qstride >> 2;  // float4 per query
    // query tile in shared memory: f32 rows -> f32 values, u8 rows -> the queries' bytes (16 per lane and step), see
    // prepare_queries; either way qs4 16-byte units per query
    float4* qs = reinterpret_cast<float4*>(smem);
    const ulonglong2* qs2 = reinterpret_cast<const ulonglong2*>(smem);
    uint64_t* tk = reinterpret_cast<uint64_t*>(smem + (size_t)NQ * p.qstride * 4);
    TopkSmem topk{tk, reinterpret_cast<uint32_t*>(tk + (size_t)NQ * p.P), p.K, p.P, NQ, p.limit};

    if (PL == 4 && p.raw_q) {
        // no tile kernel in front of this launch: the tile is the queries' bytes, zero padded to qstride * 4 per query
        const uint32_t qbytes = p.qstride * 4;
        for (uint32_t i = threadIdx.x; i < NQ * qbytes; i += blockDim.x) {
            const uint32_t qi = i / qbytes, off = i - qi * qbytes;
            smem[i] = (qi < p.nq_valid && off < p.raw_dim) ? p.raw_q[(size_t)qi * p.raw_dim + off] : (uint8_t)0;
        }
    } else {
        for (uint32_t i = threadIdx.x; i < NQ * qs4; i += blockDim.x)
            qs[i] = (i / qs4 < p.nq_valid) ? reinterpret_cast<const float4*>(p.q)[i] : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    if constexpr (EMIT) __syncthreads();
    else topk.init();

    const int pidx = lane >> SH;
    const int my_r = pidx / NQ, my_q = pidx % NQ;
    const bool emitter = (lane & ((1 << SH) - 1)) == 0 && my_q < (int)p.nq_valid;
    float qn = 0.f;
    if (METRIC == VDB_COSINE && my_q < (int)p.nq_valid) qn = p.qcache[my_q];

    const uint64_t total_warps = (uint64_t)gridDim.x * SCAN_WARPS;
    const uint64_t last_row = p.n - 1;

    // The (row group, 512-byte chunk) steps of a warp form one flat sequence; step t is computed from register buffer
    // t & 1 while the loads of step t + 1 land in the other buffer, so nothing is copied between buffers and the
    // prefetch runs across group boundaries. Addressing is incremental: one pointer per lane, rows of the group at
    // r * pitch from it; the clamped (last group) and ragged (row end inside the last chunk) cases take a slow path.
    constexpr bool SINGLE = PL == 4 && NQ >= 4;  // one buffer for u8 rows with 4-8 queries (measured with the earlier FP32 u8 arithmetic: 0.98 -> 0.89 ms; f32 rows lose)
    // 4 f32 queries: 32 accumulator registers leave room for a third buffer, i.e. two 512-byte steps in flight per
    // warp (64 KB per SM like the 1- and 2-query variants with their 8-row groups)
    constexpr bool TRIPLE = NQ == 4 && PL == 1;
    uint4 bufA[R], bufB[SINGLE ? 1 : R], bufC[TRIPLE ? R : 1];
    const uint32_t tail_lanes = p.nvec - (p.nit - 1) * 32;  // lanes with data in a row's last chunk (1..32)
    uint64_t pg = (uint64_t)blockIdx.x * SCAN_WARPS + warp;  // group being prefetched
    uint32_t pit = 0;                                        // its chunk iteration
    const uint8_t* pptr = nullptr;
    bool pclamp = false;
    auto issue = [&](uint4 (&dst)[R]) {
        if (pit == 0) {
            const uint64_t row0 = pg * R;
            pclamp = row0 + (R - 1) > last_row;
            pptr = p.rows + (row0 < last_row ? row0 : last_row) * p.pitch_bytes + (size_t)lane * 16;
        }
        if (!pclamp && (pit + 1 < p.nit || tail_lanes == 32)) {
#pragma unroll
            for (int r = 0; r < R; ++r) dst[r] = ldg_stream_u4(pptr + (size_t)r * p.pitch_bytes);
        } else if (!pclamp) {
            // a row's last, ragged chunk (every other step of a 960-byte u8 row): same addressing, lanes past the end
            // of the row load nothing
            const bool in = (uint32_t)lane < tail_lanes;
#pragma unroll
            for (int r = 0; r < R; ++r)
                dst[r] = in ? ldg_stream_u4(pptr + (size_t)r * p.pitch_bytes) : make_uint4(0u, 0u, 0u, 0u);
        } else {
            const bool in = pit + 1 < p.nit || (uint32_t)lane < tail_lanes;
            const uint64_t row0 = pg * R;
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const uint64_t row = row0 + r < last_row ? row0 + r : last_row;
                dst[r] = in ? ldg_stream_u4(p.rows + row * p.pitch_bytes + ((size_t)pit * 32 + lane) * 16)
                            : make_uint4(0u, 0u, 0u, 0u);
            }
        }
        pptr += 512;
        if (++pit == p.nit) {
            pit = 0;
            pg += total_warps;
        }
    };

    // f32 rows: (even, odd) partial sums in packed pairs; u8 rows: exact integer sums (scanmath.cuh)
    constexpr bool U8 = PL == 4;
    f32x2 acc2[U8 ? 1 : V], xx2[U8 ? 1 : R];
    uint32_t acci[U8 ? V : 1], xxi[U8 ? R : 1];
    if constexpr (U8) {
#pragma unroll
        for (int i = 0; i < V; ++i) acci[i] = 0u;
#pragma unroll
        for (int r = 0; r < R; ++r) xxi[r] = 0u;
    } else {
#pragma unroll
        for (int i = 0; i < V; ++i) acc2[i] = 0ull;
#pragma unroll
        for (int r = 0; r < R; ++r) xx2[r] = 0ull;
    }
    uint64_t g = pg;   // group being computed
    uint32_t it = 0, gi = 0;
    const ulonglong2* qp = qs2 + lane;  // this lane's chunk of query 0, plane 0
    bool want = false;

    auto accumulate = [&](const uint4 (&cur)[R]) {
        if constexpr (U8) {
            const uint4* qp4 = reinterpret_cast<const uint4*>(qp);
            if (METRIC == VDB_COSINE) {
#pragma unroll
                for (int r = 0; r < R; ++r) xxi[r] = u8x16_acc<false>(xxi[r], cur[r], cur[r]);
            }
#pragma unroll
            for (int qi = 0; qi < NQ; ++qi) {
                const uint4 q = qp4[(size_t)qi * qs4];
#pragma unroll
                for (int r = 0; r < R; ++r) acci[r * NQ + qi] = u8x16_acc<METRIC == VDB_L2SQR>(acci[r * NQ + qi], cur[r], q);
            }
        } else {
            f32x2 x01[R], x23[R];
#pragma unroll
            for (int r = 0; r < R; ++r) row_pairs(cur[r], x01[r], x23[r]);
            if (METRIC == VDB_COSINE) {
#pragma unroll
                for (int r = 0; r < R; ++r) xx2[r] = chunk_acc<false>(xx2[r], x01[r], x23[r], x01[r], x23[r]);
            }
#pragma unroll
            for (int qi = 0; qi < NQ; ++qi) {
                const ulonglong2 q = qp[(size_t)qi * qs4];
#pragma unroll
                for (int r = 0; r < R; ++r)
                    acc2[r * NQ + qi] = chunk_acc<METRIC == VDB_L2SQR>(acc2[r * NQ + qi], x01[r], x23[r], q.x, q.y);
            }
        }
        qp += 32;
    };
    auto finish = [&]() {
        if (++it < p.nit) return;
        // ---- end of a row group: cross-lane reduction, lane L then holds the total of (row my_r, query my_q) ----
        float tot, xr = 0.f;
        if constexpr (U8) {
            uint32_t ti[V], xi[R];
#pragma unroll
            for (int i = 0; i < V; ++i) {
                ti[i] = acci[i];
                acci[i] = 0u;
            }
#pragma unroll
            for (int r = 0; r < R; ++r) {
                xi[r] = xxi[r];
                xxi[r] = 0u;
            }
            tot = (float)warp_reduce_scatter<V>(ti, lane);   // integer total, converted once
            if (METRIC == VDB_COSINE) {
                const uint32_t xs = warp_reduce_scatter<R>(xi, lane);
                xr = (float)__shfl_sync(0xffffffffu, xs, my_r << SHR);
            }
        } else {
            float acc[V], xx[R];
#pragma unroll
            for (int i = 0; i < V; ++i) {
                acc[i] = sum2(acc2[i]);
                acc2[i] = 0ull;
            }
#pragma unroll
            for (int r = 0; r < R; ++r) {
                xx[r] = sum2(xx2[r]);
                xx2[r] = 0ull;
            }
            tot = warp_reduce_scatter<V>(acc, lane);
            if (METRIC == VDB_COSINE) {
                const float xs = warp_reduce_scatter<R>(xx, lane);
                xr = __shfl_sync(0xffffffffu, xs, my_r << SHR);
            }
        }
        if (METRIC == VDB_COSINE) tot = 1.0f - tot / fmaxf(sqrtf(xr) * qn, 1e-10f);
        const uint64_t row = g * R + my_r;
        if (emitter && row < p.n) {
            const uint64_t key = make_key(tot, p.id_base + (uint32_t)row);
            if constexpr (EMIT) p.emit[(size_t)my_q * p.n + row] = key;
            else if (key < topk.tau(my_q)) want |= topk.push(my_q, key);
        }
        if (!EMIT && (gi + 1) % p.sync_every == 0) {
            topk.maybe_flush(want);
            want = false;
        }
        it = 0;
        ++gi;
        g += total_warps;
        qp = qs2 + lane;
    };

    const uint32_t steps = p.iters * p.nit;  // identical for every warp of the CTA (the flush barriers rely on it)
    if (steps) issue(bufA);
    if constexpr (SINGLE) {
        // FP32-bound variants: one register buffer, reloaded as soon as the step's arithmetic has consumed it; the
        // other warps of the scheduler cover the load latency, and the registers of a second buffer go to the schedule
        for (uint32_t t = 0; t < steps; ++t) {
            accumulate(bufA);
            if (t + 1 < steps) issue(bufA);
            finish();
        }
    } else if constexpr (TRIPLE) {
        if (steps > 1) issue(bufB);
        for (uint32_t t = 0; t < steps; t += 3) {
            if (t + 2 < steps) issue(bufC);
            accumulate(bufA);
            finish();
            if (t + 1 < steps) {
                if (t + 3 < steps) issue(bufA);
                accumulate(bufB);
                finish();
                if (t + 2 < steps) {
                    if (t + 4 < steps) issue(bufB);
                    accumulate(bufC);
                    finish();
                }
            }
        }
    } else {
        for (uint32_t t = 0; t < steps; t += 2) {
            if (t + 1 < steps) issue(bufB);
            accumulate(bufA);
            finish();
            if (t + 1 < steps) {
                if (t + 2 < steps) issue(bufA);
                accumulate(bufB);
                finish();
            }
        }
    }
    if constexpr (EMIT) return;
    topk.final_flush();
    for (uint32_t i = threadIdx.x; i < p.nq_valid * p.K; i += blockDim.x) {
        const uint32_t qi = i / p.K, j = i - qi * p.K;
        p.partial[((size_t)qi * gridDim.x + blockIdx.x) * p.K + j] = topk.seg(qi)[j];
    }
    if (p.done == nullptr) return;
    // ---- fused tail: last CTA done -> merge of the gridDim.x lists per query + decode (no further launches) ----
    __shared__ uint32_t s_last, s_valid[8];
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(p.done, 1u) == gridDim.x - 1 ? 1u : 0u;
    if (threadIdx.x < 8) s_valid[threadIdx.x] = 0;
    __syncthreads();
    if (!s_last) return;
    scan_tail(ScanTailArgs{p.partial, p.nq_valid, p.K, p.P, p.limit, p.out_keys, p.out_ids, p.out_dist, p.out_counts}, topk, s_valid);
}

// ---- merge of key lists ------------------------------------------------------------------------
constexpr int MERGE_THREADS = 256;
constexpr int MERGE_UNROLL = 1;
__global__ void __launch_bounds__(MERGE_THREADS, 8) merge_keys_kernel(
    const uint64_t* __restrict__ keys, uint32_t nlists, uint32_t nq, uint32_t len, int list_major,
    const uint64_t* __restrict__ seg_off, const uint32_t* __restrict__ seg_cnt, uint32_t K, uint32_t P, uint32_t limit,
    uint64_t* __restrict__ out_keys, uint64_t* __restrict__ ids, float* __restrict__ dist, uint32_t* __restrict__ counts,
    const MergeFinish fin) {
    extern __shared__ __align__(16) uint8_t smem[];
    uint64_t* tk = reinterpret_cast<uint64_t*>(smem);
    const uint32_t q = blockIdx.x;
    // seg_off != nullptr: one variable-length list per query, keys[seg_off[q] .. seg_off[q+1]);
    // seg_cnt != nullptr: the first min(seg_cnt[q], len) keys of the fixed-pitch list keys[q * len ..]
    const bool seg = seg_off != nullptr || seg_cnt != nullptr;
    const uint64_t seg_base = seg_off ? seg_off[q] : (seg_cnt ? (uint64_t)q * len : 0);
    const uint64_t total = seg_off ? seg_off[q + 1] - seg_base
                                   : (seg_cnt ? (uint64_t)min(seg_cnt[q], len) : (uint64_t)nlists * len);
    // a short list is sorted once in the smallest power-of-two segment that holds it (no intermediate flush)
    uint32_t Pq = P, lim = limit;
    if (total + K <= P) {
        const uint32_t need = (uint32_t)total + K;
        Pq = need <= 64 ? 64u : (1u << (32 - __clz(need - 1)));
        lim = Pq - K;
    }
    TopkSmem topk{tk, reinterpret_cast<uint32_t*>(tk + P), K, Pq, 1, lim};
    topk.init();
    // one key per thread and round; the next round's key is loaded before this round's CTA-wide flush test so
    // the load latency overlaps the barrier
    const uint64_t rounds = (total + blockDim.x - 1) / blockDim.x;
    auto load_key = [&](uint64_t r) -> uint64_t {
        const uint64_t i = r * blockDim.x + threadIdx.x;
        if (i >= total) return KEY_NONE;
        const uint64_t l = seg ? 0 : i / len, j = seg ? 0 : i - l * len;
        const uint64_t src = seg ? seg_base + i
                                     : (list_major ? ((l * nq + q) * len + j) : (((uint64_t)q * nlists + l) * len + j));
        return keys[src];
    };
    if (total + K <= P) {
        // everything fits next to the K best: four rounds of loads in flight at a time, no flush test, one sort
        for (uint64_t r0 = 0; r0 < rounds; r0 += 4) {
            uint64_t kk[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) kk[u] = r0 + u < rounds ? load_key(r0 + u) : KEY_NONE;
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (kk[u] != KEY_NONE) topk.push(0, kk[u]);
        }
    } else {
        uint64_t next = rounds ? load_key(0) : KEY_NONE;
        for (uint64_t r = 0; r < rounds; ++r) {
            const uint64_t key = next;
            if (r + 1 < rounds) next = load_key(r + 1);
            bool want = false;
            if (key < topk.tau(0)) want = topk.push(0, key);
            topk.maybe_flush(want);
        }
    }
    topk.final_flush();
    uint32_t valid = 0;
    for (uint32_t j = threadIdx.x; j < K; j += blockDim.x) {
        const uint64_t key = topk.seg(0)[j];
        const bool ok = key != KEY_NONE;
        valid += ok;
        if (out_keys) out_keys[(size_t)q * K + j] = key;
        if (ids) ids[(size_t)q * K + j] = ok ? (uint64_t)key_id(key) : KEY_NONE;
        if (dist) dist[(size_t)q * K + j] = ok ? key_dist(key) : __uint_as_float(0x7fc00000u);
    }
    __shared__ uint32_t total_valid;
    if (threadIdx.x == 0) total_valid = 0;
    __syncthreads();
    if (valid) atomicAdd(&total_valid, valid);
    __syncthreads();
    if (threadIdx.x == 0 && counts) counts[q] = total_valid;
    if (fin.cnt_raw && threadIdx.x == 0) {
        // the same tests as overflow_kernel / check_kernel (flat_gemm.cu), on the keys still in shared memory
        const bool ovf = fin.cnt_raw[q] > fin.cap || (fin.qbad && fin.qbad[q]);
        if (fin.overflow) fin.overflow[q] = ovf ? 1u : 0u;
        if (fin.cand_total) atomicAdd(fin.cand_total, (unsigned long long)min((uint64_t)fin.cap, total));
        if (fin.redo) {
            const uint32_t need = (uint32_t)((uint64_t)K < fin.n_total ? (uint64_t)K : fin.n_total);
            bool ok = !ovf;
            if (ok && need) {
                const uint64_t kk = topk.seg(0)[need - 1];
                ok = kk != KEY_NONE;
                if (ok) {
                    const float dk = key_dist(kk);
                    const float shift = fin.qsq ? fin.qsq[q] : 0.f;
                    const float slack = 2e-5f * (fabsf(dk) + shift + fabsf(fin.tau[q]));
                    ok = (dk - shift) < fin.tau[q] - slack;
                }
            }
            if (fin.force_mod && q % fin.force_mod == 0) ok = false;
            if (!ok) fin.redo[atomicAdd(fin.nredo, 1u)] = q;
        }
    }
}

constexpr size_t MERGE_SMEM_MAX = 200 * 1024;
// the check of launch_merge_keys below for an input of more than 1024 keys per query (shorter inputs always fit)
bool merge_keys_fits(uint32_t k) { return TopkSmem::bytes(1, topk_segment_size(k, MERGE_THREADS)) <= MERGE_SMEM_MAX; }

void launch_merge_keys(const uint64_t* d_keys, uint32_t nlists, uint32_t nq, uint32_t len, bool list_major,
                       uint32_t k, uint64_t* d_out_keys, uint64_t* d_ids, float* d_dist,
                       uint32_t* d_counts, cudaStream_t stream, const uint64_t* d_seg_off, const uint32_t* d_seg_cnt,
                       const MergeFinish* finish) {
    if (nq == 0 || k == 0) return;
    // segment size: small inputs (K + all keys of a query fit in 1024 slots) are loaded completely and sorted once
    // in the smallest power-of-two segment; larger inputs stream through a K + 2 * 256 slot segment
    const uint64_t total_max = (uint64_t)nlists * len;  // per query (an upper bound when segment offsets are used)
    uint32_t P, limit;
    if (total_max + k <= 1024) {
        P = std::max(64u, next_pow2((uint32_t)total_max + k));
        limit = P - k;  // never reached: no intermediate flush
    } else {
        P = topk_segment_size(k, MERGE_THREADS);
        limit = P - k - MERGE_THREADS;
    }
    const size_t smem = TopkSmem::bytes(1, P);
    VDB_REQUIRE(smem <= MERGE_SMEM_MAX, "k=%u too large for the fused top-k (max %u)", k, 20000u);
    if (smem > 48 * 1024)
        VDB_CUDA(cudaFuncSetAttribute(merge_keys_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)smem));
    // short inputs (the sample lists of the tensor path: 16-300 keys per query, 10 000 queries): a CTA of one or two warps
    // per query instead of eight - four times as many queries resident per SM and nearly free barriers
    uint32_t threads = MERGE_THREADS;
    if (total_max + k <= 1024) threads = P <= 128 ? 32u : (P <= 256 ? 64u : (P <= 512 ? 128u : 256u));
    // counted lists (the tensor path's final selection: ~1.3 k live keys of a cap-sized list per query): the sort is over
    // <= 256 slots for k <= 128, so 4 warps do it as fast as 8 and twice as many queries are resident (a shorter period
    // than the limit assumes is always safe)
    else if (d_seg_cnt && k <= 128) threads = 128;
    ProfScope prof("merge", stream);
    merge_keys_kernel<<<nq, threads, smem, stream>>>(d_keys, nlists, nq, len, list_major ? 1 : 0, d_seg_off, d_seg_cnt,
                                                           k, P, limit, d_out_keys, d_ids,
                                                           d_dist, d_counts, finish ? *finish : MergeFinish{});
    VDB_LAUNCHED();
}

// ---- merge of SORTED lists (the per-shard [nq, k] results after the all-gather) -------------------------------------
// Every key finds its rank in the union by binary searches in the other lists (ties between lists go to the lower
// list index: stable), so there is no sort: nlists * len * (nlists - 1) * log2(len) shared-memory reads per query.
// Lists are ascending with KEY_NONE padding at the end (the contract of vdb_*_keys_dev).
__global__ void __launch_bounds__(256) merge_sorted_kernel(const uint64_t* __restrict__ keys, uint32_t nlists, uint32_t nq, uint32_t len,
                                                          uint32_t k, uint64_t* __restrict__ out_keys, uint64_t* __restrict__ ids,
                                                          float* __restrict__ dist, uint32_t* __restrict__ counts) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    uint64_t* s = reinterpret_cast<uint64_t*>(smem_raw);  // [nlists][len]
    uint64_t* o = s + (size_t)nlists * len;               // [k]
    const uint32_t q = blockIdx.x, T = nlists * len;
    __shared__ uint32_t valid;
    if (threadIdx.x == 0) valid = 0;
    for (uint32_t t = threadIdx.x; t < T; t += blockDim.x) {
        const uint32_t l = t / len, i = t - l * len;
        s[t] = keys[((size_t)l * nq + q) * len + i];
    }
    for (uint32_t j = threadIdx.x; j < k; j += blockDim.x) o[j] = KEY_NONE;
    __syncthreads();
    uint32_t mine = 0;
    for (uint32_t t = threadIdx.x; t < T; t += blockDim.x) {
        const uint64_t x = s[t];
        if (x == KEY_NONE) continue;
        ++mine;
        const uint32_t l = t / len;
        uint32_t rank = t - l * len;
        for (uint32_t l2 = 0; l2 < nlists && rank < k; ++l2) {
            if (l2 == l) continue;
            const uint64_t* lst = s + (size_t)l2 * len;
            uint32_t lo = 0, hi = len;
            if (l2 < l) {  // elements <= x
                while (lo < hi) {
                    const uint32_t mid = (lo + hi) >> 1;
                    if (lst[mid] <= x) lo = mid + 1;
                    else hi = mid;
                }
            } else {       // elements < x
                while (lo < hi) {
                    const uint32_t mid = (lo + hi) >> 1;
                    if (lst[mid] < x) lo = mid + 1;
                    else hi = mid;
                }
            }
            rank += lo;
        }
        if (rank < k) o[rank] = x;
    }
    if (mine) atomicAdd(&valid, mine);
    __syncthreads();
    for (uint32_t j = threadIdx.x; j < k; j += blockDim.x) {
        const uint64_t key = o[j];
        if (out_keys) out_keys[(size_t)q * k + j] = key;
        if (ids) {
            const bool ok = key != KEY_NONE;
            ids[(size_t)q * k + j] = ok ? (uint64_t)key_id(key) : KEY_NONE;
            dist[(size_t)q * k + j] = ok ? key_dist(key) : __uint_as_float(0x7fc00000u);
        }
    }
    if (threadIdx.x == 0 && counts) counts[q] = min(valid, k);
}

// list-major [nlists][nq][len] ascending lists -> the k smallest per query; falls back to the generic merge when the
// lists of a query do not fit in shared memory, and to select + sort in global memory when k does not fit the generic merge
void launch_merge_sorted(const uint64_t* d_keys, uint32_t nlists, uint32_t nq, uint32_t len, uint32_t k, uint64_t* d_out_keys,
                         uint64_t* d_ids, float* d_dist, uint32_t* d_counts, cudaStream_t stream) {
    if (nq == 0 || k == 0) return;
    if (!merge_keys_fits(k)) {
        large_k_select(d_keys, nlists, nq, len, k, d_out_keys, d_ids, d_dist, d_counts, stream);
        return;
    }
    static const int generic = getenv("VDB_MERGE_GENERIC") ? atoi(getenv("VDB_MERGE_GENERIC")) : 0;
    const size_t smem = ((size_t)nlists * len + k) * 8;
    if (generic || nlists == 1 || smem > 96 * 1024) {
        launch_merge_keys(d_keys, nlists, nq, len, true, k, d_out_keys, d_ids, d_dist, d_counts, stream);
        return;
    }
    if (smem > 48 * 1024)
        VDB_CUDA(cudaFuncSetAttribute(merge_sorted_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ProfScope prof("merge", stream);
    merge_sorted_kernel<<<nq, 256, smem, stream>>>(d_keys, nlists, nq, len, k, d_out_keys, d_ids, d_dist, d_counts);
    VDB_LAUNCHED();
}

__global__ void decode_keys_kernel(const uint64_t* __restrict__ keys, uint32_t nq, uint32_t k,
                                   uint64_t* __restrict__ ids, float* __restrict__ dist,
                                   uint32_t* __restrict__ counts) {
    const uint32_t q = blockIdx.x;
    uint32_t valid = 0;
    for (uint32_t j = threadIdx.x; j < k; j += blockDim.x) {
        const uint64_t key = keys[(size_t)q * k + j];
        const bool ok = key != KEY_NONE;
        valid += ok;
        ids[(size_t)q * k + j] = ok ? (uint64_t)key_id(key) : KEY_NONE;
        dist[(size_t)q * k + j] = ok ? key_dist(key) : __uint_as_float(0x7fc00000u);
    }
    __shared__ uint32_t total_valid;
    if (threadIdx.x == 0) total_valid = 0;
    __syncthreads();
    if (valid) atomicAdd(&total_valid, valid);
    __syncthreads();
    if (threadIdx.x == 0 && counts) counts[q] = total_valid;
}

void decode_keys(const uint64_t* d_keys, uint32_t nq, uint32_t k, uint64_t* d_ids, float* d_dist,
                 uint32_t* d_counts, cudaStream_t st) {
    if (nq == 0) return;
    if (k == 0) {
        if (d_counts) VDB_CUDA(cudaMemsetAsync(d_counts, 0, (size_t)nq * 4, st));
        return;
    }
    decode_keys_kernel<<<nq, 128, 0, st>>>(d_keys, nq, k, d_ids, d_dist, d_counts);
    VDB_LAUNCHED();
}

// ---- query tile preparation ---------------------------------------------------------------------
template <typename T>
__global__ void prepare_queries_kernel(const T* __restrict__ src, uint32_t dim, uint32_t vec, uint32_t nit,
                                       uint32_t qstride, int metric, float* __restrict__ tile,
                                       float* __restrict__ qcache, uint32_t* __restrict__ zero_word) {
    const uint32_t q = blockIdx.x;
    if (zero_word && q == 0 && threadIdx.x == 0) *zero_word = 0u;
    const uint32_t plane = nit * 32 * 4;  // floats per plane
    float ss = 0.f;
    for (uint32_t i = threadIdx.x; i < qstride; i += blockDim.x) {
        const uint32_t pl = i / plane, rem = i - pl * plane;
        const uint32_t c = rem >> 2, comp = rem & 3;
        const uint32_t e = c * vec + pl * 4 + comp;
        const float v = e < dim ? (float)src[(size_t)q * dim + e] : 0.f;
        tile[(size_t)q * qstride + i] = v;
        ss = fmaf(v, v, ss);
    }
    __shared__ float red[32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ss;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.f;
        for (uint32_t w = 0; w < blockDim.x / 32; ++w) t += red[w];
        qcache[q] = metric == VDB_COSINE ? sqrtf(t) : t;
    }
}

// u8 sets: the tile holds the queries' BYTES, zero padded to nit * 512 bytes per query (lane L of step it reads bytes
// [(it*32 + L) * 16, +16), exactly the bytes it loads from a row), and the cache is computed in integers (exact)
__global__ void prepare_queries_u8_kernel(const uint8_t* __restrict__ src, uint32_t dim, uint32_t qbytes, int metric,
                                          uint8_t* __restrict__ tile, float* __restrict__ qcache,
                                          uint32_t* __restrict__ zero_word) {
    const uint32_t q = blockIdx.x;
    if (zero_word && q == 0 && threadIdx.x == 0) *zero_word = 0u;
    __shared__ unsigned long long total;
    if (threadIdx.x == 0) total = 0;
    __syncthreads();
    uint32_t ss = 0;   // <= 64 bytes per thread (dim <= 65536, 1024 threads): 64 * 255^2 fits
    for (uint32_t i = threadIdx.x; i < qbytes; i += blockDim.x) {
        const uint32_t v = i < dim ? src[(size_t)q * dim + i] : 0u;
        tile[(size_t)q * qbytes + i] = (uint8_t)v;
        ss += v * v;
    }
    ss = __reduce_add_sync(0xffffffffu, ss);
    if ((threadIdx.x & 31) == 0 && ss) atomicAdd(&total, (unsigned long long)ss);
    __syncthreads();
    if (threadIdx.x == 0) qcache[q] = metric == VDB_COSINE ? sqrtf((float)total) : (float)total;
}

// geometry of the tile only (no buffers, no launch)
static QueryTile query_tile_shape(const vdb_dataset* ds) {
    QueryTile t;
    const uint32_t vec = vec_elems(ds->dtype);
    t.nvec = ds->pitch / vec;
    t.nit = ceil_div(t.nvec, 32u);
    // floats per query for f32 sets; for u8 sets the same count of 4-byte words (= nit * 512 bytes of query bytes), so
    // qstride * 4 is the tile's size in bytes per query for both
    t.qstride = ds->dtype == VDB_F32 ? t.nit * 32 * vec : t.nit * 32 * 4;
    return t;
}

QueryTile prepare_queries(const vdb_dataset* ds, const void* d_queries, uint32_t nq, cudaStream_t st, uint32_t* d_zero_word) {
    QueryTile t = query_tile_shape(ds);
    const uint32_t vec = vec_elems(ds->dtype);
    t.q = DevBuf((size_t)nq * t.qstride * 4, st);
    t.qcache = DevBuf((size_t)nq * 4, st);
    if (nq == 0) return t;
    if (ds->dtype == VDB_F32) {
        prepare_queries_kernel<float><<<nq, 256, 0, st>>>((const float*)d_queries, ds->dim, vec, t.nit,
                                                         t.qstride, ds->metric, t.q.as<float>(),
                                                         t.qcache.as<float>(), d_zero_word);
    } else {
        VDB_REQUIRE(ds->dim <= 65536, "u8 rows: dim %u too large for the 32-bit integer sums (max 65536)", ds->dim);
        // one byte per thread and pass when the query is short: the loads of a query are all in flight at once
        prepare_queries_u8_kernel<<<nq, 1024, 0, st>>>((const uint8_t*)d_queries, ds->dim, t.qstride * 4, ds->metric,
                                                      t.q.as<uint8_t>(), t.qcache.as<float>(), d_zero_word);
    }
    VDB_LAUNCHED();
    return t;
}

// ---- host launcher ------------------------------------------------------------------------------
template <int NQ, int R, int METRIC, int PL, bool EMIT>
static void launch_scan(const ScanParams& p, uint32_t grid, size_t smem, cudaStream_t st) {
    auto kern = flat_scan_kernel<NQ, R, METRIC, PL, EMIT>;
    static std::atomic<size_t> configured[VDB_MAX_DEVICES];
    if (smem > 48 * 1024) ensure_dyn_smem(kern, smem, configured);
    ProfScope prof(EMIT ? "flat_scan_emit" : "flat_scan", st);
    kern<<<grid, SCAN_THREADS, smem, st>>>(p);
    VDB_LAUNCHED();
}

template <int METRIC, int PL, bool EMIT = false>
static void dispatch_scan(int nqt, const ScanParams& p, uint32_t grid, size_t smem, cudaStream_t st) {
    switch (nqt) {
        case 1: launch_scan<1, 8, METRIC, PL, EMIT>(p, grid, smem, st); break;
        case 2: launch_scan<2, 8, METRIC, PL, EMIT>(p, grid, smem, st); break;
        case 4: launch_scan<4, 4, METRIC, PL, EMIT>(p, grid, smem, st); break;
        default: launch_scan<8, 4, METRIC, PL, EMIT>(p, grid, smem, st); break;
    }
}
template <bool EMIT = false>
static void dispatch_scan_ds(const vdb_dataset* ds, int nqt, const ScanParams& p, uint32_t grid, size_t smem, cudaStream_t st) {
    if (ds->dtype == VDB_F32) {
        if (ds->metric == VDB_L2SQR) dispatch_scan<VDB_L2SQR, 1, EMIT>(nqt, p, grid, smem, st);
        else dispatch_scan<VDB_COSINE, 1, EMIT>(nqt, p, grid, smem, st);
    } else {
        if (ds->metric == VDB_L2SQR) dispatch_scan<VDB_L2SQR, 4, EMIT>(nqt, p, grid, smem, st);
        else dispatch_scan<VDB_COSINE, 4, EMIT>(nqt, p, grid, smem, st);
    }
}
static int rows_per_group(int nqt) { return nqt <= 2 ? 8 : 4; }
// query tile + top-k segments (P = 0: the emit instantiation, no segments)
static size_t scan_smem(const QueryTile& qt, int nqt, uint32_t P) {
    return (size_t)nqt * qt.qstride * 4 + (P ? TopkSmem::bytes(nqt, P) : 0);
}

constexpr size_t SCAN_SMEM_MAX = 200 * 1024;

// The CTA-wide flush test (a barrier) runs every `sync_every` row groups: often enough that a query's segment cannot
// overflow between two tests (at most `period` appends), but not more often than every ~8 steps of 512 bytes - short
// rows (u8 x 960 = 2 steps per group, 128-d f32 = 1) otherwise meet at a barrier after every group and lose the overlap
// between warps (measured neutral for u8 x 960, where something else bounds the pass at 0.253 ms).
static uint32_t sync_every_for(uint32_t nit, uint32_t R) {
    return std::max(std::max(1u, 64u / (SCAN_WARPS * R)), ceil_div(8u, nit));
}
// shared memory of the fused scan: the top-k segment size and the largest query template (<= 8) that fits
struct ScanFit {
    uint32_t period, P;
    int nqt;
    bool fits;
};
static ScanFit scan_fit(const QueryTile& qt, uint32_t k) {
    ScanFit f;
    f.period = std::max(sync_every_for(qt.nit, 4) * SCAN_WARPS * 4, sync_every_for(qt.nit, 8) * SCAN_WARPS * 8);
    f.P = topk_segment_size(k, f.period);
    f.nqt = 8;
    while (f.nqt > 1 && scan_smem(qt, f.nqt, f.P) > SCAN_SMEM_MAX) f.nqt >>= 1;
    f.fits = scan_smem(qt, f.nqt, f.P) <= SCAN_SMEM_MAX;
    return f;
}
static bool scan_fuse_on() {
    const char* fuse_s = getenv("VDB_SCAN_FUSE");   // read per call: the tests toggle it in one process
    return !(fuse_s && !atoi(fuse_s));
}

bool fused_topk_fits(const vdb_dataset* ds, uint32_t nq, uint32_t k) {
    if (nq == 0 || k == 0 || ds->n == 0) return true;
    const ScanFit f = scan_fit(query_tile_shape(ds), k);
    if (!f.fits) return false;
    // the per-CTA lists are merged by launch_merge_keys unless the whole batch is one launch with the fused tail
    const bool merged = !(scan_fuse_on() && nq <= 8 && nq <= (uint32_t)f.nqt);
    return !merged || merge_keys_fits(k);
}

// Large-k path: the emit instantiation of the scan writes the key of every (query, row) of a chunk of queries to global
// memory - one rows pass per <= 8 queries, as in the fused scan - and large_k_select reduces each query's n keys to its
// k best. Emitted keys take at most LARGE_K_EMIT_BYTES per chunk (at least one query).
constexpr uint64_t LARGE_K_EMIT_BYTES = 1ull << 30;
static void flat_large_k_keys(const vdb_dataset* ds, const void* d_queries, uint32_t nq, uint32_t k, uint64_t* d_keys,
                              cudaStream_t st) {
    const QueryTile qt = prepare_queries(ds, d_queries, nq, st);
    int nqt = 8;
    while (nqt > 1 && scan_smem(qt, nqt, 0) > SCAN_SMEM_MAX) nqt >>= 1;
    VDB_REQUIRE(scan_smem(qt, nqt, 0) <= SCAN_SMEM_MAX, "flat scan: dim=%u does not fit in shared memory", ds->dim);
    const uint64_t per_query = ds->n * 8;
    uint32_t chunk = (uint32_t)std::min<uint64_t>(nq, std::max<uint64_t>(1, LARGE_K_EMIT_BYTES / per_query));
    if (chunk > 8) chunk = chunk / 8 * 8;   // whole 8-query passes
    DevBuf emit((size_t)chunk * per_query, st);
    const int sms = sm_count();
    ScanParams p{};
    p.rows = (const uint8_t*)ds->d_rows;
    p.n = ds->n;
    p.pitch_bytes = ds->pitch_bytes();
    p.nvec = qt.nvec;
    p.nit = qt.nit;
    p.qstride = qt.qstride;
    p.raw_dim = ds->dim;
    p.sync_every = 1;
    p.id_base = (uint32_t)ds->id_base;
    for (uint32_t q0 = 0; q0 < nq; q0 += chunk) {
        const uint32_t qn = std::min(chunk, nq - q0);
        for (uint32_t qq = 0; qq < qn;) {
            const uint32_t left = qn - qq;
            int t = nqt;
            while (t > 1 && (uint32_t)(t >> 1) >= left) t >>= 1;
            const uint32_t now = std::min<uint32_t>(left, t);
            const uint64_t ngroups = ceil_div<uint64_t>(ds->n, rows_per_group(t));
            const uint32_t grid = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(2 * sms, ceil_div<uint64_t>(ngroups, SCAN_WARPS)));
            p.iters = (uint32_t)ceil_div<uint64_t>(ngroups, (uint64_t)grid * SCAN_WARPS);
            p.q = qt.q.as<float>() + (size_t)(q0 + qq) * qt.qstride;
            p.qcache = qt.qcache.as<float>() + (q0 + qq);
            p.nq_valid = now;
            p.emit = emit.as<uint64_t>() + (size_t)qq * ds->n;
            dispatch_scan_ds<true>(ds, t, p, grid, scan_smem(qt, t, 0), st);
            qq += now;
        }
        large_k_select(emit.as<uint64_t>(), 1, qn, ds->n, k, d_keys + (size_t)q0 * k, nullptr, nullptr, nullptr, st);
    }
}

bool flat_scan_keys(const vdb_dataset* ds, const void* d_queries, uint32_t nq, uint32_t k,
                    uint64_t* d_keys, cudaStream_t st, const ScanOut* out) {
    if (nq == 0 || k == 0) return false;
    if (ds->n == 0) {
        VDB_CUDA(cudaMemsetAsync(d_keys, 0xff, (size_t)nq * k * 8, st));
        return false;
    }
    if (!fused_topk_fits(ds, nq, k)) {
        flat_large_k_keys(ds, d_queries, nq, k, d_keys, st);
        return false;
    }
    const bool fuse_on = scan_fuse_on();
    DevBuf done(fuse_on && nq <= 8 ? 4 : 0, st);   // arrival counter of the fused tail (cleared by the tile kernel)
    // u8 rows under L2Sqr in one launch (the trait's single-query call): the scan CTAs read the caller's query bytes
    // themselves and the counter is cleared by a 4-byte memset - no tile kernel in front of the scan
    const bool raw_q = ds->dtype == VDB_U8 && ds->metric == VDB_L2SQR && nq <= 8 && done.p != nullptr;
    QueryTile qt;
    if (raw_q) {
        qt = query_tile_shape(ds);
        VDB_REQUIRE(ds->dim <= 65536, "u8 rows: dim %u too large for the 32-bit integer sums (max 65536)", ds->dim);
        VDB_CUDA(cudaMemsetAsync(done.p, 0, 4, st));
    } else {
        qt = prepare_queries(ds, d_queries, nq, st, done.as<uint32_t>());
    }

    // queries per pass: as many as fit (<= 8) next to the top-k segments in shared memory (fused_topk_fits held)
    const ScanFit fit = scan_fit(qt, k);
    const uint32_t period = fit.period, P = fit.P;
    const int nqt = fit.nqt;
    auto smem_for = [&](int t) { return scan_smem(qt, t, P); };

    const int sms = sm_count();
    ScanParams p{};
    p.rows = (const uint8_t*)ds->d_rows;
    p.n = ds->n;
    p.pitch_bytes = ds->pitch_bytes();
    p.nvec = qt.nvec;
    p.nit = qt.nit;
    p.qstride = qt.qstride;
    p.K = k;
    p.P = P;
    p.limit = P - k - period;
    p.id_base = (uint32_t)ds->id_base;

    // passes are grouped in chunks so the partial lists stay small
    const uint32_t max_grid = 2 * sms;
    const size_t partial_per_query = (size_t)max_grid * k * 8;
    uint32_t chunk = (uint32_t)std::max<size_t>(8, (size_t)(64u << 20) / partial_per_query);
    chunk = std::min(round_up(chunk, 8u), round_up(nq, 8u));
    DevBuf partial(partial_per_query * chunk, st);
    bool fused = false;

    for (uint32_t q0 = 0; q0 < nq; q0 += chunk) {
        const uint32_t qn = std::min(chunk, nq - q0);
        uint32_t grid_used = 0;
        for (uint32_t qq = 0; qq < qn;) {
            const uint32_t left = qn - qq;
            int t = nqt;
            while (t > 1 && (uint32_t)(t >> 1) >= left) t >>= 1;  // smallest template that covers `left`
            const uint32_t now = std::min<uint32_t>(left, t);
            const int R = rows_per_group(t);
            const uint64_t ngroups = ceil_div<uint64_t>(ds->n, R);
            const uint32_t grid = (uint32_t)std::max<uint64_t>(
                1, std::min<uint64_t>(max_grid, ceil_div<uint64_t>(ngroups, SCAN_WARPS)));
            // every pass of a chunk must use the same grid so the partial layout is uniform
            if (grid_used == 0) grid_used = grid;
            p.iters = (uint32_t)ceil_div<uint64_t>(ngroups, (uint64_t)grid_used * SCAN_WARPS);
            p.sync_every = sync_every_for(qt.nit, (uint32_t)R);
            p.q = raw_q ? nullptr : qt.q.as<float>() + (size_t)(q0 + qq) * qt.qstride;
            p.qcache = raw_q ? nullptr : qt.qcache.as<float>() + (q0 + qq);
            p.raw_q = raw_q ? (const uint8_t*)d_queries + (size_t)(q0 + qq) * ds->dim : nullptr;
            p.raw_dim = ds->dim;
            p.nq_valid = now;
            p.partial = partial.as<uint64_t>() + (size_t)qq * grid_used * k;
            // the whole batch in this one launch: its last CTA merges and decodes
            fused = done.p != nullptr && q0 == 0 && qq == 0 && now == nq;
            p.done = fused ? done.as<uint32_t>() : nullptr;
            p.out_keys = d_keys;
            p.out_ids = fused && out ? out->ids : nullptr;
            p.out_dist = fused && out ? out->dist : nullptr;
            p.out_counts = fused && out ? out->counts : nullptr;
            dispatch_scan_ds(ds, t, p, grid_used, smem_for(t), st);
            qq += now;
        }
        if (!fused)
            launch_merge_keys(partial.as<uint64_t>(), grid_used, qn, k, false, k, d_keys + (size_t)q0 * k,
                              nullptr, nullptr, nullptr, st);
    }
    return fused && out != nullptr;
}

}  // namespace vdb
