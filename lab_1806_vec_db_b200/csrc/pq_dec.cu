// pq_dec.cu — K8d: the 4-bit PQ ADC scan of a query batch as a tensor-core contraction over DECODED rows (L2Sqr tables,
// sub-vectors of 4 dimensions: the reference's bench configuration m = dim / 4, config/bench_pq_240_hnsw.toml:16-23).
//
// In real arithmetic the ADC distance (reference src/distance/pq_table.rs:239-301: sum over the groups of the lookup
// table entry l2(q_g, c_{g, code})) is ||q - x^||^2 = ||q||^2 - 2 q.x^ + ||x^||^2 with x^ = the row's centroids
// concatenated. K8t (pq_gemm.cu) evaluates it as <onehot(row), LUT_q> over K = 16 m columns; here the contraction is the
// plain dot product q.x^ over K = dim columns — FOUR TIMES fewer MMAs and generated tiles — and the decoded operand never
// exists in HBM: generator warps expand the code nibbles of a 128-row tile into FP16 centroid values (codebooks in
// shared memory, 8 bytes per (group, centroid)) directly in the 128-byte-swizzled A tile the MMA reads. Memory stays
// the table's: 0.5 byte per (row, group) + 8 bytes per row of norms.
//
// The tensor cores only PRUNE. With q~ = fp16(q s_q), c~ = fp16(c s_c) (powers of two), acc = q~.x^~ in fp32:
//   |q.x^ - acc / (s_q s_c)| <= ACC qn' xn' + qn' ex + eq xn'      (as in flat_gemm.cu; ex <= EX = the worst-case
//   decode error norm over all code words, xn = ||x^||, ACC = dim 2^-23)
// so S' = ||x^||^2 - 2 acc / (s_q s_c) - (qab EX + qb xn) <= adc_real - ||q||^2, and the reference's f32 evaluation of
// the same sum of non-negative terms is within (m + 8) 2^-24 relative of adc_real. Rows with
// S' <= tau_q (1 + 5e-5) - ||q||^2 (1 - 5e-5) become coarse candidates; their ADC value is then re-evaluated with the
// reference's arithmetic (pq_exact_cands_kernel, pq_gemm.cu) and the rows with adc <= tau_q go on exactly as in the FP32
// scan: the candidate set, hence every id and distance bit, is unchanged (tests/test_index_gpu.py).
//
// Kernel (sm_100a, one CTA per SM, 704 threads): warps 0-3 epilogue (thread = row, registers = queries), warp 4 TMA
// producer of the FP16 query tile (256 queries x 64 dims), warp 5 one thread issuing tcgen05.mma.kind::f16 (M = 128
// rows, N = 256 queries, K = 16, four per k-block) into double-buffered TMEM accumulators, warps 6-21 four generator
// groups taking the k-blocks round-robin (thread = row: one 8-byte load of 16 code nibbles, 16 LDS.64 of centroid
// values, 8 conflict-free STS.128, fence.proxy.async, mbarrier arrive).
#include <cuda.h>
#include <cuda_fp16.h>

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <memory>
#include <mutex>
#include <vector>

#include "index.cuh"
#include "tc.cuh"
#include "topk.cuh"

namespace vdb {

constexpr int DM = 128;                     // rows per tile (TMEM lanes)
constexpr int DN = 256;                     // queries per tile (TMEM columns per accumulator)
constexpr int DK = 64;                      // fp16 columns per k-block = 16 groups x 4 dims = 128 bytes
constexpr int D_A_BYTES = DM * DK * 2;      // 16 KB generated tile
constexpr int D_B_BYTES = DN * DK * 2;      // 32 KB query tile
constexpr int D_STAGE_BYTES = D_A_BYTES + D_B_BYTES;
constexpr int D_STAGES = 4;
constexpr int D_GG = 4;                     // generator groups of 4 warps
constexpr int D_BASE_THREADS = 192;
constexpr int D_THREADS = D_BASE_THREADS + 128 * D_GG;
constexpr int D_TMEM_COLS = 512;
constexpr uint32_t D_MAX_M = 240;           // codebooks (128 B per group) + 4 stages + thresholds fit 227 KB of shared memory
// instruction descriptor: D = F32, A = B = F16, both K-major, N >> 3, M >> 4
constexpr uint32_t D_IDESC = (1u << 4) | ((uint32_t)(DN >> 3) << 17) | ((uint32_t)(DM >> 4) << 24);

static size_t dec_smem_bytes(uint32_t m) { return 1024 + (size_t)D_STAGES * D_STAGE_BYTES + (size_t)m * 128 + 3 * DN * 4 + 256; }

struct PqDecParams {
    const uint8_t* codes;     // [n][enc] reference layout (low nibble = even group)
    uint64_t n;
    uint32_t enc, m, kblocks, nq;
    const uint2* cb16;        // [m][16] four fp16 values (c s_c) per (group, centroid)
    const float* row_r;       // [n] ||x^||^2
    const float* row_xn;      // [n] ||x^||
    const float* qd;          // [nq] -2 / (s_q s_c)
    const float* qb;          // [nq] coefficient of xn in the bound
    const float* qt;          // [nq] MODE 1: threshold of the score; MODE 0: ||q||^2 + qab EX
    uint32_t* ccnt;           // [nq] coarse candidate counters
    uint32_t* ccand;          // [nq][ccap] rows
    uint32_t ccap;
    uint32_t tiles_per_item, nrow_items, nqt;
    float* all_out;           // MODE 0: [nq][n] upper bounds of the exact ADC values (sample pass); MODE 2: [nq][n] scores
    // MODE 1 output: one record per (row, chunk of 32 queries) with any passing score - the per-query candidate lists are
    // filled from the records by pq_dec_expand_kernel. (Appending to the per-query lists from the epilogue costs one
    // atomic round trip per passing score in divergent code: at 0.25 % passing scores the four epilogue warps needed
    // twice the time of the tile's MMAs.)
    uint64_t* rec;            // [rec_cap] row << 16 | chunk index (query = chunk * 32 + bit)
    uint32_t* rec_mask;       // [rec_cap] passing queries of the chunk
    uint32_t* rec_count;      // records written (may exceed rec_cap: then every list is declared overflowed)
    uint32_t rec_cap;
};

// MODE 0: store an upper bound of every ADC value (sample pass), 1: filter, 2: store every filter score (test hook)
template <int MODE>
__global__ void __launch_bounds__(D_THREADS, 1) pq_dec_kernel(const __grid_constant__ CUtensorMap map_q, const PqDecParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t* stage_base = smem;
    uint2* cb_s = reinterpret_cast<uint2*>(smem + D_STAGES * D_STAGE_BYTES);   // [m][16]
    float* qd_s = reinterpret_cast<float*>(cb_s + (size_t)p.m * 16);           // [DN]
    float* qb_s = qd_s + DN;
    float* qt_s = qb_s + DN;
    uint64_t* bars = reinterpret_cast<uint64_t*>(qt_s + DN);
    uint64_t* full_bar = bars;                  // [D_STAGES]
    uint64_t* empty_bar = bars + D_STAGES;      // [D_STAGES]
    uint64_t* tfull_bar = bars + 2 * D_STAGES;  // [2]
    uint64_t* tempty_bar = tfull_bar + 2;       // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int s = 0; s < D_STAGES; ++s) {
            mbar_init(&full_bar[s], 1 + 4);   // TMA expect_tx arrive + one arrive per warp of the generating group
            mbar_init(&empty_bar[s], 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&tfull_bar[a], 1);
            mbar_init(&tempty_bar[a], 4);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (uint32_t e = threadIdx.x; e < p.m * 16; e += blockDim.x) cb_s[e] = p.cb16[e];
    if (warp == 5) tmem_alloc(tmem_slot, D_TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t nitems = p.nrow_items * p.nqt;

    if (warp == 4) {
        // ===== TMA producer: the FP16 query tile of every k-block =====
        if (lane == 0) {
            uint32_t stage = 0, phase = 0;
            for (uint32_t item = blockIdx.x; item < nitems; item += gridDim.x) {
                const uint32_t ri = item / p.nqt, qt = item - ri * p.nqt;
                const uint64_t r0 = (uint64_t)ri * p.tiles_per_item * DM;
                const uint32_t ntile = (uint32_t)min((uint64_t)p.tiles_per_item, (p.n - r0 + DM - 1) / DM);
                for (uint32_t t = 0; t < ntile; ++t)
                    for (uint32_t kb = 0; kb < p.kblocks; ++kb) {
                        mbar_wait(&empty_bar[stage], phase ^ 1);
                        mbar_expect_tx(&full_bar[stage], D_B_BYTES);
                        tma_load_2d(smem_u32(stage_base + stage * D_STAGE_BYTES) + D_A_BYTES, &map_q, (int)(kb * DK), (int)(qt * DN),
                                    &full_bar[stage]);
                        if (++stage == D_STAGES) stage = 0, phase ^= 1;
                    }
            }
        }
    } else if (warp == 5) {
        // ===== MMA issuer =====
        if (lane == 0) {
            uint32_t stage = 0, phase = 0, acc = 0, acc_phase = 0;
            for (uint32_t item = blockIdx.x; item < nitems; item += gridDim.x) {
                const uint32_t ri = item / p.nqt;
                const uint64_t r0 = (uint64_t)ri * p.tiles_per_item * DM;
                const uint32_t ntile = (uint32_t)min((uint64_t)p.tiles_per_item, (p.n - r0 + DM - 1) / DM);
                for (uint32_t t = 0; t < ntile; ++t) {
                    mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
                    tc_fence_after();
                    const uint32_t d_tmem = tmem_base + acc * DN;
                    for (uint32_t kb = 0; kb < p.kblocks; ++kb) {
                        mbar_wait(&full_bar[stage], phase);
                        tc_fence_after();
                        const uint32_t sa = smem_u32(stage_base + stage * D_STAGE_BYTES);
                        const uint64_t da = umma_desc(sa), db = umma_desc(sa + D_A_BYTES);
#pragma unroll
                        for (int k = 0; k < DK / 16; ++k) umma_f16(d_tmem, da + 2 * k, db + 2 * k, D_IDESC, (kb | k) != 0);
                        umma_commit(&empty_bar[stage]);
                        if (++stage == D_STAGES) stage = 0, phase ^= 1;
                    }
                    umma_commit(&tfull_bar[acc]);
                    if (++acc == 2) acc = 0, acc_phase ^= 1;
                }
            }
        }
    } else if (warp >= 6) {
        // ===== generators: 16 code nibbles -> 64 fp16 centroid values of the row, written in the 128B-swizzle layout =====
        const uint32_t gt = threadIdx.x - D_BASE_THREADS;
        const uint32_t gg = gt >> 7;   // generator group
        const uint32_t r = gt & 127;   // row of the tile
        uint32_t kbc = 0;              // running k-block counter (all groups count alike)
        for (uint32_t item = blockIdx.x; item < nitems; item += gridDim.x) {
            const uint32_t ri = item / p.nqt;
            const uint64_t r0 = (uint64_t)ri * p.tiles_per_item * DM;
            const uint32_t ntile = (uint32_t)min((uint64_t)p.tiles_per_item, (p.n - r0 + DM - 1) / DM);
            for (uint32_t t = 0; t < ntile; ++t) {
                const uint64_t row = r0 + (uint64_t)t * DM + r;
                const bool row_ok = row < p.n;
                const uint2* my = reinterpret_cast<const uint2*>(p.codes + (row_ok ? row : 0) * p.enc);   // enc % 8 == 0
                // the code words of this thread's k-blocks of the tile (every 4th), all loads in flight together; the next
                // tile's row is on its way to L1 meanwhile (the rows of an item are consecutive)
                const uint32_t first = (gg + D_GG - (kbc % D_GG)) % D_GG;
                uint2 cw[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const uint32_t kb = first + D_GG * i;
                    cw[i] = (row_ok && kb < p.kblocks) ? __ldg(my + kb) : make_uint2(0u, 0u);
                }
                if (row + DM < p.n && gg == 0) {
                    const uint8_t* nxt = p.codes + (row + DM) * p.enc;
                    asm volatile("prefetch.global.L1 [%0];" ::"l"(nxt));
                    asm volatile("prefetch.global.L1 [%0];" ::"l"(nxt + p.enc - 1));
                }
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const uint32_t kb = first + D_GG * i;
                    if (kb >= p.kblocks) break;
                    const uint32_t c = kbc + kb;
                    const uint32_t stage = c % D_STAGES, phase = (c / D_STAGES) & 1;
                    mbar_wait(&empty_bar[stage], phase ^ 1);
                    uint8_t* arow = stage_base + stage * D_STAGE_BYTES + r * 128;
                    const uint2* cbk = cb_s + (size_t)kb * 16 * 16;   // 16 groups of this k-block
#pragma unroll
                    for (int j = 0; j < 8; ++j) {   // chunk j = groups 2j (low nibble) and 2j + 1 (high nibble) of byte j
                        const uint32_t byte = ((j < 4 ? cw[i].x : cw[i].y) >> (8 * (j & 3))) & 0xffu;
                        const uint2 a = cbk[(2 * j) * 16 + (byte & 0xfu)];
                        const uint2 b = cbk[(2 * j + 1) * 16 + (byte >> 4)];
                        const uint4 v = row_ok ? make_uint4(a.x, a.y, b.x, b.y) : make_uint4(0u, 0u, 0u, 0u);
                        *reinterpret_cast<uint4*>(arow + ((j ^ (r & 7)) << 4)) = v;
                    }
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> visible to the MMA
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&full_bar[stage]);
                }
                kbc += p.kblocks;
            }
        }
    } else {
        // ===== epilogue: warps 0-3, thread = row (TMEM lane), registers = queries =====
        uint32_t acc = 0, acc_phase = 0;
        const uint32_t lane_base = (uint32_t)warp * 32;
        for (uint32_t item = blockIdx.x; item < nitems; item += gridDim.x) {
            const uint32_t ri = item / p.nqt, qt = item - ri * p.nqt;
            const uint64_t r0 = (uint64_t)ri * p.tiles_per_item * DM;
            const uint32_t ntile = (uint32_t)min((uint64_t)p.tiles_per_item, (p.n - r0 + DM - 1) / DM);
            const uint32_t q0 = qt * DN;
            asm volatile("bar.sync 1, 128;" ::: "memory");  // the previous item's per-query scalars are no longer read
            for (uint32_t c = threadIdx.x; c < DN; c += 128) {
                const bool ok = (q0 + c) < p.nq;
                qd_s[c] = ok ? p.qd[q0 + c] : 0.f;
                qb_s[c] = ok ? p.qb[q0 + c] : 0.f;
                qt_s[c] = ok ? p.qt[q0 + c] : __uint_as_float(0xff800000u);  // -inf: nothing passes
            }
            asm volatile("bar.sync 1, 128;" ::: "memory");
            const uint32_t qd_a = smem_u32(qd_s), qb_a = smem_u32(qb_s), qt_a = smem_u32(qt_s);
            for (uint32_t t = 0; t < ntile; ++t) {
                const uint64_t row = r0 + (uint64_t)t * DM + threadIdx.x;
                const bool row_ok = row < p.n;
                const float rr = row_ok ? p.row_r[row] : 0.f, xn = row_ok ? p.row_xn[row] : 0.f;
                mbar_wait(&tfull_bar[acc], acc_phase);
                tc_fence_after();
                const uint32_t taddr = tmem_base + (lane_base << 16) + acc * DN;
                constexpr int HC = DN / 64;   // chunks of 32 queries per half tile
                auto flush = [&](const uint32_t (&msk)[HC], int half) {
                    // records of this half tile: ONE atomic per warp reserves their slots
                    uint32_t cnt = 0;
#pragma unroll
                    for (int ci = 0; ci < HC; ++ci) cnt += msk[ci] != 0u;
                    uint32_t incl = cnt;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const uint32_t y = __shfl_up_sync(0xffffffffu, incl, o);
                        if (lane >= o) incl += y;
                    }
                    const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
                    if (total == 0) return;
                    uint32_t base = 0;
                    if (lane == 31) base = atomicAdd(p.rec_count, total);
                    base = __shfl_sync(0xffffffffu, base, 31);
                    uint32_t idx = base + incl - cnt;
#pragma unroll
                    for (int ci = 0; ci < HC; ++ci) {
                        if (msk[ci]) {
                            if (idx < p.rec_cap) {
                                p.rec[idx] = ((uint64_t)row << 16) | (uint64_t)(qt * (DN / 32) + half * HC + ci);
                                p.rec_mask[idx] = msk[ci];
                            }
                            ++idx;
                        }
                    }
                };
#pragma unroll 1
                for (int half = 0; half < 2; ++half) {
                    uint32_t msk[HC];
#pragma unroll
                    for (int ci = 0; ci < HC; ++ci) {
                        msk[ci] = 0u;
                        const int c0 = (half * HC + ci) * 32;
                        uint32_t v[32];
                        tmem_ld32(taddr + c0, v);
                        if (row_ok) {
#pragma unroll
                            for (int j4 = 0; j4 < 32; j4 += 4) {
                                const float4 d4 = lds_f4(qd_a + (c0 + j4) * 4), b4 = lds_f4(qb_a + (c0 + j4) * 4),
                                             t4 = lds_f4(qt_a + (c0 + j4) * 4);
                                const float dv[4] = {d4.x, d4.y, d4.z, d4.w}, bv[4] = {b4.x, b4.y, b4.z, b4.w},
                                            tv[4] = {t4.x, t4.y, t4.z, t4.w};
#pragma unroll
                                for (int jj = 0; jj < 4; ++jj) {
                                    const int j = j4 + jj;
                                    const float dot = __uint_as_float(v[j]);
                                    if (MODE == 2) {
                                        const uint32_t q = q0 + c0 + j;
                                        if (q < p.nq) p.all_out[(size_t)q * p.n + row] = fmaf(dv[jj], dot, fmaf(-bv[jj], xn, rr));
                                    } else if (MODE == 0) {
                                        // upper bound of the reference's ADC value; a warp stores 32 consecutive rows of a query
                                        const uint32_t q = q0 + c0 + j;
                                        const float up = (fmaf(dv[jj], dot, fmaf(bv[jj], xn, rr)) + tv[jj]) * 1.00005f + 1e-30f;
                                        if (q < p.nq) p.all_out[(size_t)q * p.n + row] = up;
                                    } else {
                                        const float sc = fmaf(dv[jj], dot, fmaf(-bv[jj], xn, rr));
                                        msk[ci] |= (sc > tv[jj] ? 0u : 1u) << j;   // also keeps NaN (the exact re-evaluation decides)
                                    }
                                }
                            }
                        }
                    }
                    if (half == 1) {   // every TMEM load of the tile is done: hand the accumulator back (one arrive per warp)
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&tempty_bar[acc]);
                        if (++acc == 2) acc = 0, acc_phase ^= 1;
                    }
                    if (MODE == 1) flush(msk, half);
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 5) tmem_dealloc(tmem_base, D_TMEM_COLS);
}

// records (row, chunk of 32 queries, passing mask) -> per-query coarse candidate lists. One thread per record: the
// atomics of a record are independent of every other thread's, so their latency is hidden by parallelism.
__global__ void pq_dec_expand_kernel(const uint64_t* __restrict__ rec, const uint32_t* __restrict__ rec_mask,
                                     const uint32_t* __restrict__ rec_count, uint32_t rec_cap, uint32_t nq,
                                     uint32_t* __restrict__ ccnt, uint32_t* __restrict__ ccand, uint32_t ccap) {
    const uint32_t total = *rec_count;
    if (total > rec_cap) {   // the record buffer overflowed: every list counts as overflowed (exact fallback)
        for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < nq; q += gridDim.x * blockDim.x) ccnt[q] = ccap + 1;
        return;
    }
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const uint64_t r = rec[i];
        const uint32_t row = (uint32_t)(r >> 16), q0 = (uint32_t)(r & 0xffffu) * 32;
        uint32_t m = rec_mask[i];
        while (m) {
            const uint32_t b = __ffs(m) - 1;
            m &= m - 1;
            const uint32_t q = q0 + b;
            const uint32_t pos = atomicAdd(&ccnt[q], 1u);
            if (pos < ccap) ccand[(size_t)q * ccap + pos] = row;
        }
    }
}

// ---- per-table side data (lazily built by the first batched search) ---------------------------------------------
// ||x^||^2 and ||x^|| of every code row: the sum of the centroids' squared norms in group order
__global__ void pq_dec_rows_kernel(const uint8_t* __restrict__ codes, uint64_t n, uint32_t enc, uint32_t m,
                                   const float* __restrict__ cn2, float* __restrict__ out_r, float* __restrict__ out_xn) {
    const uint64_t row = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= n) return;
    const uint8_t* cr = codes + row * enc;
    float s = 0.f;
    for (uint32_t g = 0; g < m; g += 2) {
        const uint32_t byte = cr[g >> 1];
        s += cn2[g * 16 + (byte & 0xfu)];
        if (g + 1 < m) s += cn2[(g + 1) * 16 + (byte >> 4)];
    }
    out_r[row] = s;
    out_xn[row] = sqrtf(s) * 1.000001f;
}

static std::mutex g_dec_mu;

bool pq_dec_supported(const vdb_pq* pq, uint32_t nq) {
    const char* off = getenv("VDB_PQ_NO_DECODE");   // read per call: the tests compare the two contractions in one process
    if (off && atoi(off)) return false;
    if (!pq_tensor_supported(pq, nq)) return false;
    if (pq->m > D_MAX_M || pq->m % 16 != 0 || pq->dim != 4 * pq->m || pq->enc % 8 != 0) return false;
    for (uint32_t g = 0; g < pq->m; ++g)
        if (pq->g_len[g] != 4) return false;
    return true;
}

static void ensure_dec_side(const vdb_pq* cpq, cudaStream_t st) {
    vdb_pq* pq = const_cast<vdb_pq*>(cpq);
    std::lock_guard<std::mutex> lk(g_dec_mu);
    if (pq->d_dec_cb16) return;
    const uint32_t tab = pq->m * 16, ne = tab * 4;
    // the codebooks are tiny (m x 16 x 4 values): converted on the host
    std::vector<float> cb(ne);
    if (pq->dtype == VDB_F32) {
        VDB_CUDA(cudaMemcpyAsync(cb.data(), pq->d_codebooks, (size_t)ne * 4, cudaMemcpyDeviceToHost, st));
        VDB_CUDA(cudaStreamSynchronize(st));
    } else {
        std::vector<uint8_t> raw(ne);
        VDB_CUDA(cudaMemcpyAsync(raw.data(), pq->d_codebooks, ne, cudaMemcpyDeviceToHost, st));
        VDB_CUDA(cudaStreamSynchronize(st));
        for (uint32_t i = 0; i < ne; ++i) cb[i] = (float)raw[i];
    }
    float amax = 0.f;
    for (float v : cb)
        if (std::isfinite(v)) amax = std::max(amax, std::fabs(v));
    float scale = 1.0f;
    if (amax > 0.f) {
        int e = 0;
        std::frexp(amax, &e);   // amax = f * 2^e, f in [0.5, 1): the largest magnitude lands in (2^13, 2^14]
        scale = std::ldexp(1.0f, std::max(-100, std::min(100, 14 - e)));
    }
    std::vector<__half> h16(ne);
    std::vector<float> cn2(tab);
    double ex2 = 0.0;   // sum over the groups of the worst centroid's squared decode error
    bool finite = true;
    for (uint32_t g = 0; g < pq->m; ++g) {
        double worst = 0.0;
        for (uint32_t c = 0; c < 16; ++c) {
            double e2 = 0.0;
            float n2 = 0.f;
            for (uint32_t j = 0; j < 4; ++j) {
                const float v = cb[((size_t)g * 16 + c) * 4 + j];
                const __half h = __float2half_rn(v * scale);
                h16[((size_t)g * 16 + c) * 4 + j] = h;
                const float back = __half2float(h) / scale;
                finite = finite && std::isfinite(v) && std::isfinite(back);
                e2 += ((double)v - back) * ((double)v - back);
                n2 += v * v;
            }
            cn2[g * 16 + c] = n2;
            worst = std::max(worst, e2);
        }
        ex2 += worst;
    }
    pq->dec_ok = finite;
    pq->dec_scale = scale;
    pq->dec_ex = (float)(std::sqrt(ex2) * 1.0001);
    if (!finite) {   // remember the decision with an empty table
        VDB_CUDA(cudaMalloc(&pq->d_dec_cb16, 16));
        return;
    }
    float* d_cn2 = nullptr;
    VDB_CUDA(cudaMalloc(&pq->d_dec_cb16, (size_t)ne * 2));
    VDB_CUDA(cudaMalloc(&d_cn2, (size_t)tab * 4));
    VDB_CUDA(cudaMalloc(&pq->d_dec_r, std::max<size_t>(4, pq->n * 4)));
    VDB_CUDA(cudaMalloc(&pq->d_dec_xn, std::max<size_t>(4, pq->n * 4)));
    VDB_CUDA(cudaMalloc(&pq->d_dec_sr, std::max<size_t>(4, (size_t)pq->sample_n * 4)));
    VDB_CUDA(cudaMalloc(&pq->d_dec_sxn, std::max<size_t>(4, (size_t)pq->sample_n * 4)));
    VDB_CUDA(cudaMemcpyAsync(pq->d_dec_cb16, h16.data(), (size_t)ne * 2, cudaMemcpyHostToDevice, st));
    VDB_CUDA(cudaMemcpyAsync(d_cn2, cn2.data(), (size_t)tab * 4, cudaMemcpyHostToDevice, st));
    pq_dec_rows_kernel<<<(uint32_t)ceil_div<uint64_t>(pq->n, 256), 256, 0, st>>>(pq->d_codes, pq->n, pq->enc, pq->m, d_cn2, pq->d_dec_r,
                                                                              pq->d_dec_xn);
    VDB_LAUNCHED();
    pq_dec_rows_kernel<<<ceil_div(pq->sample_n, 256u), 256, 0, st>>>(pq->d_sample, pq->sample_n, pq->enc, pq->m, d_cn2, pq->d_dec_sr,
                                                                     pq->d_dec_sxn);
    VDB_LAUNCHED();
    VDB_CUDA(cudaStreamSynchronize(st));
    cudaFree(d_cn2);
}

void pq_dec_destroy(vdb_pq* pq) {
    cudaFree(pq->d_dec_cb16);
    cudaFree(pq->d_dec_r);
    cudaFree(pq->d_dec_xn);
    cudaFree(pq->d_dec_sr);
    cudaFree(pq->d_dec_sxn);
    pq->d_dec_cb16 = nullptr;
    pq->d_dec_r = pq->d_dec_xn = pq->d_dec_sr = pq->d_dec_sxn = nullptr;
}

// ---- query side: FP16 operand (one power-of-two scale per query), ||q||^2, the operand error and the coefficients ------
template <typename T>
__global__ void __launch_bounds__(256) pq_dec_query_kernel(const T* __restrict__ src, uint32_t nq, uint32_t dim, float cb_scale,
                                                           float ex_max, float acc, __half* __restrict__ q16,
                                                           float* __restrict__ qsq, float* __restrict__ qd, float* __restrict__ qb,
                                                           float* __restrict__ qab) {
    const uint32_t q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (q >= nq) return;
    const T* row = src + (size_t)q * dim;
    float m = 0.f;
    bool finite = true;
    for (uint32_t e = lane; e < dim; e += 32) {
        const float v = fabsf((float)row[e]);
        finite = finite && (v <= 3.0e38f);
        m = fmaxf(m, v <= 3.0e38f ? v : 0.f);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    float scale = 1.0f;
    if (m > 0.f) {
        int e2 = (int)((__float_as_uint(m) >> 23) & 0xff) - 126;   // m = f * 2^e2, f in [0.5, 1) (normal m)
        e2 = max(-100, min(100, 14 - e2));
        scale = __uint_as_float((uint32_t)(e2 + 127) << 23);
    }
    const float inv = 1.0f / scale;
    float s = 0.f, ee = 0.f;
    for (uint32_t e = lane; e < dim; e += 32) {
        const float v = (float)row[e];
        const __half h = __float2half_rn(v * scale);
        q16[(size_t)q * dim + e] = h;
        const float d = v - __half2float(h) * inv;
        s = fmaf(v, v, s);
        ee = fmaf(d, d, ee);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, o);
        ee += __shfl_xor_sync(0xffffffffu, ee, o);
    }
    finite = __all_sync(0xffffffffu, finite);
    if (lane == 0) {
        const float eq = sqrtf(ee) * 1.0001f;
        const float qn1 = (sqrtf(s) + eq) * 1.0001f;
        const float b = 2.0f * (acc * qn1 + eq) * 1.0001f;
        qsq[q] = s;
        // a non-finite query keeps every row (NaN coefficients fail no comparison): the exact re-evaluation decides
        qd[q] = finite ? -2.0f * inv / cb_scale : __uint_as_float(0x7fc00000u);
        // coefficient of ||x^||: the bound's own (b, with xn' = xn + EX folded into qab) + the rounding of ||x^||^2 itself
        qb[q] = b + 4e-6f * qn1;
        qab[q] = (2.0f * qn1 + b) * ex_max;   // (coefficient of the decode error) x (its worst case over all code words)
    }
}
// MODE 1 threshold of the score for the ADC threshold tau (non-decreasing in tau)
__device__ __forceinline__ float dec_score_threshold(float tau, float qsq, float qab) {
    return tau * 1.00005f - qsq * 0.99995f + qab + 1e-30f;
}
// MODE 1 threshold of the score / MODE 0 additive constant of the upper bound
__global__ void pq_dec_thresholds_kernel(const float* __restrict__ tau, const float* __restrict__ qsq, const float* __restrict__ qab,
                                         uint32_t nq, float* __restrict__ out) {
    const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    if (tau) out[q] = dec_score_threshold(tau[q], qsq[q], qab[q]);
    else out[q] = qsq[q] * 1.00005f + qab[q];
}
// test hook: filter score -> the smallest ADC threshold tau at which the filter keeps the row (its lower bound of the
// ADC value in the units of the other paths): bisection over the ordered float bit patterns, the threshold being
// non-decreasing in tau. NaN scores are kept at every threshold (-inf).
__global__ void pq_dec_lower_kernel(float* __restrict__ v, uint32_t nq, uint64_t n, const float* __restrict__ qsq,
                                    const float* __restrict__ qab) {
    const uint64_t total = (uint64_t)nq * n;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t q = (uint32_t)(i / n);
        const float sc = v[i];
        uint32_t lo = f32_order_bits(__uint_as_float(0xff800000u)), hi = f32_order_bits(__uint_as_float(0x7f800000u));
        if (!(sc > dec_score_threshold(f32_from_order_bits(lo), qsq[q], qab[q]))) hi = lo;
        while (hi - lo > 1) {   // invariant: the row is dropped at lo, kept at hi
            const uint32_t mid = lo + (hi - lo) / 2;
            if (sc > dec_score_threshold(f32_from_order_bits(mid), qsq[q], qab[q])) lo = mid;
            else hi = mid;
        }
        v[i] = f32_from_order_bits(hi);
    }
}

struct PqDecQueries {
    DevBuf q16, qsq, qd, qb, qab, qt;
};

static void launch_dec(int mode, const vdb_pq* pq, const PqDecQueries& Q, uint32_t nq, const uint8_t* codes, uint64_t n,
                       const float* row_r, const float* row_xn, PqDecParams p, cudaStream_t st) {
    const CUtensorMap map = make_map_f16(Q.q16.p, pq->dim, nq, (uint64_t)pq->dim * 2, DN);
    p.codes = codes;
    p.n = n;
    p.enc = pq->enc;
    p.m = pq->m;
    p.kblocks = pq->m / 16;
    p.nq = nq;
    p.cb16 = reinterpret_cast<const uint2*>(pq->d_dec_cb16);
    p.row_r = row_r;
    p.row_xn = row_xn;
    p.qd = Q.qd.as<float>();
    p.qb = Q.qb.as<float>();
    p.qt = Q.qt.as<float>();
    p.nqt = ceil_div(nq, (uint32_t)DN);
    const uint32_t units = (uint32_t)sm_count();
    const uint64_t row_tiles = ceil_div<uint64_t>(n, DM);
    p.tiles_per_item = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(8, row_tiles * p.nqt / ((uint64_t)units * 4)));
    p.nrow_items = (uint32_t)ceil_div<uint64_t>(row_tiles, p.tiles_per_item);
    const size_t smem = dec_smem_bytes(pq->m);
    const uint32_t grid = std::min<uint32_t>(units, p.nrow_items * p.nqt);
    ProfScope prof("pq_gemm", st);
    if (mode == 0) {
        static std::atomic<size_t> configured[VDB_MAX_DEVICES];
        ensure_dyn_smem(pq_dec_kernel<0>, dec_smem_bytes(D_MAX_M), configured);
        pq_dec_kernel<0><<<grid, D_THREADS, smem, st>>>(map, p);
    } else if (mode == 2) {
        static std::atomic<size_t> configured[VDB_MAX_DEVICES];
        ensure_dyn_smem(pq_dec_kernel<2>, dec_smem_bytes(D_MAX_M), configured);
        pq_dec_kernel<2><<<grid, D_THREADS, smem, st>>>(map, p);
    } else {
        static std::atomic<size_t> configured[VDB_MAX_DEVICES];
        ensure_dyn_smem(pq_dec_kernel<1>, dec_smem_bytes(D_MAX_M), configured);
        pq_dec_kernel<1><<<grid, D_THREADS, smem, st>>>(map, p);
    }
    VDB_LAUNCHED();
}

// query context of one batch (opaque to pq.cu)
void* pq_dec_begin(const vdb_pq* pq, const void* d_queries, uint32_t nq, cudaStream_t st) {
    ensure_dec_side(pq, st);
    if (!pq->dec_ok) return nullptr;
    auto Q = new PqDecQueries();
    try {
        Q->q16 = DevBuf((size_t)nq * pq->dim * 2, st);
        for (DevBuf* b : {&Q->qsq, &Q->qd, &Q->qb, &Q->qab, &Q->qt}) *b = DevBuf((size_t)nq * 4, st);
        const float acc = (float)pq->dim * ldexpf(1.0f, -23);
        const uint32_t grid = ceil_div(nq, 8u);
        if (pq->dtype == VDB_F32)
            pq_dec_query_kernel<float><<<grid, 256, 0, st>>>((const float*)d_queries, nq, pq->dim, pq->dec_scale, pq->dec_ex, acc,
                                                             Q->q16.as<__half>(), Q->qsq.as<float>(), Q->qd.as<float>(),
                                                             Q->qb.as<float>(), Q->qab.as<float>());
        else
            pq_dec_query_kernel<uint8_t><<<grid, 256, 0, st>>>((const uint8_t*)d_queries, nq, pq->dim, pq->dec_scale, pq->dec_ex, acc,
                                                               Q->q16.as<__half>(), Q->qsq.as<float>(), Q->qd.as<float>(),
                                                               Q->qb.as<float>(), Q->qab.as<float>());
        VDB_LAUNCHED();
    } catch (...) {
        delete Q;
        throw;
    }
    return Q;
}
void pq_dec_end(void* ctx) { delete static_cast<PqDecQueries*>(ctx); }

// SAMPLE step: upper bounds of the ADC values of the sampled rows, [nq][sample_n]
void pq_dec_sample(const vdb_pq* pq, void* ctx, uint32_t nq, float* d_all, cudaStream_t st) {
    auto& Q = *static_cast<PqDecQueries*>(ctx);
    pq_dec_thresholds_kernel<<<ceil_div(nq, 256u), 256, 0, st>>>(nullptr, Q.qsq.as<float>(), Q.qab.as<float>(), nq, Q.qt.as<float>());
    VDB_LAUNCHED();
    PqDecParams p{};
    p.all_out = d_all;
    launch_dec(0, pq, Q, nq, pq->d_sample, pq->sample_n, pq->d_dec_sr, pq->d_dec_sxn, p, st);
}

// FILTER step: coarse candidates from the decoded contraction, then the exact re-evaluation of pq_gemm.cu: on return
// cnt[q] / cand[q][] hold exactly the rows with adc <= tau_q (as keys), or cnt[q] > cap when a list overflowed
void pq_dec_filter(const vdb_pq* pq, void* ctx, const float* d_lut, uint32_t nq, const float* d_tau, uint32_t id_base,
                   uint32_t* d_cnt, uint64_t* d_cand, uint32_t cap, cudaStream_t st) {
    auto& Q = *static_cast<PqDecQueries*>(ctx);
    const uint32_t ccap = 2 * cap;
    DevBuf ccnt((size_t)nq * 4, st), ccand((size_t)nq * ccap * 4, st);
    VDB_CUDA(cudaMemsetAsync(ccnt.p, 0, (size_t)nq * 4, st));
    pq_dec_thresholds_kernel<<<ceil_div(nq, 256u), 256, 0, st>>>(d_tau, Q.qsq.as<float>(), Q.qab.as<float>(), nq, Q.qt.as<float>());
    VDB_LAUNCHED();
    // one record per (row, 32-query chunk) with a passing score; at most one per candidate, so nq * ccap records hold
    // every case in which no list overflows
    const uint64_t rec_cap64 = std::min<uint64_t>((uint64_t)nq * ccap, 1ull << 28);
    const uint32_t rec_cap = (uint32_t)rec_cap64;
    DevBuf rec((size_t)rec_cap * 8, st), rec_mask((size_t)rec_cap * 4, st), rec_count(4, st);
    VDB_CUDA(cudaMemsetAsync(rec_count.p, 0, 4, st));
    PqDecParams p{};
    p.ccnt = ccnt.as<uint32_t>();
    p.ccand = ccand.as<uint32_t>();
    p.ccap = ccap;
    p.rec = rec.as<uint64_t>();
    p.rec_mask = rec_mask.as<uint32_t>();
    p.rec_count = rec_count.as<uint32_t>();
    p.rec_cap = rec_cap;
    launch_dec(1, pq, Q, nq, pq->d_codes, pq->n, pq->d_dec_r, pq->d_dec_xn, p, st);
    pq_dec_expand_kernel<<<(uint32_t)sm_count() * 8, 256, 0, st>>>(rec.as<uint64_t>(), rec_mask.as<uint32_t>(), rec_count.as<uint32_t>(),
                                                                  rec_cap, nq, ccnt.as<uint32_t>(), ccand.as<uint32_t>(), ccap);
    VDB_LAUNCHED();
    pq_exact_candidates(pq, d_lut, d_tau, nq, ccnt.as<uint32_t>(), ccand.as<uint32_t>(), ccap, id_base, d_cnt, d_cand, cap, st);
}

// test hook: the filter's lower bound (pq_dec_lower_kernel) and the sample pass's upper bound of the ADC value of every
// (query, row) of the table, [nq][n] each, from the same kernel and coefficients as pq_dec_filter / pq_dec_sample
void pq_dec_bounds(const vdb_pq* pq, const void* d_queries, uint32_t nq, float* d_lower, float* d_upper, cudaStream_t st) {
    VDB_REQUIRE(pq_dec_supported(pq, UINT32_MAX), "decoded PQ contraction: unsupported table");
    const std::unique_ptr<PqDecQueries> ctx(static_cast<PqDecQueries*>(pq_dec_begin(pq, d_queries, nq, st)));
    VDB_REQUIRE(ctx, "decoded PQ contraction: codebooks not representable in FP16");
    auto& Q = *ctx;
    pq_dec_thresholds_kernel<<<ceil_div(nq, 256u), 256, 0, st>>>(nullptr, Q.qsq.as<float>(), Q.qab.as<float>(), nq, Q.qt.as<float>());
    VDB_LAUNCHED();
    PqDecParams p{};
    p.all_out = d_upper;
    launch_dec(0, pq, Q, nq, pq->d_codes, pq->n, pq->d_dec_r, pq->d_dec_xn, p, st);
    p.all_out = d_lower;
    launch_dec(2, pq, Q, nq, pq->d_codes, pq->n, pq->d_dec_r, pq->d_dec_xn, p, st);
    pq_dec_lower_kernel<<<(uint32_t)sm_count() * 8, 256, 0, st>>>(d_lower, nq, pq->n, Q.qsq.as<float>(), Q.qab.as<float>());
    VDB_LAUNCHED();
    VDB_CUDA(cudaStreamSynchronize(st));
}

}  // namespace vdb
