// flat_gemm.cu — K2: batched Flat L2 kNN as a tensor-core contraction + exact FP32 rerank.
//
// Replaces FlatIndex::knn (reference src/index_algorithm/flat_index.rs:48-57) for large query batches
// (the additive batch entry; the reference batches with rayon, examples/bench.rs:414-418).
//
// Pipeline (all on the caller's stream):
//   1. side arrays per dataset: ||x||^2 and ||x|| (fp32), built once and cached on the handle
//   2. SAMPLE pass  : S' over a strided row sample, per query the j-th smallest S' becomes tau_q
//   3. FILTER pass  : for every (query, row): S' = ||x||^2 - 2 q~.x~ - b(q, x)  (a LOWER bound of d(q,x) - ||q||^2:
//                     q~, x~ are the operands the tensor core consumes - FP16 copies scaled by exact powers of two,
//                     or the fp32 values truncated to TF32 by the hardware - and
//                     b = 2 (||q~|| ||x - x~|| + ||q - q~|| ||x~|| + dim 2^-23 ||q~|| ||x~||) uses the EXACT per-row /
//                     per-query operand errors ||x - x~||, ||q - q~|| (Cauchy-Schwarz), not a worst-case constant);
//                     rows with S' < tau_q are appended to the query's candidate list
//   4. RERANK       : exact difference-form distances of the candidates (pairs.cu), top-k by (d, id)
//   5. CHECK        : the candidate set is provably complete iff  d_k - ||q||^2 < tau_q  (every excluded
//                     row has d - ||q||^2 >= S' >= tau_q); queries that fail (or overflowed their list)
//                     are re-run through the exact streaming scan (K1) — still on the GPU.
// Results are therefore identical to the exact scan: the tensor cores only PRUNE.
//
// The contraction kernel is hand-written for sm_100a: TMA (cp.async.bulk.tensor, 128B swizzle) feeds a
// 4-stage shared-memory ring, one elected thread issues tcgen05.mma.kind::tf32 (M=128 queries x N=256 rows,
// K=8 per instruction) into double-buffered TMEM accumulators, four epilogue warps read them back with
// tcgen05.ld (thread = query, registers = rows) and apply the per-query threshold in registers.
#include <cuda.h>
#include <cuda_fp16.h>

#include <cmath>
#include <cstdlib>
#include <algorithm>
#include <mutex>
#include <vector>

#include "index.cuh"
#include "tc.cuh"
#include "topk.cuh"

namespace vdb {

// ---- tile configuration ---------------------------------------------------------------------------------
constexpr int GM = 128;              // queries per tile (TMEM lanes)
constexpr int GN = 256;              // database rows per tile (TMEM columns per accumulator)
constexpr int GKB = 128;             // bytes of one operand row per k-block = one 128-byte swizzle row
constexpr int G_A_BYTES = GM * GKB;  // 16 KB: 128 queries x 128 B
// operand kinds of the contraction. FP16 has TF32's 10 mantissa bits at twice the tensor rate and half the operand
// bytes; its 5-bit exponent is handled by exact power-of-two scales per dataset / per query, and whatever the
// conversion loses (underflow included) is measured per row and folded into the pruning bound.
enum { KIND_TF32 = 0, KIND_F16 = 1 };
template <int KIND> struct KindCfg {
    static constexpr int ELEM = KIND == KIND_F16 ? 2 : 4;       // bytes per operand element
    static constexpr int GKE = GKB / ELEM;                      // elements per k-block: 32 (tf32) / 64 (f16)
    static constexpr uint32_t FMT = KIND == KIND_F16 ? 0u : 2u;  // UMMA a/b format: F16 = 0, TF32 = 2
};
// filter (mode 1): passing scores are staged per epilogue warp in shared memory (list owner + key) and their list slots
// reserved by ALL lanes at once when the buffer fills, so the ~700-cycle atomic round trip is paid once per G_STG_CAP
// candidates instead of once per 32-score chunk with a hit
constexpr int G_STG_CAP = 256;
constexpr int G_THREADS = 192;       // warps 0-3 epilogue, warp 4 TMA producer, warp 5 MMA issuer
constexpr int G_TMEM_COLS = 512;     // 2 accumulators x 256 columns
constexpr int G_MAX_STAGES = 6;
// CTAS = 1: one CTA computes a 128 x 256 tile. CTAS = 2: a CTA pair (cta_group::2) computes 256 x 256, each CTA
// loads its own 128 queries and HALF of the 256 database rows, so the shared-memory fill per MMA cycle drops 1.5x.
template <int CTAS, int KIND = KIND_TF32> struct GemmCfg {
    static constexpr int B_ROWS = GN / CTAS;                    // database rows loaded per CTA and k-block
    static constexpr int B_BYTES = B_ROWS * GKB;
    static constexpr int STAGE_BYTES = G_A_BYTES + B_BYTES;     // 48 KB / 32 KB
    static constexpr int STAGES = CTAS == 1 ? 4 : 6;            // 192 KB either way
    static constexpr uint32_t SMEM = 1024 /*align*/ + STAGES * STAGE_BYTES + 2 * 3 * GN * 4 /*row-scalar tiles*/ + 512 /*barriers*/;
    static constexpr uint32_t SMEM_STAGED = SMEM + 4 * G_STG_CAP * 12;   // + candidate staging of the 4 epilogue warps
    // instruction descriptor (cute::UMMA::InstrDescriptor): D=F32, A=B=TF32 or F16, both K-major, N>>3, M>>4
    static constexpr uint32_t IDESC = (1u << 4) | (KindCfg<KIND>::FMT << 7) | (KindCfg<KIND>::FMT << 10) |
                                      ((uint32_t)(GN >> 3) << 17) | ((uint32_t)((GM * CTAS) >> 4) << 24);
};
constexpr uint32_t G_SAMPLE = 32768;  // sampled rows for the thresholds
constexpr int G_TOPJ = 16;             // order statistics kept in registers by the sample pass (mode 2)
constexpr int G_ITEMQ = 4;              // depth of the dynamic-scheduler item queue
constexpr uint32_t G_NO_ITEM = 0xFFFFFFFFu;
constexpr uint32_t PEER_MASK = 0xFEFFFFFFu;  // clears the CTA-pair peer bit of a shared::cluster address (-> even CTA)

// ---- kernel ----------------------------------------------------------------------------------------------------
// one unit of work: query rows [q0, q_end) (at most GM * CTAS of them) against database rows [r0, r_end)
struct GemmItem {
    uint32_t q0, q_end;
    uint64_t r0, r_end;
};
struct ItemView {
    uint32_t q0, q_end, ntile, slab;
    uint64_t r0, r_end;
};

struct GemmParams {
    uint32_t nq;            // queries
    uint64_t nrows;         // rows addressed by the B tensor map (sample rows or all rows)
    uint32_t row_stride;    // database row of B row i is i * row_stride
    uint32_t kblocks;       // ceil(dim / elements per k-block)
    uint32_t ntiles;        // ceil(nrows / GN)
    uint32_t nqt;           // query-tile UNITS: ceil(nq / (GM * CTAS))
    uint32_t tiles_per_slab;
    uint32_t nslabs;        // slabs covered by this launch
    uint32_t slab0;         // first slab of this launch (the filter pass may be cut into row parts)
    // S' = sqnorm[x] + qd[q] * acc - qab[q] * ex[x] - qb[q] * rnorm[x]                       (L2Sqr)
    // S' = qb[q] - (qd[q] * sqnorm[x]) * acc - qab[q] * ex[x]                                (cosine)
    const float* sqnorm;    // [n] L2Sqr: ||x||^2;  cosine: 1 / ||x|| (0 for zero rows)
    const float* rnorm;     // [n] ||x||
    const float* ex;        // [n] L2Sqr: ||x - x~||;  cosine: ||x - x~|| / ||x||   (x~ = the operand the MMA consumes)
    const float* qd;        // [nq] L2Sqr: -2 / (s_q s_x);  cosine: 1 / (s_q s_x ||q||)   (s = power-of-two operand scales)
    const float* qab;       // [nq] coefficient of ex
    const float* qb;        // [nq] L2Sqr: coefficient of ||x||;  cosine: 1 - (query-side share of the error bound)
    const float* qnorm;     // [nq] cosine: ||q||
    // mode 0: store keys (S', sample index) to out_keys[nq][nrows]
    // mode 2: per (query, slab) the G_TOPJ smallest S' as keys to out_keys[nq][nslabs][G_TOPJ]
    uint64_t* out_keys;
    // mode 1: filter
    const float* tau;       // [nq]
    uint32_t* cand_cnt;     // [nq]
    uint64_t* cand;         // [nq][cap]  (S' bits << 32 | local row)
    uint32_t cap;
    uint32_t* work_counter; // dynamic item scheduler (zeroed before the launch)
    // table mode (IVF: one rectangular block per (list, query group)): explicit items instead of the slab x unit grid
    const GemmItem* items;  // nullptr -> the grid of plan_gemm
    uint32_t nitems;
    const uint32_t* qmap;   // table mode: row of the gathered query matrix -> query that owns the candidate list
    uint32_t rare_per_score;  // filter's rare path: 0 one atomic per thread and 32-score chunk, 1 one per score, 2 staged per warp
};

template <int CTAS>
__device__ __forceinline__ ItemView decode_item(const GemmParams& p, uint32_t item) {
    ItemView v;
    if (p.items) {
        const GemmItem it = p.items[item];
        v.q0 = it.q0;
        v.q_end = it.q_end;
        v.r0 = it.r0;
        v.r_end = it.r_end;
        v.slab = 0;  // mode 2: every gathered query row belongs to exactly one item
    } else {
        const uint32_t sl = item / p.nqt;
        v.slab = p.slab0 + sl;
        v.q0 = (item - sl * p.nqt) * GM * CTAS;
        v.q_end = p.nq;
        v.r0 = (uint64_t)v.slab * p.tiles_per_slab * GN;
        v.r_end = min(p.nrows, v.r0 + (uint64_t)p.tiles_per_slab * GN);
    }
    v.ntile = (uint32_t)((v.r_end - v.r0 + GN - 1) / GN);
    return v;
}

// STAGED (filter only): passing scores go through the per-warp staging buffer (G_STG_CAP). A separate instantiation: as
// a run-time switch inside the one kernel it cost the sparse full pass ~7 % (194 instead of 168 registers, 12 % more
// executed instructions, tensor pipe 73 -> 66 %: round-2 re-capture), so the full pass keeps its own code.
template <int MODE, int CTAS, int METRIC, int KIND, bool STAGED = false>
__global__ void __launch_bounds__(G_THREADS, 1)
flat_gemm_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_x, const GemmParams p) {
    using Cfg = GemmCfg<CTAS, KIND>;
    constexpr int GKE = KindCfg<KIND>::GKE;
    constexpr int STAGES = Cfg::STAGES;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t* stage_base = smem;
    float* norm_tiles = reinterpret_cast<float*>(smem + STAGES * Cfg::STAGE_BYTES);  // [2 acc][3 arrays][GN]
    uint64_t* bars = reinterpret_cast<uint64_t*>(norm_tiles + 2 * 3 * GN);
    uint64_t* full_bar = bars;                       // [STAGES]  (pair mode: the leader's copy is the live one)
    uint64_t* empty_bar = bars + G_MAX_STAGES;       // [STAGES]  per CTA
    uint64_t* tfull_bar = bars + 2 * G_MAX_STAGES;   // [2]       per CTA
    uint64_t* tempty_bar = tfull_bar + 2;            // [2]       (pair mode: the leader's copy is the live one)
    uint64_t* iq_full = tempty_bar + 2;              // [G_ITEMQ] per CTA: an item id has been published
    uint64_t* iq_empty = iq_full + G_ITEMQ;          // [G_ITEMQ] (leader's copy is live): every reader took it
    uint32_t* item_ring = reinterpret_cast<uint32_t*>(iq_empty + G_ITEMQ);  // [G_ITEMQ]
    uint32_t* tmem_slot = item_ring + G_ITEMQ;
    uint8_t* stg_base = reinterpret_cast<uint8_t*>(bars) + 512;   // [4 warps][G_STG_CAP] keys (8 B), then owners (4 B)

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t cta_rank = CTAS == 2 ? cluster_ctarank() : 0u;
    const bool leader = cta_rank == 0;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&tfull_bar[a], 1);
            mbar_init(&tempty_bar[a], 4 * CTAS);  // one arrive per epilogue warp of every CTA in the group
        }
        for (int i = 0; i < G_ITEMQ; ++i) {
            mbar_init(&iq_full[i], 1);
            // readers of a published item: MMA thread + 4 epilogue warps (+ the peer's producer and 4 epilogue warps)
            mbar_init(&iq_empty[i], CTAS == 1 ? 5 : 10);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 5) {
        if (CTAS == 2) tmem_alloc2(tmem_slot, G_TMEM_COLS);
        else tmem_alloc(tmem_slot, G_TMEM_COLS);
    }
    tc_fence_before();
    __syncthreads();
    if (CTAS == 2) cluster_sync_all();  // the peer's barriers are initialised before any remote arrive / TMA
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    const uint32_t items = p.items ? p.nitems : p.nqt * p.nslabs;
    // ---- dynamic scheduler: the leader's producer draws item ids from a global counter and publishes them to
    // every role of the CTA (pair) through a small shared-memory queue. Items are taken in global order, so the
    // CTAs in flight always work on neighbouring slabs (shared in L2) no matter how their speeds drift apart.
    const uint32_t leader_empty_base = CTAS == 2 ? mapa_cluster(smem_u32(iq_empty), 0) : smem_u32(iq_empty);
    auto take_item = [&](uint32_t n) -> uint32_t {  // called by ONE thread of a reader role, n = 0, 1, 2, ...
        const uint32_t slot = n % G_ITEMQ, ph = (n / G_ITEMQ) & 1;
        if (CTAS == 2) mbar_wait_cluster(&iq_full[slot], ph);
        else mbar_wait(&iq_full[slot], ph);
        const uint32_t item = ((volatile uint32_t*)item_ring)[slot];
        if (CTAS == 2) mbar_arrive_cluster_release(leader_empty_base + slot * 8);
        else mbar_arrive(&iq_empty[slot]);
        return item;
    };

    if (warp == 4) {
        // ===== TMA producer (every CTA loads its own queries and its share of the database rows) =====
        if (lane == 0) {
            uint32_t stage = 0, phase = 0;
            for (uint32_t n = 0;; ++n) {
                uint32_t item;
                if (leader) {
                    const uint32_t slot = n % G_ITEMQ, ph = (n / G_ITEMQ) & 1;
                    mbar_wait_cluster(&iq_empty[slot], ph ^ 1);
                    item = atomicAdd(p.work_counter, 1u);
                    if (item >= items) item = G_NO_ITEM;
                    item_ring[slot] = item;
                    mbar_arrive(&iq_full[slot]);
                    if (CTAS == 2) {
                        st_cluster_u32(mapa_cluster(smem_u32(&item_ring[slot]), 1), item);
                        mbar_arrive_cluster_release(mapa_cluster(smem_u32(&iq_full[slot]), 1));
                    }
                } else {
                    item = take_item(n);
                }
                if (item == G_NO_ITEM) break;
                const ItemView iv = decode_item<CTAS>(p, item);
                const int qrow = (int)(iv.q0 + cta_rank * GM);
                for (uint32_t t = 0; t < iv.ntile; ++t) {
                    const int brow = (int)(iv.r0 + (uint64_t)t * GN + cta_rank * Cfg::B_ROWS);
                    for (uint32_t kb = 0; kb < p.kblocks; ++kb) {
                        mbar_wait(&empty_bar[stage], phase ^ 1);
                        const uint32_t sa = smem_u32(stage_base + stage * Cfg::STAGE_BYTES);
                        if (CTAS == 1) {
                            mbar_expect_tx(&full_bar[stage], Cfg::STAGE_BYTES);
                            tma_load_2d(sa, &map_q, (int)(kb * GKE), qrow, &full_bar[stage]);
                            tma_load_2d(sa + G_A_BYTES, &map_x, (int)(kb * GKE), brow, &full_bar[stage]);
                        } else {
                            // both CTAs' bytes are accounted on the LEADER's barrier
                            if (leader) mbar_expect_tx(&full_bar[stage], Cfg::STAGE_BYTES * CTAS);
                            const uint32_t lbar = smem_u32(&full_bar[stage]) & PEER_MASK;
                            tma_load_2d_2sm(sa, &map_q, (int)(kb * GKE), qrow, lbar);
                            tma_load_2d_2sm(sa + G_A_BYTES, &map_x, (int)(kb * GKE), brow, lbar);
                        }
                        if (++stage == STAGES) stage = 0, phase ^= 1;
                    }
                }
            }
        }
    } else if (warp == 5) {
        // ===== MMA issuer (one elected thread of the leader CTA) =====
        if (lane == 0 && leader) {
            uint32_t stage = 0, phase = 0, acc = 0, acc_phase = 0;
            for (uint32_t n = 0;; ++n) {
                const uint32_t item = take_item(n);
                if (item == G_NO_ITEM) break;
                const ItemView iv = decode_item<CTAS>(p, item);
                for (uint32_t t = 0; t < iv.ntile; ++t) {
                    mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
                    tc_fence_after();
                    const uint32_t d_tmem = tmem_base + acc * GN;
                    for (uint32_t kb = 0; kb < p.kblocks; ++kb) {
                        mbar_wait(&full_bar[stage], phase);
                        tc_fence_after();
                        const uint32_t sa = smem_u32(stage_base + stage * Cfg::STAGE_BYTES);
                        const uint64_t da = umma_desc(sa), db = umma_desc(sa + G_A_BYTES);
#pragma unroll
                        for (int k = 0; k < GKB / 32; ++k) {  // one MMA consumes 32 bytes of K (8 tf32 / 16 f16): 2 x 16B units
                            if (KIND == KIND_F16) {
                                if (CTAS == 1) umma_f16(d_tmem, da + 2 * k, db + 2 * k, Cfg::IDESC, (kb | k) != 0);
                                else umma_f16_2sm(d_tmem, da + 2 * k, db + 2 * k, Cfg::IDESC, (kb | k) != 0);
                            } else {
                                if (CTAS == 1) umma_tf32(d_tmem, da + 2 * k, db + 2 * k, Cfg::IDESC, (kb | k) != 0);
                                else umma_tf32_2sm(d_tmem, da + 2 * k, db + 2 * k, Cfg::IDESC, (kb | k) != 0);
                            }
                        }
                        // frees the smem stage (in both CTAs) when these MMAs retire
                        if (CTAS == 1) umma_commit(&empty_bar[stage]);
                        else umma_commit_2sm(&empty_bar[stage]);
                        if (++stage == STAGES) stage = 0, phase ^= 1;
                    }
                    // accumulator ready for the epilogue warps (of both CTAs)
                    if (CTAS == 1) umma_commit(&tfull_bar[acc]);
                    else umma_commit_2sm(&tfull_bar[acc]);
                    if (++acc == 2) acc = 0, acc_phase ^= 1;
                }
            }
        }
    } else {
        // ===== epilogue: warps 0-3, thread = query (TMEM lane), registers = database rows =====
        uint32_t acc = 0, acc_phase = 0;
        const uint32_t lane_base = (uint32_t)warp * 32;
        // (dead code unless STAGED: the flush lambda and the buffer pointers are only used by that instantiation)
        uint64_t* stg_key = reinterpret_cast<uint64_t*>(stg_base) + warp * G_STG_CAP;
        uint32_t* stg_own = reinterpret_cast<uint32_t*>(stg_base + 4 * G_STG_CAP * 8) + warp * G_STG_CAP;
        uint32_t stg_fill = 0;   // warp-uniform
        auto stg_flush = [&]() {
            __syncwarp();
            uint32_t pos[G_STG_CAP / 32];
#pragma unroll
            for (int u = 0; u < G_STG_CAP / 32; ++u) {   // every round trip of the buffer is in flight at once
                const uint32_t e = u * 32 + lane;
                pos[u] = e < stg_fill ? atomicAdd(&p.cand_cnt[stg_own[e]], 1u) : 0xffffffffu;
            }
#pragma unroll
            for (int u = 0; u < G_STG_CAP / 32; ++u) {
                const uint32_t e = u * 32 + lane;
                if (e < stg_fill && pos[u] < p.cap) p.cand[(uint64_t)stg_own[e] * p.cap + pos[u]] = stg_key[e];
            }
            __syncwarp();
            stg_fill = 0;
        };
        for (uint32_t n = 0;; ++n) {
            uint32_t item = 0;
            if (lane == 0) item = take_item(n);
            item = __shfl_sync(0xffffffffu, item, 0);
            if (item == G_NO_ITEM) break;
            const ItemView iv = decode_item<CTAS>(p, item);
            const uint32_t slab = iv.slab;
            const uint32_t q = iv.q0 + cta_rank * GM + threadIdx.x;   // row of the (gathered) query matrix
            const bool qok = q < iv.q_end;
            const uint32_t oq = (qok && p.qmap) ? p.qmap[q] : q;        // query that owns the candidate list
            const float qd = qok ? p.qd[q] : 0.f, qab = qok ? p.qab[q] : 0.f, qb = qok ? p.qb[q] : 0.f;
            const float qn = (METRIC == VDB_COSINE && qok) ? p.qnorm[q] : 0.f;
            float tau = 0.f;
            if (MODE == 1) tau = qok ? p.tau[q] : __uint_as_float(0xff800000u);  // -inf: nothing passes
            float best[MODE == 2 ? G_TOPJ : 1];     // mode 2: this query's smallest scores of the slab, ascending,
            uint32_t bidx[MODE == 2 ? G_TOPJ : 1];  // and the rows (of the B tensor) they belong to
            if (MODE == 2) {
#pragma unroll
                for (int i = 0; i < (MODE == 2 ? G_TOPJ : 1); ++i) best[i] = __uint_as_float(0x7f800000u), bidx[i] = 0xffffffffu;
            }
            // Row scalars of a tile (3 x GN floats: two rows per thread and array). The loads of tile t + 1 are issued
            // before tile t is scored and stored to the other buffer after it, so their latency hides under the
            // scoring loop; only an item's first tile pays it.
            float pre[6];
            auto load_scalars = [&](uint32_t t) {
                const uint64_t tile_row0 = iv.r0 + (uint64_t)t * GN;
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const uint64_t brow = tile_row0 + threadIdx.x + h * 128;
                    const bool ok = brow < iv.r_end;
                    const uint64_t row = brow * p.row_stride;
                    if (METRIC == VDB_L2SQR) {
                        pre[h * 3 + 0] = ok ? p.sqnorm[row] : __uint_as_float(0x7f800000u);  // +inf: never a candidate
                        pre[h * 3 + 1] = ok ? p.rnorm[row] : 0.f;
                        pre[h * 3 + 2] = ok ? p.ex[row] : 0.f;
                    } else {   // padding: S' = qb - 0 * acc - qab * (-inf) = +inf, and never under the norm clamp
                        pre[h * 3 + 0] = ok ? p.sqnorm[row] : 0.f;
                        pre[h * 3 + 1] = ok ? p.rnorm[row] : __uint_as_float(0x7f800000u);
                        pre[h * 3 + 2] = ok ? p.ex[row] : __uint_as_float(0xff800000u);
                    }
                }
            };
            auto store_scalars = [&](uint32_t buf) {
                const uint32_t base = smem_u32(norm_tiles + buf * 3 * GN) + threadIdx.x * 4;
#pragma unroll
                for (int h = 0; h < 2; ++h)
#pragma unroll
                    for (int a = 0; a < 3; ++a) sts_f32(base + (a * GN + h * 128) * 4, pre[h * 3 + a]);
            };
            load_scalars(0);
            store_scalars(acc);
            for (uint32_t t = 0; t < iv.ntile; ++t) {
                const uint64_t tile_row0 = iv.r0 + (uint64_t)t * GN;
                asm volatile("bar.sync 1, 128;" ::: "memory");   // every warp has stored this tile's scalars and left tile t - 1
                const bool more = t + 1 < iv.ntile;
                if (more) load_scalars(t + 1);
                mbar_wait(&tfull_bar[acc], acc_phase);
                tc_fence_after();
                const uint32_t taddr = tmem_base + (lane_base << 16) + acc * GN;
                // the row scalars are read with 128-bit SHARED loads (every lane reads the same address: one broadcast
                // wavefront per 4 rows and array). Reading them through generic pointers costs a generic-space LD per
                // row and array, which made this loop - not the MMAs - the bound of the whole kernel.
                const uint32_t sq_s = smem_u32(norm_tiles + acc * 3 * GN), rn_s = sq_s + GN * 4, ex_s = rn_s + GN * 4;
                // cosine: a row is under the reference's 1e-10 norm-product clamp iff ||x|| < 2e-10 / ||q|| (always kept)
                const float rthr = METRIC == VDB_COSINE ? (qn > 0.f ? 2e-10f / qn : __uint_as_float(0x7f800000u)) : 0.f;
                uint32_t va[32], vb[32];
                tmem_ld32_issue(taddr, va);
                tmem_ld_wait(va);
                // scores of the 32 columns in v[]: 3 FMAs + one predicate-chained compare per score, a flag per group of 8
                auto score = [&](uint32_t (&v)[32], int c0) {
                    constexpr bool staged = MODE == 1 && STAGED;   // every lane of the warp takes part
                    if (!qok && !staged) return;
                    const float thr = MODE == 1 ? tau : (MODE == 2 ? best[MODE == 2 ? G_TOPJ - 1 : 0] : 0.f);
                    bool none[4] = {true, true, true, true};
#pragma unroll
                    for (int j4 = 0; j4 < 32; j4 += 4) {
                        const float4 sq4 = lds_f4(sq_s + (c0 + j4) * 4), rn4 = lds_f4(rn_s + (c0 + j4) * 4),
                                     ex4 = lds_f4(ex_s + (c0 + j4) * 4);
                        const float sqv[4] = {sq4.x, sq4.y, sq4.z, sq4.w}, rnv[4] = {rn4.x, rn4.y, rn4.z, rn4.w},
                                    exv[4] = {ex4.x, ex4.y, ex4.z, ex4.w};
#pragma unroll
                        for (int jj = 0; jj < 4; ++jj) {
                            const int j = j4 + jj;
                            const float dot = __uint_as_float(v[j]);
                            float sc;
                            if (METRIC == VDB_L2SQR) {
                                // S' = ||x||^2 - 2 q~.x~ / (s_q s_x) - b(q, x)   (lower bound of d - ||q||^2)
                                sc = fmaf(qd, dot, fmaf(-qab, exv[jj], fmaf(-qb, rnv[jj], sqv[jj])));
                            } else {
                                // S' = (1 - bound) - q~.x~ / (s_q s_x ||q|| ||x||)  (lower bound of the cosine distance;
                                // sq = 1/||x||). Padding rows are staged with ex = -inf: S' = +inf.
                                sc = fmaf(-(qd * sqv[jj]), dot, fmaf(-qab, exv[jj], qb));
                                if (rnv[jj] < rthr) sc = __uint_as_float(0xff800000u);
                            }
                            v[j] = __float_as_uint(sc);
                            if (MODE != 0) none[j >> 3] = none[j >> 3] && (sc >= thr);   // a NaN score fails the test
                        }
                    }
                    if (MODE == 0) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            const uint64_t brow = tile_row0 + c0 + j;
                            if (brow < iv.r_end) p.out_keys[(uint64_t)q * p.nrows + brow] = make_key(__uint_as_float(v[j]), (uint32_t)brow);
                        }
                    } else if constexpr (staged) {
                        const bool mine = qok && !(none[0] && none[1] && none[2] && none[3]);
                        if (__any_sync(0xffffffffu, mine)) {
                            uint32_t pass = 0;
                            if (mine) {
#pragma unroll
                                for (int g = 0; g < 4; ++g) {
                                    if (none[g]) continue;
#pragma unroll
                                    for (int j = g * 8; j < g * 8 + 8; ++j) pass |= (__uint_as_float(v[j]) >= tau ? 0u : 1u) << j;
                                }
                            }
                            const uint32_t cnt = (uint32_t)__popc(pass);
                            uint32_t inc = cnt;
#pragma unroll
                            for (int d = 1; d < 32; d <<= 1) {
                                const uint32_t up = __shfl_up_sync(0xffffffffu, inc, d);
                                if (lane >= d) inc += up;
                            }
                            const uint32_t total = __shfl_sync(0xffffffffu, inc, 31);
                            if (total) {
                                if (stg_fill + total > (uint32_t)G_STG_CAP) stg_flush();
                                if (total > (uint32_t)G_STG_CAP) {
                                    // denser than the buffer (a threshold of +inf): slots reserved per thread
                                    if (pass) {
                                        uint32_t pos = atomicAdd(&p.cand_cnt[oq], cnt);
                                        uint64_t* list = p.cand + (uint64_t)oq * p.cap;
#pragma unroll
                                        for (int j = 0; j < 32; ++j) {
                                            if ((pass >> j) & 1u) {
                                                if (pos < p.cap) list[pos] = ((uint64_t)v[j] << 32) | (uint32_t)(tile_row0 + c0 + j);
                                                ++pos;
                                            }
                                        }
                                    }
                                } else {
                                    uint32_t e = stg_fill + inc - cnt;
#pragma unroll
                                    for (int g = 0; g < 4; ++g) {
                                        if (((pass >> (g * 8)) & 0xffu) == 0u) continue;
#pragma unroll
                                        for (int j = g * 8; j < g * 8 + 8; ++j) {
                                            if ((pass >> j) & 1u) {
                                                stg_key[e] = ((uint64_t)v[j] << 32) | (uint32_t)(tile_row0 + c0 + j);
                                                stg_own[e] = oq;
                                                ++e;
                                            }
                                        }
                                    }
                                    stg_fill += total;
                                }
                            }
                        }
                    } else if (MODE == 1 && !p.rare_per_score && !(none[0] && none[1] && none[2] && none[3])) {
                        // rare path of the filter: the passing (or NaN: the exact rerank decides) scores of the flagged groups
                        // of 8 are collected in a bit mask and the thread reserves all their list slots with ONE atomic. (One
                        // atomic per score serialises its ~700-cycle round trips in divergent code: the sample pass of the
                        // two-level selection, where 0.6 % of the scores pass, ran at a third of the MMA rate.)
                        uint32_t pass = 0;
#pragma unroll
                        for (int g = 0; g < 4; ++g) {
                            if (none[g]) continue;
#pragma unroll
                            for (int j = g * 8; j < g * 8 + 8; ++j) pass |= (__uint_as_float(v[j]) >= tau ? 0u : 1u) << j;
                        }
                        if (pass) {
                            uint32_t pos = atomicAdd(&p.cand_cnt[oq], (uint32_t)__popc(pass));
                            uint64_t* list = p.cand + (uint64_t)oq * p.cap;
#pragma unroll
                            for (int j = 0; j < 32; ++j) {
                                if ((pass >> j) & 1u) {
                                    if (pos < p.cap) list[pos] = ((uint64_t)v[j] << 32) | (uint32_t)(tile_row0 + c0 + j);
                                    ++pos;
                                }
                            }
                        }
                    } else if (MODE == 2 && !(none[0] && none[1] && none[2] && none[3])) {
                        // Top-G_TOPJ epilogue: the flagged scores go to this thread's private row of a shared-memory scratch and
                        // are inserted from there in column order. Walking the 32 columns in unrolled code made the WARP pay an
                        // insertion chain for every column in which ANY lane had a new best (nearly every row of a tile's first
                        // slabs); the per-thread loop makes it pay max-over-lanes(insertions) chains per chunk instead.
                        float* row = reinterpret_cast<float*>(stg_base) + threadIdx.x * 33;
                        const float last = best[MODE == 2 ? G_TOPJ - 1 : 0];
                        uint32_t mask = 0;
#pragma unroll
                        for (int g = 0; g < 4; ++g) {
                            if (none[g]) continue;
#pragma unroll
                            for (int j = g * 8; j < g * 8 + 8; ++j) {
                                const float sc = __uint_as_float(v[j]);
                                row[j] = sc;
                                mask |= (sc < last ? 1u : 0u) << j;
                            }
                        }
                        while (mask) {
                            const int j = __ffs(mask) - 1;
                            mask &= mask - 1;
                            const float sc = row[j];
                            if (sc < best[MODE == 2 ? G_TOPJ - 1 : 0]) {  // bubble (sc, row) into place
                                // (measured: computing the rank with 16 independent compares and rewriting the slots
                                // independently executes ~50 % more instructions and is 15-20 % SLOWER than this chain)
                                float w = sc;
                                uint32_t wi = (uint32_t)(tile_row0 + c0 + j);
#pragma unroll
                                for (int i = 0; i < (MODE == 2 ? G_TOPJ : 1); ++i) {
                                    const bool lt = w < best[i];
                                    const float lo = lt ? w : best[i], hi = lt ? best[i] : w;
                                    const uint32_t loi = lt ? wi : bidx[i], hii = lt ? bidx[i] : wi;
                                    best[i] = lo, bidx[i] = loi, w = hi, wi = hii;
                                }
                            }
                        }
                    } else if (MODE != 2 && !(none[0] && none[1] && none[2] && none[3])) {
                        // rare path: only the groups of 8 in which this thread saw a passing (or NaN) score are walked again
#pragma unroll
                        for (int g = 0; g < 4; ++g) {
                            if (none[g]) continue;
#pragma unroll
                            for (int j = g * 8; j < g * 8 + 8; ++j) {
                                const float sc = __uint_as_float(v[j]);
                                if (MODE == 2) {
                                    if (sc < best[MODE == 2 ? G_TOPJ - 1 : 0]) {  // bubble (sc, row) into place
                                        // (measured: computing the rank with 16 independent compares and rewriting the slots
                                        // independently executes ~50 % more instructions and is 15-20 % SLOWER than this chain)
                                        float w = sc;
                                        uint32_t wi = (uint32_t)(tile_row0 + c0 + j);
#pragma unroll
                                        for (int i = 0; i < (MODE == 2 ? G_TOPJ : 1); ++i) {
                                            const bool lt = w < best[i];
                                            const float lo = lt ? w : best[i], hi = lt ? best[i] : w;
                                            const uint32_t loi = lt ? wi : bidx[i], hii = lt ? bidx[i] : wi;
                                            best[i] = lo, bidx[i] = loi, w = hi, wi = hii;
                                        }
                                    }
                                } else if (!(sc >= tau)) {   // NaN scores (non-finite rows / queries) are kept: the exact rerank decides
                                    const uint32_t pos = atomicAdd(&p.cand_cnt[oq], 1u);
                                    if (pos < p.cap)
                                        p.cand[(uint64_t)oq * p.cap + pos] =
                                            ((uint64_t)__float_as_uint(sc) << 32) | (uint32_t)(tile_row0 + c0 + j);
                                }
                            }
                        }
                    }
                };
                // the TMEM load of chunk c + 1 is in flight while chunk c is scored
#pragma unroll 1
                for (int c0 = 0; c0 < GN; c0 += 64) {
                    tmem_ld32_issue(taddr + c0 + 32, vb);
                    score(va, c0);
                    tmem_ld_wait(vb);
                    if (c0 + 64 < GN) tmem_ld32_issue(taddr + c0 + 64, va);
                    score(vb, c0 + 32);
                    if (c0 + 64 < GN) tmem_ld_wait(va);
                }
                // hand the accumulator back to the MMA issuer: one arrive per warp, on the leader's barrier
                tc_fence_before();
                __syncwarp();
                if (lane == 0) {
                    if (CTAS == 1) mbar_arrive(&tempty_bar[acc]);
                    else mbar_arrive_cluster(smem_u32(&tempty_bar[acc]) & PEER_MASK);
                }
                if (more) store_scalars(acc ^ 1);
                if (++acc == 2) acc = 0, acc_phase ^= 1;
            }
            if (MODE == 2 && qok) {
#pragma unroll
                for (int i = 0; i < (MODE == 2 ? G_TOPJ : 1); ++i)
                    p.out_keys[((uint64_t)q * p.nslabs + slab) * G_TOPJ + i] =
                        bidx[i] == 0xffffffffu ? KEY_NONE : make_key(best[i], bidx[i]);
            }
        }
        if (MODE == 1 && STAGED && stg_fill) stg_flush();
    }
    tc_fence_before();
    __syncthreads();
    if (CTAS == 2) cluster_sync_all();  // neither CTA may exit (or free TMEM) while its peer still uses it
    if (warp == 5) {
        if (CTAS == 2) tmem_dealloc2(tmem_base, G_TMEM_COLS);
        else tmem_dealloc(tmem_base, G_TMEM_COLS);
    }
}

// ---- host side ------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) mean_kernel(const float* __restrict__ v, uint64_t n, uint64_t stride, float* out) {
    __shared__ float red[32];
    float s = 0.f;
    uint32_t cnt = 0;
    for (uint64_t i = (uint64_t)threadIdx.x * stride; i < n; i += (uint64_t)blockDim.x * stride) s += v[i], ++cnt;
    __shared__ uint32_t total;
    if (threadIdx.x == 0) total = 0;
    __syncthreads();
    atomicAdd(&total, cnt);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.f;
        for (int w = 0; w < 32; ++w) t += red[w];
        *out = t / (float)max(total, 1u);
    }
}

// ---- operand copies and per-row error norms ---------------------------------------------------------------------------
// One warp per row. FP16 kind: writes x~ = fp16(x * s_x) (s_x an exact power of two) and ||x - x~ / s_x||; TF32 kind: the
// hardware truncates the fp32 bits to TF32 itself (no copy), the error of THAT truncation is what is measured (a
// round-to-nearest unit would err less than truncation on every element, so the norm bounds it too). u8 rows are exact
// in FP16. Non-finite rows get sqnorm = -inf ("always a candidate": the exact rerank decides) and error 0.
// Norm sums follow row_cache's arithmetic (lane-strided fma chain + xor butterfly).
template <typename T, int KIND>
__global__ void __launch_bounds__(256) row_side_kernel(const T* __restrict__ rows, uint64_t n, uint32_t dim, uint32_t pitch,
                                                       float scale, uint32_t op_pitch, __half* __restrict__ op,
                                                       int cosine, float* __restrict__ colA, float* __restrict__ rn,
                                                       float* __restrict__ ex) {
    const uint64_t row = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (row >= n) return;
    const T* src = rows + row * pitch;
    const float inv_scale = 1.0f / scale;
    float ss = 0.f, ee = 0.f;
    bool finite = true;
    const uint32_t span = KIND == KIND_F16 ? op_pitch : dim;
    for (uint32_t e = lane; e < span; e += 32) {
        const float v = e < dim ? (float)src[e] : 0.f;
        float back;
        if (KIND == KIND_F16) {
            const __half h = __float2half_rn(v * scale);
            op[row * op_pitch + e] = h;
            back = __half2float(h) * inv_scale;
        } else {
            back = __uint_as_float(__float_as_uint(v) & 0xffffe000u);
        }
        finite = finite && (fabsf(v) <= 3.0e38f) && (fabsf(back) <= 3.0e38f);
        const float d = v - back;
        ss = fmaf(v, v, ss);
        ee = fmaf(d, d, ee);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        ss += __shfl_xor_sync(0xffffffffu, ss, o);
        ee += __shfl_xor_sync(0xffffffffu, ee, o);
    }
    finite = __all_sync(0xffffffffu, finite);
    if (lane == 0) {
        const float norm = sqrtf(ss);
        float err = sqrtf(ee) * 1.0001f;
        if (!finite) {
            colA[row] = cosine ? 0.f : __uint_as_float(0xff800000u);
            rn[row] = 0.f;     // cosine: a zero norm product puts the row under the reference's clamp -> always kept
            ex[row] = 0.f;
            return;
        }
        rn[row] = norm;
        if (cosine) {
            colA[row] = norm > 0.f ? 1.0f / norm : 0.f;
            ex[row] = norm > 0.f ? err / norm * 1.0001f : 0.f;
        } else {
            colA[row] = ss;
            ex[row] = err;
        }
    }
}

// max |x| over the set (non-finite values ignored), as raw float bits (non-negative floats order like integers)
template <typename T>
__global__ void __launch_bounds__(256) absmax_kernel(const T* __restrict__ rows, uint64_t n, uint32_t dim, uint32_t pitch,
                                                     uint32_t* __restrict__ out) {
    float m = 0.f;
    const uint64_t total = n * pitch;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (uint64_t)gridDim.x * blockDim.x) {
        const float v = fabsf((float)rows[i]);
        if (v <= 3.0e38f) m = fmaxf(m, v);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(out, __float_as_uint(m));
}

// exact power of two that brings a largest magnitude `m` to (2^13, 2^14]: a factor 4 under FP16's largest finite value
static float f16_scale_for(float m) {
    if (!(m > 0.f) || !std::isfinite(m)) return 1.0f;
    int e = 0;
    std::frexp(m, &e);   // m = f * 2^e, f in [0.5, 1)
    return std::ldexp(1.0f, std::max(-100, std::min(100, 14 - e)));
}

// stratified random sample: one row per bucket of n/ns consecutive rows, at a hashed offset inside the bucket
// (a plain stride would alias with periodic data). Operand rows are copied as 16-byte units.
__global__ void gather_sample_kernel(const uint4* __restrict__ op_rows, uint32_t row_u4, const float* __restrict__ colA,
                                     const float* __restrict__ rnorm, const float* __restrict__ ex, uint64_t n, uint32_t ns,
                                     uint4* __restrict__ out, float* __restrict__ out_sq, float* __restrict__ out_rn,
                                     float* __restrict__ out_ex, uint32_t* __restrict__ out_row) {
    const uint32_t i = blockIdx.x;
    if (i >= ns) return;
    const uint64_t lo = (uint64_t)i * n / ns, hi = (uint64_t)(i + 1) * n / ns;
    uint64_t h = (i + 0x9E3779B97F4A7C15ull) * 0xBF58476D1CE4E5B9ull;
    h ^= h >> 31;
    h *= 0x94D049BB133111EBull;
    h ^= h >> 29;
    const uint64_t row = lo + h % (hi > lo ? hi - lo : 1);
    for (uint32_t e = threadIdx.x; e < row_u4; e += blockDim.x) out[(size_t)i * row_u4 + e] = op_rows[row * row_u4 + e];
    if (threadIdx.x == 0) {
        out_sq[i] = colA[row];
        out_rn[i] = rnorm[row];
        out_ex[i] = ex[row];
        out_row[i] = (uint32_t)row;
    }
}

void drop_side_arrays(vdb_dataset* ds) {
    for (void* p : {(void*)ds->d_lo, (void*)ds->d_sqnorm, (void*)ds->d_ex, ds->d_op, ds->d_sample, (void*)ds->d_sample_sq,
                    (void*)ds->d_sample_rn, (void*)ds->d_sample_ex, (void*)ds->d_sample_row})
        if (p) cudaFree(p);
    ds->d_lo = ds->d_sqnorm = ds->d_ex = ds->d_sample_sq = ds->d_sample_rn = ds->d_sample_ex = nullptr;
    ds->d_op = ds->d_sample = nullptr;
    ds->d_sample_row = nullptr;
    ds->sample_n = 0;
    ds->side_n = 0;
}

static int forced_kind() {   // VDB_GEMM_KIND = tf32 | f16 (tests / tuning); default: chosen per dataset
    const char* e = getenv("VDB_GEMM_KIND");
    if (!e) return -1;
    return (e[0] == 't' || e[0] == '0') ? KIND_TF32 : KIND_F16;
}

static std::mutex g_side_mu;
// per-row scalars, the MMA operand (an FP16 copy, or the fp32 rows in place for the TF32 kind) and the threshold
// sample, cached on the (logically const) dataset handle; `kind` < 0: choose
static void ensure_side_arrays(const vdb_dataset* cds, cudaStream_t st, int kind = -1) {
    vdb_dataset* ds = const_cast<vdb_dataset*>(cds);
    std::lock_guard<std::mutex> lk(g_side_mu);
    if (kind < 0) kind = forced_kind();
    if (ds->d_sqnorm && ds->side_n == ds->n && (kind < 0 || kind == ds->op_kind)) return;
    drop_side_arrays(ds);
    const bool u8 = ds->dtype == VDB_U8;
    const bool cosine = ds->metric == VDB_COSINE;
    if (u8) kind = KIND_F16;   // 8-bit values are exact in FP16; there is no in-place operand for bytes
    const uint64_t n = ds->n;
    VDB_CUDA(cudaMalloc(&ds->d_sqnorm, n * 4));
    VDB_CUDA(cudaMalloc(&ds->d_lo, n * 4));
    VDB_CUDA(cudaMalloc(&ds->d_ex, n * 4));
    const uint32_t grid = (uint32_t)ceil_div<uint64_t>(n, 8);   // 8 warps per CTA, one row each
    auto means = [&](float* m_norm, float* m_ex) {
        DevBuf m(8, st);
        const uint64_t stride = std::max<uint64_t>(1, n / 65536);
        mean_kernel<<<1, 1024, 0, st>>>(ds->d_lo, n, stride, m.as<float>());
        VDB_LAUNCHED();
        mean_kernel<<<1, 1024, 0, st>>>(ds->d_ex, n, stride, m.as<float>() + 1);
        VDB_LAUNCHED();
        float h[2];
        VDB_CUDA(cudaMemcpyAsync(h, m.p, 8, cudaMemcpyDeviceToHost, st));
        VDB_CUDA(cudaStreamSynchronize(st));
        *m_norm = h[0];
        *m_ex = h[1];
    };
    auto build_f16 = [&]() {
        float scale = 1.0f;
        if (!u8) {
            DevBuf mx(4, st);
            VDB_CUDA(cudaMemsetAsync(mx.p, 0, 4, st));
            absmax_kernel<float><<<(uint32_t)sm_count() * 8, 256, 0, st>>>((const float*)ds->d_rows, n, ds->dim, ds->pitch, mx.as<uint32_t>());
            VDB_LAUNCHED();
            float h = 0.f;
            VDB_CUDA(cudaMemcpyAsync(&h, mx.p, 4, cudaMemcpyDeviceToHost, st));
            VDB_CUDA(cudaStreamSynchronize(st));
            scale = f16_scale_for(h);
        }
        ds->op_scale = scale;
        ds->op_pitch = round_up(ds->dim, 8u);   // 16-byte rows for the TMA
        VDB_CUDA(cudaMalloc(&ds->d_op, n * (size_t)ds->op_pitch * 2));
        if (u8)
            row_side_kernel<uint8_t, KIND_F16><<<grid, 256, 0, st>>>((const uint8_t*)ds->d_rows, n, ds->dim, ds->pitch, scale, ds->op_pitch,
                                                                     (__half*)ds->d_op, cosine, ds->d_sqnorm, ds->d_lo, ds->d_ex);
        else
            row_side_kernel<float, KIND_F16><<<grid, 256, 0, st>>>((const float*)ds->d_rows, n, ds->dim, ds->pitch, scale, ds->op_pitch,
                                                                   (__half*)ds->d_op, cosine, ds->d_sqnorm, ds->d_lo, ds->d_ex);
        VDB_LAUNCHED();
        ds->op_kind = KIND_F16;
        ds->op_owned = true;
    };
    auto build_tf32 = [&]() {
        row_side_kernel<float, KIND_TF32><<<grid, 256, 0, st>>>((const float*)ds->d_rows, n, ds->dim, ds->pitch, 1.0f, 0, nullptr, cosine,
                                                                ds->d_sqnorm, ds->d_lo, ds->d_ex);
        VDB_LAUNCHED();
        ds->op_kind = KIND_TF32;
        ds->op_scale = 1.0f;
        ds->op_pitch = ds->pitch;
        ds->d_op = nullptr;     // the fp32 rows themselves are the operand
        ds->op_owned = false;
    };
    if (kind == KIND_TF32) {
        build_tf32();
        means(&ds->mean_norm, &ds->mean_ex);
    } else {
        build_f16();
        means(&ds->mean_norm, &ds->mean_ex);
        // FP16 carries TF32's mantissa: its measured error norm sits at ~2^-12 of the row norm. Rows whose dynamic range
        // exceeds FP16's exponent (tiny components flushed next to large ones) show up as a larger norm; then the TF32
        // kind (8-bit exponent, operand = the fp32 rows in place) prunes better.
        const float rel = cosine ? ds->mean_ex : (ds->mean_norm > 0.f ? ds->mean_ex / ds->mean_norm : 0.f);
        if (kind < 0 && !u8 && rel > 1.0e-3f) {
            cudaFree(ds->d_op);
            ds->d_op = nullptr;
            build_tf32();
            means(&ds->mean_norm, &ds->mean_ex);
        }
    }
    // ~3 % of the shard, so the sample pass stays a small fixed fraction of the filter pass on every shard size
    static const uint32_t sample_env = getenv("VDB_GEMM_SAMPLE_N") ? (uint32_t)atoi(getenv("VDB_GEMM_SAMPLE_N")) : 0;
    const uint64_t sample_max = sample_env ? sample_env : G_SAMPLE;
    ds->sample_n = (uint32_t)std::min<uint64_t>(std::min<uint64_t>(sample_max, n / 2), std::max<uint64_t>(2048, n / 30));
    const size_t op_row_bytes = ds->op_kind == KIND_F16 ? (size_t)ds->op_pitch * 2 : ds->pitch_bytes();
    VDB_CUDA(cudaMalloc(&ds->d_sample, (size_t)ds->sample_n * op_row_bytes));
    VDB_CUDA(cudaMalloc(&ds->d_sample_sq, (size_t)ds->sample_n * 4));
    VDB_CUDA(cudaMalloc(&ds->d_sample_rn, (size_t)ds->sample_n * 4));
    VDB_CUDA(cudaMalloc(&ds->d_sample_ex, (size_t)ds->sample_n * 4));
    VDB_CUDA(cudaMalloc(&ds->d_sample_row, (size_t)ds->sample_n * 4));
    gather_sample_kernel<<<ds->sample_n, 128, 0, st>>>((const uint4*)(ds->op_kind == KIND_F16 ? ds->d_op : ds->d_rows),
                                                       (uint32_t)(op_row_bytes / 16), ds->d_sqnorm, ds->d_lo, ds->d_ex, n, ds->sample_n,
                                                       (uint4*)ds->d_sample, ds->d_sample_sq, ds->d_sample_rn, ds->d_sample_ex, ds->d_sample_row);
    VDB_LAUNCHED();
    VDB_CUDA(cudaStreamSynchronize(st));
    ds->side_n = n;
}

// tensor map of `nrows` operand rows of the dataset's kind starting at `base` (row pitch in bytes)
static CUtensorMap make_op_map(int kind, const void* base, uint32_t dim, uint64_t nrows, uint64_t pitch_bytes, uint32_t box_rows) {
    return kind == KIND_F16 ? make_map_f16(base, dim, nrows, pitch_bytes, box_rows) : make_map(base, dim, nrows, pitch_bytes, box_rows);
}
static const void* op_rows_of(const vdb_dataset* ds) { return ds->op_kind == KIND_F16 ? ds->d_op : ds->d_rows; }
static size_t op_row_bytes_of(const vdb_dataset* ds) {
    return ds->op_kind == KIND_F16 ? (size_t)ds->op_pitch * 2 : ds->pitch_bytes();
}
static uint32_t kblocks_of(int kind, uint32_t dim) { return ceil_div(dim, kind == KIND_F16 ? 64u : 32u); }

static int gemm_ctas();
// tiling of one pass: query-tile units x row slabs (small slabs, query tile fastest: the CTAs in flight share a few
// row tiles and all query tiles in L2)
static void plan_gemm(GemmParams& p, int ctas_sel = 0, uint32_t tps_want = 0) {
    const uint32_t ctas = (uint32_t)(ctas_sel ? ctas_sel : gemm_ctas());
    const uint32_t sms = (uint32_t)sm_count();
    p.ntiles = (uint32_t)ceil_div<uint64_t>(p.nrows, GN);
    p.nqt = ceil_div<uint32_t>(p.nq, GM * ctas);
    static const uint32_t tps_env = getenv("VDB_GEMM_TPS") ? (uint32_t)atoi(getenv("VDB_GEMM_TPS")) : 0;
    const uint32_t tps = tps_want ? tps_want : (tps_env ? tps_env : 4u);
    p.tiles_per_slab = std::max(1u, std::min(tps, ceil_div(p.ntiles * p.nqt, sms / ctas)));
    p.nslabs = ceil_div(p.ntiles, p.tiles_per_slab);
}

static int gemm_ctas() {
    static const int v = getenv("VDB_GEMM_CTAS") ? atoi(getenv("VDB_GEMM_CTAS")) : 2;
    return v == 1 ? 1 : 2;
}

template <int MODE, int CTAS, int METRIC, int KIND, bool STAGED = false>
static void launch_gemm_t(const CUtensorMap& mq, const CUtensorMap& mx, GemmParams p, cudaStream_t st, const char* prof_name) {
    using Cfg = GemmCfg<CTAS, KIND>;
    auto kern = flat_gemm_kernel<MODE, CTAS, METRIC, KIND, STAGED>;
    static std::atomic<size_t> configured[VDB_MAX_DEVICES];
    // + the staging buffers (STAGED filter) or the top-G_TOPJ epilogue's per-thread score rows (mode 2: 128 x 33 floats)
    constexpr uint32_t SMEM = (STAGED ? Cfg::SMEM_STAGED : Cfg::SMEM) + (MODE == 2 ? 128 * 33 * 4 : 0);
    ensure_dyn_smem(kern, SMEM, configured);
    const uint32_t sms = (uint32_t)sm_count();
    const uint32_t units = std::min(sms / CTAS, p.items ? p.nitems : p.nqt * p.nslabs);
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(units * CTAS);
    cfg.blockDim = dim3(G_THREADS);
    cfg.dynamicSmemBytes = SMEM;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CTAS;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    DevBuf counter(4, st);
    VDB_CUDA(cudaMemsetAsync(counter.p, 0, 4, st));
    p.work_counter = counter.as<uint32_t>();
    ProfScope prof(prof_name, st);
    VDB_CUDA(cudaLaunchKernelEx(&cfg, kern, mq, mx, p));
    VDB_LAUNCHED();
}

template <int MODE, int CTAS, bool STAGED = false>
static void launch_gemm_mk(int metric, int kind, const CUtensorMap& mq, const CUtensorMap& mx, const GemmParams& p, cudaStream_t st,
                           const char* prof_name) {
    if (metric == VDB_COSINE) {
        if (kind == KIND_F16) launch_gemm_t<MODE, CTAS, VDB_COSINE, KIND_F16, STAGED>(mq, mx, p, st, prof_name);
        else launch_gemm_t<MODE, CTAS, VDB_COSINE, KIND_TF32, STAGED>(mq, mx, p, st, prof_name);
    } else {
        if (kind == KIND_F16) launch_gemm_t<MODE, CTAS, VDB_L2SQR, KIND_F16, STAGED>(mq, mx, p, st, prof_name);
        else launch_gemm_t<MODE, CTAS, VDB_L2SQR, KIND_TF32, STAGED>(mq, mx, p, st, prof_name);
    }
}

// mode 0 = store every score, 1 = filter, 2 = per-slab smallest scores; `p` must have been planned (plan_gemm)
static void launch_gemm(int mode, int metric, int kind, const CUtensorMap& mq, const CUtensorMap& mx, const GemmParams& p,
                        cudaStream_t st, int ctas = 0, const char* prof_name = "flat_gemm") {
    const bool pair = (ctas ? ctas : gemm_ctas()) == 2;
    if (mode == 1 && p.rare_per_score == 2) {   // filter with staged candidate slots (its own instantiation)
        if (pair) launch_gemm_mk<1, 2, true>(metric, kind, mq, mx, p, st, prof_name);
        else launch_gemm_mk<1, 1, true>(metric, kind, mq, mx, p, st, prof_name);
        return;
    }
    switch (mode * 2 + (pair ? 1 : 0)) {
        case 0: launch_gemm_mk<0, 1>(metric, kind, mq, mx, p, st, prof_name); break;
        case 1: launch_gemm_mk<0, 2>(metric, kind, mq, mx, p, st, prof_name); break;
        case 2: launch_gemm_mk<1, 1>(metric, kind, mq, mx, p, st, prof_name); break;
        case 3: launch_gemm_mk<1, 2>(metric, kind, mq, mx, p, st, prof_name); break;
        case 4: launch_gemm_mk<2, 1>(metric, kind, mq, mx, p, st, prof_name); break;
        default: launch_gemm_mk<2, 2>(metric, kind, mq, mx, p, st, prof_name); break;
    }
}

// Query side of the tensor path in one pass (one warp per query): padded fp32 copy (exact rerank), the MMA operand
// q~ (FP16 of q * s_q with s_q an exact power of two chosen per query, or q rounded to TF32), ||q||^2, the operand
// error ||q - q~|| and a flag for non-finite queries (they are answered by the exact scan). The norm is summed exactly
// like row_cache's PM_SQNORM kernel (lane-strided fma chain + xor butterfly), so thresholds do not depend on which of
// the two produced it.
template <typename T, int KIND>
__global__ void __launch_bounds__(256) tq_prepare_kernel(const T* __restrict__ src, uint32_t nq, uint32_t dim, uint32_t qpitch,
                                                         uint32_t op_pitch, float* __restrict__ qcopy, void* __restrict__ qop,
                                                         float* __restrict__ qsq, float* __restrict__ qerr,
                                                         float* __restrict__ qscale, uint32_t* __restrict__ qbad) {
    const uint32_t q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (q >= nq) return;
    const T* row = src + (size_t)q * dim;
    float scale = 1.0f;
    bool finite = true;
    if (KIND == KIND_F16) {
        float m = 0.f;
        for (uint32_t e = lane; e < dim; e += 32) {
            const float v = fabsf((float)row[e]);
            finite = finite && (v <= 3.0e38f);
            m = fmaxf(m, v <= 3.0e38f ? v : 0.f);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        if (m > 0.f) {
            int e2 = (int)((__float_as_uint(m) >> 23) & 0xff) - 126;   // m = f * 2^e2, f in [0.5, 1) (normal m)
            e2 = max(-100, min(100, 14 - e2));
            scale = __uint_as_float((uint32_t)(e2 + 127) << 23);
        }
    }
    const float inv_scale = 1.0f / scale;
    float s = 0.f, ee = 0.f;
    const uint32_t span = max(qpitch, op_pitch);
    for (uint32_t e = lane; e < span; e += 32) {
        const float v = e < dim ? (float)row[e] : 0.f;
        float back;
        if (KIND == KIND_F16) {
            const __half h = __float2half_rn(v * scale);
            if (e < op_pitch) reinterpret_cast<__half*>(qop)[(size_t)q * op_pitch + e] = h;
            back = __half2float(h) * inv_scale;
        } else {
            uint32_t r;
            asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
            if (e < op_pitch) reinterpret_cast<float*>(qop)[(size_t)q * op_pitch + e] = __uint_as_float(r);
            back = __uint_as_float(r);
        }
        if (e < qpitch) qcopy[(size_t)q * qpitch + e] = v;
        finite = finite && (fabsf(v) <= 3.0e38f);
        if (e < dim) {
            const float d = v - back;
            s = fmaf(v, v, s);
            ee = fmaf(d, d, ee);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, o);
        ee += __shfl_xor_sync(0xffffffffu, ee, o);
    }
    finite = __all_sync(0xffffffffu, finite);
    if (lane == 0) {
        qsq[q] = s;
        qerr[q] = sqrtf(ee) * 1.0001f;
        qscale[q] = scale;
        qbad[q] = finite ? 0u : 1u;
    }
}

// Pruning-bound coefficients per query (see GemmParams). With q = q~/s_q + dq, x = x~/s_x + dx, ||dq|| = eq, ||dx|| = ex and
// the fp32 accumulation error of the contraction bounded by ACC * ||q~|| ||x~|| (ACC = dim * 2^-23):
//   |q.x - acc / (s_q s_x)| <= ACC qn' xn' + qn' ex + eq xn',   qn' = ||q|| + eq,  xn' = ||x|| + ex
// L2Sqr:  S' = ||x||^2 - 2 acc / (s_q s_x) - 2 (that bound) = sq + qd acc - qab ex - qb rn  with
//         qd = -2 / (s_q s_x), qb = 2 (ACC qn' + eq), qab = 2 qn' + qb
// cosine: S' = 1 - acc / (s_q s_x ||q|| ||x||) - bound / (||q|| ||x||) - 1e-6 = qb - (qd / ||x||) acc - qab exr  with eqr = eq / ||q||,
//         exr = ex / ||x||, qd = 1 / (s_q s_x ||q||), qb = 1 - 1e-6 - (ACC (1 + eqr) + eqr), qab = (1 + eqr)(1 + ACC) + eqr
__global__ void tq_coeff_kernel(const float* __restrict__ qsq, const float* __restrict__ qerr, const float* __restrict__ qscale,
                                const float* __restrict__ qnorm_cos, uint32_t nq, float acc, float row_scale,
                                float* __restrict__ qd, float* __restrict__ qab, float* __restrict__ qb) {
    const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    const float eq = qerr[q];
    const float inv_scales = 1.0f / (qscale[q] * row_scale);   // powers of two: exact
    if (!qnorm_cos) {
        const float qn1 = (sqrtf(qsq[q]) + eq) * 1.0001f;
        const float b = 2.0f * (acc * qn1 + eq) * 1.0001f;
        qd[q] = -2.0f * inv_scales;
        qb[q] = b;
        qab[q] = 2.0f * qn1 + b;
    } else {
        const float qn = qnorm_cos[q];
        const float eqr = qn > 0.f ? eq / qn * 1.0001f : 0.f;
        qd[q] = qn > 0.f ? inv_scales / qn : 0.f;
        qb[q] = 1.0f - 1e-6f - (acc * (1.0f + eqr) + eqr) * 1.0001f;
        qab[q] = ((1.0f + eqr) * (1.0f + acc) + eqr) * 1.0001f;
    }
}
// IVF probe scan: tau_q = (j0-th smallest sampled S') + margin. j0 is chosen so that the k-th best S' of the probed rows
// is <= S'_(j0) with high probability; because S <= S' + 2 b(q, x), the margin (3 x the pruning bound at the mean row
// error / mean row norm) keeps the k-th EXACT distance inside the threshold. The check kernel verifies it per query.
__global__ void tau_from_keys_kernel(const uint64_t* __restrict__ keys, uint32_t nq, uint32_t j, uint32_t j0,
                                     const float* __restrict__ qab, const float* __restrict__ qb, float mean_norm, float mean_ex,
                                     int cosine, float* __restrict__ tau) {
    const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    const uint64_t kk = keys[(size_t)q * j + (j0 - 1)];
    const float s = kk == KEY_NONE ? __uint_as_float(0x7f800000u) : key_dist(kk);
    const float b = cosine ? (1.0f - qb[q]) + qab[q] * mean_ex : qab[q] * mean_ex + qb[q] * mean_norm;
    tau[q] = s + 3.0f * b;
}
// Flat: the sample keys carry EXACT distances (the j best sampled rows by pruning score are re-evaluated in fp32), so
// tau_q = d_(j0) - ||q||^2 (cosine: d_(j0)) needs no margin: every row x of the true top-k has S'(x) <= d(x) - ||q||^2
// <= d_k - ||q||^2 <= d_(j0) - ||q||^2 whenever the j0-th sampled distance is not better than the k-th best of the set
// (probability > 1 - 2e-5 by the choice of j0, verified per query by the check kernel). The slack keeps the check's
// strict comparison satisfiable when the j0-th sampled row IS the k-th best.
__device__ __forceinline__ float tau_of_key(uint64_t kk, float shift) {
    if (kk == KEY_NONE) return __uint_as_float(0x7f800000u);   // fewer than j0 sampled rows: keep everything
    const float d = key_dist(kk);
    return (d - shift) + 1e-4f * (fabsf(d) + shift) + 1e-30f;
}
__global__ void tau_exact_kernel(const uint64_t* __restrict__ keys, uint32_t nq, uint32_t j, uint32_t j0,
                                 const float* __restrict__ qsq, float* __restrict__ tau) {
    const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    tau[q] = tau_of_key(keys[(size_t)q * j + (j0 - 1)], qsq ? qsq[q] : 0.f);
}
// Tail of the sample phase for j <= 32, one warp per query: exact distances of the j best sampled rows -> keys -> ascending
// (rank by counting, ties cannot occur: the ids differ) -> optionally tau_q from the j0-th. Replaces a re-keying launch, a
// one-CTA-per-query merge and the tau launch.
__global__ void __launch_bounds__(256) sample_finish_kernel(const float* __restrict__ dist, const uint32_t* __restrict__ rid,
                                                            const uint8_t* __restrict__ valid, uint32_t id_base, uint32_t nq,
                                                            uint32_t j, uint64_t* __restrict__ jkeys, uint32_t j0,
                                                            const float* __restrict__ qsq, float* __restrict__ tau) {
    const uint32_t q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (q >= nq) return;   // warp-uniform
    const size_t i = (size_t)q * j + lane;
    const uint64_t mine = (lane < j && valid[i]) ? make_key(dist[i], id_base + rid[i]) : KEY_NONE;
    uint32_t rank = 0;
    for (uint32_t m = 0; m < j; ++m) {
        const uint64_t other = __shfl_sync(0xffffffffu, mine, m);
        rank += (other < mine || (other == mine && m < lane)) ? 1u : 0u;
    }
    if (lane < j) {
        jkeys[(size_t)q * j + rank] = mine;
        if (tau && rank == j0 - 1) tau[q] = tau_of_key(mine, qsq ? qsq[q] : 0.f);
    }
}
// two-level sample selection: coarse threshold = the j1-th smallest sub-sample score, nudged up so that the strict
// comparison of the filter keeps the row it came from (+inf when the sub-sample holds fewer than j1 rows)
__global__ void tau_coarse_kernel(const uint64_t* __restrict__ keys, uint32_t nq, uint32_t j1, float* __restrict__ tau) {
    const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    const uint64_t kk = keys[(size_t)q * j1 + (j1 - 1)];
    const float s = key_dist(kk);
    tau[q] = kk == KEY_NONE ? __uint_as_float(0x7f800000u) : s + 1e-6f * fabsf(s) + 1e-30f;
}
// filter-mode candidates (raw score bits << 32 | row of the B tensor) -> sortable keys, in place
__global__ void cand_sortable_kernel(uint64_t* __restrict__ cand, const uint32_t* __restrict__ cnt, uint32_t cap) {
    const uint32_t q = blockIdx.x, c = min(cnt[q], cap);
    for (uint32_t j = threadIdx.x; j < c; j += blockDim.x) {
        const uint64_t e = cand[(uint64_t)q * cap + j];
        cand[(uint64_t)q * cap + j] = make_key(__uint_as_float((uint32_t)(e >> 32)), (uint32_t)e);
    }
}
// ---- candidate pruning by score bounds -------------------------------------------------------------------------------
// The filter keeps every row whose LOWER bound S' of the (shifted) distance is under tau_q; tau_q comes from a sample, so a
// list holds several times k rows. The same contraction also gives an UPPER bound: the score without its error term lies
// within +-B(q, x) of the exact value, so U = S' + 2 B (plus the rounding slack of the check kernel) >= d(q, x) - shift. At
// least k rows of the list have a distance <= U_(k), the k-th smallest U, hence d_k - shift <= U_(k) and no row with
// S' > U_(k) can be among the k best: it is dropped BEFORE the exact rerank (HBM gathers of whole rows). One CTA per
// query: U of every candidate -> radix select of U_(k) in shared memory -> in-place compaction. Lists of <= k entries and
// NaN scores (non-finite rows; the rerank decides) are kept whole.
// order bits of the upper bound U of a candidate's shifted distance (see above); rows that must be kept whatever their
// score (NaN / -inf: cosine rows under the reference's norm clamp) get the largest value: no upper bound
template <int METRIC>
__device__ __forceinline__ uint32_t cand_upper_bits(uint64_t e, float a, float b, float shift, const float* __restrict__ rnorm,
                                                    const float* __restrict__ ex) {
    const uint32_t row = (uint32_t)e;
    const float sp = __uint_as_float((uint32_t)(e >> 32));
    const float bound = METRIC == VDB_L2SQR ? fmaf(a, ex[row], b * rnorm[row]) : (1.0f - b) + a * ex[row];
    float up = sp + 2.0002f * bound;
    up += 2e-5f * (fabsf(up) + shift) + 1e-30f;
    return fabsf(sp) <= 3.0e38f ? f32_order_bits(up) : 0xffffffffu;
}
// Row-sharded search, first half of the global pruning: per query the upper bounds of ranks m, 2m, ..., T m of this shard's
// candidate list, ascending (order bits; 0xffffffff where the list is shorter, and everywhere for lists too long to sort
// here - they only weaken the bound). One CTA per query, bitonic sort of the list's U in shared memory.
constexpr uint32_t PRUNE_SORT_MAX = 2048;
template <int METRIC>
__global__ void __launch_bounds__(256) prune_stats_kernel(const uint64_t* __restrict__ cand, const uint32_t* __restrict__ cnt,
                                                          uint32_t cap, uint32_t m, uint32_t T, const float* __restrict__ rnorm,
                                                          const float* __restrict__ ex, const float* __restrict__ qab,
                                                          const float* __restrict__ qb, const float* __restrict__ qsq,
                                                          uint32_t* __restrict__ stats) {
    __shared__ uint32_t u[PRUNE_SORT_MAX];
    const uint32_t q = blockIdx.x, tid = threadIdx.x;
    const uint32_t c = min(cnt[q], cap);
    uint32_t* out = stats + (size_t)q * T;
    if (c > PRUNE_SORT_MAX || c == 0) {
        for (uint32_t i = tid; i < T; i += blockDim.x) out[i] = 0xffffffffu;
        return;
    }
    const uint32_t n = c <= 32 ? 32u : (1u << (32 - __clz(c - 1)));
    const uint64_t* list = cand + (uint64_t)q * cap;
    const float a = qab[q], b = qb[q], shift = qsq ? qsq[q] : 0.f;
    for (uint32_t j = tid; j < n; j += blockDim.x) u[j] = j < c ? cand_upper_bits<METRIC>(list[j], a, b, shift, rnorm, ex) : 0xffffffffu;
    __syncthreads();
    for (uint32_t size = 2; size <= n; size <<= 1)
        for (uint32_t st = size >> 1; st > 0; st >>= 1) {
            for (uint32_t t = tid; t < (n >> 1); t += blockDim.x) {
                const uint32_t i = ((t & ~(st - 1)) << 1) | (t & (st - 1)), l = i | st;
                const uint32_t x = u[i], y = u[l];
                if ((x > y) == ((i & size) == 0)) u[i] = y, u[l] = x;
            }
            __syncthreads();
        }
    for (uint32_t i = tid; i < T; i += blockDim.x) {
        const uint32_t r = (i + 1) * m - 1;
        out[i] = r < c ? u[r] : 0xffffffffu;
    }
}
template <int METRIC>
__global__ void __launch_bounds__(256) cand_prune_kernel(uint64_t* __restrict__ cand, const uint32_t* __restrict__ cnt, uint32_t cap,
                                                         uint32_t k, const float* __restrict__ rnorm, const float* __restrict__ ex,
                                                         const float* __restrict__ qab, const float* __restrict__ qb,
                                                         const float* __restrict__ qsq, uint32_t* __restrict__ cnt_out,
                                                         uint64_t* __restrict__ off, unsigned long long* __restrict__ pair_total,
                                                         uint32_t* __restrict__ qidx, uint32_t* __restrict__ rid,
                                                         const uint32_t* __restrict__ gstats, uint32_t gshards, uint32_t gT,
                                                         uint32_t gnq) {
    extern __shared__ uint32_t prune_u[];   // [min(cnt, cap)] order bits of U
    __shared__ uint32_t hist[256];
    __shared__ uint32_t s_bin, s_k, s_warp[8], s_base;
    __shared__ unsigned long long s_off;
    const uint32_t q = blockIdx.x, tid = threadIdx.x;
    const uint32_t c = min(cnt[q], cap);
    uint64_t* list = cand + (uint64_t)q * cap;
    // off != nullptr: the surviving (query, row) pairs go straight to the rerank's input arrays, at a range claimed with
    // one atomic per query (the order of the ranges does not matter: every pair carries its query) - no separate
    // prefix-sum and pair-building launches
    auto emit_pairs = [&](uint32_t count) {
        if (!off) return;
        if (tid == 0) {
            s_off = atomicAdd(pair_total, (unsigned long long)count);
            off[q] = s_off;
        }
        __syncthreads();
        const unsigned long long o = s_off;
        for (uint32_t j = tid; j < count; j += blockDim.x) {
            qidx[o + j] = q;
            rid[o + j] = (uint32_t)list[j];
        }
    };
    if (c <= k && !gstats) {
        if (tid == 0) cnt_out[q] = c;
        emit_pairs(c);
        return;
    }
    uint32_t thr;
    if (gstats) {
        // Row-sharded search: every shard sent the upper bounds U of ranks m, 2m, ..., T m of ITS list (order bits, ascending,
        // padded with the largest value; prune_stats_kernel). The i-th entry of a shard's row certifies (i + 1) m rows with
        // d - shift <= that value, so the T-th smallest of all G T entries certifies >= T m >= k rows of the WHOLE set: no row
        // with S' above it can be among the k best - the local list is cut against the global bound, not the shard's own.
        const uint32_t GT = gshards * gT;
        for (uint32_t i = tid; i < GT; i += blockDim.x) {
            const uint32_t sh = i / gT, t = i - sh * gT;
            prune_u[i] = gstats[((size_t)sh * gnq + q) * gT + t];
        }
        __syncthreads();
        if (tid == 0) s_bin = 0xffffffffu;
        __syncthreads();
        for (uint32_t i = tid; i < GT; i += blockDim.x) {
            const uint32_t v = prune_u[i];
            uint32_t r = 0;
            for (uint32_t j = 0; j < GT; ++j) {
                const uint32_t w = prune_u[j];
                r += (w < v || (w == v && j < i)) ? 1u : 0u;
            }
            if (r == gT - 1) s_bin = v;   // exactly one entry has this rank
        }
        __syncthreads();
        thr = s_bin;
        __syncthreads();
    } else {
    const float a = qab[q], b = qb[q], shift = qsq ? qsq[q] : 0.f;
    for (uint32_t j = tid; j < c; j += blockDim.x) prune_u[j] = cand_upper_bits<METRIC>(list[j], a, b, shift, rnorm, ex);
    // radix select: the k-th smallest (1-based) of prune_u[0, c), 8 bits per pass from the top
    uint32_t prefix = 0, mask = 0, kk = k;
    for (int sh = 24; sh >= 0; sh -= 8) {
        hist[tid] = 0;
        __syncthreads();
        for (uint32_t j = tid; j < c; j += blockDim.x) {
            const uint32_t v = prune_u[j];
            if ((v & mask) == prefix) atomicAdd(&hist[(v >> sh) & 255u], 1u);
        }
        __syncthreads();
        if (tid < 32) {   // warp 0: bin that holds the kk-th element (inclusive scan over 8 bins per lane)
            uint32_t loc[8], sum = 0;
#pragma unroll
            for (int i = 0; i < 8; ++i) loc[i] = hist[tid * 8 + i], sum += loc[i];
            uint32_t incl = sum;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t y = __shfl_up_sync(0xffffffffu, incl, o);
                if ((int)tid >= o) incl += y;
            }
            const uint32_t before = incl - sum;
            if (before < kk && kk <= incl) {   // exactly one lane
                uint32_t run = before;
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    if (run < kk && kk <= run + loc[i]) s_bin = tid * 8 + i, s_k = kk - run;
                    run += loc[i];
                }
            }
        }
        __syncthreads();
        prefix |= s_bin << sh;
        mask |= 0xffu << sh;
        kk = s_k;
        __syncthreads();
    }
    thr = prefix;
    }
    // stable in-place compaction (a chunk is read completely before anything is written at or below it)
    if (tid == 0) s_base = 0;
    __syncthreads();
    for (uint32_t j0 = 0; j0 < c; j0 += blockDim.x) {
        const uint32_t j = j0 + tid;
        const uint64_t e = j < c ? list[j] : 0;
        const float sp = __uint_as_float((uint32_t)(e >> 32));
        const bool keep = j < c && (sp != sp || f32_order_bits(sp) <= thr);
        const uint32_t bal = __ballot_sync(0xffffffffu, keep);
        const uint32_t lane = tid & 31, w = tid >> 5;
        if (lane == 0) s_warp[w] = __popc(bal);
        __syncthreads();
        uint32_t off = s_base, total = 0;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            if (i < (int)w) off += s_warp[i];
            total += s_warp[i];
        }
        if (keep) list[off + __popc(bal & ((1u << lane) - 1u))] = e;
        __syncthreads();
        if (tid == 0) s_base += total;
        __syncthreads();
    }
    if (tid == 0) cnt_out[q] = s_base;
    emit_pairs(s_base);   // the loop's last barrier ordered the compacted list
}
// (query, source row) pairs of the j best sampled rows of every query; KEY_NONE entries are masked out
__global__ void sample_pairs_kernel(const uint64_t* __restrict__ keys, uint64_t count, uint32_t j,
                                    const uint32_t* __restrict__ sample_row, uint32_t* __restrict__ qidx,
                                    uint32_t* __restrict__ rid, uint8_t* __restrict__ valid) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t kk = keys[i];
        const bool ok = kk != KEY_NONE;
        qidx[i] = (uint32_t)(i / j);
        rid[i] = ok ? sample_row[key_id(kk)] : 0u;
        valid[i] = ok;
    }
}
// exclusive scan of min(cnt, cap) over the queries (one block; nq is at most a few 100k)
__global__ void __launch_bounds__(1024) cand_offsets_kernel(const uint32_t* __restrict__ cnt, uint32_t nq, uint32_t cap,
                                                            uint64_t* __restrict__ off) {
    __shared__ uint64_t warp_sums[32];
    __shared__ uint64_t carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (uint32_t base = 0; base < nq; base += blockDim.x) {
        const uint32_t q = base + threadIdx.x;
        const uint64_t v = q < nq ? min(cnt[q], cap) : 0u;
        uint64_t x = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint64_t y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += y;
        }
        if (lane == 31) warp_sums[warp] = x;
        __syncthreads();
        if (warp == 0) {
            uint64_t w = warp_sums[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint64_t y = __shfl_up_sync(0xffffffffu, w, o);
                if (lane >= o) w += y;
            }
            warp_sums[lane] = w;
        }
        __syncthreads();
        const uint64_t before = carry + (warp ? warp_sums[warp - 1] : 0) + x - v;
        if (q < nq) off[q] = before;
        __syncthreads();
        if (threadIdx.x == blockDim.x - 1) carry = before + v;
        __syncthreads();
    }
    if (threadIdx.x == 0) off[nq] = carry;
}
// ---- row-part pipeline of the filter pass: candidates [prev[q], cur[q]) of every query (one row part) -------------
// exclusive scan of the part's candidate counts; prev == nullptr -> 0
__global__ void __launch_bounds__(1024) part_offsets_kernel(const uint32_t* __restrict__ prev, const uint32_t* __restrict__ cur,
                                                            uint32_t nq, uint32_t cap, uint64_t* __restrict__ off) {
    __shared__ uint64_t warp_sums[32];
    __shared__ uint64_t carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (uint32_t base = 0; base < nq; base += blockDim.x) {
        const uint32_t q = base + threadIdx.x;
        const uint64_t v = q < nq ? min(cur[q], cap) - (prev ? min(prev[q], cap) : 0u) : 0u;
        uint64_t x = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint64_t y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += y;
        }
        if (lane == 31) warp_sums[warp] = x;
        __syncthreads();
        if (warp == 0) {
            uint64_t w = warp_sums[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint64_t y = __shfl_up_sync(0xffffffffu, w, o);
                if (lane >= o) w += y;
            }
            warp_sums[lane] = w;
        }
        __syncthreads();
        const uint64_t before = carry + (warp ? warp_sums[warp - 1] : 0) + x - v;
        if (q < nq) off[q] = before;
        __syncthreads();
        if (threadIdx.x == blockDim.x - 1) carry = before + v;
        __syncthreads();
    }
    if (threadIdx.x == 0) off[nq] = carry;
}
__global__ void part_to_pairs_kernel(const uint64_t* __restrict__ cand, const uint32_t* __restrict__ prev,
                                     const uint32_t* __restrict__ cur, uint32_t cap, const uint64_t* __restrict__ off,
                                     uint32_t* __restrict__ qidx, uint32_t* __restrict__ rid) {
    const uint32_t q = blockIdx.x;
    const uint32_t j0 = prev ? min(prev[q], cap) : 0u, j1 = min(cur[q], cap);
    const uint64_t o = off[q];
    for (uint32_t j = j0 + threadIdx.x; j < j1; j += blockDim.x) {
        qidx[o + (j - j0)] = q;
        rid[o + (j - j0)] = (uint32_t)cand[(uint64_t)q * cap + j];
    }
}
// exact distances of the part's pairs -> final keys, written over the candidate entries they came from
__global__ void part_rekey_kernel(const float* __restrict__ dist, const uint32_t* __restrict__ qidx,
                                  const uint32_t* __restrict__ rid, const uint64_t* __restrict__ off, uint32_t nq,
                                  const uint32_t* __restrict__ prev, uint32_t cap, uint32_t id_base,
                                  uint64_t* __restrict__ cand, const uint64_t* __restrict__ n_ptr) {
    const uint64_t n = n_ptr ? *n_ptr : off[nq];
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t q = qidx[i];
        const uint32_t j = (prev ? min(prev[q], cap) : 0u) + (uint32_t)(i - off[q]);
        cand[(uint64_t)q * cap + j] = make_key(dist[i], id_base + rid[i]);
    }
}
// candidate (S', local row) lists -> dense rerank inputs at off[q]
__global__ void cand_to_pairs_kernel(const uint64_t* __restrict__ cand, const uint32_t* __restrict__ cnt, uint32_t cap,
                                     const uint64_t* __restrict__ off, const uint32_t* __restrict__ pos_to_row,
                                     uint32_t* __restrict__ qidx, uint32_t* __restrict__ rid) {
    const uint32_t q = blockIdx.x;
    const uint32_t c = min(cnt[q], cap);
    const uint64_t o = off[q];
    for (uint32_t j = threadIdx.x; j < c; j += blockDim.x) {
        qidx[o + j] = q;
        const uint32_t pos = (uint32_t)cand[(uint64_t)q * cap + j];
        rid[o + j] = pos_to_row ? pos_to_row[pos] : pos;  // IVF: list-order position -> row id
    }
}
__global__ void rekey_dev_count_kernel(const float* __restrict__ dist, const uint32_t* __restrict__ ids, uint32_t id_base,
                                       const uint64_t* __restrict__ count, uint64_t* __restrict__ keys) {
    const uint64_t n = *count;
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (uint64_t)gridDim.x * blockDim.x)
        keys[j] = make_key(dist[j], ids[j] + id_base);
}
// completeness check; failing queries are appended to redo[]
// keys / overflow are indexed by the LOCAL query i of the checked range [q0, q0 + cnt) (a row-sharded search checks
// only the slice of queries a GPU owns); tau / qsq by the batch index q0 + i, which is also what redo[] receives.
__global__ void check_kernel(const uint64_t* __restrict__ keys, uint32_t q0, uint32_t cnt, uint32_t k, uint64_t n,
                             const uint32_t* __restrict__ overflow, const float* __restrict__ tau,
                             const float* __restrict__ qsq, uint32_t force_mod, uint32_t* __restrict__ redo,
                             uint32_t* __restrict__ nredo) {
    // qsq == nullptr: cosine (scores bound the distance itself); else L2Sqr (scores bound d - ||q||^2)
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= cnt) return;
    const uint32_t q = q0 + i;
    const uint32_t need = (uint32_t)((uint64_t)k < n ? (uint64_t)k : n);
    bool ok = !(overflow && overflow[i]);
    if (ok && need) {
        const uint64_t kk = keys[(size_t)i * k + (need - 1)];
        ok = kk != KEY_NONE;  // fewer than `need` candidates survived the filter
        if (ok) {
            const float dk = key_dist(kk);
            const float shift = qsq ? qsq[q] : 0.f;
            const float slack = 2e-5f * (fabsf(dk) + shift + fabsf(tau[q]));
            ok = (dk - shift) < tau[q] - slack;
        }
    }
    if (force_mod && q % force_mod == 0) ok = false;
    if (!ok) redo[atomicAdd(nredo, 1u)] = q;
}
__global__ void gather_rows_kernel(const uint8_t* __restrict__ src, uint32_t row_bytes, const uint32_t* __restrict__ idx,
                                   uint32_t cnt, uint8_t* __restrict__ dst) {
    const uint32_t i = blockIdx.x;
    if (i >= cnt) return;
    for (uint32_t e = threadIdx.x; e < row_bytes; e += blockDim.x)
        dst[(size_t)i * row_bytes + e] = src[(size_t)idx[i] * row_bytes + e];
}
__global__ void scatter_keys_kernel(const uint64_t* __restrict__ src, uint32_t k, const uint32_t* __restrict__ idx,
                                    uint32_t cnt, uint64_t* __restrict__ dst) {
    const uint32_t i = blockIdx.x;
    if (i >= cnt) return;
    for (uint32_t e = threadIdx.x; e < k; e += blockDim.x) dst[(size_t)idx[i] * k + e] = src[(size_t)i * k + e];
}

constexpr uint32_t G_MAX_K = 1024;

bool flat_gemm_supported(const vdb_dataset* ds, uint32_t nq, uint32_t k) {
    return (ds->dtype == VDB_F32 || ds->dtype == VDB_U8) && k >= 1 && k <= G_MAX_K && ds->n >= 65536 &&
           nq >= 1 && ((uintptr_t)ds->d_rows & 15) == 0;
}

std::atomic<uint64_t> g_gemm_redo{0};  // queries that needed the exact fallback (instrumentation)
std::atomic<uint64_t> g_gemm_cands{0}; // candidates reranked (instrumentation)
std::atomic<uint64_t> g_gemm_queries{0};
// test hook (vdb_debug_force_redo): every query whose index is a multiple of m fails the completeness check, so
// the exact re-scan of flagged queries (single-GPU and sharded) can be exercised on purpose; 0 = off
std::atomic<uint32_t> g_debug_force_redo{0};

// ---- phases (also exported one by one for the row-sharded search, sharded.py) -------------------------------
// j0: smallest order statistic of an `ns`-row uniform sample whose rank among the `n` rows is >= k with high
// probability: P(rank < k) = P(Poisson(k*ns/n) >= j0) < eps (2e-5 by default)
uint32_t tensor_j0(uint32_t k, uint64_t ns, uint64_t n, double eps) {
    uint32_t j0 = 1;
    const double x = (double)k * (double)ns / (double)n;
    double term = exp(-x), cdf = term;
    while (1.0 - cdf >= eps && j0 < 4096) {
        term *= x / j0;
        cdf += term;
        ++j0;
    }
    return (uint32_t)std::min<uint64_t>(j0, ns);
}

}  // namespace vdb

// per-call query context of the tensor path: padded fp32 copy (exact rerank), the MMA operand q~, ||q||^2, the
// pruning-bound coefficients and the TMA descriptor of the operand
struct vdb_tq {
    const vdb_dataset* ds = nullptr;
    const void* d_queries = nullptr;
    uint32_t nq = 0, qpitch = 0, op_pitch = 0;
    int kind = 0;
    cudaStream_t st = nullptr;
    vdb::DevBuf qcopy, qop, qsq, qerr, qscale, qbad, qd, qab, qb, cnt;
    vdb::QueryTile qtile;   // cosine: ||q|| exactly as the streaming scan computes it
    CUtensorMap mq;
    uint32_t cap = 0;
    int ctas = 2;   // CTAs per work unit: pairs (M = 256 queries), single CTAs (M = 128) for batches of <= 128 queries
    // row-sharded search with the global pruning bound: the filter is split around one peer exchange
    // (tensor_filter_begin / tensor_filter_finish); these live from the one to the other
    vdb::DevBuf f_cand, f_stats;
    uint32_t f_k = 0, f_m = 0, f_T = 0;
    const float* f_tau = nullptr;
};

namespace vdb {
// tq->cnt: [nq] candidate-list lengths, then (8-byte aligned) the number of reranked candidates (u64) and the number of
// queries that failed the completeness check (u32). The filter clears all of it with one memset.
static size_t tq_cnt_bytes(uint32_t nq) { return ((size_t)round_up(nq, 2u) + 6) * 4; }
// ... and the number of (query, row) pairs the pruning kernel handed to the rerank (u64)
static uint64_t* tq_pairs_ptr(const vdb_tq* tq) { return reinterpret_cast<uint64_t*>(tq->cnt.as<uint32_t>() + round_up(tq->nq, 2u) + 4); }
uint64_t* tensor_cand_total_ptr(const vdb_tq* tq) { return reinterpret_cast<uint64_t*>(tq->cnt.as<uint32_t>() + round_up(tq->nq, 2u)); }
uint32_t* tensor_nredo_ptr(const vdb_tq* tq) { return tq->cnt.as<uint32_t>() + round_up(tq->nq, 2u) + 2; }

}  // namespace vdb

namespace vdb {

vdb_tq* tensor_begin(const vdb_dataset* ds, const void* d_queries, uint32_t nq, cudaStream_t st, bool any_size) {
    VDB_REQUIRE(any_size || flat_gemm_supported(ds, nq, 1), "tensor-core Flat path: unsupported dataset");
    ensure_side_arrays(ds, st, any_size ? ds->op_kind : -1);
    const uint32_t dim = ds->dim;
    const float acc = (float)dim * ldexpf(1.0f, -23);   // fp32 accumulation of the contraction
    auto tq = new vdb_tq();
    try {
        tq->ds = ds;
        tq->d_queries = d_queries;
        tq->nq = nq;
        tq->st = st;
        tq->kind = ds->op_kind;
        tq->qpitch = round_up(dim, 4u);
        tq->op_pitch = tq->kind == KIND_F16 ? round_up(dim, 8u) : tq->qpitch;
        tq->qcopy = DevBuf((size_t)nq * tq->qpitch * 4, st);
        tq->qop = DevBuf((size_t)nq * tq->op_pitch * (tq->kind == KIND_F16 ? 2 : 4), st);
        for (DevBuf* b : {&tq->qsq, &tq->qerr, &tq->qscale, &tq->qbad, &tq->qd, &tq->qab, &tq->qb})
            *b = DevBuf((size_t)nq * 4, st);
        tq->cnt = DevBuf(tq_cnt_bytes(nq), st);   // list lengths + the call's two counters, cleared by one memset
        const bool l2 = ds->metric == VDB_L2SQR;
        const uint32_t pgrid = ceil_div(nq, 8u);   // 8 warps per CTA, one query each
        auto prep = [&](auto kern, auto* src) {
            kern<<<pgrid, 256, 0, st>>>(src, nq, dim, tq->qpitch, tq->op_pitch, tq->qcopy.as<float>(), tq->qop.p, tq->qsq.as<float>(),
                                        tq->qerr.as<float>(), tq->qscale.as<float>(), tq->qbad.as<uint32_t>());
            VDB_LAUNCHED();
        };
        if (ds->dtype == VDB_U8) prep(tq_prepare_kernel<uint8_t, KIND_F16>, (const uint8_t*)d_queries);
        else if (tq->kind == KIND_F16) prep(tq_prepare_kernel<float, KIND_F16>, (const float*)d_queries);
        else prep(tq_prepare_kernel<float, KIND_TF32>, (const float*)d_queries);
        if (!l2) tq->qtile = prepare_queries(ds, d_queries, nq, st);
        tq_coeff_kernel<<<ceil_div(nq, 256u), 256, 0, st>>>(tq->qsq.as<float>(), tq->qerr.as<float>(), tq->qscale.as<float>(),
                                                            l2 ? nullptr : tq->qtile.qcache.as<float>(), nq, acc, ds->op_scale,
                                                            tq->qd.as<float>(), tq->qab.as<float>(), tq->qb.as<float>());
        VDB_LAUNCHED();
        tq->mq = make_op_map(tq->kind, tq->qop.p, dim, nq, (uint64_t)tq->op_pitch * (tq->kind == KIND_F16 ? 2 : 4), GM);
        // a batch that fits one 128-query tile runs on single CTAs: a CTA pair would spend half of its MMAs on padding
        // (the pass is then HBM-bound on the operand rows instead of tensor-bound)
        static const bool small_single = !(getenv("VDB_GEMM_SMALL_PAIRS") && atoi(getenv("VDB_GEMM_SMALL_PAIRS")));
        tq->ctas = (small_single && nq <= (uint32_t)GM) ? 1 : gemm_ctas();
    } catch (...) {
        delete tq;
        throw;
    }
    return tq;
}
void tensor_end(vdb_tq* tq) { delete tq; }
void operand_info(const vdb_dataset* ds, int* kind, float* scale, float* mean_norm, float* mean_ex, uint64_t* side_bytes) {
    std::lock_guard<std::mutex> lk(g_side_mu);
    const bool built = ds->d_sqnorm && ds->side_n == ds->n;
    if (kind) *kind = built ? ds->op_kind : -1;
    if (scale) *scale = ds->op_scale;
    if (mean_norm) *mean_norm = ds->mean_norm;
    if (mean_ex) *mean_ex = ds->mean_ex;
    if (side_bytes)
        *side_bytes = built ? ds->n * 12 + (ds->op_kind == KIND_F16 ? ds->n * (uint64_t)ds->op_pitch * 2 : 0) +
                                  (uint64_t)ds->sample_n * (op_row_bytes_of(ds) + 12)
                            : 0;
}
void tensor_info(const vdb_dataset* ds, uint64_t* n, uint32_t* sample_n, float* mean_norm, float* mean_ex, cudaStream_t st) {
    VDB_REQUIRE(flat_gemm_supported(ds, 1, 1), "tensor-core Flat path: unsupported dataset");
    ensure_side_arrays(ds, st);
    if (n) *n = ds->n;
    if (sample_n) *sample_n = ds->sample_n;
    if (mean_norm) *mean_norm = ds->mean_norm;
    if (mean_ex) *mean_ex = ds->mean_ex;
}

static GemmParams base_params(const vdb_tq* tq) {
    GemmParams p{};
    p.nq = tq->nq;
    p.kblocks = kblocks_of(tq->kind, tq->ds->dim);
    p.qd = tq->qd.as<float>();
    p.qab = tq->qab.as<float>();
    p.qb = tq->qb.as<float>();
    p.qnorm = tq->ds->metric == VDB_COSINE ? tq->qtile.qcache.as<float>() : nullptr;
    // The filter over the whole set passes ~0.05 % of its scores: there the per-score path (1) is faster (A/B in one process,
    // 1M x 960, 10k queries: 14.7 vs 16.6 ms per pass with the per-thread mask path 0, 16.4 vs 16.9 with the staged path 2);
    // the sample pass of the two-level selection passes ~0.6 % and takes the staged path. At 0.34 % (a 125k-row shard under
    // its LOCAL threshold) staged is 2.9 vs 4.0-4.6 ms. VDB_GEMM_RARE_PER_SCORE = 0 / 1 / 2 overrides both (read per call).
    const char* rare = getenv("VDB_GEMM_RARE_PER_SCORE");
    p.rare_per_score = rare ? (uint32_t)std::min(2, std::max(0, atoi(rare))) : 1u;
    return p;
}

// SAMPLE: the j best sampled rows of every query by pruning score, re-evaluated exactly: d_jkeys [nq][j] = keys
// (exact distance, global row id), ascending, KEY_NONE padded
void tensor_sample_keys(vdb_tq* tq, uint32_t j, uint64_t* d_jkeys, float* d_tau, uint32_t j0) {
    const vdb_dataset* ds = tq->ds;
    cudaStream_t st = tq->st;
    const uint64_t ns = ds->sample_n;
    VDB_REQUIRE(j >= 1 && j <= ns, "sample order statistic %u out of range (sample %llu)", j, (unsigned long long)ns);
    const CUtensorMap ms = make_op_map(tq->kind, ds->d_sample, ds->dim, ns, op_row_bytes_of(ds), GN / tq->ctas);
    GemmParams ps = base_params(tq);
    ps.nrows = ns;
    ps.row_stride = 1;
    ps.sqnorm = ds->d_sample_sq;
    ps.rnorm = ds->d_sample_rn;
    ps.ex = ds->d_sample_ex;
    // The top-G_TOPJ epilogue pays a warp-wide insertion whenever ANY of its 32 queries sees a new best: ~512 (1 + ln(T / 512))
    // times per slab of T rows, i.e. on nearly every row of a 1024-row slab but on a quarter of an 8192-row one. Long slabs
    // (as long as the items still cover the SMs about twice) keep the sample pass near the filter pass's rate per row.
    static const uint32_t stps_env = getenv("VDB_GEMM_SAMPLE_TPS") ? (uint32_t)atoi(getenv("VDB_GEMM_SAMPLE_TPS")) : 0;
    uint32_t stps = 4;
    if (j <= (uint32_t)G_TOPJ) {
        const uint32_t ntiles = (uint32_t)ceil_div<uint64_t>(ns, GN), nqt = ceil_div(tq->nq, (uint32_t)(GM * tq->ctas));
        const uint32_t units = (uint32_t)sm_count() / tq->ctas;
        // (plan_gemm still caps the slab at ceil(tiles x query tiles / units), so small batches keep one tile per CTA; a
        // floor of 12 instead of 4 gives a 125k-row shard 2 slabs instead of 5: sample phase 0.333 -> 0.296 ms)
        stps = stps_env ? stps_env : std::max(12u, std::min(32u, (uint32_t)((uint64_t)ntiles * nqt / (2 * units))));
    }
    plan_gemm(ps, tq->ctas, stps);
    const uint64_t cnt = (uint64_t)tq->nq * j;
    DevBuf skeys(cnt * 8, st);
    // Two-level selection (default): the register top-G_TOPJ epilogue (mode 2) runs at a fraction of the MMA rate (its
    // insertions are warp-wide: 4 ms for 32768 sampled rows x 10 000 queries, a fifth of the whole step), and storing
    // every sampled score (mode 0) is nq * ns * 8 bytes. Instead: (1) every SUB-th sample row is scored (~1024 rows) and
    // the j1-th smallest score per query - j1 = the order statistic of the sub-sample whose rank in the sample is >= j
    // with probability > 1 - 1e-5 - becomes a coarse threshold; (2) the whole sample is FILTERED against it at the full
    // MMA rate (mode 1, ~j1 * SUB survivors per query); (3) the j smallest survivors are selected. A query that ends up
    // with fewer than j survivors (or an overflowed list) only gets a looser tau: the completeness check of the search
    // decides, as always.
    // Batches of <= 128 queries (single CTAs, HBM-bound on the operand rows) keep the one-launch register epilogue.
    // End of round 2: with the per-thread insertion loop of the top-G_TOPJ epilogue (mode 2) ONE launch over the whole sample
    // beats the two levels whenever j fits the registers (10k queries x 33k sampled rows: 0.87 + 0.22 ms against 1.11 + 0.35
    // for gemms + merges; a 125k-row shard 0.33 against 0.46 ms per sample phase), so the two levels are now only the way
    // to handle j > G_TOPJ (k beyond ~200). VDB_GEMM_SAMPLE_2L=1 forces them as before, =0 forbids them.
    const char* two_level_s = getenv("VDB_GEMM_SAMPLE_2L");   // read per call: the tests toggle it in one process
    const bool two_level_forced = two_level_s && atoi(two_level_s);
    const bool two_level = two_level_s ? two_level_forced : j > (uint32_t)G_TOPJ;
    static const uint32_t sub_env = getenv("VDB_GEMM_SAMPLE_SUBN") ? (uint32_t)atoi(getenv("VDB_GEMM_SAMPLE_SUBN")) : 0;
    const uint32_t SUB = (uint32_t)std::max<uint64_t>(2, ns / (sub_env ? sub_env : 1024));   // sub-sample of ~1024 rows
    if (two_level && ns >= 2048 && (tq->ctas == 2 || j > (uint32_t)G_TOPJ)) {
        const uint64_t ns1 = ns / SUB;
        const uint32_t j1 = tensor_j0(j, ns1, ns, 1e-5);
        const CUtensorMap m1 = make_op_map(tq->kind, ds->d_sample, ds->dim, ns1, op_row_bytes_of(ds) * SUB, GN / tq->ctas);
        GemmParams p1 = ps;
        p1.nrows = ns1;
        p1.row_stride = SUB;
        plan_gemm(p1, tq->ctas);
        DevBuf k1((size_t)tq->nq * j1 * 8, st), tau1((size_t)tq->nq * 4, st);
        if (j1 <= (uint32_t)G_TOPJ) {   // ~1024 rows: the register epilogue costs 1/32 of what it did on the whole sample
            DevBuf part1((size_t)tq->nq * p1.nslabs * G_TOPJ * 8, st);
            p1.out_keys = part1.as<uint64_t>();
            launch_gemm(2, ds->metric, tq->kind, tq->mq, m1, p1, st, tq->ctas, "flat_gemm_sample");
            launch_merge_keys(part1.as<uint64_t>(), p1.nslabs, tq->nq, G_TOPJ, false, j1, k1.as<uint64_t>(), nullptr, nullptr, nullptr, st);
        } else {
            DevBuf all1((size_t)tq->nq * ns1 * 8, st);
            p1.out_keys = all1.as<uint64_t>();
            launch_gemm(0, ds->metric, tq->kind, tq->mq, m1, p1, st, tq->ctas, "flat_gemm_sample");
            launch_merge_keys(all1.as<uint64_t>(), 1, tq->nq, (uint32_t)ns1, false, j1, k1.as<uint64_t>(), nullptr, nullptr, nullptr, st);
        }
        tau_coarse_kernel<<<ceil_div(tq->nq, 256u), 256, 0, st>>>(k1.as<uint64_t>(), tq->nq, j1, tau1.as<float>());
        VDB_LAUNCHED();
        const uint32_t cap2 = next_pow2(std::max<uint32_t>(256, 4 * j1 * SUB));
        DevBuf cand2((size_t)tq->nq * cap2 * 8, st), cnt2((size_t)tq->nq * 4, st);
        VDB_CUDA(cudaMemsetAsync(cnt2.p, 0, (size_t)tq->nq * 4, st));
        GemmParams p2 = ps;
        p2.tau = tau1.as<float>();
        p2.cand_cnt = cnt2.as<uint32_t>();
        p2.cand = cand2.as<uint64_t>();
        p2.cap = cap2;
        // ~0.6-1.6 % of the sample's scores pass the coarse threshold: staged slots (A/B on one box, 10k queries: 1.39 ->
        // 1.25 ms for the 33k-row sample; the per-thread mask path 0 and the per-score path 1 stay selectable)
        if (!getenv("VDB_GEMM_RARE_PER_SCORE")) p2.rare_per_score = 2;
        plan_gemm(p2, tq->ctas);
        launch_gemm(1, ds->metric, tq->kind, tq->mq, ms, p2, st, tq->ctas, "flat_gemm_sample");
        cand_sortable_kernel<<<tq->nq, 128, 0, st>>>(cand2.as<uint64_t>(), cnt2.as<uint32_t>(), cap2);
        VDB_LAUNCHED();
        launch_merge_keys(cand2.as<uint64_t>(), 1, tq->nq, cap2, false, j, skeys.as<uint64_t>(), nullptr, nullptr, nullptr, st,
                          nullptr, cnt2.as<uint32_t>());
    } else if (j <= (uint32_t)G_TOPJ) {
        // the epilogue keeps each query's G_TOPJ smallest scores per slab in registers: nothing but
        // nq * nslabs * G_TOPJ keys ever reaches HBM
        DevBuf part((size_t)tq->nq * ps.nslabs * G_TOPJ * 8, st);
        ps.out_keys = part.as<uint64_t>();
        launch_gemm(2, ds->metric, tq->kind, tq->mq, ms, ps, st, tq->ctas, "flat_gemm_sample");
        launch_merge_keys(part.as<uint64_t>(), ps.nslabs, tq->nq, G_TOPJ, false, j, skeys.as<uint64_t>(), nullptr, nullptr, nullptr, st);
    } else {
        DevBuf all((size_t)tq->nq * ns * 8, st);
        ps.out_keys = all.as<uint64_t>();
        launch_gemm(0, ds->metric, tq->kind, tq->mq, ms, ps, st, tq->ctas, "flat_gemm_sample");
        launch_merge_keys(all.as<uint64_t>(), 1, tq->nq, (uint32_t)ns, false, j, skeys.as<uint64_t>(), nullptr, nullptr, nullptr, st);
    }
    // exact fp32 distances of those rows (the rerank's arithmetic), sorted ascending per query
    DevBuf qidx(cnt * 4, st), rid(cnt * 4, st), valid(cnt, st), dist(cnt * 4, st), ekeys(cnt * 8, st);
    sample_pairs_kernel<<<(uint32_t)std::min<uint64_t>(ceil_div<uint64_t>(cnt, 256), 65535), 256, 0, st>>>(
        skeys.as<uint64_t>(), cnt, j, ds->d_sample_row, qidx.as<uint32_t>(), rid.as<uint32_t>(), valid.as<uint8_t>());
    VDB_LAUNCHED();
    exact_pair_distances_masked(ds, tq->qcopy.p, tq->qpitch, qidx.as<uint32_t>(), rid.as<uint32_t>(), valid.as<uint8_t>(), cnt,
                                dist.as<float>(), st, nullptr, ds->metric == VDB_COSINE ? tq->qtile.qcache.as<float>() : nullptr);
    const float* qsq = ds->metric == VDB_COSINE ? nullptr : tq->qsq.as<float>();
    if (j <= 32) {
        VDB_REQUIRE(!d_tau || (j0 >= 1 && j0 <= j), "j0 out of range");
        sample_finish_kernel<<<ceil_div(tq->nq, 8u), 256, 0, st>>>(dist.as<float>(), rid.as<uint32_t>(), valid.as<uint8_t>(),
                                                                  (uint32_t)ds->id_base, tq->nq, j, d_jkeys, j0, qsq, d_tau);
        VDB_LAUNCHED();
        return;
    }
    rekey_based(dist.as<float>(), rid.as<uint32_t>(), (uint32_t)ds->id_base, valid.as<uint8_t>(), cnt, ekeys.as<uint64_t>(), st);
    launch_merge_keys(ekeys.as<uint64_t>(), 1, tq->nq, j, false, j, d_jkeys, nullptr, nullptr, nullptr, st);
    if (d_tau) {
        tau_exact_kernel<<<ceil_div(tq->nq, 256u), 256, 0, st>>>(d_jkeys, tq->nq, j, j0, qsq, d_tau);
        VDB_LAUNCHED();
    }
}

// TAU: merge `nlists` shards' [nq][j] exact sample keys (list-major) and set tau_q from the j0-th smallest
void tensor_tau(vdb_tq* tq, const uint64_t* d_lists, uint32_t nlists, uint32_t j, uint32_t j0, float* d_tau) {
    cudaStream_t st = tq->st;
    VDB_REQUIRE(j0 >= 1 && j0 <= (uint64_t)j * nlists, "j0 out of range");
    const uint32_t jj = std::min<uint64_t>(j0, (uint64_t)j * nlists);
    const float* qsq = tq->ds->metric == VDB_COSINE ? nullptr : tq->qsq.as<float>();
    if (nlists == 1) {   // a single ascending [nq][j] list: its jj-th entry is the order statistic, nothing to merge
        tau_exact_kernel<<<ceil_div(tq->nq, 256u), 256, 0, st>>>(d_lists, tq->nq, j, jj, qsq, d_tau);
        VDB_LAUNCHED();
        return;
    }
    DevBuf merged((size_t)tq->nq * jj * 8, st);
    launch_merge_sorted(d_lists, nlists, tq->nq, j, jj, merged.as<uint64_t>(), nullptr, nullptr, nullptr, st);  // per-shard lists are ascending
    tau_exact_kernel<<<ceil_div(tq->nq, 256u), 256, 0, st>>>(merged.as<uint64_t>(), tq->nq, jj, jj, qsq, d_tau);
    VDB_LAUNCHED();
}

// number of sampled rows re-evaluated per query for the order statistic j0: a few more than j0 when they come for free
// (the epilogue keeps G_TOPJ per slab anyway), because the j0-th smallest EXACT distance need not be among the j0
// smallest pruning scores
uint32_t tensor_sample_j(uint32_t j0, uint64_t sample_n) {
    const uint32_t j = j0 <= (uint32_t)G_TOPJ ? std::min<uint32_t>(G_TOPJ, j0 + 4) : j0 + j0 / 4;
    return (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(j, sample_n));
}

// side stream of the filter pass (per host thread and device): reranks row part i under the contraction of part i + 1
struct SideStream {
    int device = -1;
    cudaStream_t s = nullptr;
    cudaEvent_t ev = nullptr, ev2 = nullptr;
    void ensure(int dev) {
        if (device == dev) return;
        release();
        VDB_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
        VDB_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        VDB_CUDA(cudaEventCreateWithFlags(&ev2, cudaEventDisableTiming));
        device = dev;
    }
    void release() {
        if (device < 0) return;
        cudaStreamDestroy(s);
        cudaEventDestroy(ev);
        cudaEventDestroy(ev2);
        device = -1;
    }
    ~SideStream() { release(); }
};
// drains the side stream if the filter pass unwinds early (its scratch is freed in stream order on the MAIN stream)
struct SideDrain {
    cudaStream_t s;
    bool armed;
    ~SideDrain() {
        if (armed) cudaStreamSynchronize(s);
    }
};
// FILTER + RERANK: rows with S' < tau_q -> exact distances -> this shard's k best keys per query.
// d_overflow[q] = 1 when the candidate list of q overflowed (its result is then incomplete).
void tensor_filter_keys(vdb_tq* tq, uint32_t k, uint32_t j0_local_hint, const float* d_tau, uint64_t* d_keys,
                        uint32_t* d_overflow, const TensorCheck* check) {
    const vdb_dataset* ds = tq->ds;
    cudaStream_t st = tq->st;
    const uint32_t nq = tq->nq, dim = ds->dim;
    const uint64_t ns = ds->sample_n;
    const uint32_t cap = (uint32_t)next_pow2((uint32_t)std::min<uint64_t>(
        ds->n, std::max<uint64_t>(8ull * std::max(j0_local_hint, 1u) * (ds->n / ns), 8192)));
    tq->cap = cap;
    DevBuf cand((size_t)nq * cap * 8, st);
    VDB_CUDA(cudaMemsetAsync(tq->cnt.p, 0, tq_cnt_bytes(nq), st));
    const CUtensorMap mx = make_op_map(tq->kind, op_rows_of(ds), dim, ds->n, op_row_bytes_of(ds), GN / tq->ctas);
    GemmParams pf = base_params(tq);
    pf.sqnorm = ds->d_sqnorm;
    pf.rnorm = ds->d_lo;
    pf.ex = ds->d_ex;
    pf.nrows = ds->n;
    pf.row_stride = 1;
    pf.tau = d_tau;
    pf.cand_cnt = tq->cnt.as<uint32_t>();
    pf.cand = cand.as<uint64_t>();
    pf.cap = cap;
    plan_gemm(pf, tq->ctas);
    // The contraction is tensor-bound and leaves HBM idle, the exact rerank of its candidates is an HBM-bound gather:
    // the pass is cut into row parts (slab ranges, so nothing is streamed twice) and the rerank of part i runs on a
    // side stream under the contraction of part i + 1 (the rerank CTAs fit next to the one persistent contraction
    // CTA per SM: 192 threads x <= 87 registers and no free shared memory needed). A part's candidates are the entries
    // [snap[i-1][q], snap[i][q]) of every query's list (counter snapshots taken between the launches); their exact
    // keys are written back over the entries they came from, so the final selection reads one [nq][cap] array.
    const uint32_t total_slabs = pf.nslabs;
    const char* parts_s = getenv("VDB_GEMM_PARTS");   // read per call: the probe scripts sweep it
    const uint32_t parts_env = parts_s ? (uint32_t)atoi(parts_s) : 0;
    const uint64_t tile_units = (uint64_t)pf.ntiles * pf.nqt;   // 256 x 256 (or 128 x 256) score tiles of the pass
    // measured (scripts/probe_parts.py, probe_shard_phases.py): 1M x 960, 10k queries 39.2 -> 38.6 ms with 3 parts (the
    // step is power-capped, so hiding the gathers slows the contraction by almost as much); a 125k-row shard with its
    // own thresholds 9.6 -> 8.0 ms; the same shard under the global thresholds of an 8-way split 4.87 -> 4.77 ms;
    // 8 parts cost more in launch tails than they hide
    // Round 2: with 2-byte operands the contraction runs at the L2 -> SM bandwidth, which the concurrent gathers
    // compete for (1M x 960, 10k queries: 20.6 ms with 3 parts, 19.8 ms unsplit), and the bound-based pruning below cuts
    // the rerank to a fraction, so the pass is NOT split by default any more (VDB_GEMM_PARTS=n brings the parts back,
    // without pruning).
    (void)tile_units;
    uint32_t parts = parts_env ? parts_env : 1u;
    parts = std::max(1u, std::min(parts, total_slabs));
    const char* prune_s = getenv("VDB_GEMM_PRUNE");   // read per call: the tests toggle it in one process
    const bool prune_on = !(prune_s && !atoi(prune_s));
    const bool prune = prune_on && parts == 1 && (size_t)cap * 4 <= 96 * 1024;
    // part i covers a share proportional to ratio^i of the slabs: the rerank of the LAST part is the only one that is
    // not hidden under a contraction launch, so later parts are made smaller
    const char* ratio_s = getenv("VDB_GEMM_PART_RATIO");
    const double ratio = ratio_s ? std::max(0.2, std::min(1.0, atof(ratio_s))) : 1.0;
    std::vector<uint32_t> part_end(parts);
    {
        double total_w = 0, w = 1.0, acc_w = 0;
        for (uint32_t i = 0; i < parts; ++i, w *= ratio) total_w += w;
        w = 1.0;
        for (uint32_t i = 0; i < parts; ++i, w *= ratio) {
            acc_w += w;
            part_end[i] = i + 1 == parts ? total_slabs : std::max<uint32_t>(i + 1, (uint32_t)std::llround(total_slabs * acc_w / total_w));
        }
        for (uint32_t i = 0; i + 1 < parts; ++i) {   // every part gets at least one slab
            if (i) part_end[i] = std::max(part_end[i], part_end[i - 1] + 1);
            part_end[i] = std::min(part_end[i], total_slabs - (parts - 1 - i));
        }
    }
    static thread_local SideStream side;
    if (parts > 1) side.ensure(ds->device);
    cudaStream_t rs = parts > 1 ? side.s : st;   // rerank stream
    DevBuf snaps((size_t)parts * nq * 4, st);
    const uint64_t total = (uint64_t)nq * cap;  // capacity bound; the live counts stay on the device
    DevBuf off((size_t)(nq + 1) * 8, st), qidx(total * 4, st), rid(total * 4, st), dist(total * 4, st);
    SideDrain drain{rs, parts > 1};
    if (parts > 1) {   // the side stream must not touch the scratch before the allocations above are ordered
        VDB_CUDA(cudaEventRecord(side.ev, st));
        VDB_CUDA(cudaStreamWaitEvent(rs, side.ev, 0));
    }
    for (uint32_t part = 0; part < parts; ++part) {
        const uint32_t s0 = part ? part_end[part - 1] : 0u, s1 = part_end[part];
        GemmParams pp = pf;
        pp.slab0 = s0;
        pp.nslabs = s1 - s0;
        launch_gemm(1, ds->metric, tq->kind, tq->mq, mx, pp, st, tq->ctas);
        uint32_t* snap = snaps.as<uint32_t>() + (size_t)part * nq;
        const uint32_t* prev = part ? snap - nq : nullptr;
        if (prune) {   // snap = the pruned list lengths
            auto kern = ds->metric == VDB_COSINE ? cand_prune_kernel<VDB_COSINE> : cand_prune_kernel<VDB_L2SQR>;
            const size_t sm = (size_t)cap * 4;
            if (sm > 48 * 1024) VDB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
            kern<<<nq, 256, sm, st>>>(cand.as<uint64_t>(), tq->cnt.as<uint32_t>(), cap, k, ds->d_lo, ds->d_ex, tq->qab.as<float>(),
                                      tq->qb.as<float>(), ds->metric == VDB_COSINE ? nullptr : tq->qsq.as<float>(), snap,
                                      off.as<uint64_t>(), reinterpret_cast<unsigned long long*>(tq_pairs_ptr(tq)),
                                      qidx.as<uint32_t>(), rid.as<uint32_t>(), nullptr, 0u, 0u, 0u);
            VDB_LAUNCHED();
        } else {
            VDB_CUDA(cudaMemcpyAsync(snap, tq->cnt.p, (size_t)nq * 4, cudaMemcpyDeviceToDevice, st));
        }
        if (parts > 1) {
            VDB_CUDA(cudaEventRecord(side.ev, st));
            VDB_CUDA(cudaStreamWaitEvent(rs, side.ev, 0));
        }
        // exact rerank of the part's candidates (compacted: only the valid pairs are touched)
        const uint64_t* n_pairs = prune ? tq_pairs_ptr(tq) : off.as<uint64_t>() + nq;   // pruned: pairs came with the pruning
        if (!prune) {
            part_offsets_kernel<<<1, 1024, 0, rs>>>(prev, snap, nq, cap, off.as<uint64_t>());
            VDB_LAUNCHED();
            part_to_pairs_kernel<<<nq, 256, 0, rs>>>(cand.as<uint64_t>(), prev, snap, cap, off.as<uint64_t>(), qidx.as<uint32_t>(),
                                                     rid.as<uint32_t>());
            VDB_LAUNCHED();
        }
        exact_pair_distances_masked(ds, tq->qcopy.p, tq->qpitch, qidx.as<uint32_t>(), rid.as<uint32_t>(), nullptr, total,
                                    dist.as<float>(), rs, n_pairs,
                                    ds->metric == VDB_COSINE ? tq->qtile.qcache.as<float>() : nullptr);
        part_rekey_kernel<<<(uint32_t)sm_count() * 8, 256, 0, rs>>>(dist.as<float>(), qidx.as<uint32_t>(), rid.as<uint32_t>(),
                                                                   off.as<uint64_t>(), nq, prev, cap, (uint32_t)ds->id_base,
                                                                   cand.as<uint64_t>(), prune ? n_pairs : nullptr);
        VDB_LAUNCHED();
    }
    if (parts > 1) {
        VDB_CUDA(cudaEventRecord(side.ev2, rs));
        VDB_CUDA(cudaStreamWaitEvent(st, side.ev2, 0));
    }
    drain.armed = false;   // from here on the main stream is ordered after the side stream
    // the k best exact keys of every query's list (its first min(cnt, cap) entries)
    const uint32_t* final_cnt = prune ? snaps.as<uint32_t>() : tq->cnt.as<uint32_t>();   // <= cap when pruned
    // the merge's CTA of a query also sets its overflow flag, counts its reranked rows and (single-GPU calls) runs the
    // completeness check on the keys it still holds: overflow_kernel + cand_total_kernel + check_kernel + a memset less
    MergeFinish fin;
    fin.cnt_raw = tq->cnt.as<uint32_t>();
    fin.qbad = tq->qbad.as<uint32_t>();
    fin.cap = cap;
    fin.overflow = d_overflow;
    fin.cand_total = reinterpret_cast<unsigned long long*>(tensor_cand_total_ptr(tq));
    if (check) {
        fin.tau = d_tau;
        fin.qsq = ds->metric == VDB_COSINE ? nullptr : tq->qsq.as<float>();
        fin.n_total = check->n_total;
        fin.force_mod = g_debug_force_redo.load();
        fin.redo = check->d_redo;
        fin.nredo = tensor_nredo_ptr(tq);
    }
    launch_merge_keys(cand.as<uint64_t>(), 1, nq, cap, false, k, d_keys, nullptr, nullptr, nullptr, st, nullptr, final_cnt, &fin);
}

// ---- the filter, split around ONE peer exchange (row-sharded search) -----------------------------------------------------
// A shard can only prune its candidate list against ITS k-th upper bound, and holds fewer than k candidates per query once
// the set is split 4 or 8 ways: nothing is pruned and the shards together gather ~4x the rows the unsharded call gathers
// (8 x B200, 10k queries, k = 100: 533 rows per query against 129). tensor_filter_begin runs the contraction and leaves T
// order statistics of the list's upper bounds per query (ranks m, 2m, ..., T m >= k; prune_stats_kernel); the caller makes
// every shard's [nq][T] block visible to every shard; tensor_filter_finish cuts the list against the bound they certify
// together (cand_prune_kernel, gstats branch) and reranks what is left. Results are the bits of the unsplit call: only rows
// that provably are not among the k best of the WHOLE set are dropped.
constexpr uint32_t GPRUNE_M = 4;
bool tensor_filter_split_supported(const vdb_tq* tq, uint32_t k) {
    const char* e = getenv("VDB_MG_GLOBAL_PRUNE");   // read per call: the tests toggle it in one process
    if (e && !atoi(e)) return false;
    const char* parts_s = getenv("VDB_GEMM_PARTS");
    const char* prune_s = getenv("VDB_GEMM_PRUNE");
    if ((parts_s && atoi(parts_s) > 1) || (prune_s && !atoi(prune_s))) return false;
    return k >= 1 && k <= 256 && tq->nq > 0;
}
const uint32_t* tensor_filter_begin(vdb_tq* tq, uint32_t k, const float* d_tau, uint32_t* T_out) {
    const vdb_dataset* ds = tq->ds;
    cudaStream_t st = tq->st;
    const uint32_t nq = tq->nq;
    const uint32_t cap = (uint32_t)next_pow2((uint32_t)std::min<uint64_t>(ds->n, 8192));   // as tensor_filter_keys with hint 0
    tq->cap = cap;
    tq->f_k = k;
    tq->f_m = GPRUNE_M;
    tq->f_T = ceil_div(k, GPRUNE_M);
    tq->f_tau = d_tau;
    tq->f_cand = DevBuf((size_t)nq * cap * 8, st);
    tq->f_stats = DevBuf((size_t)nq * tq->f_T * 4, st);
    VDB_CUDA(cudaMemsetAsync(tq->cnt.p, 0, tq_cnt_bytes(nq), st));
    const CUtensorMap mx = make_op_map(tq->kind, op_rows_of(ds), ds->dim, ds->n, op_row_bytes_of(ds), GN / tq->ctas);
    GemmParams pf = base_params(tq);
    pf.sqnorm = ds->d_sqnorm;
    pf.rnorm = ds->d_lo;
    pf.ex = ds->d_ex;
    pf.nrows = ds->n;
    pf.row_stride = 1;
    pf.tau = d_tau;
    pf.cand_cnt = tq->cnt.as<uint32_t>();
    pf.cand = tq->f_cand.as<uint64_t>();
    pf.cap = cap;
    plan_gemm(pf, tq->ctas);
    launch_gemm(1, ds->metric, tq->kind, tq->mq, mx, pf, st, tq->ctas);
    auto kern = ds->metric == VDB_COSINE ? prune_stats_kernel<VDB_COSINE> : prune_stats_kernel<VDB_L2SQR>;
    kern<<<nq, 256, 0, st>>>(tq->f_cand.as<uint64_t>(), tq->cnt.as<uint32_t>(), cap, tq->f_m, tq->f_T, ds->d_lo, ds->d_ex,
                             tq->qab.as<float>(), tq->qb.as<float>(), ds->metric == VDB_COSINE ? nullptr : tq->qsq.as<float>(),
                             tq->f_stats.as<uint32_t>());
    VDB_LAUNCHED();
    *T_out = tq->f_T;
    return tq->f_stats.as<uint32_t>();
}
// d_stats_all: [shards][nq][T] (every shard's block, this one's included)
void tensor_filter_finish(vdb_tq* tq, const uint32_t* d_stats_all, uint32_t shards, uint64_t* d_keys, uint32_t* d_overflow) {
    const vdb_dataset* ds = tq->ds;
    cudaStream_t st = tq->st;
    const uint32_t nq = tq->nq, cap = tq->cap, k = tq->f_k;
    VDB_REQUIRE(tq->f_cand.p && shards >= 1 && (size_t)shards * tq->f_T * 4 <= (size_t)cap * 4, "tensor_filter_finish without begin");
    const uint64_t total = (uint64_t)nq * cap;
    DevBuf snap((size_t)nq * 4, st), off((size_t)(nq + 1) * 8, st), qidx(total * 4, st), rid(total * 4, st), dist(total * 4, st);
    {
        auto kern = ds->metric == VDB_COSINE ? cand_prune_kernel<VDB_COSINE> : cand_prune_kernel<VDB_L2SQR>;
        const size_t sm = (size_t)cap * 4;
        if (sm > 48 * 1024) VDB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
        kern<<<nq, 256, sm, st>>>(tq->f_cand.as<uint64_t>(), tq->cnt.as<uint32_t>(), cap, k, ds->d_lo, ds->d_ex, tq->qab.as<float>(),
                                  tq->qb.as<float>(), ds->metric == VDB_COSINE ? nullptr : tq->qsq.as<float>(), snap.as<uint32_t>(),
                                  off.as<uint64_t>(), reinterpret_cast<unsigned long long*>(tq_pairs_ptr(tq)), qidx.as<uint32_t>(),
                                  rid.as<uint32_t>(), d_stats_all, shards, tq->f_T, nq);
        VDB_LAUNCHED();
    }
    const uint64_t* n_pairs = tq_pairs_ptr(tq);
    exact_pair_distances_masked(ds, tq->qcopy.p, tq->qpitch, qidx.as<uint32_t>(), rid.as<uint32_t>(), nullptr, total, dist.as<float>(),
                                st, n_pairs, ds->metric == VDB_COSINE ? tq->qtile.qcache.as<float>() : nullptr);
    part_rekey_kernel<<<(uint32_t)sm_count() * 8, 256, 0, st>>>(dist.as<float>(), qidx.as<uint32_t>(), rid.as<uint32_t>(),
                                                               off.as<uint64_t>(), nq, nullptr, cap, (uint32_t)ds->id_base,
                                                               tq->f_cand.as<uint64_t>(), n_pairs);
    VDB_LAUNCHED();
    MergeFinish fin;
    fin.cnt_raw = tq->cnt.as<uint32_t>();
    fin.qbad = tq->qbad.as<uint32_t>();
    fin.cap = cap;
    fin.overflow = d_overflow;
    fin.cand_total = reinterpret_cast<unsigned long long*>(tensor_cand_total_ptr(tq));
    launch_merge_keys(tq->f_cand.as<uint64_t>(), 1, nq, cap, false, k, d_keys, nullptr, nullptr, nullptr, st, nullptr,
                      snap.as<uint32_t>(), &fin);
    tq->f_cand = DevBuf();   // stream-ordered frees
    tq->f_stats = DevBuf();
}

// CHECK: the (merged) result of q is provably exact iff no shard overflowed and d_k - ||q||^2 < tau_q
void tensor_check(vdb_tq* tq, const uint64_t* d_keys, uint32_t k, uint64_t n_total, const float* d_tau,
                  const uint32_t* d_overflow, uint32_t* d_redo, uint32_t* d_nredo) {
    tensor_check_range(tq, 0, tq->nq, d_keys, k, n_total, d_tau, d_overflow, d_redo, d_nredo);
}
// the same for the queries [q0, q0 + cnt) of the batch: d_keys [cnt][k] and d_overflow [cnt] are local to the range,
// d_tau is the whole batch's; d_redo receives batch indices
void tensor_check_range(vdb_tq* tq, uint32_t q0, uint32_t cnt, const uint64_t* d_keys, uint32_t k, uint64_t n_total,
                        const float* d_tau, const uint32_t* d_overflow, uint32_t* d_redo, uint32_t* d_nredo) {
    VDB_CUDA(cudaMemsetAsync(d_nredo, 0, 4, tq->st));
    if (cnt == 0) return;
    check_kernel<<<ceil_div(cnt, 256u), 256, 0, tq->st>>>(d_keys, q0, cnt, k, n_total, d_overflow, d_tau,
                                                          tq->ds->metric == VDB_COSINE ? nullptr : tq->qsq.as<float>(),
                                                          g_debug_force_redo.load(), d_redo, d_nredo);
    VDB_LAUNCHED();
}

// One chunk of the batch, enqueued WITHOUT a host synchronisation: sample -> tau -> filter -> rerank -> check.
struct ChunkState {
    vdb_tq* tq = nullptr;
    DevBuf redo;
    const void* d_queries = nullptr;
    uint64_t* d_keys = nullptr;
    uint32_t nq = 0;
    uint32_t h_redo = 0;
    uint64_t h_cands = 0;
};

static void chunk_enqueue(const vdb_dataset* ds, const void* d_queries, uint32_t nq, uint32_t k, uint64_t* d_keys,
                          cudaStream_t st, ChunkState& cs) {
    cs.d_queries = d_queries;
    cs.d_keys = d_keys;
    cs.nq = nq;
    cs.tq = tensor_begin(ds, d_queries, nq, st);
    const uint32_t j0 = tensor_j0(k, ds->sample_n, ds->n), j = tensor_sample_j(j0, ds->sample_n);
    DevBuf jkeys((size_t)nq * j * 8, st), tau((size_t)nq * 4, st);
    cs.redo = DevBuf((size_t)nq * 4, st);
    tensor_sample_keys(cs.tq, j, jkeys.as<uint64_t>(), tau.as<float>(), std::min(j0, j));   // tau from the same launch
    const TensorCheck chk{ds->n, cs.redo.as<uint32_t>()};
    tensor_filter_keys(cs.tq, k, j0, tau.as<float>(), d_keys, nullptr, &chk);   // check fused into the final merge
}

// worker streams of the chunk pipeline (per host thread and device)
struct ChunkStreams {
    int device = -1;
    cudaStream_t s[2] = {nullptr, nullptr};
    cudaEvent_t fork = nullptr, join[2] = {nullptr, nullptr};
    void ensure(int dev) {
        if (device == dev) return;
        release();
        for (int i = 0; i < 2; ++i) {
            VDB_CUDA(cudaStreamCreateWithFlags(&s[i], cudaStreamNonBlocking));
            VDB_CUDA(cudaEventCreateWithFlags(&join[i], cudaEventDisableTiming));
        }
        VDB_CUDA(cudaEventCreateWithFlags(&fork, cudaEventDisableTiming));
        device = dev;
    }
    void release() {
        if (device < 0) return;
        for (int i = 0; i < 2; ++i) {
            cudaStreamDestroy(s[i]);
            cudaEventDestroy(join[i]);
        }
        cudaEventDestroy(fork);
        device = -1;
    }
    ~ChunkStreams() { release(); }
};

// Batches are cut into chunks of at most 16384 queries (bounds the candidate / rerank scratch, ~5 GB per chunk); all
// completeness checks are read back once, after the last chunk. VDB_GEMM_CHUNKS=c (c > 1) additionally splits the
// batch into c chunks that alternate between two worker streams, so the tail of one chunk (rerank gathers, merges,
// check) runs under the contraction of the next. Measured on B200 (1M x 960, 10k queries): 39.4 ms unsplit, 39.9 ms
// with 4 chunks, 55.8 ms with 8 — the rerank gathers and the contraction compete for the same L2 bandwidth and every
// chunk re-streams the database, so the pipeline is OFF by default.
constexpr uint32_t G_QUERY_CHUNK = 16384;

void flat_gemm_keys(const vdb_dataset* ds, const void* d_queries, uint32_t nq, uint32_t k, uint64_t* d_keys,
                    cudaStream_t st) {
    VDB_REQUIRE(flat_gemm_supported(ds, nq, k), "tensor-core Flat path: unsupported dataset/k");
    static const uint32_t chunks_env = getenv("VDB_GEMM_CHUNKS") ? (uint32_t)atoi(getenv("VDB_GEMM_CHUNKS")) : 0;
    uint32_t csize = (chunks_env > 1 && nq >= 4096) ? std::max(1024u, round_up(ceil_div(nq, chunks_env), 256u)) : nq;
    csize = std::min(csize, G_QUERY_CHUNK);
    const uint32_t nchunks = ceil_div(nq, csize);
    const size_t row_bytes = (size_t)ds->dim * ds->elem_size();
    std::vector<ChunkState> cs(nchunks);
    static thread_local ChunkStreams ws;
    const bool pipelined = nchunks > 1 && chunks_env > 1;
    auto cleanup = [&]() {
        for (auto& c : cs)
            if (c.tq) tensor_end(c.tq), c.tq = nullptr;
    };
    try {
        if (pipelined) {
            ws.ensure(ds->device);
            VDB_CUDA(cudaEventRecord(ws.fork, st));
            for (int i = 0; i < 2; ++i) VDB_CUDA(cudaStreamWaitEvent(ws.s[i], ws.fork, 0));
        }
        for (uint32_t c = 0; c < nchunks; ++c) {
            const uint32_t q0 = c * csize, cn = std::min(csize, nq - q0);
            chunk_enqueue(ds, (const uint8_t*)d_queries + (size_t)q0 * row_bytes, cn, k, d_keys + (size_t)q0 * k,
                          pipelined ? ws.s[c & 1] : st, cs[c]);
        }
        if (pipelined)
            for (int i = 0; i < 2; ++i) {
                VDB_CUDA(cudaEventRecord(ws.join[i], ws.s[i]));
                VDB_CUDA(cudaStreamWaitEvent(st, ws.join[i], 0));
            }
        for (auto& c : cs) {
            VDB_CUDA(cudaMemcpyAsync(&c.h_redo, tensor_nredo_ptr(c.tq), 4, cudaMemcpyDeviceToHost, st));
            VDB_CUDA(cudaMemcpyAsync(&c.h_cands, tensor_cand_total_ptr(c.tq), 8, cudaMemcpyDeviceToHost, st));
        }
        VDB_CUDA(cudaStreamSynchronize(st));
        for (auto& c : cs) {
            g_gemm_redo += c.h_redo;
            g_gemm_cands += c.h_cands;
            g_gemm_queries += c.nq;
            if (c.h_redo) {  // exact streaming scan for the queries whose candidate set could not be proven complete
                DevBuf rq((size_t)c.h_redo * row_bytes, st), rkeys((size_t)c.h_redo * k * 8, st);
                gather_rows_kernel<<<c.h_redo, 128, 0, st>>>((const uint8_t*)c.d_queries, (uint32_t)row_bytes, c.redo.as<uint32_t>(),
                                                             c.h_redo, rq.as<uint8_t>());
                VDB_LAUNCHED();
                flat_scan_keys(ds, rq.p, c.h_redo, k, rkeys.as<uint64_t>(), st);
                scatter_keys_kernel<<<c.h_redo, 128, 0, st>>>(rkeys.as<uint64_t>(), k, c.redo.as<uint32_t>(), c.h_redo, c.d_keys);
                VDB_LAUNCHED();
            }
        }
    } catch (...) {
        cudaDeviceSynchronize();  // worker streams may still hold work that references the chunk scratch
        cleanup();
        throw;
    }
    cleanup();
}


// ---- IVF probe scan on the tensor cores ---------------------------------------------------------------------------
// A batch of queries probing nlist lists is a block-sparse contraction: list l's rows x the queries that probe l.
// Rows and norms are kept a second time in LIST ORDER (position p <-> members[p]) so every list is a contiguous row
// range the TMA can tile; the queries are gathered list by list into one matrix; the work items of the contraction
// kernel are (list, tile of gathered queries, range of row tiles). Query tiles of <= 128 rows run on single CTAs
// (M = 128), larger ones on CTA pairs (M = 256). Thresholds:
//   k/64 small (j0 <= 16): a stratified 1/64 sample of every list (also kept in list order) is scored first, the
//     j0-th smallest sampled S' over the probed lists (+ margin) is tau, as in the Flat path;
//   else: tau = the k-th smallest EXACT distance over the first S rows of the visit sequence (complete by construction).
// Candidates are reranked with the FP32 list scan's arithmetic; queries failing the completeness check or overflowing
// their candidate list are redone by the FP32 list scan.
constexpr uint32_t IVF_SAMPLE_RATE = 64;   // round 2: 16 -> 64. The register top-16 epilogue pays per sampled row (594 us of a
// 2.1 ms 1000-query batch at 1/16); a sparser sample loosens tau (more candidates), which the upper-bound pruning takes back

__global__ void gather_op_rows_kernel(const uint4* __restrict__ op_rows, uint32_t row_u4, const float* __restrict__ colA,
                                      const float* __restrict__ rn, const float* __restrict__ ex,
                                      const uint32_t* __restrict__ members, uint64_t n, uint4* __restrict__ out,
                                      float* __restrict__ outA, float* __restrict__ outR, float* __restrict__ outE) {
    const uint64_t p = blockIdx.x;
    if (p >= n) return;
    const uint64_t row = members[p];
    for (uint32_t e = threadIdx.x; e < row_u4; e += blockDim.x) out[p * row_u4 + e] = op_rows[row * row_u4 + e];
    if (threadIdx.x == 0) {
        outA[p] = colA[row];
        outR[p] = rn[row];
        outE[p] = ex[row];
    }
}
// sample row s of list l = one hashed position out of the s-th bucket of IVF_SAMPLE_RATE consecutive list positions
__global__ void ivf_sample_gather_kernel(const uint4* __restrict__ rows_lo, uint32_t row_u4, const float* __restrict__ colA_lo,
                                         const float* __restrict__ rn_lo, const float* __restrict__ ex_lo,
                                         const uint64_t* __restrict__ offsets, const uint64_t* __restrict__ soff, uint32_t nlist,
                                         uint4* __restrict__ out, float* __restrict__ outA, float* __restrict__ outR,
                                         float* __restrict__ outE) {
    const uint64_t s = blockIdx.x;
    uint32_t lo = 0, hi = nlist;  // largest l with soff[l] <= s
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) / 2;
        if (soff[mid] <= s) lo = mid;
        else hi = mid;
    }
    const uint64_t b0 = offsets[lo] + (s - soff[lo]) * IVF_SAMPLE_RATE;
    const uint64_t b1 = min(offsets[lo + 1], b0 + IVF_SAMPLE_RATE);
    uint64_t h = (s + 0x9E3779B97F4A7C15ull) * 0xBF58476D1CE4E5B9ull;
    h ^= h >> 31;
    h *= 0x94D049BB133111EBull;
    h ^= h >> 29;
    const uint64_t pos = b0 + h % (b1 - b0);
    for (uint32_t e = threadIdx.x; e < row_u4; e += blockDim.x) out[s * row_u4 + e] = rows_lo[pos * row_u4 + e];
    if (threadIdx.x == 0) {
        outA[s] = colA_lo[pos];
        outR[s] = rn_lo[pos];
        outE[s] = ex_lo[pos];
    }
}

std::mutex g_ivf_side_mu;
static void ensure_ivf_side(const vdb_dataset* ds, const vdb_ivf* civf, cudaStream_t st) {
    const std::vector<uint64_t>& h_off = civf->h_off;
    vdb_ivf* ivf = const_cast<vdb_ivf*>(civf);
    std::lock_guard<std::mutex> lk(g_ivf_side_mu);
    ensure_side_arrays(ds, st);
    if (ivf->d_rows_lo && ivf->op_kind == ds->op_kind) return;
    VDB_REQUIRE(!ivf->d_rows_lo, "IVF tensor path: the dataset's operand kind changed under a built index");
    const size_t rowb = op_row_bytes_of(ds);
    const uint32_t row_u4 = (uint32_t)(rowb / 16);
    void* rows = nullptr;
    float *colA = nullptr, *rn = nullptr, *ex = nullptr;
    VDB_CUDA(cudaMalloc(&rows, ds->n * rowb));
    VDB_CUDA(cudaMalloc(&colA, ds->n * 4));
    VDB_CUDA(cudaMalloc(&rn, ds->n * 4));
    VDB_CUDA(cudaMalloc(&ex, ds->n * 4));
    gather_op_rows_kernel<<<(uint32_t)ds->n, 128, 0, st>>>((const uint4*)op_rows_of(ds), row_u4, ds->d_sqnorm, ds->d_lo, ds->d_ex,
                                                          ivf->d_members, ds->n, (uint4*)rows, colA, rn, ex);
    VDB_LAUNCHED();
    ivf->h_samp_off.assign(ivf->nlist + 1, 0);
    for (uint32_t l = 0; l < ivf->nlist; ++l)
        ivf->h_samp_off[l + 1] = ivf->h_samp_off[l] + ceil_div<uint64_t>(h_off[l + 1] - h_off[l], IVF_SAMPLE_RATE);
    ivf->samp_n = ivf->h_samp_off[ivf->nlist];
    VDB_CUDA(cudaMalloc(&ivf->d_samp_rows, std::max<uint64_t>(ivf->samp_n, 1) * rowb));
    VDB_CUDA(cudaMalloc(&ivf->d_samp_colA, std::max<uint64_t>(ivf->samp_n, 1) * 4));
    VDB_CUDA(cudaMalloc(&ivf->d_samp_rn, std::max<uint64_t>(ivf->samp_n, 1) * 4));
    VDB_CUDA(cudaMalloc(&ivf->d_samp_ex, std::max<uint64_t>(ivf->samp_n, 1) * 4));
    if (ivf->samp_n) {
        DevBuf soff((size_t)(ivf->nlist + 1) * 8, st);
        VDB_CUDA(cudaMemcpyAsync(soff.p, ivf->h_samp_off.data(), (size_t)(ivf->nlist + 1) * 8, cudaMemcpyHostToDevice, st));
        ivf_sample_gather_kernel<<<(uint32_t)ivf->samp_n, 128, 0, st>>>((const uint4*)rows, row_u4, colA, rn, ex, ivf->d_offsets,
                                                                       soff.as<uint64_t>(), ivf->nlist, (uint4*)ivf->d_samp_rows,
                                                                       ivf->d_samp_colA, ivf->d_samp_rn, ivf->d_samp_ex);
        VDB_LAUNCHED();
        VDB_CUDA(cudaStreamSynchronize(st));
    }
    VDB_CUDA(cudaStreamSynchronize(st));
    ivf->d_colA_lo = colA;
    ivf->d_rn_lo = rn;
    ivf->d_ex_lo = ex;
    ivf->op_kind = ds->op_kind;
    ivf->d_rows_lo = rows;
}

// first S rows of every query's visit sequence (probed lists in probe order) as rerank pairs
__global__ void ivf_subset_kernel(const uint64_t* __restrict__ probes, uint32_t nprobe, const uint64_t* __restrict__ offsets,
                                  const uint32_t* __restrict__ members, uint32_t S, uint32_t* __restrict__ qidx,
                                  uint32_t* __restrict__ rid, uint8_t* __restrict__ valid) {
    const uint32_t q = blockIdx.x;
    for (uint32_t s = threadIdx.x; s < S; s += blockDim.x) {
        uint32_t left = s, row = 0;
        bool ok = false;
        for (uint32_t j = 0; j < nprobe && !ok; ++j) {
            const uint64_t pk = probes[(size_t)q * nprobe + j];
            if (pk == KEY_NONE) break;
            const uint32_t c = key_id(pk);
            const uint64_t len = offsets[c + 1] - offsets[c];
            if (left < len) {
                row = members[offsets[c] + left];
                ok = true;
            } else {
                left -= (uint32_t)len;
            }
        }
        qidx[(size_t)q * S + s] = q;
        rid[(size_t)q * S + s] = row;
        valid[(size_t)q * S + s] = ok;
    }
}
// tau' in the units of the pruning score: L2Sqr: d_k - ||q||^2, cosine: d_k; +inf when fewer than k rows are probed
__global__ void ivf_tau_kernel(const uint64_t* __restrict__ keys, uint32_t nq, uint32_t k, const float* __restrict__ qsq,
                               float* __restrict__ tau) {
    const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    const uint64_t kk = keys[(size_t)q * k + (k - 1)];
    if (kk == KEY_NONE) {
        tau[q] = __uint_as_float(0x7f800000u);
        return;
    }
    const float dk = key_dist(kk);
    const float shift = qsq ? qsq[q] : 0.f;
    tau[q] = (dk - shift) + 2e-5f * (fabsf(dk) + shift) + 1e-30f;
}
// the 16 smallest sampled scores of every probed list of a query, side by side: [nq][nprobe][G_TOPJ]
__global__ void ivf_collect_sample_kernel(const uint64_t* __restrict__ skeys, const uint32_t* __restrict__ gpos, uint32_t nprobe,
                                          uint64_t* __restrict__ out) {
    const uint32_t q = blockIdx.x;
    for (uint32_t e = threadIdx.x; e < nprobe * G_TOPJ; e += blockDim.x) {
        const uint32_t g = gpos[(size_t)q * nprobe + e / G_TOPJ];
        out[(size_t)q * nprobe * G_TOPJ + e] = g == 0xffffffffu ? KEY_NONE : skeys[(size_t)g * G_TOPJ + e % G_TOPJ];
    }
}
__global__ void gather_query_side_kernel(const uint4* __restrict__ qop, uint32_t row_u4, const float* __restrict__ qd,
                                         const float* __restrict__ qab, const float* __restrict__ qb,
                                         const float* __restrict__ qnorm, const uint32_t* __restrict__ qmap, uint32_t G,
                                         uint4* __restrict__ outq, float* __restrict__ out_qd, float* __restrict__ out_qab,
                                         float* __restrict__ out_qb, float* __restrict__ out_qnorm) {
    const uint32_t g = blockIdx.x;
    if (g >= G) return;
    const uint32_t q = qmap[g];
    for (uint32_t e = threadIdx.x; e < row_u4; e += blockDim.x) outq[(size_t)g * row_u4 + e] = qop[(size_t)q * row_u4 + e];
    if (threadIdx.x == 0) {
        out_qd[g] = qd[q];
        out_qab[g] = qab[q];
        out_qb[g] = qb[q];
        if (qnorm) out_qnorm[g] = qnorm[q];
    }
}
__global__ void gather_f32_kernel(const float* __restrict__ src, const uint32_t* __restrict__ idx, uint32_t cnt,
                                  float* __restrict__ dst) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < cnt) dst[i] = src[idx[i]];
}
// completeness: no overflow, and (unless the threshold is complete by construction) the k-th exact distance lies
// strictly inside the threshold; tau = +inf keeps every probed row, so short visit sets pass
__global__ void ivf_check_kernel(const uint64_t* __restrict__ keys, uint32_t nq, uint32_t k, const uint32_t* __restrict__ cnt,
                                 uint32_t cap, const float* __restrict__ tau, const float* __restrict__ qsq, int by_construction,
                                 uint32_t* __restrict__ redo, uint32_t* __restrict__ nredo) {
    const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    bool ok = cnt[q] <= cap;
    if (ok && !by_construction && tau[q] != __uint_as_float(0x7f800000u)) {
        const uint64_t kk = keys[(size_t)q * k + (k - 1)];
        ok = kk != KEY_NONE;
        if (ok) {
            const float dk = key_dist(kk);
            const float shift = qsq ? qsq[q] : 0.f;
            const float slack = 2e-5f * (fabsf(dk) + shift + fabsf(tau[q]));
            ok = (dk - shift) < tau[q] - slack;
        }
    }
    if (!ok) redo[atomicAdd(nredo, 1u)] = q;
}

bool ivf_tensor_keys(const vdb_dataset* ds, const vdb_ivf* ivf, const void* d_queries, const uint64_t* d_probes,
                     const uint64_t* h_probes, uint32_t nq, uint32_t nprobe, uint32_t k, uint64_t* d_keys, cudaStream_t st) {
    if (!flat_gemm_supported(ds, nq, k) || k > 512) return false;
    ensure_ivf_side(ds, ivf, st);
    const std::vector<uint64_t>& h_off = ivf->h_off;
    // ---- host: group the (query, list) pairs by list (counting sort), build the gathered query order and the work
    // items. Everything the device needs - qmap | gpos | the four item tables - is laid out in ONE page-locked staging
    // block and uploaded with one copy (round 1: vectors of vectors and four pageable copies, ~0.4 ms per 1000 queries).
    const size_t npairs = (size_t)nq * nprobe;
    std::vector<uint32_t> lcount(ivf->nlist + 1, 0);
    for (size_t e = 0; e < npairs; ++e) {
        const uint64_t pk = h_probes[e];
        if (pk != KEY_NONE) ++lcount[key_id(pk) + 1];
    }
    for (uint32_t l = 0; l < ivf->nlist; ++l) lcount[l + 1] += lcount[l];   // lcount[l] = first gathered row of list l
    const uint32_t G = lcount[ivf->nlist];
    // Query tiles run on single CTAs (M = 128) by default: the probe scan of a batch is bound by streaming the lists
    // and by per-item latency, not by the MMAs, and one launch per pass beats a single-CTA + a CTA-pair launch (measured,
    // 1M x 960, nlist 128: 1000 queries nprobe 8 1.47 -> 1.27 ms, 10 000 queries nprobe 24 11.8 -> 11.7 ms).
    // VDB_IVF_CTAS=0: 256-row tiles on CTA pairs with the remainder on single CTAs; =2: pairs only.
    static const uint32_t force_ctas = getenv("VDB_IVF_CTAS") ? (uint32_t)atoi(getenv("VDB_IVF_CTAS")) : 1;
    const uint32_t tiles_per_item = 8;
    // item counts first (the staging block is sized from them)
    size_t n_items[2] = {0, 0}, n_sitems[2] = {0, 0};
    for (uint32_t l = 0; l < ivf->nlist; ++l) {
        const uint64_t r0 = h_off[l], r1 = h_off[l + 1];
        const uint32_t cnt = lcount[l + 1] - lcount[l];
        if (r1 == r0 || cnt == 0) continue;
        const uint64_t row_groups = ceil_div<uint64_t>(r1 - r0, (uint64_t)tiles_per_item * GN);
        for (uint32_t g = 0; g < cnt;) {
            const uint32_t left = cnt - g;
            const uint32_t pair = force_ctas ? force_ctas - 1 : (left > GM ? 1u : 0u);
            n_items[pair] += row_groups;
            n_sitems[pair] += 1;
            g += std::min(left, pair ? 2u * GM : (uint32_t)GM);
        }
    }
    static thread_local PinnedStage table_stage;
    const size_t off_qmap = 0, off_gpos = off_qmap + round_up<size_t>((size_t)G * 4, 16);
    size_t off_items[2], off_sitems[2], at = off_gpos + round_up<size_t>(npairs * 4, 16);
    for (int t = 0; t < 2; ++t) off_items[t] = at, at += n_items[t] * sizeof(GemmItem);
    for (int t = 0; t < 2; ++t) off_sitems[t] = at, at += n_sitems[t] * sizeof(GemmItem);
    const size_t stage_bytes = std::max<size_t>(at, 16);
    uint8_t* stage = (uint8_t*)table_stage.get(stage_bytes);
    uint32_t* qmap = (uint32_t*)(stage + off_qmap);
    uint32_t* gpos = (uint32_t*)(stage + off_gpos);
    GemmItem* items[2] = {(GemmItem*)(stage + off_items[0]), (GemmItem*)(stage + off_items[1])};
    GemmItem* sitems[2] = {(GemmItem*)(stage + off_sitems[0]), (GemmItem*)(stage + off_sitems[1])};
    {
        std::vector<uint32_t> fill(lcount.begin(), lcount.end() - 1);   // next free gathered row of every list
        for (size_t e = 0; e < npairs; ++e) {
            const uint64_t pk = h_probes[e];
            if (pk == KEY_NONE) {
                gpos[e] = 0xffffffffu;
                continue;
            }
            const uint32_t pos = fill[key_id(pk)]++;
            gpos[e] = pos;
            qmap[pos] = (uint32_t)(e / nprobe);
        }
    }
    size_t w_items[2] = {0, 0}, w_sitems[2] = {0, 0};
    for (uint32_t l = 0; l < ivf->nlist; ++l) {
        const uint64_t r0 = h_off[l], r1 = h_off[l + 1];
        const uint32_t g0 = lcount[l], g1 = lcount[l + 1];
        if (r1 == r0 || g1 == g0) continue;
        const uint64_t s0 = ivf->h_samp_off[l], s1 = ivf->h_samp_off[l + 1];
        // query tiles: 256 rows on a CTA pair, a remainder of <= 128 rows on a single CTA
        for (uint32_t g = g0; g < g1;) {
            const uint32_t left = g1 - g;
            const uint32_t pair = force_ctas ? force_ctas - 1 : (left > GM ? 1u : 0u);
            const uint32_t len = std::min(left, pair ? 2u * GM : (uint32_t)GM);
            for (uint64_t r = r0; r < r1; r += (uint64_t)tiles_per_item * GN)
                items[pair][w_items[pair]++] = GemmItem{g, g + len, r, std::min<uint64_t>(r1, r + (uint64_t)tiles_per_item * GN)};
            sitems[pair][w_sitems[pair]++] = GemmItem{g, g + len, s0, s1};
            g += len;
        }
    }
    if (G == 0) {
        VDB_CUDA(cudaMemsetAsync(d_keys, 0xff, (size_t)nq * k * 8, st));
        return true;
    }
    vdb_tq* tq = tensor_begin(ds, d_queries, nq, st);
    try {
        const bool cosine = ds->metric == VDB_COSINE;
        // ---- gathered query matrix, its per-row scalars, item tables ----
        const size_t q_rowb = (size_t)tq->op_pitch * (tq->kind == KIND_F16 ? 2 : 4);
        DevBuf d_stage(stage_bytes, st), qg((size_t)G * q_rowb, st), qd_g((size_t)G * 4, st), qab_g((size_t)G * 4, st),
            qb_g((size_t)G * 4, st), qn_g((size_t)G * 4, st), tau_g((size_t)G * 4, st), tau((size_t)nq * 4, st);
        VDB_CUDA(cudaMemcpyAsync(d_stage.p, stage, stage_bytes, cudaMemcpyHostToDevice, st));
        const uint32_t* d_qmap = (const uint32_t*)((const uint8_t*)d_stage.p + off_qmap);
        const uint32_t* d_gpos = (const uint32_t*)((const uint8_t*)d_stage.p + off_gpos);
        const GemmItem* d_items[2] = {(const GemmItem*)((const uint8_t*)d_stage.p + off_items[0]),
                                      (const GemmItem*)((const uint8_t*)d_stage.p + off_items[1])};
        const GemmItem* d_sitems[2] = {(const GemmItem*)((const uint8_t*)d_stage.p + off_sitems[0]),
                                       (const GemmItem*)((const uint8_t*)d_stage.p + off_sitems[1])};
        gather_query_side_kernel<<<G, 128, 0, st>>>((const uint4*)tq->qop.p, (uint32_t)(q_rowb / 16), tq->qd.as<float>(),
                                                    tq->qab.as<float>(), tq->qb.as<float>(),
                                                    cosine ? tq->qtile.qcache.as<float>() : nullptr, d_qmap, G,
                                                    (uint4*)qg.p, qd_g.as<float>(), qab_g.as<float>(), qb_g.as<float>(), qn_g.as<float>());
        VDB_LAUNCHED();
        const CUtensorMap mq = make_op_map(tq->kind, qg.p, ds->dim, G, q_rowb, GM);
        GemmParams base{};
        base.nq = G;
        base.kblocks = kblocks_of(tq->kind, ds->dim);
        base.qd = qd_g.as<float>();
        base.qab = qab_g.as<float>();
        base.qb = qb_g.as<float>();
        base.qnorm = cosine ? qn_g.as<float>() : nullptr;
        base.row_stride = 1;
        base.qmap = d_qmap;
        base.nslabs = 1;
        auto run_items = [&](int mode, const GemmItem* const* tabs, const size_t* counts, const void* rows, uint64_t nrows,
                             GemmParams p) {
            for (uint32_t pair = 0; pair < 2; ++pair) {
                if (counts[pair] == 0) continue;
                const CUtensorMap mx = make_op_map(tq->kind, rows, ds->dim, nrows, op_row_bytes_of(ds), GN / (pair + 1));
                p.nrows = nrows;
                p.items = tabs[pair];
                p.nitems = (uint32_t)counts[pair];
                launch_gemm(mode, ds->metric, tq->kind, mq, mx, p, st, (int)pair + 1);
            }
        };
        // ---- thresholds ----
        const uint32_t j0 = tensor_j0(k, 1u << 20, (uint64_t)IVF_SAMPLE_RATE << 20);
        static const int force_subset = getenv("VDB_IVF_SUBSET") ? atoi(getenv("VDB_IVF_SUBSET")) : 0;
        const bool by_sample = j0 <= (uint32_t)G_TOPJ && ivf->samp_n > 0 && !force_subset;
        if (by_sample) {
            DevBuf skeys((size_t)G * G_TOPJ * 8, st), ckeys((size_t)nq * nprobe * G_TOPJ * 8, st), jkeys((size_t)nq * j0 * 8, st);
            VDB_CUDA(cudaMemsetAsync(skeys.p, 0xff, (size_t)G * G_TOPJ * 8, st));
            GemmParams ps = base;
            ps.sqnorm = ivf->d_samp_colA;
            ps.rnorm = ivf->d_samp_rn;
            ps.ex = ivf->d_samp_ex;
            ps.out_keys = skeys.as<uint64_t>();
            run_items(2, d_sitems, n_sitems, ivf->d_samp_rows, ivf->samp_n, ps);
            ivf_collect_sample_kernel<<<nq, 128, 0, st>>>(skeys.as<uint64_t>(), d_gpos, nprobe, ckeys.as<uint64_t>());
            VDB_LAUNCHED();
            launch_merge_keys(ckeys.as<uint64_t>(), 1, nq, nprobe * G_TOPJ, false, j0, jkeys.as<uint64_t>(), nullptr, nullptr,
                              nullptr, st);
            // +inf when the probed lists hold fewer than j0 sampled rows
            tau_from_keys_kernel<<<ceil_div(nq, 256u), 256, 0, st>>>(jkeys.as<uint64_t>(), nq, j0, j0, tq->qab.as<float>(),
                                                                    tq->qb.as<float>(), ds->mean_norm, ds->mean_ex, cosine ? 1 : 0,
                                                                    tau.as<float>());
            VDB_LAUNCHED();
        } else {
            // S balances the two exact-distance passes: S subset rows against ~k * visited / S surviving candidates
            const double visited = (double)nprobe * (double)ds->n / (double)ivf->nlist;
            const uint32_t S = force_subset > 1
                                   ? (uint32_t)force_subset
                                   : std::min(4096u, (uint32_t)next_pow2(std::max<uint32_t>(
                                                         std::max(256u, 2 * k), (uint32_t)std::sqrt((double)k * visited))));
            const uint64_t cnt = (uint64_t)nq * S;
            DevBuf qidx(cnt * 4, st), rid(cnt * 4, st), valid(cnt, st), dist(cnt * 4, st), skeys(cnt * 8, st), kkeys((size_t)nq * k * 8, st);
            ivf_subset_kernel<<<nq, 128, 0, st>>>(d_probes, nprobe, ivf->d_offsets, ivf->d_members, S, qidx.as<uint32_t>(),
                                                  rid.as<uint32_t>(), valid.as<uint8_t>());
            VDB_LAUNCHED();
            exact_pair_distances_masked(ds, tq->qcopy.p, tq->qpitch, qidx.as<uint32_t>(), rid.as<uint32_t>(), valid.as<uint8_t>(),
                                        cnt, dist.as<float>(), st, nullptr, cosine ? tq->qtile.qcache.as<float>() : nullptr);
            rekey_based(dist.as<float>(), rid.as<uint32_t>(), 0, valid.as<uint8_t>(), cnt, skeys.as<uint64_t>(), st);
            launch_merge_keys(skeys.as<uint64_t>(), 1, nq, S, false, k, kkeys.as<uint64_t>(), nullptr, nullptr, nullptr, st);
            ivf_tau_kernel<<<ceil_div(nq, 256u), 256, 0, st>>>(kkeys.as<uint64_t>(), nq, k, cosine ? nullptr : tq->qsq.as<float>(),
                                                              tau.as<float>());
            VDB_LAUNCHED();
        }
        gather_f32_kernel<<<ceil_div(G, 256u), 256, 0, st>>>(tau.as<float>(), d_qmap, G, tau_g.as<float>());
        VDB_LAUNCHED();
        // ---- filter pass over the probed (list, query tile) blocks ----
        const uint32_t cap = 8192;
        DevBuf cand((size_t)nq * cap * 8, st);
        VDB_CUDA(cudaMemsetAsync(tq->cnt.p, 0, (size_t)nq * 4, st));
        {
            GemmParams pf = base;
            pf.sqnorm = ivf->d_colA_lo;
            pf.rnorm = ivf->d_rn_lo;
            pf.ex = ivf->d_ex_lo;
            pf.tau = tau_g.as<float>();
            pf.cand_cnt = tq->cnt.as<uint32_t>();
            pf.cand = cand.as<uint64_t>();
            pf.cap = cap;
            run_items(1, d_items, n_items, ivf->d_rows_lo, ds->n, pf);
        }
        // ---- candidates that cannot be among the k best by their score bounds are dropped (cand_prune_kernel) ----
        DevBuf pcnt((size_t)nq * 4, st);
        {
            auto kern = cosine ? cand_prune_kernel<VDB_COSINE> : cand_prune_kernel<VDB_L2SQR>;
            kern<<<nq, 256, (size_t)cap * 4, st>>>(cand.as<uint64_t>(), tq->cnt.as<uint32_t>(), cap, k, ivf->d_rn_lo, ivf->d_ex_lo,
                                                   tq->qab.as<float>(), tq->qb.as<float>(), cosine ? nullptr : tq->qsq.as<float>(),
                                                   pcnt.as<uint32_t>(), nullptr, nullptr, nullptr, nullptr, nullptr, 0u, 0u, 0u);
            VDB_LAUNCHED();
        }
        // ---- exact rerank (the FP32 list scan's arithmetic) and top-k ----
        const uint64_t total = (uint64_t)nq * cap;
        DevBuf off((size_t)(nq + 1) * 8, st), qidx(total * 4, st), rid(total * 4, st), dist(total * 4, st), keys2(total * 8, st);
        cand_offsets_kernel<<<1, 1024, 0, st>>>(pcnt.as<uint32_t>(), nq, cap, off.as<uint64_t>());
        VDB_LAUNCHED();
        cand_to_pairs_kernel<<<nq, 256, 0, st>>>(cand.as<uint64_t>(), pcnt.as<uint32_t>(), cap, off.as<uint64_t>(),
                                                 ivf->d_members, qidx.as<uint32_t>(), rid.as<uint32_t>());
        VDB_LAUNCHED();
        const uint64_t* d_total = off.as<uint64_t>() + nq;
        exact_pair_distances_masked(ds, tq->qcopy.p, tq->qpitch, qidx.as<uint32_t>(), rid.as<uint32_t>(), nullptr, total,
                                    dist.as<float>(), st, d_total, cosine ? tq->qtile.qcache.as<float>() : nullptr);
        rekey_dev_count_kernel<<<(uint32_t)sm_count() * 8, 256, 0, st>>>(dist.as<float>(), rid.as<uint32_t>(),
                                                                        (uint32_t)ds->id_base, d_total, keys2.as<uint64_t>());
        VDB_LAUNCHED();
        launch_merge_keys(keys2.as<uint64_t>(), 1, nq, cap, false, k, d_keys, nullptr, nullptr, nullptr, st, off.as<uint64_t>());
        // ---- completeness check; failing queries: FP32 list scan ----
        DevBuf redo((size_t)nq * 4, st), nredo(4, st);
        VDB_CUDA(cudaMemsetAsync(nredo.p, 0, 4, st));
        ivf_check_kernel<<<ceil_div(nq, 256u), 256, 0, st>>>(d_keys, nq, k, tq->cnt.as<uint32_t>(), cap, tau.as<float>(),
                                                            cosine ? nullptr : tq->qsq.as<float>(), by_sample ? 0 : 1,
                                                            redo.as<uint32_t>(), nredo.as<uint32_t>());
        VDB_LAUNCHED();
        uint32_t h_n = 0;
        uint64_t h_cands = 0;
        VDB_CUDA(cudaMemcpyAsync(&h_n, nredo.p, 4, cudaMemcpyDeviceToHost, st));
        VDB_CUDA(cudaMemcpyAsync(&h_cands, d_total, 8, cudaMemcpyDeviceToHost, st));
        VDB_CUDA(cudaStreamSynchronize(st));
        g_gemm_redo += h_n;
        g_gemm_cands += h_cands;
        g_gemm_queries += nq;
        if (h_n) {
            std::vector<uint32_t> sel(h_n);
            VDB_CUDA(cudaMemcpyAsync(sel.data(), redo.p, (size_t)h_n * 4, cudaMemcpyDeviceToHost, st));
            VDB_CUDA(cudaStreamSynchronize(st));
            std::sort(sel.begin(), sel.end());
            DevBuf rk((size_t)h_n * k * 8, st), dsel((size_t)h_n * 4, st);
            ivf_list_major_subset(ds, ivf, d_queries, d_probes, sel.data(), h_n, nprobe, k, rk.as<uint64_t>(), st);
            VDB_CUDA(cudaMemcpyAsync(dsel.p, sel.data(), (size_t)h_n * 4, cudaMemcpyHostToDevice, st));
            scatter_keys_kernel<<<h_n, 128, 0, st>>>(rk.as<uint64_t>(), k, dsel.as<uint32_t>(), h_n, d_keys);
            VDB_LAUNCHED();
            VDB_CUDA(cudaStreamSynchronize(st));
        }
    } catch (...) {
        tensor_end(tq);
        throw;
    }
    tensor_end(tq);
    return true;
}

// debug / test entry: the pruning scores S' of every (query, strided row) pair as keys, [nq][n / row_stride] (mode 0 of
// the kernel), computed by the very pipeline of the search (operand copies, error norms, coefficients) with the operand
// kind forced to `kind` (0 = TF32 on the fp32 rows in place, 1 = FP16 copy; < 0: the dataset's own choice)
void flat_gemm_store(const vdb_dataset* ds, const void* d_queries, uint32_t nq, uint32_t row_stride, int kind,
                     uint64_t* d_out_keys, cudaStream_t st) {
    VDB_REQUIRE(row_stride >= 1 && ds->n >= row_stride, "flat_gemm_store: bad row stride");
    ensure_side_arrays(ds, st, kind);
    vdb_tq* tq = tensor_begin(ds, d_queries, nq, st, true);   // the debug entry also serves sets of < 65536 rows
    try {
        const uint64_t ns = ds->n / row_stride;
        GemmParams p = base_params(tq);
        p.sqnorm = ds->d_sqnorm;
        p.rnorm = ds->d_lo;
        p.ex = ds->d_ex;
        p.nrows = ns;
        p.row_stride = row_stride;
        p.out_keys = d_out_keys;
        const CUtensorMap ms = make_op_map(tq->kind, op_rows_of(ds), ds->dim, ns, op_row_bytes_of(ds) * row_stride, GN / gemm_ctas());
        plan_gemm(p);
        launch_gemm(0, ds->metric, tq->kind, tq->mq, ms, p, st);
        VDB_CUDA(cudaStreamSynchronize(st));
    } catch (...) {
        tensor_end(tq);
        throw;
    }
    tensor_end(tq);
}

}  // namespace vdb
