// pq_gemm.cu — K4t: the 4-bit PQ ADC scan of a query batch as a tensor-core contraction (L2Sqr tables).
//
// Replaces the inner loop of PQTable::k_nearest over all rows (reference src/index_algorithm/pq_table.rs, ADC lookup
// d(q, row) = sum_g LUT_q[g][code(row, g)], flat_index.rs knn_pq) for large batches. The lookup is a dot product
// with a ONE-HOT vector: adc(q, row) = < onehot(row), LUT_q > over K = m * 16 columns. The tensor cores evaluate it
// in BF16 and only PRUNE: every LUT entry of an L2Sqr table is >= 0, so the BF16 rounding of the table is a RELATIVE
// error (< 2^-8 per entry: BF16 keeps 8 significant bits, so round-to-nearest moves a value by up to half of its 2^-7
// spacing; one-hot entries are exact) and
//     S' = S_bf16 * (1 - 2^-8 * 1.05 - m * 2^-21) - 1e-35  <=  adc_exact(q, row)
// holds for every pair. Rows with S' <= tau_q (tau_q: the exact-ADC threshold of the global-threshold scan, pq.cu)
// become coarse candidates; their ADC value is then re-evaluated with the reference's arithmetic (sequential f32 sum
// in group order) and the rows with adc <= tau_q go on exactly as in the FP32 scan — the candidate set is identical.
//
// Kernel (sm_100a, one CTA per SM, 320 threads):
//   warps 6-9  generators: thread = row of the 128-row tile; per k-block (4 groups = 64 bf16 columns = one 128-byte
//              swizzle row) they expand 4 code nibbles into the one-hot A tile directly in shared memory
//              (8 x 16-byte chunks, chunk j of row r at position j ^ (r & 7): the layout TMA's 128B swizzle produces),
//              fence.proxy.async, arrive on the stage's full barrier
//   warp 4     TMA producer: LUT tile (256 queries x 64 columns, bf16) of the k-block, same barrier (expect_tx)
//   warp 5     one thread issues tcgen05.mma.kind::f16 (M = 128 rows, N = 256 queries, K = 16 x 4 per k-block)
//              into double-buffered TMEM accumulators; tcgen05.commit frees the stage / publishes the accumulator
//   warps 0-3  epilogue: tcgen05.ld (thread = row, registers = queries), threshold test, candidate append
#include <cuda.h>
#include <cuda_bf16.h>

#include <algorithm>
#include <cstdlib>

#include "index.cuh"
#include "tc.cuh"
#include "topk.cuh"

namespace vdb {

constexpr int PM = 128;                    // rows per CTA and tile (TMEM lanes)
constexpr int PN = 256;                    // queries per tile (TMEM columns per accumulator)
constexpr int PK = 64;                     // bf16 columns per k-block = 4 groups x 16 centroids = 128 bytes
constexpr int P_A_BYTES = PM * PK * 2;     // 16 KB generated one-hot tile
constexpr int P_BASE_THREADS = 192;        // warps 0-3 epilogue, 4 TMA producer, 5 MMA issuer; then GG x 4 generator warps
constexpr int P_TMEM_COLS = 512;
constexpr uint32_t P_MAX_ENC = 256;        // m <= 512 groups (the code tile of 128 rows must fit beside the stages)
constexpr int P_MAX_STAGES = 6;
// CTAS = 1: one CTA computes 128 rows x 256 queries. CTAS = 2: a CTA pair (cta_group::2) computes 256 rows x 256
// queries; each CTA generates the one-hot rows of its own 128 rows and loads HALF of the LUT tile, so the shared-memory
// traffic per MMA cycle drops 1.5x (ncu: the single-CTA kernel keeps the tensor pipe only 56 % busy at 103 B/clk of
// shared-memory traffic).
template <int CTAS> struct PqCfg {
    static constexpr int B_ROWS = PN / CTAS;                   // queries loaded per CTA and k-block
    static constexpr int B_BYTES = B_ROWS * PK * 2;
    static constexpr int STAGE_BYTES = P_A_BYTES + B_BYTES;    // 48 KB / 32 KB
    static constexpr int STAGES = CTAS == 1 ? 4 : 6;           // 192 KB either way
    static constexpr uint32_t smem_bytes(uint32_t enc) {  // align + stages + code tile + thresholds + barriers
        return 1024 + STAGES * STAGE_BYTES + ((PM * enc + 15u) & ~15u) + PN * 4 + 256;
    }
    // instruction descriptor: D = F32, A = B = BF16, both K-major, N >> 3, M >> 4
    static constexpr uint32_t IDESC = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(PN >> 3) << 17) |
                                      ((uint32_t)((PM * CTAS) >> 4) << 24);
};
constexpr uint32_t P_PEER_MASK = 0xFEFFFFFFu;  // clears the CTA-pair peer bit of a shared::cluster address (-> even CTA)

__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
        : "memory");
}
__device__ __forceinline__ void umma_bf16_2sm(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
        : "memory");
}

struct PqGemmParams {
    const uint8_t* codes;   // [n][enc] reference layout (low nibble = even group)
    uint64_t n;
    uint32_t enc, m, kblocks;
    uint32_t nq;
    const float* tau;       // [nq] exact-ADC thresholds
    float factor;           // 1 - relative bound of the bf16 evaluation
    uint32_t* ccnt;         // [nq] coarse candidate counters
    uint32_t* ccand;        // [nq][ccap] rows
    uint32_t ccap;
    uint32_t tiles_per_item, nrow_items, nqt;
    float* all_out;         // MODE 0: [nq][n] upper bounds of the exact ADC values (sample pass); MODE 2: [nq][n] S'
    float up_factor;        // MODE 0: 1 + relative bound
};

// relative bound of the bf16 evaluation (see the top of the file)
static float pq_rel_bound(uint32_t m) { return ldexpf(1.05f, -8) + (float)m * ldexpf(1.0f, -21); }
// the filter's lower bound S' of the exact ADC value, from the fp32 accumulator of the contraction
__device__ __forceinline__ float pq_filter_score(float acc, float factor) { return fmaf(acc, factor, -1e-35f); }

// MODE 0: store every score (sample pass), 1: filter against tau, 2: store every S' of the filter (test hook). GG generator groups of 4 warps take the k-blocks
// round-robin: one group's chain per k-block (wait -> LDS -> STS -> proxy fence -> arrive) is longer than the MMAs of a
// k-block, so several chains have to be in flight.
template <int MODE, int CTAS, int GG>
__global__ void __launch_bounds__(P_BASE_THREADS + 128 * GG, 1) pq_gemm_kernel(const __grid_constant__ CUtensorMap map_lut, const PqGemmParams p) {
    using Cfg = PqCfg<CTAS>;
    constexpr int STAGES = Cfg::STAGES;
    constexpr uint32_t TM = PM * CTAS;  // rows per tile of the CTA (pair)
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t* stage_base = smem;
    uint8_t* codes_s = smem + STAGES * Cfg::STAGE_BYTES;                  // [PM][enc]
    float* tau_s = reinterpret_cast<float*>(codes_s + ((PM * p.enc + 15u) & ~15u));  // [PN]
    uint64_t* bars = reinterpret_cast<uint64_t*>(tau_s + PN);
    uint64_t* full_bar = bars;                      // [STAGES]  (pair mode: the leader's copy is the live one)
    uint64_t* empty_bar = bars + P_MAX_STAGES;      // [STAGES]  per CTA
    uint64_t* tfull_bar = bars + 2 * P_MAX_STAGES;  // [2]       per CTA
    uint64_t* tempty_bar = tfull_bar + 2;           // [2]       (pair mode: the leader's copy is the live one)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t cta_rank = CTAS == 2 ? cluster_ctarank() : 0u;
    const bool leader = cta_rank == 0;
    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&full_bar[s], 1 + 4 * CTAS);  // TMA expect_tx arrive + one arrive per generator warp (of every CTA)
            mbar_init(&empty_bar[s], 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&tfull_bar[a], 1);
            mbar_init(&tempty_bar[a], 4 * CTAS);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 5) {
        if (CTAS == 2) tmem_alloc2(tmem_slot, P_TMEM_COLS);
        else tmem_alloc(tmem_slot, P_TMEM_COLS);
    }
    tc_fence_before();
    __syncthreads();
    if (CTAS == 2) cluster_sync_all();  // the peer's barriers are initialised before any remote arrive / TMA
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t nitems = p.nrow_items * p.nqt;
    const uint32_t unit = blockIdx.x / CTAS, nunits = gridDim.x / CTAS;  // a unit = one CTA or one CTA pair

    if (warp == 4) {
        // ===== TMA producer: this CTA's share of the LUT tile of every k-block =====
        if (lane == 0) {
            uint32_t stage = 0, phase = 0;
            for (uint32_t item = unit; item < nitems; item += nunits) {
                const uint32_t ri = item / p.nqt, qt = item - ri * p.nqt;
                const uint64_t r0 = (uint64_t)ri * p.tiles_per_item * TM;
                const uint32_t ntile = (uint32_t)min((uint64_t)p.tiles_per_item, (p.n - r0 + TM - 1) / TM);
                const int qrow = (int)(qt * PN + cta_rank * Cfg::B_ROWS);
                for (uint32_t t = 0; t < ntile; ++t)
                    for (uint32_t kb = 0; kb < p.kblocks; ++kb) {
                        mbar_wait(&empty_bar[stage], phase ^ 1);
                        const uint32_t dst = smem_u32(stage_base + stage * Cfg::STAGE_BYTES) + P_A_BYTES;
                        if (CTAS == 1) {
                            mbar_expect_tx(&full_bar[stage], Cfg::B_BYTES);
                            tma_load_2d(dst, &map_lut, (int)(kb * PK), qrow, &full_bar[stage]);
                        } else {
                            // both CTAs' bytes are accounted on the LEADER's barrier
                            if (leader) mbar_expect_tx(&full_bar[stage], Cfg::B_BYTES * CTAS);
                            tma_load_2d_2sm(dst, &map_lut, (int)(kb * PK), qrow, smem_u32(&full_bar[stage]) & P_PEER_MASK);
                        }
                        if (++stage == STAGES) stage = 0, phase ^= 1;
                    }
            }
        }
    } else if (warp == 5) {
        // ===== MMA issuer (one elected thread of the leader CTA) =====
        if (lane == 0 && leader) {
            uint32_t stage = 0, phase = 0, acc = 0, acc_phase = 0;
            for (uint32_t item = unit; item < nitems; item += nunits) {
                const uint32_t ri = item / p.nqt;
                const uint64_t r0 = (uint64_t)ri * p.tiles_per_item * TM;
                const uint32_t ntile = (uint32_t)min((uint64_t)p.tiles_per_item, (p.n - r0 + TM - 1) / TM);
                for (uint32_t t = 0; t < ntile; ++t) {
                    if (CTAS == 2) mbar_wait_cluster(&tempty_bar[acc], acc_phase ^ 1);
                    else mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
                    tc_fence_after();
                    const uint32_t d_tmem = tmem_base + acc * PN;
                    for (uint32_t kb = 0; kb < p.kblocks; ++kb) {
                        // the peer's generators arrive with release.cluster: acquire at cluster scope
                        if (CTAS == 2) mbar_wait_cluster(&full_bar[stage], phase);
                        else mbar_wait(&full_bar[stage], phase);
                        tc_fence_after();
                        const uint32_t sa = smem_u32(stage_base + stage * Cfg::STAGE_BYTES);
                        const uint64_t da = umma_desc(sa), db = umma_desc(sa + P_A_BYTES);
#pragma unroll
                        for (int k = 0; k < PK / 16; ++k) {  // 16 bf16 = 32 bytes (2 x 16 B units) per K step
                            if (CTAS == 1) umma_bf16(d_tmem, da + 2 * k, db + 2 * k, Cfg::IDESC, (kb | k) != 0);
                            else umma_bf16_2sm(d_tmem, da + 2 * k, db + 2 * k, Cfg::IDESC, (kb | k) != 0);
                        }
                        if (CTAS == 1) umma_commit(&empty_bar[stage]);
                        else umma_commit_2sm(&empty_bar[stage]);  // frees the stage in both CTAs
                        if (++stage == STAGES) stage = 0, phase ^= 1;
                    }
                    if (CTAS == 1) umma_commit(&tfull_bar[acc]);
                    else umma_commit_2sm(&tfull_bar[acc]);
                    if (++acc == 2) acc = 0, acc_phase ^= 1;
                }
            }
        }
    } else if (warp >= 6) {
        // ===== generators: code nibbles -> one-hot bf16 rows, written in the 128B-swizzle layout =====
        const uint32_t gt = threadIdx.x - P_BASE_THREADS;
        const uint32_t gg = gt >> 7;   // generator group
        const uint32_t r = gt & 127;   // row of this CTA's half of the tile
        uint32_t kbc = 0;              // running k-block counter of this CTA (all groups count alike)
        for (uint32_t item = unit; item < nitems; item += nunits) {
            const uint32_t ri = item / p.nqt;
            const uint64_t r0 = (uint64_t)ri * p.tiles_per_item * TM;
            const uint32_t ntile = (uint32_t)min((uint64_t)p.tiles_per_item, (p.n - r0 + TM - 1) / TM);
            for (uint32_t t = 0; t < ntile; ++t) {
                const uint64_t row0 = r0 + (uint64_t)t * TM + cta_rank * PM;
                const uint32_t rows = row0 < p.n ? (uint32_t)min((uint64_t)PM, p.n - row0) : 0u;
                // every generator is done with the previous code tile
                asm volatile("bar.sync 2, %0;" ::"n"(128 * GG) : "memory");
                {
                    const uint32_t bytes = rows * p.enc;          // contiguous in the reference layout
                    const uint8_t* src = p.codes + row0 * p.enc;  // row0 * enc is a multiple of 128
                    const uint32_t vec = bytes / 16;
                    for (uint32_t e = gt; e < vec; e += 128 * GG)
                        reinterpret_cast<uint4*>(codes_s)[e] = __ldg(reinterpret_cast<const uint4*>(src) + e);
                    for (uint32_t e = vec * 16 + gt; e < bytes; e += 128 * GG) codes_s[e] = __ldg(src + e);
                }
                asm volatile("bar.sync 2, %0;" ::"n"(128 * GG) : "memory");
                const bool row_ok = r < rows;
                const uint8_t* my = codes_s + r * p.enc;
                for (uint32_t kb = 0; kb < p.kblocks; ++kb, ++kbc) {
                    if (kbc % GG != gg) continue;
                    const uint32_t stage = kbc % STAGES, phase = (kbc / STAGES) & 1;
                    mbar_wait(&empty_bar[stage], phase ^ 1);
                    uint8_t* arow = stage_base + stage * Cfg::STAGE_BYTES + r * 128;
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const uint32_t g = kb * 4 + i;
                        const bool ok = row_ok && g < p.m;
                        const uint32_t byte = ok ? my[g >> 1] : 0u;
                        const uint32_t c = (g & 1) ? (byte >> 4) : (byte & 0xfu);
                        const uint32_t one = ok ? (0x3F80u << ((c & 1) * 16)) : 0u;  // bf16 1.0 in the low / high half
                        const uint32_t w = (c & 7) >> 1;
                        uint4 v;
                        v.x = w == 0 ? one : 0u;
                        v.y = w == 1 ? one : 0u;
                        v.z = w == 2 ? one : 0u;
                        v.w = w == 3 ? one : 0u;
                        const uint4 z = make_uint4(0u, 0u, 0u, 0u);
                        const uint32_t j0 = 2 * i, j1 = 2 * i + 1;
                        *reinterpret_cast<uint4*>(arow + ((j0 ^ (r & 7)) << 4)) = c < 8 ? v : z;
                        *reinterpret_cast<uint4*>(arow + ((j1 ^ (r & 7)) << 4)) = c < 8 ? z : v;
                    }
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> visible to the MMA
                    __syncwarp();
                    if (lane == 0) {
                        if (CTAS == 1) mbar_arrive(&full_bar[stage]);
                        else mbar_arrive_cluster_release(smem_u32(&full_bar[stage]) & P_PEER_MASK);
                    }
                }
            }
        }
    } else {
        // ===== epilogue: warps 0-3, thread = row (TMEM lane), registers = queries =====
        uint32_t acc = 0, acc_phase = 0;
        const uint32_t lane_base = (uint32_t)warp * 32;
        for (uint32_t item = unit; item < nitems; item += nunits) {
            const uint32_t ri = item / p.nqt, qt = item - ri * p.nqt;
            const uint64_t r0 = (uint64_t)ri * p.tiles_per_item * TM;
            const uint32_t ntile = (uint32_t)min((uint64_t)p.tiles_per_item, (p.n - r0 + TM - 1) / TM);
            const uint32_t q0 = qt * PN;
            asm volatile("bar.sync 1, 128;" ::: "memory");  // previous item's thresholds are no longer read
            if (MODE == 1)
                for (uint32_t c = threadIdx.x; c < PN; c += 128)
                    tau_s[c] = (q0 + c) < p.nq ? p.tau[q0 + c] : __uint_as_float(0xff800000u);  // -inf: nothing passes
            asm volatile("bar.sync 1, 128;" ::: "memory");
            for (uint32_t t = 0; t < ntile; ++t) {
                const uint64_t row = r0 + (uint64_t)t * TM + cta_rank * PM + threadIdx.x;
                const bool row_ok = row < p.n;
                mbar_wait(&tfull_bar[acc], acc_phase);
                tc_fence_after();
                const uint32_t taddr = tmem_base + (lane_base << 16) + acc * PN;
#pragma unroll 1
                for (int c0 = 0; c0 < PN; c0 += 32) {
                    uint32_t v[32];
                    tmem_ld32(taddr + c0, v);
                    if (row_ok) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            if (MODE != 1) {
                                // a warp stores 32 consecutive rows of one query: 128-byte segments
                                const uint32_t q = q0 + c0 + j;
                                const float x = __uint_as_float(v[j]);
                                if (q < p.nq) p.all_out[(size_t)q * p.n + row] = MODE == 0 ? x * p.up_factor : pq_filter_score(x, p.factor);
                                continue;
                            }
                            const float s = pq_filter_score(__uint_as_float(v[j]), p.factor);
                            if (!(s > tau_s[c0 + j])) {  // also keeps NaN (the exact re-evaluation decides)
                                const uint32_t q = q0 + c0 + j;
                                if (q < p.nq) {
                                    const uint32_t pos = atomicAdd(&p.ccnt[q], 1u);
                                    if (pos < p.ccap) p.ccand[(size_t)q * p.ccap + pos] = (uint32_t)row;
                                }
                            }
                        }
                    }
                }
                // hand the accumulator back to the MMA issuer: one arrive per warp, on the leader's barrier
                tc_fence_before();
                __syncwarp();
                if (lane == 0) {
                    if (CTAS == 1) mbar_arrive(&tempty_bar[acc]);
                    else mbar_arrive_cluster_release(smem_u32(&tempty_bar[acc]) & P_PEER_MASK);
                }
                if (++acc == 2) acc = 0, acc_phase ^= 1;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (CTAS == 2) cluster_sync_all();  // neither CTA may exit (or free TMEM) while its peer still uses it
    if (warp == 5) {
        if (CTAS == 2) tmem_dealloc2(tmem_base, P_TMEM_COLS);
        else tmem_dealloc(tmem_base, P_TMEM_COLS);
    }
}

// [nq][m*16] f32 -> [nq][kpad] bf16 (round to nearest), zero padded to whole k-blocks
__global__ void lut_to_bf16_kernel(const float* __restrict__ lut, uint32_t tab, uint32_t kpad, uint64_t count,
                                   __nv_bfloat16* __restrict__ out) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t q = i / kpad;
        const uint32_t e = (uint32_t)(i - q * kpad);
        out[i] = __float2bfloat16_rn(e < tab ? lut[q * tab + e] : 0.f);
    }
}

// exact ADC (reference arithmetic: sequential f32 sum in group order) of the coarse candidates; rows with
// adc <= tau join the candidate list of the global-threshold scan. One CTA per query, its LUT in shared memory.
__global__ void __launch_bounds__(256, 4) pq_exact_cands_kernel(const uint8_t* __restrict__ codes, uint32_t enc, uint32_t m,
                                                             const float* __restrict__ lut, const float* __restrict__ tau,
                                                             const uint32_t* __restrict__ ccnt, const uint32_t* __restrict__ ccand,
                                                             uint32_t ccap, uint32_t id_base, uint32_t* __restrict__ cnt,
                                                             uint64_t* __restrict__ cand, uint32_t cap) {
    extern __shared__ __align__(16) float s_lut[];
    const uint32_t q = blockIdx.x, tab = m * 16;
    for (uint32_t e = threadIdx.x; e < tab; e += blockDim.x) s_lut[e] = lut[(size_t)q * tab + e];
    __syncthreads();
    const uint32_t total = ccnt[q];
    if (total > ccap) {  // coarse list overflowed: force the redo path
        if (threadIdx.x == 0) cnt[q] = cap + 1;
        return;
    }
    const float t = tau[q];
    const bool wide = (enc & 7u) == 0 && enc <= 128;   // code rows as 8-byte words, all loads of a row in flight together
    for (uint32_t i = threadIdx.x; i < total; i += blockDim.x) {
        const uint32_t row = ccand[(size_t)q * ccap + i];
        const uint8_t* cr = codes + (size_t)row * enc;
        float s = 0.f;
        if (wide) {
            // (byte loads inside the summation loop cost a global-memory round trip per pair of groups: 392 us per 1000
            // queries of ~2500 candidates; the sum itself stays the reference's sequential f32 chain in group order)
            uint2 w[16];
            const uint32_t nw = enc >> 3;
#pragma unroll
            for (int k = 0; k < 16; ++k)   // unconditional (clamped) loads: ptxas hoists them ahead of the lookups
                w[k] = __ldg(reinterpret_cast<const uint2*>(cr) + min((uint32_t)k, nw - 1));
#pragma unroll
            for (int k = 0; k < 16; ++k) {
                if ((uint32_t)k >= nw) break;
#pragma unroll
                for (int b = 0; b < 8; ++b) {
                    const uint32_t g = (uint32_t)(k * 16 + b * 2);
                    const uint32_t byte = ((b < 4 ? w[k].x : w[k].y) >> (8 * (b & 3))) & 0xffu;
                    if (g < m) s = __fadd_rn(s, s_lut[g * 16 + (byte & 0xfu)]);
                    if (g + 1 < m) s = __fadd_rn(s, s_lut[(g + 1) * 16 + (byte >> 4)]);
                }
            }
        } else {
            for (uint32_t g = 0; g < m; g += 2) {
                const uint32_t byte = cr[g >> 1];
                s = __fadd_rn(s, s_lut[g * 16 + (byte & 0xfu)]);
                if (g + 1 < m) s = __fadd_rn(s, s_lut[(g + 1) * 16 + (byte >> 4)]);
            }
        }
        if (!(s > t)) {
            const uint32_t pos = atomicAdd(&cnt[q], 1u);
            if (pos < cap) cand[(size_t)q * cap + pos] = make_key(s, id_base + row);
        }
    }
}

bool pq_tensor_supported(const vdb_pq* pq, uint32_t nq) {
    static const int off = getenv("VDB_PQ_NO_TENSOR") ? atoi(getenv("VDB_PQ_NO_TENSOR")) : 0;
    static const int min_nq = getenv("VDB_PQ_TENSOR_MIN_NQ") ? atoi(getenv("VDB_PQ_TENSOR_MIN_NQ")) : 32;
    return !off && pq->n_bits == 4 && pq->metric == VDB_L2SQR && pq->enc <= P_MAX_ENC && pq->n >= 65536 && nq >= (uint32_t)min_nq &&
           ((uintptr_t)pq->d_codes & 15) == 0 && pq->d_sample != nullptr;
}

static uint32_t pq_kpad(const vdb_pq* pq) { return ceil_div(pq->m, 4u) * PK; }

// bf16 copy of the batch's lookup tables, [nq][kpad]
void pq_tensor_lut(const vdb_pq* pq, const float* d_lut, uint32_t nq, DevBuf& lut16, cudaStream_t st) {
    const uint32_t kpad = pq_kpad(pq);
    lut16 = DevBuf((size_t)nq * kpad * 2, st);
    const uint64_t count = (uint64_t)nq * kpad;
    lut_to_bf16_kernel<<<(uint32_t)std::min<uint64_t>(ceil_div<uint64_t>(count, 256), (uint64_t)sm_count() * 16), 256, 0, st>>>(
        d_lut, pq->m * 16, kpad, count, lut16.as<__nv_bfloat16>());
    VDB_LAUNCHED();
}

static int pq_ctas() {
    static const int v = getenv("VDB_PQ_CTAS") ? atoi(getenv("VDB_PQ_CTAS")) : 1;
    return v == 2 ? 2 : 1;
}

template <int MODE, int CTAS, int GG>
static void launch_pq_gemm_t(const vdb_pq* pq, const DevBuf& lut16, uint32_t nq, const uint8_t* codes, uint64_t n, PqGemmParams p,
                             cudaStream_t st) {
    using Cfg = PqCfg<CTAS>;
    const uint32_t kpad = pq_kpad(pq);
    const CUtensorMap map = make_map_bf16(lut16.p, kpad, nq, (uint64_t)kpad * 2, Cfg::B_ROWS);
    p.codes = codes;
    p.n = n;
    p.enc = pq->enc;
    p.m = pq->m;
    p.kblocks = kpad / PK;
    p.nq = nq;
    p.nqt = ceil_div(nq, (uint32_t)PN);
    const uint32_t units = (uint32_t)sm_count() / CTAS;
    const uint64_t row_tiles = ceil_div<uint64_t>(n, PM * CTAS);
    // items small enough that every unit gets several, large enough to amortise the threshold-tile reload
    p.tiles_per_item = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(8, row_tiles * p.nqt / ((uint64_t)units * 4)));
    p.nrow_items = (uint32_t)ceil_div<uint64_t>(row_tiles, p.tiles_per_item);
    auto kern = pq_gemm_kernel<MODE, CTAS, GG>;
    static std::atomic<size_t> configured[VDB_MAX_DEVICES];
    ensure_dyn_smem(kern, Cfg::smem_bytes(P_MAX_ENC), configured);
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(std::min<uint32_t>(units, p.nrow_items * p.nqt) * CTAS);
    cfg.blockDim = dim3(P_BASE_THREADS + 128 * GG);
    cfg.dynamicSmemBytes = Cfg::smem_bytes(pq->enc);
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CTAS;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    ProfScope prof("pq_gemm", st);
    VDB_CUDA(cudaLaunchKernelEx(&cfg, kern, map, p));
    VDB_LAUNCHED();
}

template <int MODE>
static void launch_pq_gemm(const vdb_pq* pq, const DevBuf& lut16, uint32_t nq, const uint8_t* codes, uint64_t n, PqGemmParams p,
                           cudaStream_t st) {
    static const int gg = getenv("VDB_PQ_GEN") ? atoi(getenv("VDB_PQ_GEN")) : 4;
    if (pq_ctas() == 2) {
        if (gg >= 4) launch_pq_gemm_t<MODE, 2, 4>(pq, lut16, nq, codes, n, p, st);
        else if (gg == 2) launch_pq_gemm_t<MODE, 2, 2>(pq, lut16, nq, codes, n, p, st);
        else launch_pq_gemm_t<MODE, 2, 1>(pq, lut16, nq, codes, n, p, st);
    } else {
        if (gg >= 4) launch_pq_gemm_t<MODE, 1, 4>(pq, lut16, nq, codes, n, p, st);
        else if (gg == 2) launch_pq_gemm_t<MODE, 1, 2>(pq, lut16, nq, codes, n, p, st);
        else launch_pq_gemm_t<MODE, 1, 1>(pq, lut16, nq, codes, n, p, st);
    }
}

// SAMPLE step: upper bounds of the ADC values of the sampled rows, [nq][sample_n]. The thresholds derived from them
// need not be exact — the count check of the scan verifies every query afterwards.
void pq_tensor_sample(const vdb_pq* pq, const DevBuf& lut16, uint32_t nq, float* d_all, cudaStream_t st) {
    PqGemmParams p{};
    p.all_out = d_all;
    p.up_factor = 1.0f + pq_rel_bound(pq->m);
    launch_pq_gemm<0>(pq, lut16, nq, pq->d_sample, pq->sample_n, p, st);
}

// FILTER step of the global-threshold scan on the tensor cores: on return cnt[q] / cand[q][] hold exactly the rows
// with adc <= tau_q (as keys), or cnt[q] > cap when a list overflowed.
void pq_tensor_filter(const vdb_pq* pq, const DevBuf& lut16, const float* d_lut, uint32_t nq, const float* d_tau, uint32_t id_base,
                      uint32_t* d_cnt, uint64_t* d_cand, uint32_t cap, cudaStream_t st) {
    const uint32_t tab = pq->m * 16;
    const uint32_t ccap = 2 * cap;
    DevBuf ccnt((size_t)nq * 4, st), ccand((size_t)nq * ccap * 4, st);
    VDB_CUDA(cudaMemsetAsync(ccnt.p, 0, (size_t)nq * 4, st));
    PqGemmParams p{};
    p.tau = d_tau;
    p.factor = 1.0f - pq_rel_bound(pq->m);
    p.ccnt = ccnt.as<uint32_t>();
    p.ccand = ccand.as<uint32_t>();
    p.ccap = ccap;
    launch_pq_gemm<1>(pq, lut16, nq, pq->d_codes, pq->n, p, st);
    (void)tab;
    pq_exact_candidates(pq, d_lut, d_tau, nq, ccnt.as<uint32_t>(), ccand.as<uint32_t>(), ccap, id_base, d_cnt, d_cand, cap, st);
}

// test hook: the filter's S' (d_lower) and the sample pass's upper bound (d_upper) of every (query, row) of the table,
// [nq][n] each, from the same kernel and constants as pq_tensor_filter / pq_tensor_sample
void pq_tensor_bounds(const vdb_pq* pq, const float* d_lut, uint32_t nq, float* d_lower, float* d_upper, cudaStream_t st) {
    DevBuf lut16;
    pq_tensor_lut(pq, d_lut, nq, lut16, st);
    PqGemmParams p{};
    p.all_out = d_upper;
    p.up_factor = 1.0f + pq_rel_bound(pq->m);
    launch_pq_gemm<0>(pq, lut16, nq, pq->d_codes, pq->n, p, st);
    p = PqGemmParams{};
    p.all_out = d_lower;
    p.factor = 1.0f - pq_rel_bound(pq->m);
    launch_pq_gemm<2>(pq, lut16, nq, pq->d_codes, pq->n, p, st);
}

void pq_exact_candidates(const vdb_pq* pq, const float* d_lut, const float* d_tau, uint32_t nq, const uint32_t* d_ccnt,
                         const uint32_t* d_ccand, uint32_t ccap, uint32_t id_base, uint32_t* d_cnt, uint64_t* d_cand,
                         uint32_t cap, cudaStream_t st) {
    const uint32_t tab = pq->m * 16;
    ProfScope prof("pq_exact", st);
    pq_exact_cands_kernel<<<nq, 256, (size_t)tab * 4, st>>>(pq->d_codes, pq->enc, pq->m, d_lut, d_tau, d_ccnt, d_ccand, ccap, id_base,
                                                          d_cnt, d_cand, cap);
    VDB_LAUNCHED();
}

}  // namespace vdb
