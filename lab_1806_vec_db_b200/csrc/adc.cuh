// adc.cuh — the per-row ADC sum shared by the Flat code scan (K8, pq.cu) and the IVF list scan (ivf_pq.cu).
#pragma once
#include "common.cuh"

namespace vdb {

constexpr int ADC_THREADS = 512;
constexpr size_t ADC_SMEM_MAX = 200 * 1024;

// ADC sums of one row against NQ lookup tables, in the reference's arithmetic (pq_table.rs:239-301): one sequential f32
// chain per query in group order, low nibble (= even group) first; cdp = the same chain over dist_cache (cosine).
// cw points at the row's first code word in the transposed layout ([block][word][lane]: word w is cw[w * 32]).
// lut = [NQ][tab] tables, dc = dist_cache [tab]: in shared memory when LUT_SMEM, else read through L1 (NQ == 1 then).
// The branch on LUT_SMEM is compile-time so the shared-memory path compiles to LDS, never to generic loads.
template <int NQ, int NBITS, int METRIC, bool LUT_SMEM>
__device__ __forceinline__ void adc_row_sum(const uint32_t* __restrict__ cw, uint32_t words, uint32_t m, uint32_t tab,
                                            const float* lut, const float* dc, float (&sum)[NQ], float& cdp) {
    constexpr int KC = NBITS == 4 ? 16 : 256;
    auto lookup = [&](uint32_t e) {
        if constexpr (LUT_SMEM) {
#pragma unroll
            for (int q = 0; q < NQ; ++q) sum[q] = __fadd_rn(sum[q], lut[q * tab + e]);
            if (METRIC == VDB_COSINE) cdp = __fadd_rn(cdp, dc[e]);
        } else {
#pragma unroll
            for (int q = 0; q < NQ; ++q) sum[q] = __fadd_rn(sum[q], __ldg(lut + (size_t)q * tab + e));
            if (METRIC == VDB_COSINE) cdp = __fadd_rn(cdp, __ldg(dc + e));
        }
    };
    uint32_t g = 0;
    uint32_t next = cw[0];
    for (uint32_t w = 0; w < words; ++w) {
        const uint32_t word = next;
        if (w + 1 < words) next = cw[(size_t)(w + 1) * 32];  // prefetch the next code word
        if (NBITS == 4) {
            if (LUT_SMEM && METRIC == VDB_L2SQR && g + 8 <= m) {
                // full word: issue all 8 x NQ table reads first, then add in the reference's group order
                float v[8][NQ];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const uint32_t e = (g + i) * KC + ((word >> (4 * i)) & 0xfu);
#pragma unroll
                    for (int q = 0; q < NQ; ++q) v[i][q] = lut[q * tab + e];
                }
#pragma unroll
                for (int i = 0; i < 8; ++i)
#pragma unroll
                    for (int q = 0; q < NQ; ++q) sum[q] = __fadd_rn(sum[q], v[i][q]);
            } else if (g + 8 <= m) {  // full word: 8 groups, no per-nibble bound checks
#pragma unroll
                for (int i = 0; i < 8; ++i) lookup((g + i) * KC + ((word >> (4 * i)) & 0xfu));
            } else {
#pragma unroll
                for (int i = 0; i < 8; ++i)
                    if (g + i < m) lookup((g + i) * KC + ((word >> (4 * i)) & 0xfu));
            }
            g += 8;
        } else {
#pragma unroll
            for (int i = 0; i < 4; ++i)
                if (g + i < m) lookup((g + i) * KC + ((word >> (8 * i)) & 0xffu));
            g += 4;
        }
    }
}

// Queries per CTA and table placement of the per-CTA ADC scans: start from `nqt` (1, 2 or 4), no wider than the batch,
// halve while the tables and top-k segments (smem_for(queries, tables in shared memory)) exceed shared memory, and read
// the tables through L1 when even one query's does not fit.
template <class F>
inline int adc_queries_per_cta(int nqt, uint32_t nq, F smem_for, bool* lut_smem) {
    while (nqt > 1 && (uint32_t)(nqt >> 1) >= nq) nqt >>= 1;
    while (nqt > 1 && smem_for(nqt, true) > ADC_SMEM_MAX) nqt >>= 1;
    *lut_smem = smem_for(nqt, true) <= ADC_SMEM_MAX;
    return nqt;
}

}  // namespace vdb
