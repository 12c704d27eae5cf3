// pq.cu — K6/K7/K8: product-quantisation encode, lookup tables and the ADC scan with top-ef + rerank.
//
// Replaces (reference paths):
//   pq_groups                         src/distance/pq_table.rs:38-53
//   pq_encode + encode loop           src/distance/pq_table.rs:66-91, 178-181 (serial over N in the reference)
//   PQTable::create_lookup            src/distance/pq_table.rs:195-224
//   ADC DistanceAdapter<[u8], LUT>    src/distance/pq_table.rs:239-301
//   FlatIndex::knn_pq + pq_resort     src/index_algorithm/flat_index.rs:84-104, candidate_pair.rs:102-108
//
// Codes, lookup tables and ADC distances are bit-exact: every sum is one thread's sequential f32 chain
// in the reference's order (group order, low nibble = even group first) with unfused multiply/add.
// Pinned by tests/test_index_gpu.py (4-bit m = 240 / 7, 8-bit m = 5) and tests/test_pq_paths_gpu.py: 8-bit codes with
// m % 4 != 0 through every pq_adc_scan_kernel<NQ = 1/2/4, 8, *, LUT_SMEM = true> and <1, 8, *, false>, u8 rows,
// 4-bit sub-vectors longer than ENC_MAXL (pq_encode_kernel), <1, 4, L2SQR, false> at m = 3000, and the top-k of
// the per-CTA scan under maximal candidate pressure.
// HBM layout of the codes for the scan: blocks of 32 rows, word-major ([block][word][lane]) so a warp's
// load of one code word for its 32 rows is a single coalesced 128-byte request; one lane owns one row, all
// lanes look up the SAME group at the same time, so the 16-entry LUT row is read conflict free.
#include <cstdlib>
#include <cstring>

#include "adc.cuh"
#include "index.cuh"
#include "topk.cuh"

namespace vdb {

void pq_groups_host(uint32_t dim, uint32_t m, std::vector<uint32_t>& lo, std::vector<uint32_t>& len) {
    VDB_REQUIRE(dim > 0, "dim must be greater than 0 in PQTable.");
    VDB_REQUIRE(m > 0, "m must be greater than 0 in PQTable.");
    VDB_REQUIRE(dim >= m, "dim must be greater than or equal to m in PQTable.");
    lo.clear();
    len.clear();
    uint32_t cur = 0;
    while (cur < dim) {
        const uint32_t rem = m - (uint32_t)lo.size();
        const uint32_t gs = (dim - cur + rem - 1) / rem;
        lo.push_back(cur);
        len.push_back(gs);
        cur += gs;
    }
}

template <typename T> __device__ __forceinline__ float pq_f32(T v) { return (float)v; }

// exact (reference-order) distance of a sub-vector against one centroid
template <typename T, int METRIC>
__device__ __forceinline__ float sub_distance(const T* __restrict__ v, const T* __restrict__ c, uint32_t len,
                                              float cnorm) {
    float s = 0.f, svv = 0.f;
    for (uint32_t j = 0; j < len; ++j) {
        const float x = pq_f32(v[j]), y = pq_f32(c[j]);
        if (METRIC == VDB_L2SQR) {
            const float df = __fsub_rn(x, y);
            s = __fadd_rn(s, __fmul_rn(df, df));
        } else {
            s = __fadd_rn(s, __fmul_rn(x, y));
            svv = __fadd_rn(svv, __fmul_rn(x, x));
        }
    }
    if (METRIC == VDB_L2SQR) return s;
    const float den = fmaxf(__fmul_rn(sqrtf(svv), cnorm), 1e-10f);
    return __fsub_rn(1.0f, __fdiv_rn(s, den));
}

// per centroid: dot(c,c) (dist_cache for cosine) and ||c||
template <typename T>
__global__ void pq_centroid_norms_kernel(const T* __restrict__ cb, const uint32_t* __restrict__ groups, uint32_t m,
                                         uint32_t kc, int metric, float* __restrict__ dist_cache,
                                         float* __restrict__ cb_norm) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m * kc) return;
    const uint32_t g = i / kc, c = i - g * kc;
    const uint32_t len = groups[3 * g + 1], off = groups[3 * g + 2];
    const T* cc = cb + off + (size_t)c * len;
    float s = 0.f;
    for (uint32_t j = 0; j < len; ++j) {
        const float y = pq_f32(cc[j]);
        s = __fadd_rn(s, __fmul_rn(y, y));
    }
    dist_cache[i] = metric == VDB_COSINE ? s : 0.f;
    cb_norm[i] = sqrtf(s);
}

// K6: one thread per (row, code byte)
template <typename T, int METRIC>
__global__ void __launch_bounds__(256) pq_encode_kernel(const T* __restrict__ rows, uint64_t n, uint64_t pitch,
                                                        const T* __restrict__ cb, const uint32_t* __restrict__ groups,
                                                        const float* __restrict__ cb_norm, uint32_t m, uint32_t n_bits,
                                                        uint32_t kc, uint32_t enc, uint8_t* __restrict__ codes) {
    const uint64_t total = n * enc;
    for (uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total;
         t += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t row = t / enc;
        const uint32_t b = (uint32_t)(t - row * enc);
        const uint32_t per = n_bits == 4 ? 2u : 1u;
        uint32_t byte = 0;
        for (uint32_t h = 0; h < per; ++h) {
            const uint32_t g = b * per + h;
            if (g >= m) break;
            const uint32_t lo = groups[3 * g], len = groups[3 * g + 1], off = groups[3 * g + 2];
            const T* v = rows + row * pitch + lo;
            unsigned long long best = KEY_NONE;
            for (uint32_t c = 0; c < kc; ++c) {
                const float d = sub_distance<T, METRIC>(v, cb + off + (size_t)c * len, len, cb_norm[g * kc + c]);
                const unsigned long long key = make_key(d, c);
                best = key < best ? key : best;
            }
            byte |= key_id(best) << (4 * h);
        }
        codes[t] = (uint8_t)byte;
    }
}

// K6b: 4-bit encode with everything staged in shared memory. The codebooks (16 x dim elements) are kept as
// [j][c][group] so the lanes of a warp - consecutive code bytes, i.e. consecutive groups - read consecutive words; a
// tile of rows is loaded with coalesced 128-bit loads. Same arithmetic as K6 (sequential f32 per sub-vector, ties to the
// lowest centroid), so the codes are bit-identical; 66 ms -> a few ms for 1M x 960 (the per-thread global re-reads of K6
// were L1-bound at 1 % of HBM bandwidth).
constexpr int ENC_MAXL = 8;   // longest sub-vector handled in registers
constexpr int ENC_ROWS = 8;   // rows per tile
// nearest of the 16 centroids of group g for the sub-vector at rowS + lo, LEN elements (reference order, ties -> lowest id)
template <int METRIC, int LEN>
__device__ __forceinline__ uint32_t encode_group(const float* __restrict__ x, const float* __restrict__ cbS, const float* __restrict__ cnS,
                                                 uint32_t mp, uint32_t g) {
    float v[LEN];
    float svv = 0.f;
#pragma unroll
    for (int j = 0; j < LEN; ++j) {
        v[j] = x[j];
        if (METRIC == VDB_COSINE) svv = __fadd_rn(svv, __fmul_rn(v[j], v[j]));
    }
    const float vn = sqrtf(svv);
    unsigned long long best = KEY_NONE;
#pragma unroll
    for (uint32_t c = 0; c < 16; ++c) {
        float sacc = 0.f;
#pragma unroll
        for (int j = 0; j < LEN; ++j) {
            const float y = cbS[((size_t)j * 16 + c) * mp + g];
            if (METRIC == VDB_L2SQR) {
                const float df = __fsub_rn(v[j], y);
                sacc = __fadd_rn(sacc, __fmul_rn(df, df));
            } else {
                sacc = __fadd_rn(sacc, __fmul_rn(v[j], y));
            }
        }
        float d = sacc;
        if (METRIC == VDB_COSINE) d = __fsub_rn(1.0f, __fdiv_rn(sacc, fmaxf(__fmul_rn(vn, cnS[c * mp + g]), 1e-10f)));
        const unsigned long long key = make_key(d, c);
        best = key < best ? key : best;
    }
    return key_id(best);
}

template <typename T, int METRIC>
__global__ void __launch_bounds__(256) pq_encode4_kernel(const T* __restrict__ rows, uint64_t n, uint64_t pitch, uint32_t dim,
                                                         const T* __restrict__ cb, const uint32_t* __restrict__ groups,
                                                         const float* __restrict__ cb_norm, uint32_t m, uint32_t enc,
                                                         uint32_t max_len, uint8_t* __restrict__ codes) {
    extern __shared__ __align__(16) uint8_t smem[];
    const uint32_t mp = m + (m & 1);                               // even: a byte's two groups always exist in the table
    float* cbS = reinterpret_cast<float*>(smem);                    // [max_len][16][mp]
    float* cnS = cbS + (size_t)max_len * 16 * mp;                   // [16][mp]  ||c|| (cosine)
    float* rowS = cnS + 16 * mp;                                    // [ENC_ROWS][dimp]
    const uint32_t dimp = (dim + 3) & ~3u;
    uint16_t* gl = reinterpret_cast<uint16_t*>(rowS + (size_t)ENC_ROWS * dimp);  // [mp][2] (lo, len)
    for (uint32_t i = threadIdx.x; i < max_len * 16 * mp; i += blockDim.x) cbS[i] = 0.f;
    for (uint32_t i = threadIdx.x; i < 16 * mp; i += blockDim.x) cnS[i] = 0.f;
    for (uint32_t g = threadIdx.x; g < mp; g += blockDim.x) {
        gl[2 * g] = g < m ? (uint16_t)groups[3 * g] : 0;
        gl[2 * g + 1] = g < m ? (uint16_t)groups[3 * g + 1] : 0;
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < m * 16; i += blockDim.x) {
        const uint32_t g = i >> 4, c = i & 15;
        const uint32_t len = groups[3 * g + 1], off = groups[3 * g + 2];
        for (uint32_t j = 0; j < len; ++j) cbS[((size_t)j * 16 + c) * mp + g] = pq_f32(cb[off + (size_t)c * len + j]);
        cnS[c * mp + g] = cb_norm[i];
    }
    __syncthreads();
    const uint64_t ntiles = (n + ENC_ROWS - 1) / ENC_ROWS;
    for (uint64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const uint64_t row0 = tile * ENC_ROWS;
        const uint32_t nr = (uint32_t)min((uint64_t)ENC_ROWS, n - row0);
        if (sizeof(T) == 4 && (dim & 3) == 0 && (pitch & 3) == 0 && (reinterpret_cast<uintptr_t>(rows) & 15) == 0) {
            const uint32_t d4 = dim >> 2;
            for (uint32_t i = threadIdx.x; i < nr * d4; i += blockDim.x) {
                const uint32_t r = i / d4, e = i - r * d4;
                reinterpret_cast<float4*>(rowS + (size_t)r * dimp)[e] =
                    __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(rows) + (row0 + r) * pitch) + e);
            }
        } else {
            for (uint32_t i = threadIdx.x; i < nr * dim; i += blockDim.x) {
                const uint32_t r = i / dim, e = i - r * dim;
                rowS[(size_t)r * dimp + e] = pq_f32(rows[(row0 + r) * pitch + e]);
            }
        }
        __syncthreads();
        for (uint32_t t = threadIdx.x; t < nr * enc; t += blockDim.x) {
            const uint32_t r = t / enc, b = t - r * enc;
            uint32_t byte = 0;
#pragma unroll
            for (uint32_t h = 0; h < 2; ++h) {
                const uint32_t g = 2 * b + h;
                if (g >= m) break;
                const uint32_t lo = gl[2 * g], len = gl[2 * g + 1];
                const float* x = rowS + (size_t)r * dimp + lo;
                uint32_t code = 0;
                switch (len) {
                    case 1: code = encode_group<METRIC, 1>(x, cbS, cnS, mp, g); break;
                    case 2: code = encode_group<METRIC, 2>(x, cbS, cnS, mp, g); break;
                    case 3: code = encode_group<METRIC, 3>(x, cbS, cnS, mp, g); break;
                    case 4: code = encode_group<METRIC, 4>(x, cbS, cnS, mp, g); break;
                    case 5: code = encode_group<METRIC, 5>(x, cbS, cnS, mp, g); break;
                    case 6: code = encode_group<METRIC, 6>(x, cbS, cnS, mp, g); break;
                    case 7: code = encode_group<METRIC, 7>(x, cbS, cnS, mp, g); break;
                    default: code = encode_group<METRIC, 8>(x, cbS, cnS, mp, g); break;
                }
                byte |= code << (4 * h);
            }
            codes[(row0 + r) * enc + b] = (uint8_t)byte;
        }
        __syncthreads();
    }
}
static size_t encode4_smem(uint32_t m, uint32_t max_len, uint32_t dim) {
    const uint32_t mp = m + (m & 1);
    return ((size_t)max_len * 16 * mp + 16 * mp + (size_t)ENC_ROWS * ((dim + 3) & ~3u)) * 4 + (size_t)mp * 4;
}

// reference layout [n][enc] -> [ceil(n/32)][words][32] u32 (zero padded)
__global__ void pq_transpose_kernel(const uint8_t* __restrict__ codes, uint64_t n, uint32_t enc, uint32_t words,
                                    uint32_t* __restrict__ out) {
    const uint64_t total = ceil_div<uint64_t>(n, 32) * words * 32;
    for (uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total;
         t += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t lane = t & 31;
        const uint64_t bw = t >> 5;
        const uint64_t blk = bw / words;
        const uint32_t w = (uint32_t)(bw - blk * words);
        const uint64_t row = blk * 32 + lane;
        uint32_t v = 0;
        if (row < n)
            for (uint32_t i = 0; i < 4; ++i) {
                const uint32_t byte = w * 4 + i;
                if (byte < enc) v |= (uint32_t)codes[row * enc + byte] << (8 * i);
            }
        out[t] = v;
    }
}

// K7: one thread per (query, group, centroid); qcache by one thread per query (sequential dot)
template <typename T>
__global__ void pq_lut_kernel(const T* __restrict__ q, uint32_t nq, uint32_t dim, const T* __restrict__ cb,
                              const uint32_t* __restrict__ groups, uint32_t m, uint32_t kc, int metric,
                              float* __restrict__ lut, float* __restrict__ qcache) {
    const uint64_t total = (uint64_t)nq * m * kc;
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < total) {
        const uint32_t qi = (uint32_t)(t / (m * kc));
        const uint32_t r = (uint32_t)(t - (uint64_t)qi * m * kc);
        const uint32_t g = r / kc, c = r - g * kc;
        const uint32_t lo = groups[3 * g], len = groups[3 * g + 1], off = groups[3 * g + 2];
        const T* v = q + (size_t)qi * dim + lo;
        const T* cc = cb + off + (size_t)c * len;
        float s = 0.f;
        for (uint32_t j = 0; j < len; ++j) {
            const float x = pq_f32(v[j]), y = pq_f32(cc[j]);
            if (metric == VDB_L2SQR) {
                const float df = __fsub_rn(x, y);
                s = __fadd_rn(s, __fmul_rn(df, df));
            } else {
                s = __fadd_rn(s, __fmul_rn(x, y));
            }
        }
        lut[t] = s;
    }
    if (t < nq) {
        float s = 0.f;
        if (metric == VDB_COSINE) {
            const T* v = q + (size_t)t * dim;
            for (uint32_t j = 0; j < dim; ++j) {
                const float x = pq_f32(v[j]);
                s = __fadd_rn(s, __fmul_rn(x, x));
            }
            s = sqrtf(s);
        }
        qcache[t] = s;
    }
}

// ---- K8: ADC scan ----------------------------------------------------------------------------------

struct AdcParams {
    const uint32_t* codes_t;
    uint64_t n;
    uint32_t words, m, kc;
    const float* lut;         // [nq][m*kc]   (blockIdx.y selects the group of NQ queries)
    const float* dist_cache;  // [m*kc]
    const float* qcache;      // [nq]
    uint32_t nq_total;        // queries of this launch
    uint32_t K, P, limit;
    uint32_t id_base;
    uint32_t iters;           // row tiles per CTA
    uint64_t* partial;        // [NQ][gridDim.x][K]
    float* all_out;           // optional: [nq_pass][n] every ADC distance (no top-k)
};

// LUT_SMEM: lookup tables staged in shared memory (4-bit codes); otherwise read through L1 (8-bit codes)
template <int NQ, int NBITS, int METRIC, bool LUT_SMEM>
__global__ void __launch_bounds__(ADC_THREADS) pq_adc_scan_kernel(AdcParams p) {
    extern __shared__ __align__(16) uint8_t smem[];
    const uint32_t tab = p.m * p.kc;
    // this CTA's group of NQ queries
    const uint32_t q_first = blockIdx.y * NQ;
    const uint32_t nq_valid = min((uint32_t)NQ, p.nq_total - q_first);
    p.lut += (size_t)q_first * tab;
    p.qcache += q_first;
    if (p.partial) p.partial += (size_t)q_first * gridDim.x * p.K;
    if (p.all_out) p.all_out += (size_t)q_first * p.n;
    float* s_lut = reinterpret_cast<float*>(smem);
    float* s_dc = s_lut + (LUT_SMEM ? (size_t)NQ * tab : 0);
    uint8_t* after = reinterpret_cast<uint8_t*>(s_dc + ((LUT_SMEM && METRIC == VDB_COSINE) ? tab : 0));
    uint64_t* tk = reinterpret_cast<uint64_t*>(after);
    TopkSmem topk{tk, reinterpret_cast<uint32_t*>(tk + (size_t)NQ * p.P), p.K, p.P, NQ, p.limit};
    if (LUT_SMEM) {
        for (uint32_t i = threadIdx.x; i < NQ * tab; i += blockDim.x)
            s_lut[i] = (i / tab < nq_valid) ? p.lut[i] : 0.f;
        if (METRIC == VDB_COSINE)
            for (uint32_t i = threadIdx.x; i < tab; i += blockDim.x) s_dc[i] = p.dist_cache[i];
    }
    const bool do_topk = p.all_out == nullptr;
    if (do_topk) topk.init();
    else __syncthreads();
    const int lane = threadIdx.x & 31;
    float qn[NQ];
#pragma unroll
    for (int q = 0; q < NQ; ++q) qn[q] = (METRIC == VDB_COSINE && q < (int)nq_valid) ? p.qcache[q] : 0.f;

    for (uint32_t it = 0; it < p.iters; ++it) {
        const uint64_t tile = (uint64_t)it * gridDim.x + blockIdx.x;
        const uint64_t row = tile * ADC_THREADS + threadIdx.x;
        const uint64_t blk = row >> 5;
        float sum[NQ];
        float cdp = 0.f;
#pragma unroll
        for (int q = 0; q < NQ; ++q) sum[q] = 0.f;
        const bool in = row < p.n;
        if (in)
            adc_row_sum<NQ, NBITS, METRIC, LUT_SMEM>(p.codes_t + blk * p.words * 32 + lane, p.words, p.m, tab,
                                                     LUT_SMEM ? s_lut : p.lut, LUT_SMEM ? s_dc : p.dist_cache, sum, cdp);
        bool want = false;
#pragma unroll
        for (int q = 0; q < NQ; ++q) {
            if (q < (int)nq_valid && in) {
                float d = sum[q];
                if (METRIC == VDB_COSINE) {
                    const float den = fmaxf(__fmul_rn(sqrtf(cdp), qn[q]), 1e-10f);
                    d = __fsub_rn(1.0f, __fdiv_rn(sum[q], den));
                }
                if (do_topk) {
                    const uint64_t key = make_key(d, p.id_base + (uint32_t)row);
                    if (key < topk.tau(q)) want |= topk.push(q, key);
                } else {
                    p.all_out[(size_t)q * p.n + row] = d;
                }
            }
        }
        if (do_topk) topk.maybe_flush(want);
    }
    if (do_topk) {
        topk.final_flush();
        for (uint32_t i = threadIdx.x; i < nq_valid * p.K; i += blockDim.x) {
            const uint32_t qi = i / p.K, j = i - qi * p.K;
            p.partial[((size_t)qi * gridDim.x + blockIdx.x) * p.K + j] = topk.seg(qi)[j];
        }
    }
}

// ---- global-threshold ADC scan (4-bit codes, batches) --------------------------------------------------------
// The per-CTA top-k of pq_adc_scan_kernel costs as much as the lookups when ef is large (every CTA sorts its own
// ef-best of ~7 k rows). Here the threshold is GLOBAL: the ADC distances of a stratified ~3 % row sample give, per
// query, a value tau_q that at least max(ef,k) rows of the shard undercut with probability > 1 - 1e-5 (ADC values
// are exact, so no margin is needed); the scan then only appends rows with adc <= tau_q to a per-query list and the
// exact top-max(ef,k) by (adc, id) is selected from that short list. Queries whose list turns out too short or
// overflows are re-run through the per-CTA kernel. The LUTs of the 4 queries of a pass are interleaved
// ([entry][query] as float4) so one LDS.128 serves all four.
constexpr int GQ = 4;
struct AdcGlobalParams {
    const uint32_t* codes_t;
    uint64_t n;
    uint32_t words, m;
    const float* lut;         // [GQ][m*16] of this pass (rows beyond nq_valid are ignored)
    const float* dist_cache;  // [m*16] (cosine)
    const float* qcache;      // [GQ]
    uint32_t nq_valid;
    uint32_t id_base;
    uint32_t iters;
    float* all_out;           // MODE 0: [GQ][n] every ADC distance
    const float* tau;         // MODE 1: [GQ]
    uint32_t* cnt;            // MODE 1: [GQ]
    uint64_t* cand;           // MODE 1: [GQ][cap]
    uint32_t cap;
};

template <int METRIC, int MODE>
__global__ void __launch_bounds__(ADC_THREADS) pq_adc_global_kernel(const AdcGlobalParams p) {
    extern __shared__ __align__(16) uint8_t smem[];
    const uint32_t tab = p.m * 16;
    float4* s_lut = reinterpret_cast<float4*>(smem);           // [tab] (q0, q1, q2, q3)
    float* s_dc = reinterpret_cast<float*>(s_lut + tab);        // [tab] (cosine)
    for (uint32_t e = threadIdx.x; e < tab; e += blockDim.x) {
        float4 v;
        v.x = p.lut[e];
        v.y = p.nq_valid > 1 ? p.lut[(size_t)tab + e] : 0.f;
        v.z = p.nq_valid > 2 ? p.lut[(size_t)2 * tab + e] : 0.f;
        v.w = p.nq_valid > 3 ? p.lut[(size_t)3 * tab + e] : 0.f;
        s_lut[e] = v;
        if (METRIC == VDB_COSINE) s_dc[e] = p.dist_cache[e];
    }
    __syncthreads();
    const int lane = threadIdx.x & 31;
    float tau[GQ], qn[GQ];
#pragma unroll
    for (int q = 0; q < GQ; ++q) {
        tau[q] = (MODE == 1 && q < (int)p.nq_valid) ? p.tau[q] : __uint_as_float(0xff800000u);
        qn[q] = (METRIC == VDB_COSINE && q < (int)p.nq_valid) ? p.qcache[q] : 0.f;
    }
    for (uint32_t it = 0; it < p.iters; ++it) {
        const uint64_t tile = (uint64_t)it * gridDim.x + blockIdx.x;
        const uint64_t row = tile * ADC_THREADS + threadIdx.x;
        if (row >= p.n) continue;
        const uint32_t* cw = p.codes_t + (row >> 5) * p.words * 32 + lane;
        float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f, cdp = 0.f;
        uint32_t g = 0;
        uint32_t next = cw[0];
        for (uint32_t w = 0; w < p.words; ++w) {
            const uint32_t word = next;
            if (w + 1 < p.words) next = cw[(size_t)(w + 1) * 32];
            const uint32_t ng = min(8u, p.m - g);
            if (ng == 8) {
                float4 v[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) v[i] = s_lut[(g + i) * 16 + ((word >> (4 * i)) & 0xfu)];
#pragma unroll
                for (int i = 0; i < 8; ++i) {  // the reference's group order, one sequential chain per query
                    s0 = __fadd_rn(s0, v[i].x);
                    s1 = __fadd_rn(s1, v[i].y);
                    s2 = __fadd_rn(s2, v[i].z);
                    s3 = __fadd_rn(s3, v[i].w);
                }
                if (METRIC == VDB_COSINE) {
#pragma unroll
                    for (int i = 0; i < 8; ++i) cdp = __fadd_rn(cdp, s_dc[(g + i) * 16 + ((word >> (4 * i)) & 0xfu)]);
                }
            } else {
                for (uint32_t i = 0; i < ng; ++i) {
                    const uint32_t e = (g + i) * 16 + ((word >> (4 * i)) & 0xfu);
                    const float4 v = s_lut[e];
                    s0 = __fadd_rn(s0, v.x);
                    s1 = __fadd_rn(s1, v.y);
                    s2 = __fadd_rn(s2, v.z);
                    s3 = __fadd_rn(s3, v.w);
                    if (METRIC == VDB_COSINE) cdp = __fadd_rn(cdp, s_dc[e]);
                }
            }
            g += 8;
        }
        float d[GQ] = {s0, s1, s2, s3};
#pragma unroll
        for (int q = 0; q < GQ; ++q) {
            if (q >= (int)p.nq_valid) continue;
            float dd = d[q];
            if (METRIC == VDB_COSINE) {
                const float den = fmaxf(__fmul_rn(sqrtf(cdp), qn[q]), 1e-10f);
                dd = __fsub_rn(1.0f, __fdiv_rn(d[q], den));
            }
            if (MODE == 0) {
                p.all_out[(size_t)q * p.n + row] = dd;
            } else if (!(dd > tau[q])) {  // adc <= tau (NaN is kept: it orders last and is dropped by the selection)
                const uint32_t pos = atomicAdd(&p.cnt[q], 1u);
                if (pos < p.cap) p.cand[(size_t)q * p.cap + pos] = make_key(dd, p.id_base + (uint32_t)row);
            }
        }
    }
}

__global__ void floats_to_keys_kernel(const float* __restrict__ v, uint64_t count, uint64_t per_q, uint64_t* __restrict__ keys) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (uint64_t)gridDim.x * blockDim.x)
        keys[i] = make_key(v[i], (uint32_t)(i % per_q));
}
__global__ void tau_from_jkeys_kernel(const uint64_t* __restrict__ jkeys, uint32_t nq, uint32_t j, float* __restrict__ tau) {
    const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q < nq) tau[q] = key_dist(jkeys[(size_t)q * j + (j - 1)]);
}
// tau[q] = the j-th smallest (1-based) of the ns sampled scores of query q: radix select over the order-preserving bit
// pattern, 11 + 11 + 10 bits, one CTA per query. (Converting the scores to keys and running the sorting top-k merge over
// 32768 of them per query cost 83 + 247 us per 1000 queries.)
__global__ void __launch_bounds__(256) select_jth_kernel(const float* __restrict__ v, uint32_t ns, uint32_t j, float* __restrict__ tau) {
    __shared__ uint32_t hist[2048];
    __shared__ uint32_t s_bin, s_k;
    const float* x = v + (size_t)blockIdx.x * ns;
    uint32_t prefix = 0, mask = 0, kk = j;
    const int shifts[3] = {21, 10, 0}, widths[3] = {11, 11, 10};
    for (int pass = 0; pass < 3; ++pass) {
        const int sh = shifts[pass];
        const uint32_t nb = 1u << widths[pass];
        for (uint32_t b = threadIdx.x; b < nb; b += blockDim.x) hist[b] = 0;
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < ns; i += blockDim.x) {
            const uint32_t o = f32_order_bits(x[i]);
            if ((o & mask) == prefix) atomicAdd(&hist[(o >> sh) & (nb - 1)], 1u);
        }
        __syncthreads();
        if (threadIdx.x < 32) {   // warp 0: the bin that holds the kk-th element
            const uint32_t per = nb / 32;
            uint32_t sum = 0;
            for (uint32_t i = 0; i < per; ++i) sum += hist[threadIdx.x * per + i];
            uint32_t incl = sum;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t y = __shfl_up_sync(0xffffffffu, incl, o);
                if ((int)threadIdx.x >= o) incl += y;
            }
            const uint32_t before = incl - sum;
            if (before < kk && kk <= incl) {   // exactly one lane
                uint32_t run = before;
                for (uint32_t i = 0; i < per; ++i) {
                    const uint32_t c = hist[threadIdx.x * per + i];
                    if (run < kk && kk <= run + c) s_bin = threadIdx.x * per + i, s_k = kk - run;
                    run += c;
                }
            }
        }
        __syncthreads();
        prefix |= s_bin << sh;
        mask |= (nb - 1) << sh;
        kk = s_k;
        __syncthreads();
    }
    if (threadIdx.x == 0) tau[blockIdx.x] = f32_from_order_bits(prefix);
}
// queries whose candidate list is too short (the threshold was too tight) or overflowed must be redone
__global__ void adc_check_kernel(const uint32_t* __restrict__ cnt, uint32_t nq, uint32_t need, uint32_t cap,
                                 uint32_t* __restrict__ redo, uint32_t* __restrict__ nredo) {
    const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q < nq && (cnt[q] < need || cnt[q] > cap)) redo[atomicAdd(nredo, 1u)] = q;
}
__global__ void gather_f32_rows_kernel(const float* __restrict__ src, uint32_t width, const uint32_t* __restrict__ idx,
                                       uint32_t cnt, float* __restrict__ dst) {
    const uint32_t i = blockIdx.x;
    if (i >= cnt) return;
    for (uint32_t e = threadIdx.x; e < width; e += blockDim.x) dst[(size_t)i * width + e] = src[(size_t)idx[i] * width + e];
}
__global__ void scatter_u64_rows_kernel(const uint64_t* __restrict__ src, uint32_t width, const uint32_t* __restrict__ idx,
                                        uint32_t cnt, uint64_t* __restrict__ dst) {
    const uint32_t i = blockIdx.x;
    if (i >= cnt) return;
    for (uint32_t e = threadIdx.x; e < width; e += blockDim.x) dst[(size_t)idx[i] * width + e] = src[(size_t)i * width + e];
}

template <int NQ>
static void adc_launch(const vdb_pq* pq, const AdcParams& p, bool lut_smem, uint32_t grid, uint32_t groups, size_t smem,
                       cudaStream_t st) {
    auto go = [&](auto kern) {
        if (smem > 48 * 1024)
            VDB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ADC_SMEM_MAX));
        ProfScope prof("pq_adc", st);
        kern<<<dim3(grid, groups), ADC_THREADS, smem, st>>>(p);
        VDB_LAUNCHED();
    };
    const bool cosine = pq->metric == VDB_COSINE;
    if (pq->n_bits == 4) {
        if (lut_smem) {
            if (cosine) go(pq_adc_scan_kernel<NQ, 4, VDB_COSINE, true>);
            else go(pq_adc_scan_kernel<NQ, 4, VDB_L2SQR, true>);
        } else {
            if (cosine) go(pq_adc_scan_kernel<NQ, 4, VDB_COSINE, false>);
            else go(pq_adc_scan_kernel<NQ, 4, VDB_L2SQR, false>);
        }
    } else {
        if (lut_smem) {
            if (cosine) go(pq_adc_scan_kernel<NQ, 8, VDB_COSINE, true>);
            else go(pq_adc_scan_kernel<NQ, 8, VDB_L2SQR, true>);
        } else {
            if (cosine) go(pq_adc_scan_kernel<NQ, 8, VDB_COSINE, false>);
            else go(pq_adc_scan_kernel<NQ, 8, VDB_L2SQR, false>);
        }
    }
}

// runs the scan for `nq` queries whose LUTs are in d_lut; either top-K keys ([nq][K]) or all distances
static void adc_scan(const vdb_pq* pq, const float* d_lut, const float* d_qcache, uint32_t nq, uint32_t K,
                     uint32_t id_base, uint64_t* d_keys, float* d_all, cudaStream_t st) {
    if (nq == 0) return;
    const uint32_t tab = pq->m * pq->kc;
    const bool topk = d_all == nullptr;
    const uint32_t P = topk ? topk_segment_size(K, ADC_THREADS) : 0;
    auto smem_for = [&](int t, bool ls) {
        size_t s = ls ? ((size_t)t * tab + (pq->metric == VDB_COSINE ? tab : 0)) * 4 : 0;
        if (topk) s += TopkSmem::bytes(t, P);
        return s;
    };
    static const int nqt_env = getenv("VDB_ADC_NQ") ? atoi(getenv("VDB_ADC_NQ")) : 0;
    bool lut_smem = true;
    const int nqt = adc_queries_per_cta((nqt_env == 1 || nqt_env == 2 || nqt_env == 4) ? nqt_env : 4, nq, smem_for, &lut_smem);
    VDB_REQUIRE(smem_for(nqt, lut_smem) <= ADC_SMEM_MAX, "ADC scan: ef=%u too large for the fused top-k", K);
    const uint64_t tiles = ceil_div<uint64_t>(pq->n, ADC_THREADS);
    // one wave: resident CTAs per SM is limited by shared memory (LUTs + top-k segments)
    const uint32_t occ = (uint32_t)std::max<size_t>(1, std::min<size_t>(8, (220 * 1024) / std::max<size_t>(smem_for(nqt, lut_smem), 1)));
    const uint32_t grid = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(tiles, (uint64_t)sm_count() * occ));
    AdcParams p{};
    p.codes_t = pq->d_codes_t;
    p.n = pq->n;
    p.words = pq->words;
    p.m = pq->m;
    p.kc = pq->kc;
    p.dist_cache = pq->d_dist_cache;
    p.K = K;
    p.P = P;
    p.limit = topk ? P - K - ADC_THREADS : 0;
    p.id_base = id_base;
    p.iters = (uint32_t)ceil_div<uint64_t>(tiles, grid);
    const size_t per_q = (size_t)grid * K * 8;
    uint32_t chunk = topk ? (uint32_t)std::max<size_t>(4, (size_t)(64u << 20) / std::max<size_t>(per_q, 1)) : nq;
    chunk = std::min(std::min(round_up(chunk, 4u), round_up(nq, 4u)), 65535u * (uint32_t)nqt);  // gridDim.y limit
    DevBuf partial(topk ? per_q * chunk : 0, st);
    for (uint32_t q0 = 0; q0 < nq; q0 += chunk) {
        const uint32_t qn = std::min(chunk, nq - q0);
        // one launch for all query groups of the chunk: blockIdx.y = group of nqt queries
        p.lut = d_lut + (size_t)q0 * tab;
        p.qcache = d_qcache + q0;
        p.nq_total = qn;
        p.partial = topk ? partial.as<uint64_t>() : nullptr;
        p.all_out = topk ? nullptr : d_all + (size_t)q0 * pq->n;
        const uint32_t groups = ceil_div(qn, (uint32_t)nqt);
        const size_t smem = smem_for(nqt, lut_smem);
        switch (nqt) {
            case 1: adc_launch<1>(pq, p, lut_smem, grid, groups, smem, st); break;
            case 2: adc_launch<2>(pq, p, lut_smem, grid, groups, smem, st); break;
            default: adc_launch<4>(pq, p, lut_smem, grid, groups, smem, st); break;
        }
        if (topk)
            launch_merge_keys(partial.as<uint64_t>(), grid, qn, K, false, K, d_keys + (size_t)q0 * K, nullptr,
                              nullptr, nullptr, st);
    }
}


static void adc_scan(const vdb_pq* pq, const float* d_lut, const float* d_qcache, uint32_t nq, uint32_t K,
                     uint32_t id_base, uint64_t* d_keys, float* d_all, cudaStream_t st);

static int adc_gq() { return GQ; }

template <int MODE>
static void launch_adc_global(const vdb_pq* pq, AdcGlobalParams p, const uint32_t* codes_t, uint64_t n, cudaStream_t st) {
    const uint32_t tab = pq->m * 16;
    const int gq = adc_gq();
    const size_t smem = (size_t)tab * 4 * gq + (pq->metric == VDB_COSINE ? (size_t)tab * 4 : 0);
    const uint64_t tiles = ceil_div<uint64_t>(n, ADC_THREADS);
    const uint32_t occ = (uint32_t)std::max<size_t>(1, std::min<size_t>(4, (220 * 1024) / std::max<size_t>(smem, 1)));
    const uint32_t grid = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(tiles, (uint64_t)sm_count() * occ));
    p.codes_t = codes_t;
    p.n = n;
    p.words = pq->words;
    p.m = pq->m;
    p.dist_cache = pq->d_dist_cache;
    p.iters = (uint32_t)ceil_div<uint64_t>(tiles, grid);
    auto go = [&](auto kern) {
        if (smem > 48 * 1024)
            VDB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ADC_SMEM_MAX));
        ProfScope prof("pq_adc", st);
        kern<<<grid, ADC_THREADS, smem, st>>>(p);
        VDB_LAUNCHED();
    };
    if (pq->metric == VDB_COSINE) go(pq_adc_global_kernel<VDB_COSINE, MODE>);
    else go(pq_adc_global_kernel<VDB_L2SQR, MODE>);
}

static bool adc_global_supported(const vdb_pq* pq, uint32_t K) {
    const size_t smem = (size_t)pq->m * 16 * 16 + (pq->metric == VDB_COSINE ? (size_t)pq->m * 16 * 4 : 0);
    return pq->n_bits == 4 && pq->d_sample_t && pq->n >= 65536 && K >= 1 && K <= 4096 && smem <= ADC_SMEM_MAX;
}

// top-K (adc, id) keys per query through the global-threshold scan; [nq][K]
struct DecCtx {   // query context of the decoded contraction (pq_dec.cu), released on every exit
    void* p = nullptr;
    ~DecCtx() {
        if (p) pq_dec_end(p);
    }
};

static void adc_topk_global(const vdb_pq* pq, const void* d_queries, const float* d_lut, const float* d_qcache, uint32_t nq,
                            uint32_t K, uint32_t id_base, uint64_t* d_keys, cudaStream_t st) {
    const uint32_t tab = pq->m * 16;
    const uint64_t ns = pq->sample_n;
    const uint32_t j0 = tensor_j0(K, ns, pq->n, 1e-5);
    const uint32_t cap = next_pow2((uint32_t)std::min<uint64_t>(pq->n, std::max<uint64_t>(4ull * j0 * (pq->n / ns), 4096)));
    DevBuf sall((size_t)nq * ns * 4, st), skeys, jkeys, tau((size_t)nq * 4, st),
        cnt((size_t)nq * 4, st), cand((size_t)nq * cap * 8, st), redo((size_t)nq * 4, st), nredo(4, st);
    VDB_CUDA(cudaMemsetAsync(cnt.p, 0, (size_t)nq * 4, st));
    VDB_CUDA(cudaMemsetAsync(cand.p, 0xff, (size_t)nq * cap * 8, st));
    VDB_CUDA(cudaMemsetAsync(nredo.p, 0, 4, st));
    // 1. thresholds from the sample
    const uint32_t gq = (uint32_t)adc_gq();
    const bool tensor = pq_tensor_supported(pq, nq);
    DevBuf lut16;
    DecCtx dec;   // sub-vectors of 4 dimensions: contraction over rows decoded on the fly (4x fewer MMAs than the one-hot form)
    if (tensor && d_queries && pq_dec_supported(pq, nq)) dec.p = pq_dec_begin(pq, d_queries, nq, st);
    if (dec.p) {
        pq_dec_sample(pq, dec.p, nq, sall.as<float>(), st);
    } else if (tensor) {
        pq_tensor_lut(pq, d_lut, nq, lut16, st);
        pq_tensor_sample(pq, lut16, nq, sall.as<float>(), st);
    } else
    for (uint32_t q0 = 0; q0 < nq; q0 += gq) {
        AdcGlobalParams p{};
        p.lut = d_lut + (size_t)q0 * tab;
        p.qcache = d_qcache + q0;
        p.nq_valid = std::min<uint32_t>(gq, nq - q0);
        p.all_out = sall.as<float>() + (size_t)q0 * ns;
        launch_adc_global<0>(pq, p, pq->d_sample_t, ns, st);
    }
    static const bool old_select = getenv("VDB_PQ_SELECT_OLD") && atoi(getenv("VDB_PQ_SELECT_OLD"));
    if (!old_select && j0 <= ns) {
        select_jth_kernel<<<nq, 256, 0, st>>>(sall.as<float>(), (uint32_t)ns, j0, tau.as<float>());
        VDB_LAUNCHED();
    } else {
        skeys = DevBuf((size_t)nq * ns * 8, st);
        jkeys = DevBuf((size_t)nq * j0 * 8, st);
        floats_to_keys_kernel<<<(uint32_t)std::min<uint64_t>(ceil_div<uint64_t>((uint64_t)nq * ns, 256), 8192), 256, 0, st>>>(
            sall.as<float>(), (uint64_t)nq * ns, ns, skeys.as<uint64_t>());
        VDB_LAUNCHED();
        launch_merge_keys(skeys.as<uint64_t>(), 1, nq, (uint32_t)ns, false, j0, jkeys.as<uint64_t>(), nullptr, nullptr, nullptr, st);
        tau_from_jkeys_kernel<<<ceil_div(nq, 256u), 256, 0, st>>>(jkeys.as<uint64_t>(), nq, j0, tau.as<float>());
        VDB_LAUNCHED();
    }
    // 2. filter scan over the shard (batches: bf16 one-hot contraction on the tensor cores + exact re-evaluation)
    if (dec.p)
        pq_dec_filter(pq, dec.p, d_lut, nq, tau.as<float>(), id_base, cnt.as<uint32_t>(), cand.as<uint64_t>(), cap, st);
    else if (tensor)
        pq_tensor_filter(pq, lut16, d_lut, nq, tau.as<float>(), id_base, cnt.as<uint32_t>(), cand.as<uint64_t>(), cap, st);
    else
    for (uint32_t q0 = 0; q0 < nq; q0 += gq) {
        AdcGlobalParams p{};
        p.lut = d_lut + (size_t)q0 * tab;
        p.qcache = d_qcache + q0;
        p.nq_valid = std::min<uint32_t>(gq, nq - q0);
        p.id_base = id_base;
        p.tau = tau.as<float>() + q0;
        p.cnt = cnt.as<uint32_t>() + q0;
        p.cand = cand.as<uint64_t>() + (size_t)q0 * cap;
        p.cap = cap;
        launch_adc_global<1>(pq, p, pq->d_codes_t, pq->n, st);
    }
    // 3. exact top-K by (adc, id) from the short lists
    launch_merge_keys(cand.as<uint64_t>(), 1, nq, cap, false, K, d_keys, nullptr, nullptr, nullptr, st);
    // 4. queries whose list is too short or overflowed: per-CTA top-k kernel
    const uint32_t need = (uint32_t)std::min<uint64_t>(K, pq->n);
    adc_check_kernel<<<ceil_div(nq, 256u), 256, 0, st>>>(cnt.as<uint32_t>(), nq, need, cap, redo.as<uint32_t>(),
                                                         nredo.as<uint32_t>());
    VDB_LAUNCHED();
    uint32_t h_redo = 0;
    VDB_CUDA(cudaMemcpyAsync(&h_redo, nredo.p, 4, cudaMemcpyDeviceToHost, st));
    VDB_CUDA(cudaStreamSynchronize(st));
    if (h_redo) {
        DevBuf rlut((size_t)h_redo * tab * 4, st), rqc((size_t)h_redo * 4, st), rkeys((size_t)h_redo * K * 8, st);
        gather_f32_rows_kernel<<<h_redo, 256, 0, st>>>(d_lut, tab, redo.as<uint32_t>(), h_redo, rlut.as<float>());
        VDB_LAUNCHED();
        gather_f32_rows_kernel<<<h_redo, 32, 0, st>>>(d_qcache, 1, redo.as<uint32_t>(), h_redo, rqc.as<float>());
        VDB_LAUNCHED();
        adc_scan(pq, rlut.as<float>(), rqc.as<float>(), h_redo, K, id_base, rkeys.as<uint64_t>(), nullptr, st);
        scatter_u64_rows_kernel<<<h_redo, 256, 0, st>>>(rkeys.as<uint64_t>(), K, redo.as<uint32_t>(), h_redo, d_keys);
        VDB_LAUNCHED();
    }
}

// top-K ADC keys: global-threshold scan for batches on large shards, per-CTA top-k otherwise
static void adc_topk(const vdb_pq* pq, const void* d_queries, const float* d_lut, const float* d_qcache, uint32_t nq, uint32_t K,
                     uint32_t id_base, uint64_t* d_keys, cudaStream_t st) {
    static const int force_old = getenv("VDB_ADC_OLD") ? atoi(getenv("VDB_ADC_OLD")) : 0;
    if (!force_old && nq >= 4 && adc_global_supported(pq, K)) {
        // chunks of 8192 queries bound the sample-score and candidate scratch (~1 GB + 8192 * cap * 12 B per chunk)
        const uint32_t tab = pq->m * pq->kc;
        for (uint32_t q0 = 0; q0 < nq; q0 += 8192) {
            const uint32_t cn = std::min(8192u, nq - q0);
            const void* dq = d_queries ? (const uint8_t*)d_queries + (size_t)q0 * pq->dim * (pq->dtype == VDB_F32 ? 4 : 1) : nullptr;
            adc_topk_global(pq, dq, d_lut + (size_t)q0 * tab, d_qcache + q0, cn, K, id_base, d_keys + (size_t)q0 * K, st);
        }
    } else {
        adc_scan(pq, d_lut, d_qcache, nq, K, id_base, d_keys, nullptr, st);
    }
}

// stratified random sample of the code rows, in the scan's transposed layout
__global__ void pq_sample_codes_kernel(const uint8_t* __restrict__ codes, uint64_t n, uint32_t enc, uint32_t ns,
                                       uint8_t* __restrict__ out) {
    const uint32_t i = blockIdx.x;
    if (i >= ns) return;
    const uint64_t lo = (uint64_t)i * n / ns, hi = (uint64_t)(i + 1) * n / ns;
    uint64_t h = (i + 0x9E3779B97F4A7C15ull) * 0xBF58476D1CE4E5B9ull;
    h ^= h >> 31;
    h *= 0x94D049BB133111EBull;
    h ^= h >> 29;
    const uint64_t row = lo + h % (hi > lo ? hi - lo : 1);
    for (uint32_t e = threadIdx.x; e < enc; e += blockDim.x) out[(size_t)i * enc + e] = codes[row * enc + e];
}

// ---- table construction -------------------------------------------------------------------------------
static std::atomic<uint64_t> g_pq_serial{0};

vdb_pq* pq_create(const vdb_dataset* ds, const void* h_codebooks, uint32_t m, uint32_t n_bits,
                  const uint8_t* h_codes_in, uint8_t* h_codes_out) {
    VDB_REQUIRE(n_bits == 4 || n_bits == 8, "n_bits must be 4 or 8 in PQTable.");
    VDB_REQUIRE(h_codebooks, "codebooks is NULL");
    auto pq = new vdb_pq();
    cudaStream_t st = nullptr;
    try {
        pq->device = ds->device;
        pq->serial = ++g_pq_serial;
        pq->dim = ds->dim;
        pq->m = m;
        pq->n_bits = n_bits;
        pq->kc = 1u << n_bits;
        pq->enc = n_bits == 4 ? (m + 1) / 2 : m;
        pq->dtype = ds->dtype;
        pq->metric = ds->metric;
        pq->n = ds->n;
        pq->words = ceil_div(pq->enc, 4u);
        pq_groups_host(ds->dim, m, pq->g_lo, pq->g_len);
        VDB_REQUIRE(pq->g_lo.size() == m, "pq_groups produced %zu groups for m=%u", pq->g_lo.size(), m);
        std::vector<uint32_t> groups(3 * m);
        uint32_t off = 0;
        for (uint32_t g = 0; g < m; ++g) {
            pq->g_off.push_back(off);
            groups[3 * g] = pq->g_lo[g];
            groups[3 * g + 1] = pq->g_len[g];
            groups[3 * g + 2] = off;
            off += pq->kc * pq->g_len[g];
            pq->max_len = std::max(pq->max_len, pq->g_len[g]);
        }
        const size_t es = ds->elem_size();
        VDB_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
        VDB_CUDA(cudaMalloc(&pq->d_codebooks, (size_t)off * es));
        VDB_CUDA(cudaMalloc(&pq->d_groups, groups.size() * 4));
        VDB_CUDA(cudaMalloc(&pq->d_dist_cache, (size_t)m * pq->kc * 4));
        VDB_CUDA(cudaMalloc(&pq->d_cb_norm, (size_t)m * pq->kc * 4));
        VDB_CUDA(cudaMalloc(&pq->d_codes, std::max<size_t>(1, pq->n * pq->enc)));
        VDB_CUDA(cudaMalloc(&pq->d_codes_t, std::max<size_t>(1, ceil_div<uint64_t>(pq->n, 32) * pq->words * 32 * 4)));
        VDB_CUDA(cudaMemcpyAsync(pq->d_codebooks, h_codebooks, (size_t)off * es, cudaMemcpyHostToDevice, st));
        VDB_CUDA(cudaMemcpyAsync(pq->d_groups, groups.data(), groups.size() * 4, cudaMemcpyHostToDevice, st));
        const uint32_t tab = m * pq->kc;
        if (ds->dtype == VDB_F32)
            pq_centroid_norms_kernel<float><<<ceil_div(tab, 256u), 256, 0, st>>>(
                (const float*)pq->d_codebooks, pq->d_groups, m, pq->kc, pq->metric, pq->d_dist_cache, pq->d_cb_norm);
        else
            pq_centroid_norms_kernel<uint8_t><<<ceil_div(tab, 256u), 256, 0, st>>>(
                (const uint8_t*)pq->d_codebooks, pq->d_groups, m, pq->kc, pq->metric, pq->d_dist_cache, pq->d_cb_norm);
        VDB_LAUNCHED();
        if (pq->n) {
            if (h_codes_in) {
                VDB_CUDA(cudaMemcpyAsync(pq->d_codes, h_codes_in, pq->n * pq->enc, cudaMemcpyHostToDevice, st));
            } else {
                const uint64_t total = pq->n * pq->enc;
                const uint32_t grid = (uint32_t)std::min<uint64_t>(ceil_div<uint64_t>(total, 256), (uint64_t)sm_count() * 32);
                ProfScope prof("pq_encode", st);
                static const int enc_old = getenv("VDB_PQ_ENCODE_OLD") ? atoi(getenv("VDB_PQ_ENCODE_OLD")) : 0;
                const size_t smem4 = encode4_smem(m, pq->max_len, ds->dim);
                const bool fast = !enc_old && n_bits == 4 && pq->max_len <= (uint32_t)ENC_MAXL && smem4 <= 200 * 1024 && ds->dim < 65536;
                auto go4 = [&](auto kern, auto* tag) {
                    using T = std::remove_pointer_t<decltype(tag)>;
                    if (smem4 > 48 * 1024) VDB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem4));
                    const uint32_t per_sm = (uint32_t)std::max<size_t>(1, std::min<size_t>(4, (220 * 1024) / smem4));
                    const uint32_t g4 = (uint32_t)std::min<uint64_t>(ceil_div<uint64_t>(pq->n, ENC_ROWS), (uint64_t)sm_count() * per_sm);
                    kern<<<g4, 256, smem4, st>>>((const T*)ds->d_rows, ds->n, (uint64_t)ds->pitch, ds->dim, (const T*)pq->d_codebooks,
                                                 pq->d_groups, pq->d_cb_norm, m, pq->enc, pq->max_len, pq->d_codes);
                };
                if (fast) {
                    if (ds->dtype == VDB_F32) {
                        if (pq->metric == VDB_L2SQR) go4(pq_encode4_kernel<float, VDB_L2SQR>, (float*)nullptr);
                        else go4(pq_encode4_kernel<float, VDB_COSINE>, (float*)nullptr);
                    } else {
                        if (pq->metric == VDB_L2SQR) go4(pq_encode4_kernel<uint8_t, VDB_L2SQR>, (uint8_t*)nullptr);
                        else go4(pq_encode4_kernel<uint8_t, VDB_COSINE>, (uint8_t*)nullptr);
                    }
                    VDB_LAUNCHED();
                }
                auto go = [&](auto kern, auto* tag) {
                    if (fast) return;
                    using T = std::remove_pointer_t<decltype(tag)>;
                    kern<<<grid, 256, 0, st>>>((const T*)ds->d_rows, ds->n, (uint64_t)ds->pitch, (const T*)pq->d_codebooks,
                                               pq->d_groups, pq->d_cb_norm, m, n_bits, pq->kc, pq->enc, pq->d_codes);
                };
                if (ds->dtype == VDB_F32) {
                    if (pq->metric == VDB_L2SQR) go(pq_encode_kernel<float, VDB_L2SQR>, (float*)nullptr);
                    else go(pq_encode_kernel<float, VDB_COSINE>, (float*)nullptr);
                } else {
                    if (pq->metric == VDB_L2SQR) go(pq_encode_kernel<uint8_t, VDB_L2SQR>, (uint8_t*)nullptr);
                    else go(pq_encode_kernel<uint8_t, VDB_COSINE>, (uint8_t*)nullptr);
                }
                if (!fast) VDB_LAUNCHED();
            }
            const uint64_t tt = ceil_div<uint64_t>(pq->n, 32) * pq->words * 32;
            pq_transpose_kernel<<<(uint32_t)std::min<uint64_t>(ceil_div<uint64_t>(tt, 256), 1u << 20), 256, 0, st>>>(
                pq->d_codes, pq->n, pq->enc, pq->words, pq->d_codes_t);
            VDB_LAUNCHED();
            if (pq->n >= 65536) {
                pq->sample_n = (uint32_t)std::min<uint64_t>(std::min<uint64_t>(32768, pq->n / 2), std::max<uint64_t>(2048, pq->n / 30));
                VDB_CUDA(cudaMalloc(&pq->d_sample, round_up((size_t)pq->sample_n * pq->enc, (size_t)16)));
                pq_sample_codes_kernel<<<pq->sample_n, 128, 0, st>>>(pq->d_codes, pq->n, pq->enc, pq->sample_n, pq->d_sample);
                VDB_LAUNCHED();
                const uint64_t ts = ceil_div<uint64_t>(pq->sample_n, 32) * pq->words * 32;
                VDB_CUDA(cudaMalloc(&pq->d_sample_t, ts * 4));
                pq_transpose_kernel<<<(uint32_t)std::min<uint64_t>(ceil_div<uint64_t>(ts, 256), 1u << 20), 256, 0, st>>>(
                    pq->d_sample, pq->sample_n, pq->enc, pq->words, pq->d_sample_t);
                VDB_LAUNCHED();
                VDB_CUDA(cudaStreamSynchronize(st));
            }
            if (h_codes_out)
                VDB_CUDA(cudaMemcpyAsync(h_codes_out, pq->d_codes, pq->n * pq->enc, cudaMemcpyDeviceToHost, st));
        }
        VDB_CUDA(cudaStreamSynchronize(st));
        cudaStreamDestroy(st);
    } catch (...) {
        if (st) cudaStreamDestroy(st);
        pq_destroy(pq);
        throw;
    }
    return pq;
}

void pq_destroy(vdb_pq* pq) {
    if (!pq) return;
    cudaFree(pq->d_codebooks);
    cudaFree(pq->d_groups);
    cudaFree(pq->d_dist_cache);
    cudaFree(pq->d_cb_norm);
    cudaFree(pq->d_codes);
    cudaFree(pq->d_codes_t);
    cudaFree(pq->d_sample_t);
    cudaFree(pq->d_sample);
    pq_dec_destroy(pq);
    delete pq;
}

void pq_lut(const vdb_pq* pq, const void* d_queries, uint32_t nq, float* d_lut, float* d_qcache, cudaStream_t st) {
    if (nq == 0) return;
    const uint64_t total = (uint64_t)nq * pq->m * pq->kc;
    const uint32_t grid = (uint32_t)ceil_div<uint64_t>(std::max<uint64_t>(total, nq), 256);
    ProfScope prof("pq_lut", st);
    if (pq->dtype == VDB_F32)
        pq_lut_kernel<float><<<grid, 256, 0, st>>>((const float*)d_queries, nq, pq->dim, (const float*)pq->d_codebooks,
                                                  pq->d_groups, pq->m, pq->kc, pq->metric, d_lut, d_qcache);
    else
        pq_lut_kernel<uint8_t><<<grid, 256, 0, st>>>((const uint8_t*)d_queries, nq, pq->dim,
                                                    (const uint8_t*)pq->d_codebooks, pq->d_groups, pq->m, pq->kc,
                                                    pq->metric, d_lut, d_qcache);
    VDB_LAUNCHED();
}

void pq_adc_all(const vdb_pq* pq, const float* d_lut, const float* d_qcache, uint32_t nq, float* d_out,
                cudaStream_t st) {
    adc_scan(pq, d_lut, d_qcache, nq, 0, 0, nullptr, d_out, st);
}

// keys -> (query index, local row, valid) for the rerank
__global__ void keys_to_pairs_kernel(const uint64_t* __restrict__ keys, uint64_t count, uint32_t per_q, uint32_t id_base,
                                     uint64_t n, uint32_t* __restrict__ qidx, uint32_t* __restrict__ rid,
                                     uint8_t* __restrict__ valid) {
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < count; j += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t k = keys[j];
        // candidates owned by another row shard (ids outside [id_base, id_base + n)) are skipped here
        const bool ok = k != KEY_NONE && key_id(k) >= id_base && (uint64_t)(key_id(k) - id_base) < n;
        qidx[j] = (uint32_t)(j / per_q);
        rid[j] = ok ? key_id(k) - id_base : 0u;
        valid[j] = ok;
    }
}
__global__ void rekey_kernel(const float* __restrict__ dist, const uint32_t* __restrict__ ids, uint32_t id_base,
                             const uint8_t* __restrict__ valid, uint64_t count, uint64_t* __restrict__ keys) {
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < count; j += (uint64_t)gridDim.x * blockDim.x)
        keys[j] = (!valid || valid[j]) ? make_key(dist[j], ids[j] + id_base) : KEY_NONE;
}
void rekey(const float* d_dist, const uint32_t* d_ids, const uint8_t* d_valid, uint64_t count, uint64_t* d_keys,
           cudaStream_t st) {
    if (count == 0) return;
    rekey_kernel<<<(uint32_t)std::min<uint64_t>(ceil_div<uint64_t>(count, 256), 4096), 256, 0, st>>>(d_dist, d_ids, 0,
                                                                                                  d_valid, count, d_keys);
    VDB_LAUNCHED();
}

void rekey_based(const float* d_dist, const uint32_t* d_ids, uint32_t id_base, const uint8_t* d_valid, uint64_t count,
                 uint64_t* d_keys, cudaStream_t st) {
    if (count == 0) return;
    rekey_kernel<<<(uint32_t)std::min<uint64_t>(ceil_div<uint64_t>(count, 256), 8192), 256, 0, st>>>(
        d_dist, d_ids, id_base, d_valid, count, d_keys);
    VDB_LAUNCHED();
}

// exact rerank of [nq][kk] candidate keys -> [nq][k] keys ordered by (exact distance, id)
void rerank_keys(const vdb_dataset* ds, const void* d_queries, uint32_t nq, const uint64_t* d_cand, uint32_t kk,
                 uint32_t k, uint64_t* d_keys, cudaStream_t st) {
    const uint64_t count = (uint64_t)nq * kk;
    if (count == 0 || k == 0) return;
    DevBuf qidx(count * 4, st), rid(count * 4, st), valid(count, st), dist(count * 4, st), keys2(count * 8, st);
    const uint32_t grid = (uint32_t)std::min<uint64_t>(ceil_div<uint64_t>(count, 256), 4096);
    keys_to_pairs_kernel<<<grid, 256, 0, st>>>(d_cand, count, kk, (uint32_t)ds->id_base, ds->n, qidx.as<uint32_t>(),
                                               rid.as<uint32_t>(), valid.as<uint8_t>());
    VDB_LAUNCHED();
    exact_pair_distances(ds, d_queries, qidx.as<uint32_t>(), rid.as<uint32_t>(), count, dist.as<float>(), st);
    rekey_kernel<<<grid, 256, 0, st>>>(dist.as<float>(), rid.as<uint32_t>(), (uint32_t)ds->id_base,
                                       valid.as<uint8_t>(), count, keys2.as<uint64_t>());
    VDB_LAUNCHED();
    launch_merge_keys(keys2.as<uint64_t>(), 1, nq, kk, false, k, d_keys, nullptr, nullptr, nullptr, st);
}

// this shard's max(ef,k) best codes per query by (ADC distance, global id): [nq][kk]
void pq_adc_keys(const vdb_dataset* ds, const vdb_pq* pq, const void* d_queries, uint32_t nq, uint32_t kk, uint64_t* d_keys,
                 cudaStream_t st) {
    VDB_REQUIRE(ds->metric == pq->metric, "Distance algorithm mismatch.");
    VDB_REQUIRE(ds->n == pq->n && ds->dim == pq->dim && ds->dtype == pq->dtype,
                "PQ table was built for a different vector set (it must be rebuilt after add/delete)");
    if (nq == 0 || kk == 0) return;
    const uint32_t tab = pq->m * pq->kc;
    DevBuf lut((size_t)nq * tab * 4, st), qcache((size_t)nq * 4, st);
    pq_lut(pq, d_queries, nq, lut.as<float>(), qcache.as<float>(), st);
    adc_topk(pq, d_queries, lut.as<float>(), qcache.as<float>(), nq, kk, (uint32_t)ds->id_base, d_keys, st);
}

void pq_knn_keys(const vdb_dataset* ds, const vdb_pq* pq, const void* d_queries, uint32_t nq, uint32_t k,
                 uint32_t ef, uint64_t* d_keys, cudaStream_t st) {
    VDB_REQUIRE(ds->metric == pq->metric, "Distance algorithm mismatch.");
    VDB_REQUIRE(ds->n == pq->n && ds->dim == pq->dim && ds->dtype == pq->dtype,
                "PQ table was built for a different vector set (it must be rebuilt after add/delete)");
    if (nq == 0 || k == 0) return;
    const uint32_t kk = std::max(ef, k);
    const uint32_t tab = pq->m * pq->kc;
    DevBuf lut((size_t)nq * tab * 4, st), qcache((size_t)nq * 4, st), cand((size_t)nq * kk * 8, st);
    pq_lut(pq, d_queries, nq, lut.as<float>(), qcache.as<float>(), st);
    adc_topk(pq, d_queries, lut.as<float>(), qcache.as<float>(), nq, kk, (uint32_t)ds->id_base, cand.as<uint64_t>(), st);
    rerank_keys(ds, d_queries, nq, cand.as<uint64_t>(), kk, k, d_keys, st);
}

}  // namespace vdb
