// ivf.cu — K9: IVF list construction and probe scan.
//
// Replaces (reference paths):
//   IVFIndex::from_vec_set (assignment + lists)   src/index_algorithm/ivf_index.rs:88-106
//   KMeans::find_n_nearest                        src/distance/k_means.rs:174-191
//   IVFIndex::knn_with_ef                         src/index_algorithm/ivf_index.rs:143-154
//
// Assignment and probe selection use the exact sequential arithmetic of kmeans.cu (bit-exact lists and
// probe order). The list scan gathers whole rows by id (a 960-d f32 row is 30 full 128-byte lines, so a
// gather at row granularity wastes no HBM traffic), one CTA per (query, slice of its visit sequence), warps
// stream 8 rows at a time, partial top-k lists are merged per query. Ties at the k-th distance are resolved
// by (distance, id) instead of the reference's visit order (documented in DESIGN.md; within the parity rule).
#include <algorithm>
#include <cstdlib>
#include <vector>

#include "index.cuh"
#include "scanmath.cuh"
#include "topk.cuh"

namespace vdb {

constexpr int IVF_THREADS = 256;
constexpr int IVF_WARPS = IVF_THREADS / 32;
constexpr int IVF_R = 8;

struct IvfScanParams {
    const uint8_t* rows;
    uint64_t pitch_bytes;
    uint32_t nvec, nit;
    const float* q;          // query tiles [nq][qstride]
    uint32_t qstride;
    const float* qcache;     // [nq]
    const uint64_t* probes;  // [nq][nprobe] keys (distance, list id), KEY_NONE padded
    uint32_t nprobe;
    const uint64_t* offsets; // [nlist+1]
    const uint32_t* members;
    uint32_t splits;         // CTAs per query
    uint32_t K, P, limit;
    uint32_t id_base;
    uint64_t* partial;       // [nq][splits][K]
};

template <int METRIC, int PL>
__global__ void __launch_bounds__(IVF_THREADS) ivf_scan_kernel(const IvfScanParams p) {
    extern __shared__ __align__(16) uint8_t smem[];
    constexpr int R = IVF_R;
    const uint32_t q = blockIdx.x / p.splits, split = blockIdx.x % p.splits;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t qs4 = p.qstride >> 2;
    float4* qs = reinterpret_cast<float4*>(smem);
    const ulonglong2* qs2 = reinterpret_cast<const ulonglong2*>(smem);
    uint64_t* tk = reinterpret_cast<uint64_t*>(smem + (size_t)p.qstride * 4);
    TopkSmem topk{tk, reinterpret_cast<uint32_t*>(tk + p.P), p.K, p.P, 1, p.limit};
    uint32_t* pre = reinterpret_cast<uint32_t*>(tk + p.P) + 4;  // [nprobe+1] prefix of probed list lengths
    uint64_t* lbase = reinterpret_cast<uint64_t*>(pre + round_up(p.nprobe + 1, 2u));  // [nprobe] list starts

    for (uint32_t i = threadIdx.x; i < qs4; i += blockDim.x)
        qs[i] = reinterpret_cast<const float4*>(p.q + (size_t)q * p.qstride)[i];
    if (threadIdx.x == 0) {
        uint32_t s = 0;
        for (uint32_t j = 0; j < p.nprobe; ++j) {
            const uint64_t pk = p.probes[(size_t)q * p.nprobe + j];
            pre[j] = s;
            if (pk != KEY_NONE) {
                const uint32_t c = key_id(pk);
                lbase[j] = p.offsets[c];
                s += (uint32_t)(p.offsets[c + 1] - p.offsets[c]);
            } else {
                lbase[j] = 0;
            }
        }
        pre[p.nprobe] = s;
    }
    topk.init();
    const uint32_t total = pre[p.nprobe];
    const float qn = METRIC == VDB_COSINE ? p.qcache[q] : 0.f;
    // this CTA's slice of the visit sequence, in groups of R positions
    const uint32_t groups = ceil_div<uint32_t>(total, R);
    const uint32_t gper = ceil_div<uint32_t>(groups, p.splits);
    const uint32_t g_lo = split * gper, g_hi = min(groups, g_lo + gper);
    const uint32_t steps = ceil_div<uint32_t>(g_hi > g_lo ? g_hi - g_lo : 0, IVF_WARPS);

    for (uint32_t s = 0; s < steps; ++s) {
        const uint32_t g = g_lo + s * IVF_WARPS + warp;
        const bool active = g < g_hi;
        uint32_t rid[R];
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const uint32_t pos = g * R + r;
            uint32_t id = 0xffffffffu;
            if (active && pos < total) {
                uint32_t j = 0;
                while (pre[j + 1] <= pos) ++j;  // nprobe is small
                id = p.members[lbase[j] + (pos - pre[j])];
            }
            rid[r] = id;
        }
        // f32 rows: (even, odd) chains of scanmath.cuh; u8 rows: exact integer sums - the streaming scan's distance bits
        constexpr bool U8 = PL == 4;
        f32x2 acc2[R], xx2[R];
        uint32_t acci[R], xxi[R];
#pragma unroll
        for (int r = 0; r < R; ++r) acc2[r] = 0ull, xx2[r] = 0ull, acci[r] = 0u, xxi[r] = 0u;
        if (active) {
            for (uint32_t it = 0; it < p.nit; ++it) {
                const uint32_t c = it * 32 + lane;
                uint4 v[R];
#pragma unroll
                for (int r = 0; r < R; ++r)
                    v[r] = (c < p.nvec && rid[r] != 0xffffffffu)
                               ? ldg_stream_u4(p.rows + (uint64_t)rid[r] * p.pitch_bytes + (size_t)c * 16)
                               : make_uint4(0u, 0u, 0u, 0u);
                if constexpr (U8) {
                    const uint4 qb = reinterpret_cast<const uint4*>(qs2)[c];
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        acci[r] = u8x16_acc<METRIC == VDB_L2SQR>(acci[r], v[r], qb);
                        if (METRIC == VDB_COSINE) xxi[r] = u8x16_acc<false>(xxi[r], v[r], v[r]);
                    }
                } else {
                    const ulonglong2 qv = qs2[c];
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        f32x2 x01, x23;
                        row_pairs(v[r], x01, x23);
                        acc2[r] = chunk_acc<METRIC == VDB_L2SQR>(acc2[r], x01, x23, qv.x, qv.y);
                        if (METRIC == VDB_COSINE) xx2[r] = chunk_acc<false>(xx2[r], x01, x23, x01, x23);
                    }
                }
            }
        }
        float tot, xs = 0.f;
        if constexpr (U8) {
            tot = (float)warp_reduce_scatter<R>(acci, lane);  // lane L holds row L >> 2
            if (METRIC == VDB_COSINE) xs = (float)warp_reduce_scatter<R>(xxi, lane);
        } else {
            float acc[R], xx[R];
#pragma unroll
            for (int r = 0; r < R; ++r) acc[r] = sum2(acc2[r]), xx[r] = sum2(xx2[r]);
            tot = warp_reduce_scatter<R>(acc, lane);  // lane L holds row L >> 2
            if (METRIC == VDB_COSINE) xs = warp_reduce_scatter<R>(xx, lane);
        }
        if (METRIC == VDB_COSINE) tot = 1.0f - tot / fmaxf(sqrtf(xs) * qn, 1e-10f);
        const int my_r = lane >> 2;
        uint32_t my_id = 0xffffffffu;
#pragma unroll
        for (int r = 0; r < R; ++r)
            if (r == my_r) my_id = rid[r];
        bool want = false;
        if ((lane & 3) == 0 && my_id != 0xffffffffu) {
            const uint64_t key = make_key(tot, p.id_base + my_id);
            if (key < topk.tau(0)) want = topk.push(0, key);
        }
        topk.maybe_flush(want);
    }
    topk.final_flush();
    for (uint32_t j = threadIdx.x; j < p.K; j += blockDim.x)
        p.partial[((size_t)q * p.splits + split) * p.K + j] = topk.seg(0)[j];
}

// ---- list-major batched scan -----------------------------------------------------------------------------------
// For a batch of queries the same list is probed by many queries. Work items are (list, group of <= LQ queries probing
// it, row range): the item's rows are streamed ONCE for all its queries (the K1 inner loop with gathered row ids), so
// the HBM traffic drops from sum_q(rows visited by q) to sum_lists(ceil(Q_list / 8) * list rows). Every item writes a
// k-best list per query slot; a per-query index of those partial lists drives the final merge.
constexpr int LR = 4;   // rows per warp step (an item holds up to LQ queries, index.cuh)

struct IvfListParams {
    const uint8_t* rows;
    uint64_t pitch_bytes;
    uint32_t nvec, nit;
    const float* q;          // query tiles [nq][qstride]
    uint32_t qstride;
    const float* qcache;
    const IvfItem* items;
    const uint32_t* members;
    uint32_t K, P, limit, sync_every;
    uint32_t id_base;
    uint64_t* partial;       // [nitems][LQ][K]
};

template <int METRIC, int PL>
__global__ void __launch_bounds__(IVF_THREADS, 2) ivf_list_scan_kernel(const IvfListParams p) {
    extern __shared__ __align__(16) uint8_t smem[];
    constexpr int NQ = LQ, R = LR, V = NQ * R;
    constexpr int SH = 5 - Log2<V>::value, SHR = 5 - Log2<R>::value;
    const IvfItem item = p.items[blockIdx.x];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t qs4 = p.qstride >> 2;
    float4* qs = reinterpret_cast<float4*>(smem);
    const ulonglong2* qs2 = reinterpret_cast<const ulonglong2*>(smem);
    uint64_t* tk = reinterpret_cast<uint64_t*>(smem + (size_t)NQ * p.qstride * 4);
    TopkSmem topk{tk, reinterpret_cast<uint32_t*>(tk + (size_t)NQ * p.P), p.K, p.P, NQ, p.limit};
    for (uint32_t i = threadIdx.x; i < NQ * qs4; i += blockDim.x) {
        const uint32_t qi = i / qs4, e = i - qi * qs4;
        qs[i] = qi < item.nq_valid ? reinterpret_cast<const float4*>(p.q + (size_t)item.qid[qi] * p.qstride)[e]
                                   : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    topk.init();
    const int pidx = lane >> SH;
    const int my_r = pidx / NQ, my_q = pidx % NQ;
    const bool emitter = (lane & ((1 << SH) - 1)) == 0 && my_q < (int)item.nq_valid;
    float qn = 0.f;
    if (METRIC == VDB_COSINE && my_q < (int)item.nq_valid) qn = p.qcache[item.qid[my_q]];
    const uint32_t groups = ceil_div<uint32_t>(item.nrows, R);
    const uint32_t iters = ceil_div<uint32_t>(groups, IVF_WARPS);
    const uint32_t* mem = p.members + item.row_begin;

    bool want = false;
    for (uint32_t gi = 0; gi < iters; ++gi) {
        const uint32_t g = gi * IVF_WARPS + warp;
        uint32_t rid[R];
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const uint32_t pos = g * R + r;
            rid[r] = pos < item.nrows ? mem[pos] : 0xffffffffu;
        }
        constexpr bool U8 = PL == 4;   // u8 rows: exact integer sums (scanmath.cuh)
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
        if (g < groups) {
            uint4 nxt[R], cur[R];
            auto load = [&](uint32_t it) {
                const uint32_t c = it * 32 + lane;
#pragma unroll
                for (int r = 0; r < R; ++r)
                    nxt[r] = (c < p.nvec && rid[r] != 0xffffffffu)
                                 ? ldg_stream_u4(p.rows + (uint64_t)rid[r] * p.pitch_bytes + (size_t)c * 16)
                                 : make_uint4(0u, 0u, 0u, 0u);
            };
            load(0);
            for (uint32_t it = 0; it < p.nit; ++it) {
#pragma unroll
                for (int r = 0; r < R; ++r) cur[r] = nxt[r];
                if (it + 1 < p.nit) load(it + 1);
                const uint32_t c = it * 32 + lane;
                if constexpr (U8) {
                    if (METRIC == VDB_COSINE) {
#pragma unroll
                        for (int r = 0; r < R; ++r) xxi[r] = u8x16_acc<false>(xxi[r], cur[r], cur[r]);
                    }
#pragma unroll
                    for (int qi = 0; qi < NQ; ++qi) {
                        const uint4 qb = reinterpret_cast<const uint4*>(qs2)[(size_t)qi * qs4 + c];
#pragma unroll
                        for (int r = 0; r < R; ++r) acci[r * NQ + qi] = u8x16_acc<METRIC == VDB_L2SQR>(acci[r * NQ + qi], cur[r], qb);
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
                        const ulonglong2 qv = qs2[(size_t)qi * qs4 + c];
#pragma unroll
                        for (int r = 0; r < R; ++r)
                            acc2[r * NQ + qi] = chunk_acc<METRIC == VDB_L2SQR>(acc2[r * NQ + qi], x01[r], x23[r], qv.x, qv.y);
                    }
                }
            }
        }
        float tot, xr = 0.f;
        if constexpr (U8) {
            tot = (float)warp_reduce_scatter<V>(acci, lane);
            if (METRIC == VDB_COSINE) {
                const uint32_t xs = warp_reduce_scatter<R>(xxi, lane);
                xr = (float)__shfl_sync(0xffffffffu, xs, my_r << SHR);
            }
        } else {
            float acc[V], xx[R];
#pragma unroll
            for (int i = 0; i < V; ++i) acc[i] = sum2(acc2[i]);
#pragma unroll
            for (int r = 0; r < R; ++r) xx[r] = sum2(xx2[r]);
            tot = warp_reduce_scatter<V>(acc, lane);
            if (METRIC == VDB_COSINE) {
                const float xs = warp_reduce_scatter<R>(xx, lane);
                xr = __shfl_sync(0xffffffffu, xs, my_r << SHR);
            }
        }
        if (METRIC == VDB_COSINE) tot = 1.0f - tot / fmaxf(sqrtf(xr) * qn, 1e-10f);
        uint32_t my_id = 0xffffffffu;
#pragma unroll
        for (int r = 0; r < R; ++r)
            if (r == my_r) my_id = rid[r];
        if (emitter && my_id != 0xffffffffu) {
            const uint64_t key = make_key(tot, p.id_base + my_id);
            if (key < topk.tau(my_q)) want |= topk.push(my_q, key);
        }
        if ((gi + 1) % p.sync_every == 0) {
            topk.maybe_flush(want);
            want = false;
        }
    }
    topk.final_flush();
    for (uint32_t i = threadIdx.x; i < NQ * p.K; i += blockDim.x) {
        const uint32_t qi = i / p.K, j = i - qi * p.K;
        p.partial[((size_t)blockIdx.x * NQ + qi) * p.K + j] = qi < item.nq_valid ? topk.seg(qi)[j] : KEY_NONE;
    }
}

// final merge: query q owns the partial lists plist[poff[q] .. poff[q+1]) (each K keys)
__global__ void __launch_bounds__(256) ivf_merge_kernel(const uint64_t* __restrict__ partial, const uint64_t* __restrict__ poff,
                                                        const uint32_t* __restrict__ plist, uint32_t K, uint32_t P,
                                                        uint32_t limit, uint64_t* __restrict__ out) {
    extern __shared__ __align__(16) uint8_t smem[];
    uint64_t* tk = reinterpret_cast<uint64_t*>(smem);
    TopkSmem topk{tk, reinterpret_cast<uint32_t*>(tk + P), K, P, 1, limit};
    topk.init();
    const uint32_t q = blockIdx.x;
    const uint64_t b = poff[q], e = poff[q + 1];
    const uint64_t total = (e - b) * K;
    const uint64_t rounds = (total + blockDim.x - 1) / blockDim.x;
    for (uint64_t r = 0; r < rounds; ++r) {
        const uint64_t i = r * blockDim.x + threadIdx.x;
        bool want = false;
        if (i < total) {
            const uint64_t l = i / K, j = i - l * K;
            const uint64_t key = partial[(uint64_t)plist[b + l] * K + j];
            if (key < topk.tau(0)) want = topk.push(0, key);
        }
        topk.maybe_flush(want);
    }
    topk.final_flush();
    for (uint32_t j = threadIdx.x; j < K; j += blockDim.x) out[(size_t)q * K + j] = topk.seg(0)[j];
}

// [nq][nlist] exact distances -> keys (distance, list id)
__global__ void probe_keys_kernel(const float* __restrict__ dist, uint64_t count, uint32_t nlist,
                                  uint64_t* __restrict__ keys) {
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < count; j += (uint64_t)gridDim.x * blockDim.x)
        keys[j] = make_key(dist[j], (uint32_t)(j % nlist));
}

// ---- exact query-centroid distances of a search batch (probe order = find_n_nearest, k_means.rs:174-191) -------------
// kmeans_assign_exact is laid out for n >> k (a 32-centroid chunk staged per CTA, one launch per chunk): a 1000-query
// batch paid 4 launches x 63 us for 0.4 GFLOP. Here the centroids are transposed once per index ([dim][nlist] f32, plus
// ||c|| for cosine), one warp takes (query, 32 centroids) with lane = centroid and the query row in shared memory, and
// every lane walks the same unfused sequential chain over the dimensions - the distances are bit-identical.
template <typename T>
__global__ void centroid_transpose_kernel(const T* __restrict__ cent, uint32_t nlist, uint32_t dim, float* __restrict__ centT,
                                          float* __restrict__ cnorm) {
    const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= nlist) return;
    float s = 0.f;
    for (uint32_t j = 0; j < dim; ++j) {
        const float v = (float)cent[(size_t)c * dim + j];
        centT[(size_t)j * nlist + c] = v;
        s = __fadd_rn(s, __fmul_rn(v, v));
    }
    cnorm[c] = sqrtf(s);
}
template <typename T, int METRIC>
__global__ void __launch_bounds__(256) probe_dist_kernel(const T* __restrict__ queries, uint32_t nq, uint32_t dim,
                                                         const float* __restrict__ centT, const float* __restrict__ cnorm,
                                                         uint32_t nlist, float* __restrict__ out) {
    extern __shared__ float probe_rows[];   // [8 warps][dim]
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t chunks = (nlist + 31) / 32;
    const uint64_t w = (uint64_t)blockIdx.x * 8 + warp;
    const uint32_t q = (uint32_t)(w / chunks), ch = (uint32_t)(w % chunks);
    if (q >= nq) return;
    float* x = probe_rows + (size_t)warp * dim;
    for (uint32_t e = lane; e < dim; e += 32) x[e] = (float)queries[(size_t)q * dim + e];
    __syncwarp();
    const uint32_t c = ch * 32 + lane, cc = min(c, nlist - 1);
    const float* col = centT + cc;
    float s = 0.f, svv = 0.f;
#pragma unroll 8
    for (uint32_t j = 0; j < dim; ++j) {
        const float xv = x[j], cv = col[(size_t)j * nlist];
        if (METRIC == VDB_L2SQR) {
            const float df = __fsub_rn(xv, cv);
            s = __fadd_rn(s, __fmul_rn(df, df));
        } else {
            s = __fadd_rn(s, __fmul_rn(xv, cv));
            svv = __fadd_rn(svv, __fmul_rn(xv, xv));
        }
    }
    float dist = s;
    if (METRIC == VDB_COSINE) {
        const float den = fmaxf(__fmul_rn(sqrtf(svv), cnorm[cc]), 1e-10f);
        dist = __fsub_rn(1.0f, __fdiv_rn(s, den));
    }
    if (c < nlist) out[(size_t)q * nlist + c] = dist;
}
static void probe_distances(const vdb_dataset* ds, const vdb_ivf* ivf, const void* d_queries, uint32_t nq, float* d_out,
                            cudaStream_t st) {
    const uint32_t chunks = (ivf->nlist + 31) / 32;
    const uint32_t grid = (uint32_t)ceil_div<uint64_t>((uint64_t)nq * chunks, 8);
    const size_t smem = (size_t)8 * ds->dim * 4;
    auto launch = [&](auto kern, auto* q) {
        if (smem > 48 * 1024) VDB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        ProfScope prof("kmeans_assign", st);
        kern<<<grid, 256, smem, st>>>(q, nq, ds->dim, ivf->d_centT, ivf->d_cnorm, ivf->nlist, d_out);
        VDB_LAUNCHED();
    };
    const bool l2 = ds->metric == VDB_L2SQR;
    if (ds->dtype == VDB_F32) {
        if (l2) launch(probe_dist_kernel<float, VDB_L2SQR>, (const float*)d_queries);
        else launch(probe_dist_kernel<float, VDB_COSINE>, (const float*)d_queries);
    } else {
        if (l2) launch(probe_dist_kernel<uint8_t, VDB_L2SQR>, (const uint8_t*)d_queries);
        else launch(probe_dist_kernel<uint8_t, VDB_COSINE>, (const uint8_t*)d_queries);
    }
}

vdb_ivf* ivf_create(const vdb_dataset* ds, const void* h_centroids, uint32_t nlist, uint32_t* h_assign_out) {
    VDB_REQUIRE(nlist > 0, "The number of clusters should be greater than 0.");
    VDB_REQUIRE(h_centroids, "centroids is NULL");
    auto ivf = new vdb_ivf();
    cudaStream_t st = nullptr;
    try {
        ivf->device = ds->device;
        ivf->nlist = nlist;
        ivf->dim = ds->dim;
        ivf->dtype = ds->dtype;
        ivf->metric = ds->metric;
        ivf->n = ds->n;
        const size_t cbytes = (size_t)nlist * ds->dim * ds->elem_size();
        VDB_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
        VDB_CUDA(cudaMalloc(&ivf->d_centroids, cbytes));
        VDB_CUDA(cudaMalloc(&ivf->d_offsets, (size_t)(nlist + 1) * 8));
        VDB_CUDA(cudaMalloc(&ivf->d_members, std::max<size_t>(4, ds->n * 4)));
        VDB_CUDA(cudaMemcpyAsync(ivf->d_centroids, h_centroids, cbytes, cudaMemcpyHostToDevice, st));
        VDB_CUDA(cudaMalloc(&ivf->d_centT, (size_t)nlist * ds->dim * 4));
        VDB_CUDA(cudaMalloc(&ivf->d_cnorm, (size_t)nlist * 4));
        if (ds->dtype == VDB_F32)
            centroid_transpose_kernel<float><<<ceil_div(nlist, 128u), 128, 0, st>>>((const float*)ivf->d_centroids, nlist, ds->dim,
                                                                                   ivf->d_centT, ivf->d_cnorm);
        else
            centroid_transpose_kernel<uint8_t><<<ceil_div(nlist, 128u), 128, 0, st>>>((const uint8_t*)ivf->d_centroids, nlist, ds->dim,
                                                                                     ivf->d_centT, ivf->d_cnorm);
        VDB_LAUNCHED();
        {
            DevBuf best(ds->n * 8, st), assign(std::max<size_t>(4, ds->n * 4), st);
            kmeans_assign_exact(ds->d_rows, ds->n, ds->pitch, ds->dtype, ds->metric, 0, ds->dim, ivf->d_centroids,
                                nlist, best.as<uint64_t>(), assign.as<uint32_t>(), nullptr, st);
            build_lists(assign.as<uint32_t>(), ds->n, nlist, ivf->d_offsets, ivf->d_members, st);
            if (h_assign_out && ds->n)
                VDB_CUDA(cudaMemcpyAsync(h_assign_out, assign.p, ds->n * 4, cudaMemcpyDeviceToHost, st));
            VDB_CUDA(cudaStreamSynchronize(st));
        }
        std::vector<uint64_t>& off = ivf->h_off;
        off.resize(nlist + 1);
        VDB_CUDA(cudaMemcpy(off.data(), ivf->d_offsets, off.size() * 8, cudaMemcpyDeviceToHost));
        for (uint32_t c = 0; c < nlist; ++c) ivf->max_list = std::max<uint32_t>(ivf->max_list, (uint32_t)(off[c + 1] - off[c]));
        VDB_CUDA(cudaStreamSynchronize(st));
        cudaStreamDestroy(st);
    } catch (...) {
        if (st) cudaStreamDestroy(st);
        ivf_destroy(ivf);
        throw;
    }
    return ivf;
}

void ivf_destroy(vdb_ivf* ivf) {
    if (!ivf) return;
    cudaFree(ivf->d_centroids);
    cudaFree(ivf->d_centT);
    cudaFree(ivf->d_cnorm);
    cudaFree(ivf->d_offsets);
    cudaFree(ivf->d_members);
    cudaFree(ivf->d_rows_lo);
    cudaFree(ivf->d_samp_rows);
    cudaFree(ivf->d_samp_colA);
    cudaFree(ivf->d_samp_rn);
    cudaFree(ivf->d_colA_lo);
    cudaFree(ivf->d_rn_lo);
    cudaFree(ivf->d_ex_lo);
    cudaFree(ivf->d_samp_ex);
    delete ivf;
}

IvfItems ivf_group_items(const vdb_ivf* ivf, const uint64_t* probes, uint32_t nq, uint32_t nprobe, uint32_t group,
                         uint32_t tile, uint32_t min_range) {
    const std::vector<uint64_t>& off = ivf->h_off;
    std::vector<std::vector<uint32_t>> by_list(ivf->nlist);
    for (uint32_t q = 0; q < nq; ++q)
        for (uint32_t j = 0; j < nprobe; ++j) {
            const uint64_t pk = probes[(size_t)q * nprobe + j];
            if (pk != KEY_NONE) by_list[key_id(pk)].push_back(q);
        }
    // row-range size: enough items to fill the GPU a few times, rows per item a multiple of the warp tile
    uint64_t work = 0;  // sum over (list, query group) of rows
    for (uint32_t l = 0; l < ivf->nlist; ++l) work += ceil_div<uint64_t>(by_list[l].size(), group) * (off[l + 1] - off[l]);
    const uint64_t target_items = (uint64_t)sm_count() * 16;
    uint32_t range = (uint32_t)std::max<uint64_t>(min_range, round_up<uint64_t>(ceil_div<uint64_t>(work, target_items), tile));
    IvfItems out;
    std::vector<IvfItem>& items = out.items;
    std::vector<std::vector<uint32_t>> qlists(nq);  // partial-list indices per query
    for (uint32_t l = 0; l < ivf->nlist; ++l) {
        const uint64_t len = off[l + 1] - off[l];
        if (len == 0) continue;
        const auto& qv = by_list[l];
        for (size_t c = 0; c < qv.size(); c += group) {
            const uint32_t nv = (uint32_t)std::min<size_t>(group, qv.size() - c);
            for (uint64_t r0 = 0; r0 < len; r0 += range) {
                IvfItem it{};
                it.row_begin = off[l] + r0;
                it.nrows = (uint32_t)std::min<uint64_t>(range, len - r0);
                it.nq_valid = nv;
                for (uint32_t s = 0; s < nv; ++s) {
                    it.qid[s] = qv[c + s];
                    qlists[qv[c + s]].push_back((uint32_t)(items.size() * group + s));
                }
                items.push_back(it);
            }
        }
    }
    out.poff.assign(nq + 1, 0);
    for (uint32_t q = 0; q < nq; ++q) out.poff[q + 1] = out.poff[q] + qlists[q].size();
    out.plist.resize(out.poff[nq]);
    for (uint32_t q = 0; q < nq; ++q) std::copy(qlists[q].begin(), qlists[q].end(), out.plist.begin() + out.poff[q]);
    return out;
}

void ivf_merge_items(const uint64_t* d_partial, const IvfItems& it, uint32_t nq, uint32_t K, uint64_t* d_keys, cudaStream_t st) {
    DevBuf d_poff(it.poff.size() * 8, st), d_plist(std::max<size_t>(4, it.plist.size() * 4), st);
    VDB_CUDA(cudaMemcpyAsync(d_poff.p, it.poff.data(), it.poff.size() * 8, cudaMemcpyHostToDevice, st));
    if (!it.plist.empty()) VDB_CUDA(cudaMemcpyAsync(d_plist.p, it.plist.data(), it.plist.size() * 4, cudaMemcpyHostToDevice, st));
    const uint32_t PM = topk_segment_size(K, 256);
    const size_t smem_m = TopkSmem::bytes(1, PM);
    VDB_REQUIRE(smem_m <= 200 * 1024, "IVF merge: k=%u too large", K);
    if (smem_m > 48 * 1024)
        VDB_CUDA(cudaFuncSetAttribute(ivf_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_m));
    ivf_merge_kernel<<<nq, 256, smem_m, st>>>(d_partial, d_poff.as<uint64_t>(), d_plist.as<uint32_t>(), K, PM, PM - K - 256,
                                              d_keys);
    VDB_LAUNCHED();
}

static void ivf_list_major(const vdb_dataset* ds, const vdb_ivf* ivf, const QueryTile& qt, const uint64_t* probes,
                           uint32_t nq, uint32_t nprobe, uint32_t k, uint64_t* d_keys, cudaStream_t st) {
    const IvfItems grouped = ivf_group_items(ivf, probes, nq, nprobe, LQ, IVF_WARPS * LR, IVF_WARPS * LR * 4);
    const std::vector<IvfItem>& items = grouped.items;
    if (items.empty()) {
        VDB_CUDA(cudaMemsetAsync(d_keys, 0xff, (size_t)nq * k * 8, st));
        return;
    }
    DevBuf d_items(items.size() * sizeof(IvfItem), st), partial(items.size() * LQ * (size_t)k * 8, st);
    VDB_CUDA(cudaMemcpyAsync(d_items.p, items.data(), items.size() * sizeof(IvfItem), cudaMemcpyHostToDevice, st));
    const uint32_t period = 64;
    const uint32_t P = topk_segment_size(k, period);
    const size_t smem = (size_t)LQ * qt.qstride * 4 + TopkSmem::bytes(LQ, P);
    VDB_REQUIRE(smem <= 200 * 1024, "IVF scan: dim=%u / k=%u do not fit in shared memory", ds->dim, k);
    IvfListParams p{};
    p.rows = (const uint8_t*)ds->d_rows;
    p.pitch_bytes = ds->pitch_bytes();
    p.nvec = qt.nvec;
    p.nit = qt.nit;
    p.q = qt.q.as<float>();
    p.qstride = qt.qstride;
    p.qcache = qt.qcache.as<float>();
    p.items = d_items.as<IvfItem>();
    p.members = ivf->d_members;
    p.K = k;
    p.P = P;
    p.limit = P - k - period;
    p.sync_every = std::max(1u, period / (IVF_WARPS * LR));
    p.id_base = (uint32_t)ds->id_base;
    p.partial = partial.as<uint64_t>();
    auto go = [&](auto kern) {
        if (smem > 48 * 1024)
            VDB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        ProfScope prof("ivf_scan", st);
        kern<<<(uint32_t)items.size(), IVF_THREADS, smem, st>>>(p);
        VDB_LAUNCHED();
    };
    if (ds->dtype == VDB_F32) {
        if (ds->metric == VDB_L2SQR) go(ivf_list_scan_kernel<VDB_L2SQR, 1>);
        else go(ivf_list_scan_kernel<VDB_COSINE, 1>);
    } else {
        if (ds->metric == VDB_L2SQR) go(ivf_list_scan_kernel<VDB_L2SQR, 4>);
        else go(ivf_list_scan_kernel<VDB_COSINE, 4>);
    }
    ivf_merge_items(partial.as<uint64_t>(), grouped, nq, k, d_keys, st);
}

__global__ void gather_bytes_rows_kernel(const uint8_t* __restrict__ src, uint32_t row_bytes, const uint32_t* __restrict__ idx,
                                         uint32_t cnt, uint8_t* __restrict__ dst) {
    const uint32_t i = blockIdx.x;
    if (i >= cnt) return;
    for (uint32_t e = threadIdx.x; e < row_bytes; e += blockDim.x)
        dst[(size_t)i * row_bytes + e] = src[(size_t)idx[i] * row_bytes + e];
}

// FP32 list-major scan of a subset of the batch (queries h_sel[0..nsel)); keys out: [nsel][k]
void ivf_list_major_subset(const vdb_dataset* ds, const vdb_ivf* ivf, const void* d_queries, const uint64_t* d_probes,
                           const uint32_t* h_sel, uint32_t nsel, uint32_t nprobe, uint32_t k, uint64_t* d_keys_sel,
                           cudaStream_t st) {
    if (nsel == 0) return;
    const uint32_t row_bytes = ds->dim * ds->elem_size();
    DevBuf sel((size_t)nsel * 4, st), q((size_t)nsel * row_bytes, st), pr((size_t)nsel * nprobe * 8, st);
    VDB_CUDA(cudaMemcpyAsync(sel.p, h_sel, (size_t)nsel * 4, cudaMemcpyHostToDevice, st));
    gather_bytes_rows_kernel<<<nsel, 128, 0, st>>>((const uint8_t*)d_queries, row_bytes, sel.as<uint32_t>(), nsel, q.as<uint8_t>());
    VDB_LAUNCHED();
    gather_bytes_rows_kernel<<<nsel, 64, 0, st>>>((const uint8_t*)d_probes, nprobe * 8, sel.as<uint32_t>(), nsel, pr.as<uint8_t>());
    VDB_LAUNCHED();
    std::vector<uint64_t> h_probes((size_t)nsel * nprobe);
    VDB_CUDA(cudaMemcpyAsync(h_probes.data(), pr.p, h_probes.size() * 8, cudaMemcpyDeviceToHost, st));
    VDB_CUDA(cudaStreamSynchronize(st));
    QueryTile qt = prepare_queries(ds, q.p, nsel, st);
    ivf_list_major(ds, ivf, qt, h_probes.data(), nsel, nprobe, k, d_keys_sel, st);
}

DevBuf ivf_probe_keys(const vdb_dataset* ds, const vdb_ivf* ivf, const void* d_queries, uint32_t nq, uint32_t nprobe,
                      cudaStream_t st) {
    // exact query-centroid distances, probe order = find_n_nearest (k_means.rs:174-191)
    DevBuf cdist((size_t)nq * ivf->nlist * 4, st), ckeys((size_t)nq * ivf->nlist * 8, st), probes((size_t)nq * nprobe * 8, st);
    probe_distances(ds, ivf, d_queries, nq, cdist.as<float>(), st);
    const uint64_t cnt = (uint64_t)nq * ivf->nlist;
    probe_keys_kernel<<<(uint32_t)std::min<uint64_t>(ceil_div<uint64_t>(cnt, 256), 4096), 256, 0, st>>>(
        cdist.as<float>(), cnt, ivf->nlist, ckeys.as<uint64_t>());
    VDB_LAUNCHED();
    launch_merge_keys(ckeys.as<uint64_t>(), 1, nq, ivf->nlist, false, nprobe, probes.as<uint64_t>(), nullptr, nullptr,
                      nullptr, st);
    return probes;
}

void ivf_knn_keys(const vdb_dataset* ds, const vdb_ivf* ivf, const void* d_queries, uint32_t nq, uint32_t k,
                  uint32_t n_probes, uint64_t* d_keys, cudaStream_t st) {
    VDB_REQUIRE(n_probes > 0, "The number of probes should be greater than 0.");
    VDB_REQUIRE(ds->n == ivf->n && ds->dim == ivf->dim && ds->dtype == ivf->dtype && ds->metric == ivf->metric,
                "IVF index was built for a different vector set");
    if (nq == 0 || k == 0) return;
    if (nq > 16384) {  // chunks bound the candidate / rerank scratch of the batched paths
        const size_t row_bytes = (size_t)ds->dim * ds->elem_size();
        for (uint32_t q0 = 0; q0 < nq; q0 += 16384)
            ivf_knn_keys(ds, ivf, (const uint8_t*)d_queries + (size_t)q0 * row_bytes, std::min(16384u, nq - q0), k, n_probes,
                         d_keys + (size_t)q0 * k, st);
        return;
    }
    const uint32_t nprobe = std::min(n_probes, ivf->nlist);
    // 1. probe order
    DevBuf probes = ivf_probe_keys(ds, ivf, d_queries, nq, nprobe, st);
    // 2. list scan
    if (nq >= 4) {
        // probe table to the host (nq * nprobe keys): the grouping by list is host work, the item tables go back
        static thread_local PinnedStage probe_stage;
        const uint64_t* h_probes = (const uint64_t*)probe_stage.get((size_t)nq * nprobe * 8);
        VDB_CUDA(cudaMemcpyAsync((void*)h_probes, probes.p, (size_t)nq * nprobe * 8, cudaMemcpyDeviceToHost, st));
        VDB_CUDA(cudaStreamSynchronize(st));
        static const int no_tensor = getenv("VDB_IVF_NO_TENSOR") ? atoi(getenv("VDB_IVF_NO_TENSOR")) : 0;
        if (!no_tensor && nq >= 16 &&
            ivf_tensor_keys(ds, ivf, d_queries, probes.as<uint64_t>(), h_probes, nq, nprobe, k, d_keys, st))
            return;
        QueryTile qt = prepare_queries(ds, d_queries, nq, st);
        ivf_list_major(ds, ivf, qt, h_probes, nq, nprobe, k, d_keys, st);
        return;
    }
    QueryTile qt = prepare_queries(ds, d_queries, nq, st);
    const uint32_t period = IVF_WARPS * IVF_R;
    const uint32_t P = topk_segment_size(k, period);
    const size_t smem = (size_t)qt.qstride * 4 + TopkSmem::bytes(1, P) + 16 + (size_t)round_up(nprobe + 1, 2u) * 4 +
                        (size_t)nprobe * 8;
    VDB_REQUIRE(smem <= 200 * 1024, "IVF scan: dim=%u / k=%u / n_probes=%u do not fit in shared memory", ds->dim, k,
                nprobe);
    const uint32_t target = (uint32_t)sm_count() * 4;
    uint32_t splits = std::max(1u, ceil_div(target, nq));
    const uint64_t max_visit = (uint64_t)ivf->max_list * nprobe;
    splits = (uint32_t)std::min<uint64_t>(splits, std::max<uint64_t>(1, max_visit / (IVF_WARPS * IVF_R)));
    DevBuf partial((size_t)nq * splits * k * 8, st);
    IvfScanParams p{};
    p.rows = (const uint8_t*)ds->d_rows;
    p.pitch_bytes = ds->pitch_bytes();
    p.nvec = qt.nvec;
    p.nit = qt.nit;
    p.q = qt.q.as<float>();
    p.qstride = qt.qstride;
    p.qcache = qt.qcache.as<float>();
    p.probes = probes.as<uint64_t>();
    p.nprobe = nprobe;
    p.offsets = ivf->d_offsets;
    p.members = ivf->d_members;
    p.splits = splits;
    p.K = k;
    p.P = P;
    p.limit = P - k - period;
    p.id_base = (uint32_t)ds->id_base;
    p.partial = partial.as<uint64_t>();
    auto go = [&](auto kern) {
        if (smem > 48 * 1024)
            VDB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        ProfScope prof("ivf_scan", st);
        kern<<<nq * splits, IVF_THREADS, smem, st>>>(p);
        VDB_LAUNCHED();
    };
    if (ds->dtype == VDB_F32) {
        if (ds->metric == VDB_L2SQR) go(ivf_scan_kernel<VDB_L2SQR, 1>);
        else go(ivf_scan_kernel<VDB_COSINE, 1>);
    } else {
        if (ds->metric == VDB_L2SQR) go(ivf_scan_kernel<VDB_L2SQR, 4>);
        else go(ivf_scan_kernel<VDB_COSINE, 4>);
    }
    launch_merge_keys(partial.as<uint64_t>(), splits, nq, k, false, k, d_keys, nullptr, nullptr, nullptr, st);
}

}  // namespace vdb
