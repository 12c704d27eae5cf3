// ivf_pq.cu — IndexPQ::knn_pq on the IVF index: an ADC scan of the probed lists' codes only.
//
// The reference has no IVF knn_pq; this library defines it (INTEGRATION.md) as FlatIndex::knn_pq
// (src/index_algorithm/flat_index.rs:84-104) restricted to the rows of the n_probes nearest lists (find_n_nearest,
// src/distance/k_means.rs:174-191): the max(ef, k) smallest (ADC, id) over those rows, re-scored exactly, the k smallest
// (distance, id) kept (pq_resort, candidate_pair.rs:102-108). That result does not depend on the visiting order, so the
// candidate keys are bit-exact and n_probes >= nlist gives exactly the Flat knn_pq result.
//
// Layout: a table's codes are copied once into list order (position p <-> row members[p]) in the scan's transposed
// layout ([block of 32 positions][word][lane]), so a warp reads one code word of 32 consecutive positions of a list as one
// coalesced 128-byte request, as K8 (pq.cu) does over the whole set. Work items are those of the batched IVF scan (list,
// up to NQ queries probing it, a position range); the row sums are K8's (adc.cuh).
#include <algorithm>
#include <type_traits>

#include "adc.cuh"
#include "index.cuh"
#include "topk.cuh"

struct IvfPqCodes {
    uint64_t serial = 0;     // vdb_pq::serial of the table the codes come from
    uint32_t* d = nullptr;   // [ceil(n/32)][words][32] u32, position p = row members[p]
    ~IvfPqCodes() { cudaFree(d); }
};

namespace vdb {

struct IvfPqParams {
    const uint32_t* codes;      // list-ordered, transposed
    const uint32_t* members;
    const IvfItem* items;
    uint32_t words, m, tab;
    const float* lut;           // [nq][tab]
    const float* dist_cache;    // [tab]
    const float* qcache;        // [nq]
    uint32_t K, P, limit;
    uint32_t id_base;
    uint64_t* partial;          // [items][NQ][K]
};

// One CTA per item. Warps take 32-position blocks, lane = position & 31; an item that starts or ends inside a block
// masks the lanes outside it. LUT_SMEM: the item's tables in shared memory, else read through L1 (then NQ == 1).
template <int NQ, int NBITS, int METRIC, bool LUT_SMEM>
__global__ void __launch_bounds__(ADC_THREADS) ivf_pq_scan_kernel(const IvfPqParams p) {
    static_assert(LUT_SMEM || NQ == 1, "tables read through L1 serve one query per CTA");
    extern __shared__ __align__(16) uint8_t smem[];
    constexpr int WARPS = ADC_THREADS / 32;
    const IvfItem& item = p.items[blockIdx.x];   // qid[] is indexed at run time: read in place, not copied to local memory
    const uint32_t tab = p.tab;
    float* s_lut = reinterpret_cast<float*>(smem);
    float* s_dc = s_lut + (LUT_SMEM ? (size_t)NQ * tab : 0);
    uint64_t* tk = reinterpret_cast<uint64_t*>(s_dc + ((LUT_SMEM && METRIC == VDB_COSINE) ? tab : 0));
    TopkSmem topk{tk, reinterpret_cast<uint32_t*>(tk + (size_t)NQ * p.P), p.K, p.P, NQ, p.limit};
    if (LUT_SMEM) {
        for (uint32_t i = threadIdx.x; i < NQ * tab; i += blockDim.x) {
            const uint32_t qi = i / tab;
            s_lut[i] = qi < item.nq_valid ? p.lut[(size_t)item.qid[qi] * tab + (i - qi * tab)] : 0.f;
        }
        if (METRIC == VDB_COSINE)
            for (uint32_t i = threadIdx.x; i < tab; i += blockDim.x) s_dc[i] = p.dist_cache[i];
    }
    topk.init();
    float qn[NQ];
#pragma unroll
    for (int q = 0; q < NQ; ++q) qn[q] = (METRIC == VDB_COSINE && q < (int)item.nq_valid) ? p.qcache[item.qid[q]] : 0.f;
    const float* lut = LUT_SMEM ? s_lut : p.lut + (size_t)item.qid[0] * tab;
    const float* dc = LUT_SMEM ? s_dc : p.dist_cache;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint64_t b = item.row_begin, e = b + item.nrows;
    const uint64_t blk0 = b >> 5;
    const uint32_t iters = (uint32_t)ceil_div<uint64_t>(((e + 31) >> 5) - blk0, WARPS);

    for (uint32_t it = 0; it < iters; ++it) {
        const uint64_t blk = blk0 + (uint64_t)it * WARPS + warp;
        const uint64_t pos = blk * 32 + lane;
        const bool in = pos >= b && pos < e;
        float sum[NQ];
        float cdp = 0.f;
#pragma unroll
        for (int q = 0; q < NQ; ++q) sum[q] = 0.f;
        if (in) adc_row_sum<NQ, NBITS, METRIC, LUT_SMEM>(p.codes + blk * p.words * 32 + lane, p.words, p.m, tab, lut, dc, sum, cdp);
        bool want = false;
        if (in) {
            const uint32_t id = p.id_base + p.members[pos];
#pragma unroll
            for (int q = 0; q < NQ; ++q) {
                if (q < (int)item.nq_valid) {
                    float d = sum[q];
                    if (METRIC == VDB_COSINE) {
                        const float den = fmaxf(__fmul_rn(sqrtf(cdp), qn[q]), 1e-10f);
                        d = __fsub_rn(1.0f, __fdiv_rn(sum[q], den));
                    }
                    const uint64_t key = make_key(d, id);
                    if (key < topk.tau(q)) want |= topk.push(q, key);
                }
            }
        }
        topk.maybe_flush(want);
    }
    topk.final_flush();
    for (uint32_t i = threadIdx.x; i < NQ * p.K; i += blockDim.x) {
        const uint32_t qi = i / p.K, j = i - qi * p.K;
        p.partial[((size_t)blockIdx.x * NQ + qi) * p.K + j] = qi < item.nq_valid ? topk.seg(qi)[j] : KEY_NONE;
    }
}

// the table's codes in list order, built on first use with this table (g_ivf_side_mu; see vdb_ivf::pq_codes)
static std::shared_ptr<const IvfPqCodes> ivf_pq_codes(const vdb_ivf* civf, const vdb_pq* pq, cudaStream_t st) {
    vdb_ivf* ivf = const_cast<vdb_ivf*>(civf);
    std::lock_guard<std::mutex> lk(g_ivf_side_mu);
    if (ivf->pq_codes && ivf->pq_codes->serial == pq->serial) return ivf->pq_codes;
    auto c = std::make_shared<IvfPqCodes>();
    c->serial = pq->serial;
    const uint64_t n = ivf->n, total = ceil_div<uint64_t>(n, 32) * pq->words * 32;
    VDB_CUDA(cudaMalloc(&c->d, std::max<uint64_t>(1, total) * 4));
    if (n) {
        DevBuf lo(n * pq->enc, st);
        gather_bytes_rows_kernel<<<(uint32_t)n, 128, 0, st>>>(pq->d_codes, pq->enc, ivf->d_members, (uint32_t)n, lo.as<uint8_t>());
        VDB_LAUNCHED();
        pq_transpose_kernel<<<(uint32_t)std::min<uint64_t>(ceil_div<uint64_t>(total, 256), 1u << 20), 256, 0, st>>>(
            lo.as<uint8_t>(), n, pq->enc, pq->words, c->d);
        VDB_LAUNCHED();
        VDB_CUDA(cudaStreamSynchronize(st));
    }
    ivf->pq_codes = c;
    return c;
}

static void check_ivf_pq(const vdb_dataset* ds, const vdb_ivf* ivf, const vdb_pq* pq, uint32_t n_probes) {
    // an index / table of a row-sharded set has no arrays of its own (its shards do)
    VDB_REQUIRE(ivf->shards.empty() && ds->n == ivf->n && ds->dim == ivf->dim && ds->dtype == ivf->dtype && ds->metric == ivf->metric,
                "IVF index was built for a different vector set");
    VDB_REQUIRE(pq->shards.empty() && ds->n == pq->n && ds->dim == pq->dim && ds->dtype == pq->dtype,
                "PQ table was built for a different vector set (it must be rebuilt after add/delete)");
    VDB_REQUIRE(ds->metric == pq->metric, "Distance algorithm mismatch.");
    VDB_REQUIRE(n_probes > 0, "The number of probes should be greater than 0.");
}

constexpr uint32_t IVF_PQ_CHUNK = 16384;   // queries per pass: bounds the candidate / rerank scratch

void ivf_pq_adc_keys(const vdb_dataset* ds, const vdb_ivf* ivf, const vdb_pq* pq, const void* d_queries, uint32_t nq,
                     uint32_t kk, uint32_t n_probes, uint64_t* d_keys, cudaStream_t st) {
    check_ivf_pq(ds, ivf, pq, n_probes);
    if (nq == 0 || kk == 0) return;
    if (nq > IVF_PQ_CHUNK) {
        const size_t row_bytes = (size_t)ds->dim * ds->elem_size();
        for (uint32_t q0 = 0; q0 < nq; q0 += IVF_PQ_CHUNK)
            ivf_pq_adc_keys(ds, ivf, pq, (const uint8_t*)d_queries + (size_t)q0 * row_bytes, std::min(IVF_PQ_CHUNK, nq - q0), kk,
                            n_probes, d_keys + (size_t)q0 * kk, st);
        return;
    }
    const uint32_t nprobe = std::min(n_probes, ivf->nlist);
    // 1. probe order; the probe table goes to the host, where the grouping by list is done
    DevBuf probes = ivf_probe_keys(ds, ivf, d_queries, nq, nprobe, st);
    static thread_local PinnedStage probe_stage;
    const uint64_t* h_probes = (const uint64_t*)probe_stage.get((size_t)nq * nprobe * 8);
    VDB_CUDA(cudaMemcpyAsync((void*)h_probes, probes.p, (size_t)nq * nprobe * 8, cudaMemcpyDeviceToHost, st));
    VDB_CUDA(cudaStreamSynchronize(st));
    const std::shared_ptr<const IvfPqCodes> codes = ivf_pq_codes(ivf, pq, st);
    // 2. lookup tables, queries per item and table placement as for K8
    const uint32_t tab = pq->m * pq->kc;
    DevBuf lut((size_t)nq * tab * 4, st), qcache((size_t)nq * 4, st);
    pq_lut(pq, d_queries, nq, lut.as<float>(), qcache.as<float>(), st);
    const uint32_t P = topk_segment_size(kk, ADC_THREADS);
    auto smem_for = [&](int t, bool ls) {
        return (ls ? ((size_t)t * tab + (pq->metric == VDB_COSINE ? tab : 0)) * 4 : 0) + TopkSmem::bytes(t, P);
    };
    bool lut_smem = true;
    const int nqt = adc_queries_per_cta(4, nq, smem_for, &lut_smem);
    const size_t smem = smem_for(nqt, lut_smem);
    VDB_REQUIRE(smem <= ADC_SMEM_MAX, "IVF ADC scan: ef=%u too large for the fused top-k", kk);
    // 3. list-major items: warps take 32-position blocks, an item is at least one full step of the CTA
    const IvfItems grouped = ivf_group_items(ivf, h_probes, nq, nprobe, (uint32_t)nqt, 32, ADC_THREADS);
    const std::vector<IvfItem>& items = grouped.items;
    if (items.empty()) {
        VDB_CUDA(cudaMemsetAsync(d_keys, 0xff, (size_t)nq * kk * 8, st));
        return;
    }
    DevBuf d_items(items.size() * sizeof(IvfItem), st), partial(items.size() * nqt * (size_t)kk * 8, st);
    VDB_CUDA(cudaMemcpyAsync(d_items.p, items.data(), items.size() * sizeof(IvfItem), cudaMemcpyHostToDevice, st));
    IvfPqParams p{};
    p.codes = codes->d;
    p.members = ivf->d_members;
    p.items = d_items.as<IvfItem>();
    p.words = pq->words;
    p.m = pq->m;
    p.tab = tab;
    p.lut = lut.as<float>();
    p.dist_cache = pq->d_dist_cache;
    p.qcache = qcache.as<float>();
    p.K = kk;
    p.P = P;
    p.limit = P - kk - ADC_THREADS;
    p.id_base = (uint32_t)ds->id_base;
    p.partial = partial.as<uint64_t>();
    auto go = [&](auto kern) {
        if (smem > 48 * 1024) VDB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ADC_SMEM_MAX));
        ProfScope prof("ivf_pq_scan", st);
        kern<<<(uint32_t)items.size(), ADC_THREADS, smem, st>>>(p);
        VDB_LAUNCHED();
    };
    auto by_metric = [&](auto nq_c, auto bits_c, auto smem_c) {
        constexpr int NQ = decltype(nq_c)::value, NB = decltype(bits_c)::value;
        constexpr bool LS = decltype(smem_c)::value;
        if (pq->metric == VDB_COSINE) go(ivf_pq_scan_kernel<NQ, NB, VDB_COSINE, LS>);
        else go(ivf_pq_scan_kernel<NQ, NB, VDB_L2SQR, LS>);
    };
    auto by_bits = [&](auto nq_c, auto smem_c) {
        if (pq->n_bits == 4) by_metric(nq_c, std::integral_constant<int, 4>{}, smem_c);
        else by_metric(nq_c, std::integral_constant<int, 8>{}, smem_c);
    };
    if (!lut_smem) by_bits(std::integral_constant<int, 1>{}, std::false_type{});
    else if (nqt == 1) by_bits(std::integral_constant<int, 1>{}, std::true_type{});
    else if (nqt == 2) by_bits(std::integral_constant<int, 2>{}, std::true_type{});
    else by_bits(std::integral_constant<int, 4>{}, std::true_type{});
    // 4. per-query merge of the items' lists
    ivf_merge_items(partial.as<uint64_t>(), grouped, nq, kk, d_keys, st);
}

void ivf_pq_knn_keys(const vdb_dataset* ds, const vdb_ivf* ivf, const vdb_pq* pq, const void* d_queries, uint32_t nq,
                     uint32_t k, uint32_t ef, uint32_t n_probes, uint64_t* d_keys, cudaStream_t st) {
    check_ivf_pq(ds, ivf, pq, n_probes);
    if (nq == 0 || k == 0) return;
    const uint32_t kk = std::max(ef, k);
    const size_t row_bytes = (size_t)ds->dim * ds->elem_size();
    for (uint32_t q0 = 0; q0 < nq; q0 += IVF_PQ_CHUNK) {
        const uint32_t cn = std::min(IVF_PQ_CHUNK, nq - q0);
        const void* dq = (const uint8_t*)d_queries + (size_t)q0 * row_bytes;
        DevBuf cand((size_t)cn * kk * 8, st);
        ivf_pq_adc_keys(ds, ivf, pq, dq, cn, kk, n_probes, cand.as<uint64_t>(), st);
        rerank_keys(ds, dq, cn, cand.as<uint64_t>(), kk, k, d_keys + (size_t)q0 * k, st);
    }
}

}  // namespace vdb
