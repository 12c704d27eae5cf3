// index.cuh — device mirrors of PQTable / IVFIndex and the k-means / pair-distance launchers.
#pragma once
#include <atomic>
#include <memory>
#include <mutex>
#include <vector>

#include "dataset.cuh"

// device mirror of PQTable<T> (reference src/distance/pq_table.rs:116-137)
struct vdb_pq {
    int device = 0;
    uint64_t serial = 0;            // process-wide creation number (keys the list-ordered copy of the codes an IVF keeps)
    uint32_t dim = 0, m = 0, n_bits = 0, kc = 0, enc = 0;  // enc = encoded_dim (bytes per row)
    int dtype = VDB_F32, metric = VDB_L2SQR;
    uint64_t n = 0;
    uint32_t words = 0;             // u32 words per row in the transposed layout
    std::vector<uint32_t> g_lo, g_len, g_off;  // per group: first dim, length, codebook element offset
    uint32_t max_len = 0;
    void* d_codebooks = nullptr;    // groups concatenated, group g = [kc][len_g] of dtype
    uint32_t* d_groups = nullptr;   // [m][3] (lo, len, off)
    float* d_dist_cache = nullptr;  // [m*kc] 0 (L2) / dot(c,c) (cosine), pq_table.rs:165-170
    float* d_cb_norm = nullptr;     // [m*kc] ||c|| for cosine encoding
    uint8_t* d_codes = nullptr;     // [n][enc] reference layout
    uint32_t* d_codes_t = nullptr;  // [ceil(n/32)][words][32] transposed for the ADC scan
    uint32_t* d_sample_t = nullptr; // the same layout for a stratified random row sample (thresholds of the scan)
    uint8_t* d_sample = nullptr;    // the sampled code rows in the reference layout [sample_n][enc] (tensor-core sample pass)
    uint32_t sample_n = 0;
    // decoded-operand contraction (pq_dec.cu), built lazily by the first batched search: FP16 codebooks scaled by a power
    // of two, ||x^||^2 and ||x^|| of every code row and of every sampled row, the worst-case decode error norm
    void* d_dec_cb16 = nullptr;
    float* d_dec_r = nullptr, *d_dec_xn = nullptr, *d_dec_sr = nullptr, *d_dec_sxn = nullptr;
    bool dec_ok = false;
    float dec_scale = 1.0f, dec_ex = 0.f;
    std::vector<vdb_pq*> shards;    // row-sharded parent (multi.cu): one table per shard, the arrays above stay empty
    const struct vdb_dataset* parent = nullptr;   // the row-sharded set a parent table was built on
};

// device mirror of IVFIndex<T> (reference src/index_algorithm/ivf_index.rs:34-47)
struct vdb_tq;  // per-call query context of the tensor path (flat_gemm.cu)
struct IvfPqCodes;  // one PQ table's codes in list order (ivf_pq.cu)

struct vdb_ivf {
    int device = 0;
    uint32_t nlist = 0, dim = 0;
    int dtype = VDB_F32, metric = VDB_L2SQR;
    uint64_t n = 0;
    void* d_centroids = nullptr;    // [nlist][dim] of dtype
    float* d_centT = nullptr;       // [dim][nlist] f32: the probe-order kernel reads a centroid per lane, coalesced
    float* d_cnorm = nullptr;       // [nlist] ||c|| (cosine), summed like assign_exact_kernel
    uint64_t* d_offsets = nullptr;  // [nlist+1]
    uint32_t* d_members = nullptr;  // [n] local row ids, ascending inside a list
    uint32_t max_list = 0;
    std::vector<uint64_t> h_off;    // host copy of d_offsets (fixed after the build)
    // lazily built for the tensor-core probe scan: rows / norms permuted into list order (position p <-> members[p])
    void* d_rows_lo = nullptr;    // [n][op row bytes] operand rows of the dataset's kind (FP16 copy / fp32 rows)
    int op_kind = 0;
    float* d_colA_lo = nullptr;   // [n] ||x||^2 (L2Sqr) or 1/||x|| (cosine)
    float* d_rn_lo = nullptr;     // [n] ||x||
    float* d_ex_lo = nullptr;     // [n] operand error norm
    // stratified 1/64 sample of every list, also in list order (threshold pass of the tensor-core probe scan)
    void* d_samp_rows = nullptr;
    float* d_samp_colA = nullptr, *d_samp_rn = nullptr, *d_samp_ex = nullptr;
    std::vector<uint64_t> h_samp_off;  // [nlist+1]
    uint64_t samp_n = 0;
    // lazily built by the first knn_pq call with a table (ivf_pq.cu), rebuilt when a call brings another table; a call
    // holds its own reference, so a rebuild never frees codes a running scan reads
    std::shared_ptr<const IvfPqCodes> pq_codes;
    std::vector<vdb_ivf*> shards;      // row-sharded parent (multi.cu): one index per shard, the arrays above stay empty
    const struct vdb_dataset* parent = nullptr;   // the sharded dataset it was built on
};

// device mirror of HNSWIndex<T> (reference src/index_algorithm/hnsw_index.rs:99-141)
struct HnswReplicas;
struct vdb_hnsw {
    int device = 0;
    uint64_t n = 0;
    uint32_t dim = 0;
    int dtype = VDB_F32, metric = VDB_L2SQR;
    uint32_t M = 0, M0 = 0, ef_construction = 0;
    std::vector<uint32_t> h_level;     // vec_level
    uint32_t* d_links0 = nullptr;      // level0_links [n][M0]
    uint32_t* d_len0 = nullptr;        // links_len[.][0]
    uint32_t* d_ulinks = nullptr;      // other_links: slot (uoff[node] + level - 1) holds M links
    uint32_t* d_ulen = nullptr;        // links_len[.][level >= 1] per slot
    uint64_t* d_uoff = nullptr;        // [n+1] prefix sum of the node levels
    uint64_t slots = 0;                // sum of the node levels
    uint32_t* d_level = nullptr;       // [n]
    float* d_cache = nullptr;          // dist_cache [n]
    uint32_t* d_overflow = nullptr;    // neighbours a search could not record in its visited set (must stay 0)
    int64_t enter_point = -1;
    int enter_level = -1;
    // index of a row-sharded set (multi.cu): the scalars above are replica 0's, the arrays stay empty
    HnswReplicas* rep = nullptr;
};

// HNSW on a row-sharded set: a graph walk needs every row, so each shard entry holds a full replica (all n rows and the
// same graph) and a search splits its batch over the replicas
struct HnswPqReplicas;   // one PQ table's codes over all rows, one vdb_pq per replica (multi.cu)
struct HnswReplicas {
    const struct vdb_dataset* parent = nullptr;   // the row-sharded set the index was built on
    std::vector<vdb_dataset*> ds;                 // replica r: all n rows on shard r's device, ids id_base + row
    std::vector<vdb_hnsw*> h;                     // replica r: the graph over ds[r]
    std::atomic<uint32_t> next{0};                // first replica of the next call with fewer queries than replicas
    std::mutex pq_mu;                             // guards `pq`
    // built by the first knn_pq call with a table, rebuilt when a call brings another table; a call holds its own
    // reference, so a rebuild never frees codes a running search reads
    std::shared_ptr<const HnswPqReplicas> pq;
};

namespace vdb {

// multi.cu: IVF / PQ on a row-sharded dataset
vdb_ivf* sharded_ivf_create(const vdb_dataset* md, const void* h_centroids, uint32_t nlist, uint32_t* h_assign_out);
void sharded_ivf_lists(const vdb_dataset* md, const vdb_ivf* ivf, uint64_t* offsets, uint32_t* members);
void sharded_ivf_knn(const vdb_dataset* md, const vdb_ivf* ivf, const void* queries, uint32_t nq, uint32_t k, uint32_t n_probes,
                     uint64_t* ids, float* dist, uint32_t* counts);
vdb_pq* sharded_pq_create(const vdb_dataset* md, const void* h_codebooks, uint32_t m, uint32_t n_bits, const uint8_t* h_codes_in,
                          uint8_t* h_codes_out);
void sharded_pq_knn(const vdb_dataset* md, const vdb_pq* pq, const void* queries, uint32_t nq, uint32_t k, uint32_t ef,
                    uint64_t* ids, float* dist, uint32_t* counts);
void sharded_ivf_knn_pq(const vdb_dataset* md, const vdb_ivf* ivf, const vdb_pq* pq, const void* queries, uint32_t nq, uint32_t k,
                        uint32_t ef, uint32_t n_probes, uint64_t* ids, float* dist, uint32_t* counts);
// multi.cu: HNSW on a row-sharded dataset (one replica per shard entry)
vdb_hnsw* sharded_hnsw_build(const vdb_dataset* md, uint32_t M, uint32_t ef_construction, const uint32_t* h_levels,
                             uint32_t max_batch);
vdb_hnsw* sharded_hnsw_from_graph(const vdb_dataset* md, uint32_t M, uint32_t ef_construction, const uint32_t* h_levels,
                                  const uint32_t* links0, const uint32_t* len0, const uint32_t* ulinks, const uint32_t* ulen,
                                  int64_t enter_point, int32_t enter_level);
void sharded_hnsw_destroy(vdb_hnsw* h);
// pq == nullptr: knn_with_ef, else knn_pq
void sharded_hnsw_knn(const vdb_dataset* md, const vdb_hnsw* h, const vdb_pq* pq, const void* queries, uint32_t nq, uint32_t k,
                      uint32_t ef, uint64_t* ids, float* dist, uint32_t* counts);

// hnsw.cu
vdb_hnsw* hnsw_build(const vdb_dataset* ds, uint32_t M, uint32_t ef_construction, const uint32_t* h_levels, uint32_t max_batch);
void hnsw_destroy(vdb_hnsw* h);
void hnsw_check_overflow(const vdb_hnsw* h, cudaStream_t st);
void hnsw_append(vdb_hnsw* h, const vdb_dataset* ds, const uint32_t* new_levels, uint32_t max_batch);
vdb_hnsw* hnsw_from_graph(const vdb_dataset* ds, uint32_t M, uint32_t ef_construction, const uint32_t* h_levels,
                          const uint32_t* links0, const uint32_t* len0, const uint32_t* ulinks, const uint32_t* ulen,
                          int64_t enter_point, int32_t enter_level);
void hnsw_knn_keys(const vdb_dataset* ds, const vdb_hnsw* h, const void* d_queries, uint32_t nq, uint32_t k, uint32_t ef,
                   uint64_t* d_keys, cudaStream_t st);
void hnsw_knn_pq_keys(const vdb_dataset* ds, const vdb_hnsw* h, const vdb_pq* pq, const void* d_queries, uint32_t nq, uint32_t k,
                      uint32_t ef, uint64_t* d_keys, cudaStream_t st);

// kmeans.cu
void kmeans_assign_exact(const void* d_rows, uint64_t n, uint64_t pitch, int dtype, int metric, uint32_t lo,
                         uint32_t d, const void* d_cent, uint32_t k, uint64_t* d_best, uint32_t* d_assign,
                         float* d_all_dist, cudaStream_t st);
void build_lists(const uint32_t* d_assign, uint64_t n, uint32_t k, uint64_t* d_offsets, uint32_t* d_members,
                 cudaStream_t st);
uint32_t kmeans_lloyd(const void* d_rows, uint64_t n, uint64_t pitch, int dtype, int metric, uint32_t lo,
                      uint32_t d, void* d_cent, uint32_t k, uint32_t max_iter, float tol, cudaStream_t st);
void kmeans_pp_weights(const void* d_rows, uint64_t n, uint64_t pitch, int dtype, int metric, uint32_t lo,
                       uint32_t d, const void* d_c, float* d_w, cudaStream_t st);

// pairs.cu
void row_cache(const vdb_dataset* ds, float* d_out, cudaStream_t st);
void exact_pair_distances(const vdb_dataset* ds, const void* d_queries, const uint32_t* d_qidx,
                          const uint32_t* d_rid, uint64_t npairs, float* d_out, cudaStream_t st);
void exact_pair_distances_masked(const vdb_dataset* ds, const void* d_queries, uint32_t qpitch, const uint32_t* d_qidx,
                                 const uint32_t* d_rid, const uint8_t* d_valid, uint64_t npairs, float* d_out,
                                 cudaStream_t st, const uint64_t* d_npairs = nullptr, const float* d_qnorm = nullptr);
void cached_pair_distances(const vdb_dataset* ds, const void* d_queries, const float* d_qcache,
                           const float* d_rowcache, const uint32_t* d_qidx, const uint32_t* d_rid,
                           uint64_t npairs, float* d_out, cudaStream_t st);
void raw_pair_distances(const void* d_a, const void* d_b, uint64_t count, uint32_t dim, int dtype, int metric,
                        float* d_out, cudaStream_t st);
void expand_offsets(const uint64_t* d_off, uint32_t nq, uint32_t* d_qidx, cudaStream_t st);

// pq.cu
void pq_groups_host(uint32_t dim, uint32_t m, std::vector<uint32_t>& lo, std::vector<uint32_t>& len);
vdb_pq* pq_create(const vdb_dataset* ds, const void* h_codebooks, uint32_t m, uint32_t n_bits,
                  const uint8_t* h_codes_in, uint8_t* h_codes_out);
void pq_destroy(vdb_pq* pq);
void pq_lut(const vdb_pq* pq, const void* d_queries, uint32_t nq, float* d_lut, float* d_qcache, cudaStream_t st);
void pq_adc_all(const vdb_pq* pq, const float* d_lut, const float* d_qcache, uint32_t nq, float* d_out,
                cudaStream_t st);
void pq_adc_keys(const vdb_dataset* ds, const vdb_pq* pq, const void* d_queries, uint32_t nq, uint32_t kk, uint64_t* d_keys,
                 cudaStream_t st);
void pq_knn_keys(const vdb_dataset* ds, const vdb_pq* pq, const void* d_queries, uint32_t nq, uint32_t k,
                 uint32_t ef, uint64_t* d_keys, cudaStream_t st);

void rerank_keys(const vdb_dataset* ds, const void* d_queries, uint32_t nq, const uint64_t* d_cand, uint32_t kk,
                 uint32_t k, uint64_t* d_keys, cudaStream_t st);
// reference layout [n][enc] -> the scan's [ceil(n/32)][words][32] u32
__global__ void pq_transpose_kernel(const uint8_t* __restrict__ codes, uint64_t n, uint32_t enc, uint32_t words,
                                    uint32_t* __restrict__ out);

// ivf.cu
vdb_ivf* ivf_create(const vdb_dataset* ds, const void* h_centroids, uint32_t nlist, uint32_t* h_assign_out);
void ivf_destroy(vdb_ivf* ivf);
// flat_gemm.cu: tensor-core probe scan for query batches (returns false when the shard / batch is not eligible)
bool ivf_tensor_keys(const vdb_dataset* ds, const vdb_ivf* ivf, const void* d_queries, const uint64_t* d_probes,
                     const uint64_t* h_probes, uint32_t nq, uint32_t nprobe, uint32_t k, uint64_t* d_keys, cudaStream_t st);
void ivf_list_major_subset(const vdb_dataset* ds, const vdb_ivf* ivf, const void* d_queries, const uint64_t* d_probes,
                           const uint32_t* h_sel, uint32_t nsel, uint32_t nprobe, uint32_t k, uint64_t* d_keys_sel,
                           cudaStream_t st);
void ivf_knn_keys(const vdb_dataset* ds, const vdb_ivf* ivf, const void* d_queries, uint32_t nq, uint32_t k,
                  uint32_t n_probes, uint64_t* d_keys, cudaStream_t st);
extern std::mutex g_ivf_side_mu;   // guards the lazily built list-ordered arrays of every vdb_ivf
__global__ void gather_bytes_rows_kernel(const uint8_t* __restrict__ src, uint32_t row_bytes, const uint32_t* __restrict__ idx,
                                         uint32_t cnt, uint8_t* __restrict__ dst);
// [nq][nprobe] keys (distance, list id) of the nprobe nearest lists per query, ascending: find_n_nearest (k_means.rs:174-191)
DevBuf ivf_probe_keys(const vdb_dataset* ds, const vdb_ivf* ivf, const void* d_queries, uint32_t nq, uint32_t nprobe,
                      cudaStream_t st);
// Work items of the list-major batched scans: (list, up to `group` <= LQ queries that probe it, a range of the list's
// positions). Query q's partial lists (one per item it is in; partial list index = item * group + query slot) are
// plist[poff[q] .. poff[q + 1]). Ranges are multiples of `tile` positions, at least `min_range`, sized so that there are
// enough items to fill the GPU a few times.
constexpr int LQ = 8;
struct IvfItem {
    uint64_t row_begin;   // offset into members[]
    uint32_t nrows;
    uint32_t nq_valid;
    uint32_t qid[LQ];
};
struct IvfItems {
    std::vector<IvfItem> items;
    std::vector<uint64_t> poff;
    std::vector<uint32_t> plist;
};
IvfItems ivf_group_items(const vdb_ivf* ivf, const uint64_t* h_probes, uint32_t nq, uint32_t nprobe, uint32_t group,
                         uint32_t tile, uint32_t min_range);
// per-query merge of the items' partial lists ([items][group][K] keys) into d_keys [nq][K]
void ivf_merge_items(const uint64_t* d_partial, const IvfItems& it, uint32_t nq, uint32_t K, uint64_t* d_keys, cudaStream_t st);
// ivf_pq.cu: IndexPQ::knn_pq restricted to the probed lists. Candidate stage: the max(ef, k) = kk best (ADC, global id)
// keys per query over the rows of the n_probes nearest lists, [nq][kk], KEY_NONE padded; then the exact rerank.
void ivf_pq_adc_keys(const vdb_dataset* ds, const vdb_ivf* ivf, const vdb_pq* pq, const void* d_queries, uint32_t nq,
                     uint32_t kk, uint32_t n_probes, uint64_t* d_keys, cudaStream_t st);
void ivf_pq_knn_keys(const vdb_dataset* ds, const vdb_ivf* ivf, const vdb_pq* pq, const void* d_queries, uint32_t nq,
                     uint32_t k, uint32_t ef, uint32_t n_probes, uint64_t* d_keys, cudaStream_t st);

// rebuilds (distance, id) keys: key[j] = valid[j] ? make_key(dist[j], id[j]) : KEY_NONE
void rekey(const float* d_dist, const uint32_t* d_ids, const uint8_t* d_valid, uint64_t count, uint64_t* d_keys,
           cudaStream_t st);

void rekey_based(const float* d_dist, const uint32_t* d_ids, uint32_t id_base, const uint8_t* d_valid, uint64_t count,
                 uint64_t* d_keys, cudaStream_t st);

// kmeans.cu: batched PQ training
bool pq_train_supported(uint32_t kc, uint32_t max_len);
void pq_train_groups(const void* d_rows, uint64_t n, uint64_t pitch, int dtype, int metric, uint32_t m, uint32_t kc, uint32_t max_len,
                     const uint32_t* d_groups, const double* d_uniforms, const void* d_init, uint32_t max_iter, float tol,
                     void* d_out, uint32_t* d_iters, cudaStream_t st);

// pq_gemm.cu
bool pq_tensor_supported(const vdb_pq* pq, uint32_t nq);
// pq_dec.cu: the same scan as a contraction over rows decoded on the fly (sub-vectors of 4 dimensions)
bool pq_dec_supported(const vdb_pq* pq, uint32_t nq);
void* pq_dec_begin(const vdb_pq* pq, const void* d_queries, uint32_t nq, cudaStream_t st);   // nullptr: not applicable
void pq_dec_end(void* ctx);
void pq_dec_sample(const vdb_pq* pq, void* ctx, uint32_t nq, float* d_all, cudaStream_t st);
void pq_dec_filter(const vdb_pq* pq, void* ctx, const float* d_lut, uint32_t nq, const float* d_tau, uint32_t id_base,
                   uint32_t* d_cnt, uint64_t* d_cand, uint32_t cap, cudaStream_t st);
void pq_dec_destroy(vdb_pq* pq);
// test hook: lower bound of the filter / upper bound of the sample pass of every (query, row), [nq][n] each
void pq_dec_bounds(const vdb_pq* pq, const void* d_queries, uint32_t nq, float* d_lower, float* d_upper, cudaStream_t st);
// exact ADC (reference arithmetic) of coarse candidate rows; survivors with adc <= tau become keys (pq_gemm.cu)
void pq_exact_candidates(const vdb_pq* pq, const float* d_lut, const float* d_tau, uint32_t nq, const uint32_t* d_ccnt,
                         const uint32_t* d_ccand, uint32_t ccap, uint32_t id_base, uint32_t* d_cnt, uint64_t* d_cand,
                         uint32_t cap, cudaStream_t st);
void pq_tensor_lut(const vdb_pq* pq, const float* d_lut, uint32_t nq, DevBuf& lut16, cudaStream_t st);
void pq_tensor_sample(const vdb_pq* pq, const DevBuf& lut16, uint32_t nq, float* d_all, cudaStream_t st);
void pq_tensor_filter(const vdb_pq* pq, const DevBuf& lut16, const float* d_lut, uint32_t nq, const float* d_tau, uint32_t id_base,
                      uint32_t* d_cnt, uint64_t* d_cand, uint32_t cap, cudaStream_t st);
void pq_tensor_bounds(const vdb_pq* pq, const float* d_lut, uint32_t nq, float* d_lower, float* d_upper, cudaStream_t st);

// flat_gemm.cu
void flat_gemm_store(const vdb_dataset* ds, const void* d_queries, uint32_t nq, uint32_t row_stride, int kind,
                     uint64_t* d_out_keys, cudaStream_t st);
extern std::atomic<uint64_t> g_gemm_redo, g_gemm_cands, g_gemm_queries;
extern std::atomic<uint32_t> g_debug_force_redo;
uint32_t tensor_j0(uint32_t k, uint64_t ns, uint64_t n, double eps = 2e-5);
vdb_tq* tensor_begin(const vdb_dataset* ds, const void* d_queries, uint32_t nq, cudaStream_t st, bool any_size = false);
void operand_info(const vdb_dataset* ds, int* kind, float* scale, float* mean_norm, float* mean_ex, uint64_t* side_bytes);
void tensor_end(vdb_tq* tq);
// d_tau != nullptr: also tau_q from the j0-th smallest exact sample distance (single-shard calls: no exchange in between)
void tensor_sample_keys(vdb_tq* tq, uint32_t j, uint64_t* d_jkeys, float* d_tau = nullptr, uint32_t j0 = 0);
void tensor_tau(vdb_tq* tq, const uint64_t* d_lists, uint32_t nlists, uint32_t j, uint32_t j0, float* d_tau);
uint32_t tensor_sample_j(uint32_t j0, uint64_t sample_n);
// check != nullptr: the completeness check runs inside the filter's final merge (queries that fail go to d_redo, their
// number to *tensor_nredo_ptr(tq)); the number of reranked candidates is always left in *tensor_cand_total_ptr(tq)
struct TensorCheck {
    uint64_t n_total;
    uint32_t* d_redo;
};
void tensor_filter_keys(vdb_tq* tq, uint32_t k, uint32_t j0_local_hint, const float* d_tau, uint64_t* d_keys,
                        uint32_t* d_overflow, const TensorCheck* check = nullptr);
// the same filter split around one peer exchange of pruning statistics (row-sharded search, see flat_gemm.cu)
bool tensor_filter_split_supported(const vdb_tq* tq, uint32_t k);
const uint32_t* tensor_filter_begin(vdb_tq* tq, uint32_t k, const float* d_tau, uint32_t* T_out);   // -> [nq][T] statistics
void tensor_filter_finish(vdb_tq* tq, const uint32_t* d_stats_all, uint32_t shards, uint64_t* d_keys, uint32_t* d_overflow);
uint64_t* tensor_cand_total_ptr(const vdb_tq* tq);
uint32_t* tensor_nredo_ptr(const vdb_tq* tq);
void tensor_check(vdb_tq* tq, const uint64_t* d_keys, uint32_t k, uint64_t n_total, const float* d_tau,
                  const uint32_t* d_overflow, uint32_t* d_redo, uint32_t* d_nredo);
void tensor_check_range(vdb_tq* tq, uint32_t q0, uint32_t cnt, const uint64_t* d_keys, uint32_t k, uint64_t n_total,
                        const float* d_tau, const uint32_t* d_overflow, uint32_t* d_redo, uint32_t* d_nredo);
void tensor_info(const vdb_dataset* ds, uint64_t* n, uint32_t* sample_n, float* mean_norm, float* mean_ex, cudaStream_t st);

}  // namespace vdb
