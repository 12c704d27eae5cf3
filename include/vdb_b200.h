/*
 * vdb_b200.h — C ABI of the B200-native search backend for lab-1806-vec-db.
 *
 * This is the drop-in boundary: plain pointers and sizes, no C++/torch types. A Rust
 * `extern "C"` block binds these 1:1 (rust_shim/ and INTEGRATION.md show the binding a
 * maintainer of the reference would add). The reference has no FFI seam of its own; each
 * entry point names the reference trait method / function it replaces (paths relative to the
 * reference repository, v0.8.1).
 *
 * Conventions
 *  - every function returns 0 (VDB_OK) or a VDB_E* code; vdb_last_error() gives the message of
 *    the last failure on the calling thread. The reference panics on misuse (assert!), so the
 *    Rust shim panics on non-zero. CUDA errors are never swallowed and there is NO CPU fallback.
 *  - host-pointer entry points copy inputs to the GPU and results back; the `_dev` variants
 *    take device pointers plus a cudaStream_t (as void*) and are fully asynchronous.
 *  - rows/queries are row-major `dim`-element vectors of `dtype` (VecSet<T>, src/vec_set.rs:15-30).
 *  - results are SoA: ids[nq*k] (u64), dist[nq*k] (f32), counts[nq] = valid entries per query
 *    (min(k, n)); entries are ascending by (distance, id) exactly like
 *    ResultSet::into_sorted_vec (src/index_algorithm/candidate_pair.rs:36-40, 76-78).
 *    Unused tail entries are id = UINT64_MAX, dist = NaN.
 *  - search calls are re-entrant on one handle (the reference calls knn from rayon workers and
 *    Python threads under a read lock: src/database/mod.rs:255, examples/bench.rs:415).
 */
#ifndef VDB_B200_H
#define VDB_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum { VDB_OK = 0, VDB_EINVAL = 1, VDB_ECUDA = 2, VDB_ENOMEM = 3, VDB_EUNSUPPORTED = 4 };
enum { VDB_L2SQR = 0, VDB_COSINE = 1 }; /* DistanceAlgorithm, src/distance/mod.rs:18-28 */
enum { VDB_F32 = 0, VDB_U8 = 1 };       /* Scalar, src/scalar.rs:117-119 */

typedef struct vdb_dataset vdb_dataset; /* device mirror of one VecSet<T> (or one row shard of it) */
typedef struct vdb_pq vdb_pq;           /* device mirror of a PQTable<T> (src/distance/pq_table.rs:116-137) */
typedef struct vdb_ivf vdb_ivf;         /* device mirror of an IVFIndex<T> (src/index_algorithm/ivf_index.rs:34-47) */
typedef struct vdb_hnsw vdb_hnsw;       /* device mirror of an HNSWIndex<T> (src/index_algorithm/hnsw_index.rs:99-141) */

/* ---- runtime ------------------------------------------------------------------------------ */
const char* vdb_last_error(void);
int vdb_version(void);
int vdb_device_count(int* out);
/* Selects the CUDA device used by handles created afterwards on this thread. */
int vdb_set_device(int device);

/* Registers the devices of this process (SURVEY.md section 8b `vdb_init(devices[], n)`) and enables peer access between
 * every pair (NVLink P2P). With n >= 2, vdb_dataset_create row-shards the set over them - contiguous blocks, shard s on
 * devices[s] (SURVEY.md section 8e) - and vdb_flat_knn on that handle is ONE call that runs on every device and merges
 * the per-GPU top-k over peer memory: the reference's `knn` (src/index_algorithm/mod.rs:84-91) stays one call whatever
 * the GPU count. A device may be listed more than once (several shards on one GPU; used by the single-GPU tests of the
 * sharded path). n == 1 selects that device for the calling thread; n == 0 returns to single-device mode. */
int vdb_init(const int* devices, uint32_t n);

/* ---- VecSet mirror -------------------------------------------------------------------------- */
/* Replaces the storage side of FlatIndex::from_vec_set (src/index_algorithm/flat_index.rs:59-70):
 * uploads `n` rows to HBM (rows padded to a 16-byte multiple so every row starts 128-bit aligned).
 * `id_base` is added to local row numbers in results (row-sharding across GPUs: shard r holds
 * rows [id_base, id_base+n)); id_base + n must be < 2^32. Host memory stays authoritative. */
int vdb_dataset_create(const void* rows, uint64_t n, uint32_t dim, int dtype, int metric,
                       uint64_t id_base, vdb_dataset** out);
/* Same, but adopts rows already resident on the device (row pitch in elements; pitch*sizeof(T)
 * must be a multiple of 16 and pad columns must be zero). The memory is NOT owned by the handle. */
int vdb_dataset_create_dev(const void* d_rows, uint64_t n, uint32_t dim, uint32_t pitch, int dtype,
                           int metric, uint64_t id_base, vdb_dataset** out);
/* Row-sharded set over rows already resident on the shards' devices: d_rows[s] holds counts[s] rows (global rows
 * [sum(counts[:s]), ...)) on devices[s], all with the same pitch. The memory is NOT owned by the handle. */
int vdb_dataset_create_sharded_dev(const void* const* d_rows, const uint64_t* counts, const int* devices, uint32_t nshards,
                                   uint32_t dim, uint32_t pitch, int dtype, int metric, uint64_t id_base, vdb_dataset** out);
/* Number of shards (0 for an unsharded set) and shard s: its own dataset handle (owned by the parent; valid for the
 * per-shard entry points such as vdb_ivf_create / vdb_pq_create), device and global row block. Outputs may be NULL. */
int vdb_dataset_shards(const vdb_dataset* ds, uint32_t* n);
int vdb_dataset_shard(const vdb_dataset* ds, uint32_t s, vdb_dataset** shard, int* device, uint64_t* row_lo, uint64_t* row_hi);
/* VecSet::push / DynamicIndex::batch_add (src/vec_set.rs:113-118, src/database/dynamic_index.rs:49-56) */
int vdb_dataset_append(vdb_dataset* ds, const void* rows, uint64_t n);
/* VecSet::swap_remove (src/vec_set.rs:131-137): row `idx` is overwritten by the last row. */
int vdb_dataset_swap_remove(vdb_dataset* ds, uint64_t idx);
int vdb_dataset_len(const vdb_dataset* ds, uint64_t* n);
int vdb_dataset_dim(const vdb_dataset* ds, uint32_t* dim);
int vdb_dataset_destroy(vdb_dataset* ds);

/* ---- distance primitives -------------------------------------------------------------------- */
/* DistanceAdapter<[T],[T]>::distance for `count` independent pairs a[i], b[i]
 * (src/distance/mod.rs:106-113; pyo3 calc_dist src/pyo3/mod.rs:43-48 is count == 1).
 * metric may also be VDB_DOT (the trait primitive dot_product, src/distance/mod.rs:43). */
enum { VDB_DOT = 2 };
int vdb_calc_dist(const void* a, const void* b, uint64_t count, uint32_t dim, int dtype, int metric,
                  float* out);
/* DistanceAlgorithm::dist_cache for every row (src/distance/mod.rs:31-36; HNSW push_init
 * src/index_algorithm/hnsw_index.rs:251-254, 371-379): L2Sqr -> ||v||^2, Cosine -> ||v||. */
int vdb_row_cache(const vdb_dataset* ds, float* out);
/* Batched HNSW candidate evaluation, cached form (src/index_algorithm/hnsw_index.rs:351-358,
 * src/distance/mod.rs:54-57, 67-69). Query j is compared with rows cand_ids[cand_off[j]..cand_off[j+1]);
 * out has cand_off[nq] entries. cand_ids are LOCAL row numbers of `ds`. */
int vdb_gather_dist(const vdb_dataset* ds, const void* queries, uint32_t nq, const uint32_t* cand_ids,
                    const uint64_t* cand_off, float* out);

/* ---- Flat ------------------------------------------------------------------------------------ */
/* IndexKNN::knn for FlatIndex (src/index_algorithm/flat_index.rs:48-57), batched over nq queries
 * (nq == 1 is the unchanged trait call; nq > 1 is the additive batch entry used by bench drivers,
 * examples/bench.rs:414-418, src/bin/gen_gnd.rs:65-68). Exact: the k smallest by (distance, id),
 * distances in the difference form sum((q-x)^2) / the 3-dot cosine form. */
int vdb_flat_knn(const vdb_dataset* ds, const void* queries, uint32_t nq, uint32_t k, uint64_t* ids,
                 float* dist, uint32_t* counts);
int vdb_flat_knn_dev(const vdb_dataset* ds, const void* d_queries, uint32_t nq, uint32_t k,
                     uint64_t* d_ids, float* d_dist, uint32_t* d_counts, void* stream);
/* The same on a row-sharded set with the batch already resident on every shard's device: d_queries[s] = the whole
 * [nq, dim] batch on shard s's device. Shard s OWNS the queries [s * per, min(nq, (s + 1) * per)), per = ceil(nq / G),
 * and receives their merged results in d_ids[s] / d_dist[s] / d_counts[s] (arrays of at least `per` rows on its
 * device). nq <= 16384 per call. Synchronous: every shard's stream has drained on return. */
int vdb_flat_knn_sharded_dev(const vdb_dataset* ds, const void* const* d_queries, uint32_t nq, uint32_t k,
                             uint64_t* const* d_ids, float* const* d_dist, uint32_t* const* d_counts);
/* Concurrent nq == 1 calls of vdb_flat_knn on one handle - the reference's call pattern: one query per knn call from
 * rayon workers / Python threads under a read lock (examples/bench.rs:410-416, src/database/mod.rs:248-256) - are
 * coalesced: calls that arrive while a database pass is running (or within <= 120 us of each other once several callers
 * have been seen) are answered by ONE pass. Results are bit-identical to individual calls. On by default;
 * vdb_set_batching(0) turns it off process-wide. vdb_batch_stats: passes run / queries served through the batcher. */
int vdb_set_batching(int on);
int vdb_batch_stats(const vdb_dataset* ds, uint64_t* batches, uint64_t* queries);
/* The rayon loop of the reference's drivers (examples/bench.rs:410-416 `-t`, src/bin/gen_gnd.rs:65-68) for hosts without
 * a native thread pool: nq queries, ONE vdb_flat_knn(nq = 1) call each, issued from `threads` native threads. Results
 * as vdb_flat_knn with nq queries; *seconds (optional) = wall time of the loop. */
int vdb_parallel_knn(const vdb_dataset* ds, const void* queries, uint32_t nq, uint32_t k, uint32_t threads, uint64_t* ids,
                     float* dist, uint32_t* counts, double* seconds);
/* Row-sharded search, step 1: this shard's k best per query as packed sortable keys
 * (high 32 bits = order-preserving distance bits, low 32 bits = global id), [nq, k], ascending,
 * padded with UINT64_MAX. Step 2 (after an NCCL all-gather of the shards' keys):
 * vdb_merge_keys_dev merges `nlists` such lists per query: keys is [nlists, nq, k]. */
int vdb_flat_knn_keys_dev(const vdb_dataset* ds, const void* d_queries, uint32_t nq, uint32_t k,
                          uint64_t* d_keys, void* stream);
int vdb_merge_keys_dev(const uint64_t* d_keys, uint32_t nlists, uint32_t nq, uint32_t k,
                       uint64_t* d_ids, float* d_dist, uint32_t* d_counts, void* stream);
/* Selects the Flat implementation: 0 = auto, 1 = FP32 streaming scan (K1), 2 = tensor-core
 * contraction + FP32 rerank (K2, batched L2Sqr f32 only). Results are identical either way. */
int vdb_flat_set_path(int path);
/* The same selection for ONE handle (-1 = follow the process default set by vdb_flat_set_path). */
int vdb_dataset_set_flat_path(vdb_dataset* ds, int path);

/* ---- k-means (IVF / PQ training) ---------------------------------------------------------- */
/* find_nearest for n rows (src/distance/k_means.rs:40-57, 117-120, 166-170;
 * src/index_algorithm/ivf_index.rs:89-93): out[i] = argmin_c d(rows[i][sel_lo..sel_hi], centroids[c])
 * by (distance, c). centroids is [k, sel_hi-sel_lo] of the rows' dtype. */
int vdb_kmeans_assign(const void* rows, uint64_t n, uint32_t dim, int dtype, int metric,
                      const void* centroids, uint32_t k, uint32_t sel_lo, uint32_t sel_hi,
                      uint32_t* out);
int vdb_kmeans_assign_ds(const vdb_dataset* ds, const void* centroids, uint32_t k, uint32_t sel_lo,
                         uint32_t sel_hi, uint32_t* out);
/* Lloyd iterations of KMeans::from_vec_set from given initial centroids
 * (src/distance/k_means.rs:108-161): assignment, per-centroid mean summed in ascending member
 * order in f32, empty clusters keep their centroid, stop when max squared shift < tol.
 * centroids: in = initial (k-means++ draws stay on the host side because they consume the
 * caller's RNG, k_means.rs:61-87), out = trained. *iters = iterations executed. */
int vdb_kmeans_train(const void* rows, uint64_t n, uint32_t dim, int dtype, int metric,
                     void* centroids, uint32_t k, uint32_t sel_lo, uint32_t sel_hi, uint32_t max_iter,
                     float tol, uint32_t* iters);
/* Same as vdb_kmeans_train with the training rows already resident in a dataset handle (PQ trains one k-means
 * per group on the same sample: pq_table.rs:154-172). */
int vdb_kmeans_train_ds(const vdb_dataset* ds, void* centroids, uint32_t k, uint32_t sel_lo, uint32_t sel_hi,
                        uint32_t max_iter, float tol, uint32_t* iters);
/* k-means++ initialisation (src/distance/k_means.rs:61-87) on device-resident rows. The random draws stay with the
 * caller: uniforms[0] picks the first row (index = floor(u * n)); round r = 1..k-1 uses uniforms[2r-1] for the
 * weighted pick (probability proportional to w[i] = min over chosen c of d(c, v_i)) and uniforms[2r] for the
 * uniform fallback the reference draws eagerly (k_means.rs:80-82; used when the weights are all zero/invalid).
 * uniforms has 2k-1 entries in [0,1). centroids receives [k, sel_hi-sel_lo] rows of the dataset dtype. */
int vdb_kmeans_pp_init_ds(const vdb_dataset* ds, uint32_t k, uint32_t sel_lo, uint32_t sel_hi, const double* uniforms,
                          void* centroids);
/* k-means++ weight update w[i] = min(w[i], d(c, rows[i][sel])) (src/distance/k_means.rs:75-77). */
int vdb_kmeans_pp_weights(const void* rows, uint64_t n, uint32_t dim, int dtype, int metric,
                          const void* centroid, uint32_t sel_lo, uint32_t sel_hi, float* weights);

/* The per-group k-means of PQTable::from_vec_set (src/distance/pq_table.rs:154-172) for ALL m groups at once on the
 * training sample `train` (device resident): k = 2^n_bits centroids per group, k-means++ (k_means.rs:61-87) driven by
 * the caller's draws - uniforms[g * (2k - 1) + ...] laid out per group as in vdb_kmeans_pp_init_ds - then Lloyd
 * (:108-161) with the reference's arithmetic. init_codebooks != NULL skips k-means++ (then uniforms may be NULL); given
 * the same initial centroids the result is bit-identical to m calls of vdb_kmeans_train_ds. codebooks (in/out layout):
 * groups concatenated, [k][len_g] of the dataset dtype. iters (optional) receives the iterations run per group.
 * Returns VDB_EUNSUPPORTED when k x max sub-dim does not fit one CTA's shared memory (use the per-group calls). */
int vdb_pq_train_ds(const vdb_dataset* train, uint32_t m, uint32_t n_bits, uint32_t max_iter, float tol,
                    const double* uniforms, const void* init_codebooks, void* codebooks, uint32_t* iters);

/* ---- PQ ------------------------------------------------------------------------------------- */
/* pq_groups (src/distance/pq_table.rs:38-53): out is [m, 2] (start, end). */
int vdb_pq_groups(uint32_t dim, uint32_t m, uint32_t* out);
/* Builds the device PQ table from trained codebooks (group g = [2^n_bits, len_g], concatenated)
 * and encodes every row of `ds` (pq_encode + the encode loop, src/distance/pq_table.rs:66-91,
 * 178-181). If `codes` is non-NULL it receives the reference-layout codes [n, encoded_dim]. */
int vdb_pq_create(const vdb_dataset* ds, const void* codebooks, uint32_t m, uint32_t n_bits,
                  uint8_t* codes, vdb_pq** out);
/* Same, from codes computed earlier (PQTable::load, src/distance/pq_table.rs:232-237). */
int vdb_pq_create_from_codes(const vdb_dataset* ds, const void* codebooks, uint32_t m, uint32_t n_bits,
                             const uint8_t* codes, vdb_pq** out);
int vdb_pq_destroy(vdb_pq* pq);
/* PQTable::create_lookup (src/distance/pq_table.rs:195-224): lut is [nq, m*2^n_bits], qcache [nq]. */
int vdb_pq_lut(const vdb_pq* pq, const void* queries, uint32_t nq, float* lut, float* qcache);
/* ADC distance of every code against query LUTs (src/distance/pq_table.rs:239-301): out [nq, n]. */
int vdb_pq_adc_all(const vdb_pq* pq, const void* queries, uint32_t nq, float* out);
/* IndexPQ::knn_pq for FlatIndex (src/index_algorithm/flat_index.rs:84-104): ADC scan into the
 * max(ef,k) best by (adc, id), then exact rerank (candidate_pair.rs:102-108). */
int vdb_pq_knn(const vdb_dataset* ds, const vdb_pq* pq, const void* queries, uint32_t nq, uint32_t k,
               uint32_t ef, uint64_t* ids, float* dist, uint32_t* counts);
int vdb_pq_knn_dev(const vdb_dataset* ds, const vdb_pq* pq, const void* d_queries, uint32_t nq,
                   uint32_t k, uint32_t ef, uint64_t* d_ids, float* d_dist, uint32_t* d_counts,
                   void* stream);

/* Row-sharded knn_pq (SURVEY 8e): (1) every shard's max(ef,k) best codes by (ADC, global id) as packed keys
 * [nq, kk]; (2) after an all-gather + vdb_merge_keys_to_keys_dev to the GLOBAL top-kk, every shard reranks the
 * candidates it owns (others become KEY_NONE) into [nq, k] keys; (3) all-gather + merge gives the reference result. */
int vdb_pq_adc_keys_dev(const vdb_dataset* ds, const vdb_pq* pq, const void* d_queries, uint32_t nq, uint32_t kk,
                        uint64_t* d_keys, void* stream);
int vdb_pq_rerank_keys_dev(const vdb_dataset* ds, const void* d_queries, uint32_t nq, const uint64_t* d_cand_keys,
                           uint32_t kk, uint32_t k, uint64_t* d_keys, void* stream);

/* ---- IVF ------------------------------------------------------------------------------------ */
/* IVFIndex::from_vec_set after training (src/index_algorithm/ivf_index.rs:88-106): assigns every
 * row to its nearest centroid and builds the inverted lists (members ascending). `assign_out`
 * (may be NULL) receives the per-row list id. */
int vdb_ivf_create(const vdb_dataset* ds, const void* centroids, uint32_t nlist, uint32_t* assign_out,
                   vdb_ivf** out);
int vdb_ivf_destroy(vdb_ivf* ivf);
/* Copies the lists out: offsets [nlist+1], members [n] (local row ids). */
int vdb_ivf_lists(const vdb_ivf* ivf, uint64_t* offsets, uint32_t* members);
/* IndexKNNWithEf::knn_with_ef for IVFIndex (src/index_algorithm/ivf_index.rs:143-154):
 * find_n_nearest centroids (src/distance/k_means.rs:174-191) then scan the probed lists. */
int vdb_ivf_knn(const vdb_dataset* ds, const vdb_ivf* ivf, const void* queries, uint32_t nq, uint32_t k,
                uint32_t n_probes, uint64_t* ids, float* dist, uint32_t* counts);
int vdb_ivf_knn_dev(const vdb_dataset* ds, const vdb_ivf* ivf, const void* d_queries, uint32_t nq,
                    uint32_t k, uint32_t n_probes, uint64_t* d_ids, float* d_dist, uint32_t* d_counts,
                    void* stream);

/* ---- IVF + PQ ------------------------------------------------------------------------------- */
/* IndexPQ::knn_pq on the IVF index. The reference has no IVF knn_pq; this library defines it as FlatIndex::knn_pq
 * (src/index_algorithm/flat_index.rs:84-104) restricted to the rows of the n_probes nearest lists (find_n_nearest,
 * src/distance/k_means.rs:174-191; n_probes clamped to nlist): the max(ef, k) smallest (ADC, id) over those rows in the
 * reference's ADC arithmetic (src/distance/pq_table.rs:239-301), re-scored exactly, the k smallest (distance, id) kept
 * (pq_resort, candidate_pair.rs:102-108); counts[q] = min(k, rows in the probed lists). Only the codes of the probed lists
 * are scanned. With n_probes >= nlist the result is bit-identical to vdb_pq_knn on the same table. The first call with a
 * table copies its codes into list order on the index (n * ceil(encoded_dim / 4) * 4 bytes; a call with another table
 * replaces the copy). Errors (VDB_EINVAL, in this order): the index or the table was built for another vector set (a
 * table must be rebuilt after add / delete), metric mismatch, n_probes == 0. On a row-sharded set vdb_ivf_knn_pq is one
 * call over all shards (index and table built on that set). */
int vdb_ivf_knn_pq(const vdb_dataset* ds, const vdb_ivf* ivf, const vdb_pq* pq, const void* queries, uint32_t nq, uint32_t k,
                   uint32_t ef, uint32_t n_probes, uint64_t* ids, float* dist, uint32_t* counts);
/* Device pointers. Like vdb_ivf_knn_dev it synchronises `stream` once: the probed lists are grouped on the host. */
int vdb_ivf_knn_pq_dev(const vdb_dataset* ds, const vdb_ivf* ivf, const vdb_pq* pq, const void* d_queries, uint32_t nq,
                       uint32_t k, uint32_t ef, uint32_t n_probes, uint64_t* d_ids, float* d_dist, uint32_t* d_counts,
                       void* stream);
/* The candidate stage alone (counterpart of vdb_pq_adc_keys_dev): d_keys [nq, kk] = the kk best (ADC, global id) packed
 * keys per query over the probed lists, ascending, UINT64_MAX padded. Synchronises `stream` once. */
int vdb_ivf_pq_adc_keys_dev(const vdb_dataset* ds, const vdb_ivf* ivf, const vdb_pq* pq, const void* d_queries, uint32_t nq,
                            uint32_t kk, uint32_t n_probes, uint64_t* d_keys, void* stream);

/* ---- tensor-core Flat path, phase by phase (row-sharded search: lab_1806_vec_db_b200/sharded.py) ---------
 * The single-GPU vdb_flat_knn runs these phases internally. Across shards the thresholds must be GLOBAL (else
 * every shard reranks its own ~750 candidates per query), so the phases are exported and the host inserts the
 * collectives:  begin -> sample -> [all-gather] -> tau -> filter -> [all-gather keys, all-reduce overflow] ->
 * vdb_merge_keys_dev -> check -> (rare) exact re-scan of the flagged queries -> end.  All pointers are device
 * pointers; everything runs on the stream given to begin. */
typedef struct vdb_tq vdb_tq;
/* n, sample size, mean row norm and mean operand-error norm of this shard (builds the side arrays on first use). */
int vdb_tq_info(const vdb_dataset* ds, uint64_t* n, uint32_t* sample_n, float* mean_norm, float* mean_ex);
/* Smallest sample order statistic whose rank among n_total rows is >= k with probability > 1 - 2e-5. */
uint32_t vdb_tq_j0(uint32_t k, uint64_t sample_total, uint64_t n_total);
int vdb_tq_begin_dev(const vdb_dataset* ds, const void* d_queries, uint32_t nq, void* stream, vdb_tq** out);
/* number of sampled rows to re-evaluate per query for the order statistic j0 (a few more than j0; at most sample_min,
 * the smallest shard's sample size) */
uint32_t vdb_tq_sample_j(uint32_t j0, uint64_t sample_min);
/* the j best sampled rows of every query by pruning score, re-evaluated exactly: d_keys [nq, j] = (exact distance,
 * global id) keys, ascending, KEY_NONE padded */
int vdb_tq_sample_dev(vdb_tq* tq, uint32_t j, uint64_t* d_keys);
/* merges nlists shards' sample keys ([nlists, nq, j]) and writes tau[q] = (j0-th smallest exact sample distance) -
 * ||q||^2 (cosine: the distance itself): every row of the true top-k has a pruning score below it whenever the j0-th
 * sampled distance is not better than the k-th best of the set (vdb_tq_j0), which vdb_tq_check_dev verifies per query */
int vdb_tq_tau_dev(vdb_tq* tq, const uint64_t* d_keys_lists, uint32_t nlists, uint32_t j, uint32_t j0, float* d_tau);
/* filter pass + exact rerank: this shard's k best keys per query ([nq, k], KEY_NONE padded) and per-query
 * overflow flags (candidate list overflowed: the result for that query is not provably complete) */
int vdb_tq_filter_dev(vdb_tq* tq, uint32_t k, const float* d_tau, uint64_t* d_keys, uint32_t* d_overflow);
/* completeness check of the MERGED keys: d_redo receives the queries that must be re-run exactly, *d_nredo their count */
int vdb_tq_check_dev(vdb_tq* tq, const uint64_t* d_merged_keys, uint32_t k, uint64_t n_total, const float* d_tau,
                     const uint32_t* d_overflow, uint32_t* d_redo, uint32_t* d_nredo);
int vdb_tq_end(vdb_tq* tq);
/* Exact streaming scan (K1) regardless of the selected Flat path: d_keys [nq, k]. */
int vdb_flat_scan_keys_dev(const vdb_dataset* ds, const void* d_queries, uint32_t nq, uint32_t k, uint64_t* d_keys,
                           void* stream);
/* Merge that returns packed keys instead of SoA results (keys [nlists, nq, k] -> d_out_keys [nq, k]). */
int vdb_merge_keys_to_keys_dev(const uint64_t* d_keys, uint32_t nlists, uint32_t nq, uint32_t k, uint64_t* d_out_keys,
                               void* stream);
/* Decodes packed keys into ids / distances / counts. */
int vdb_decode_keys_dev(const uint64_t* d_keys, uint32_t nq, uint32_t k, uint64_t* d_ids, float* d_dist,
                        uint32_t* d_counts, void* stream);

/* ---- tensor-core path internals (tests / tuning) ---------------------------------------------- */
/* Pruning scores of the tensor-core Flat path: out_keys[q * ns + i] = key(S'(q, row i*row_stride), i) for the
 * ns = n / row_stride strided rows. S' is the search's own lower bound of d(q, x) - ||q||^2 (L2Sqr) / of the cosine
 * distance, from the tensor-core contraction of the operand kind `kind` (0 = TF32: the fp32 rows in place, truncated by
 * the hardware; 1 = FP16 copy scaled by a power of two; < 0 = the dataset's own choice) minus the rigorous bound built
 * from the measured per-row / per-query operand errors. d_queries: device [nq, dim] of the dataset dtype. Synchronous. */
int vdb_debug_gemm_scores_dev(const vdb_dataset* ds, const void* d_queries, uint32_t nq, uint32_t row_stride,
                              int kind, uint64_t* d_out_keys, void* stream);
/* Bounds of the tensor-core PQ filter (4-bit L2Sqr tables of >= 65536 rows): for every (query, row) of the table,
 * d_lower[q * n + row] = the filter's lower bound S' of the exact ADC value (a row is dropped iff S' > tau_q) and
 * d_upper[q * n + row] = the sample pass's upper bound U of it, from the kernels and constants of the search.
 * path 0 = one-hot contraction over the BF16 lookup tables, 1 = contraction over decoded rows (sub-vectors of 4 dims;
 * its score is mapped back to the smallest tau_q at which the filter keeps the row). d_queries: device [nq, dim] of
 * the table's dtype; d_lower / d_upper: device [nq, n] f32. Synchronous. */
int vdb_debug_pq_bounds_dev(const vdb_pq* pq, const void* d_queries, uint32_t nq, int path, float* d_lower,
                            float* d_upper, void* stream);
/* Side arrays of the tensor-core path of an (unsharded) dataset, built lazily by the first batched search and dropped on
 * mutation: operand kind (-1 = not built, 0 = TF32: the fp32 rows in place, 1 = FP16 copy), its power-of-two scale, the
 * mean row norm / mean operand-error norm, and the HBM bytes they occupy (FP16 kind: 2 bytes per element + 12 bytes per
 * row, i.e. +50 % of an f32 set, +200 % of a u8 set; TF32 kind: 12 bytes per row). Outputs may be NULL. */
int vdb_dataset_operand_info(const vdb_dataset* ds, int* kind, float* scale, float* mean_norm, float* mean_ex,
                             uint64_t* side_bytes);
/* Frees them (they are rebuilt by the next batched search). Not re-entrant with searches on the handle. */
int vdb_dataset_drop_side_arrays(vdb_dataset* ds);
/* Queries that failed the tensor path's completeness check and were re-run through the exact scan. */
uint64_t vdb_flat_gemm_fallbacks(void);
/* Cumulative counters of the tensor path: queries served, candidates reranked, queries re-run exactly. */
int vdb_flat_gemm_stats(uint64_t* queries, uint64_t* candidates, uint64_t* fallbacks);

/* Test hook: every query whose batch index is a multiple of `every` fails the tensor path's completeness check and is
 * re-run through the exact scan (0 = off), so that the fallback of the single-GPU and the sharded search can be tested. */
int vdb_debug_force_redo(uint32_t every);

/* Row-sharded IVF: this shard's [nq, k] packed keys (merge the shards' lists with vdb_merge_keys_dev). */
int vdb_ivf_knn_keys_dev(const vdb_dataset* ds, const vdb_ivf* ivf, const void* d_queries, uint32_t nq, uint32_t k,
                         uint32_t n_probes, uint64_t* d_keys, void* stream);

/* ---- HNSW ------------------------------------------------------------------------------------- */
/* HNSWIndex::build_on_vec_set (src/index_algorithm/hnsw_index.rs:585-600; IndexBuilder::new :495-537, add :538-572,
 * add_parallel :399-457) over the rows of `ds` in row order, graph resident on the device. M / ef_construction as in
 * HNSWConfig (:41-59; max_m0 = 2 M, ef_construction = max(ef_construction, 2 M)). levels[i] = rand_level (:145-149)
 * of row i, drawn by the CALLER's RNG in row order (floor(-ln(u) / ln M)); host array of n entries. A batch of new
 * nodes (at most max_batch, and at most inserted / M as in next_batch_size :389-395) is searched read-only on the
 * current graph plus brute force inside the batch, then linked in batch order - the reference's batch semantics. */
int vdb_hnsw_build(const vdb_dataset* ds, uint32_t M, uint32_t ef_construction, const uint32_t* levels,
                   uint32_t max_batch, vdb_hnsw** out);
int vdb_hnsw_destroy(vdb_hnsw* h);
/* IndexBuilder::add / batch_add on a built index (:538-575; DynamicIndex::HNSW add, src/database/dynamic_index.rs:44-55):
 * inserts the rows appended to `ds` since the build (vdb_dataset_append), rows [n_index, n_ds), with new_levels[i] =
 * rand_level of row n_index + i. Same batch pipeline as the build. Not re-entrant with searches on the same handle
 * (the reference holds the table's write lock here, database/mod.rs:217). */
int vdb_hnsw_append(vdb_hnsw* h, const vdb_dataset* ds, const uint32_t* new_levels, uint32_t max_batch);
/* n, M, effective ef_construction, enter_point (-1 when empty), enter_level. Any pointer may be NULL. */
int vdb_hnsw_info(const vdb_hnsw* h, uint64_t* n, uint32_t* M, uint32_t* ef_construction, int64_t* enter_point,
                  int32_t* enter_level);
/* level-0 adjacency as the reference stores it (level0_links :110-112, links_len): links0[n * 2M], len0[n]. */
int vdb_hnsw_links0(const vdb_hnsw* h, uint32_t* links0, uint32_t* len0);
/* Upper levels (other_links :113-119, links_len): for every node its level_i lists of M links, nodes in row order,
 * levels 1..level_i in order: ulinks[sum(levels) * M], ulen[sum(levels)]. levels[n] is filled when non-NULL; a call
 * with only `levels` (ulinks == ulen == NULL) returns the levels so that the caller can size the other two arrays. */
int vdb_hnsw_upper(const vdb_hnsw* h, uint32_t* levels, uint32_t* ulinks, uint32_t* ulen);
/* An index built elsewhere - e.g. deserialised from the reference's bincode file (IndexSerdeExternalVecSet
 * :641-668) - over the rows of `ds`: same layouts as vdb_hnsw_links0 / vdb_hnsw_upper. */
int vdb_hnsw_create_from_graph(const vdb_dataset* ds, uint32_t M, uint32_t ef_construction, const uint32_t* levels,
                               const uint32_t* links0, const uint32_t* len0, const uint32_t* ulinks, const uint32_t* ulen,
                               int64_t enter_point, int32_t enter_level, vdb_hnsw** out);
/* IndexKNNWithEf::knn_with_ef (:616-625) for nq queries: greedy descent from the enter point, search_on_level with
 * max(ef, k) on level 0, the k best by (distance, id). Distances are the cached form (dist_with_cache :351-355). */
int vdb_hnsw_knn(const vdb_dataset* ds, const vdb_hnsw* h, const void* queries, uint32_t nq, uint32_t k, uint32_t ef,
                 uint64_t* ids, float* dist, uint32_t* counts);
int vdb_hnsw_knn_dev(const vdb_dataset* ds, const vdb_hnsw* h, const void* d_queries, uint32_t nq, uint32_t k,
                     uint32_t ef, uint64_t* d_ids, float* d_dist, uint32_t* d_counts, void* stream);

/* Visited sets: the reference's is unbounded (:258-291); here a search keeps it in shared memory up to ef = 896 and in
 * global memory (4 ef 2M slots per search) beyond. A neighbour that cannot be recorded because a set is 7/8 full would
 * cost recall, so it is never dropped silently: vdb_hnsw_build / _append / _knn / _knn_pq fail with VDB_EUNSUPPORTED;
 * after the asynchronous `_dev` searches the count since the last check is read with vdb_hnsw_overflow (must be 0). */
int vdb_hnsw_overflow(const vdb_hnsw* h, uint32_t* count);
/* Instrumentation: rows whose distance the search_on_level loops of this handle have evaluated (builds and searches) since
 * the last reset - each is one dependent gather of a row (dim x sizeof(T) + 4 bytes: SURVEY.md section 8d's HNSW unit). */
int vdb_hnsw_evals(const vdb_hnsw* h, uint64_t* count, int reset);

/* IndexPQ::knn_pq on the graph (:672-697): the walk uses ADC distances of the 4-bit codes, all max(ef, k) results
 * are then re-scored exactly and the k best returned (ResultSet::pq_resort, candidate_pair.rs:102-108). */
int vdb_hnsw_knn_pq(const vdb_dataset* ds, const vdb_hnsw* h, const vdb_pq* pq, const void* queries, uint32_t nq,
                    uint32_t k, uint32_t ef, uint64_t* ids, float* dist, uint32_t* counts);
int vdb_hnsw_knn_pq_dev(const vdb_dataset* ds, const vdb_hnsw* h, const vdb_pq* pq, const void* d_queries, uint32_t nq,
                        uint32_t k, uint32_t ef, uint64_t* d_ids, float* d_dist, uint32_t* d_counts, void* stream);

/* ---- instrumentation ------------------------------------------------------------------------ */
/* Number of kernels this library has launched on the calling process since load. */
uint64_t vdb_launch_count(void);
/* Per-kernel device timing for the roofline report: when enabled, the library brackets its hot
 * kernels with CUDA events on the launching stream. vdb_prof_read synchronises the device, then
 * returns the accumulated milliseconds and launch count of kernel `name` since the last reset
 * (names: "flat_scan", "flat_gemm", "rerank", "merge", "pq_adc", "pq_encode", "ivf_scan",
 * "kmeans_assign", "pq_gemm", "pq_exact", "pq_lut", "pq_train", "hnsw_search", "hnsw_select", "hnsw_arrange", "ivf_pq_scan"). */
int vdb_prof_enable(int on);
int vdb_prof_reset(void);
int vdb_prof_read(const char* name, double* ms, uint64_t* launches);

#ifdef __cplusplus
}
#endif
#endif /* VDB_B200_H */
