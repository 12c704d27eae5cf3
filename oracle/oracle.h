/*
 * oracle.h — C ABI of the CPU oracle (TEST INFRASTRUCTURE, not product code).
 *
 * The oracle is a CPU restatement of the search hot path of
 * pku-lab-1806-llm/lab-1806-vec-db v0.8.1 (pure Rust). It exists only so that
 * tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
 * legs can check or time the reference's algorithm. Nothing under
 * lab_1806_vec_db_b200/ links, imports or calls it.
 *
 * PINNING STATUS (see DESIGN.md "Oracle"): the Rust reference cannot be built in
 * this image (no cargo/rustc), so the oracle is pinned against
 *   - every RNG-free known-answer test the reference holds for this path
 *     (distance/mod.rs:138-150, pq_table.rs:312-322, pq_table.rs:324-372,
 *      flat_index.rs:157-167, ivf_index.rs:222-232), and
 *   - an independent numpy float32 emulation of the sequential reductions on the
 *     reference's own fixtures (tests/golden/, SHA-256 anchors of SURVEY.md §8c).
 * RNG-dependent artefacts (k-means++ draws, random_sample) are "parity unpinned":
 * the reference uses rand 0.8.5 StdRng (ChaCha12), which is not restated here.
 *
 * Arithmetic contract: every f32 reduction is left-to-right with a separately
 * rounded multiply and add (rustc never contracts to FMA, never reassociates).
 * Build with -O3 -ffp-contract=off and without -ffast-math (oracle/Makefile).
 */
#ifndef VDB_ORACLE_H
#define VDB_ORACLE_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum { ORC_L2SQR = 0, ORC_COSINE = 1 };      /* DistanceAlgorithm, distance/mod.rs:18-28 */
enum { ORC_F32 = 0, ORC_U8 = 1 };            /* Scalar, scalar.rs:117-119 */

/* distance/mod.rs:41-95 */
float orc_dot(const void* a, const void* b, size_t dim, int dtype);
float orc_l2_sqr(const void* a, const void* b, size_t dim, int dtype);
float orc_vec_norm(const void* a, size_t dim, int dtype);
float orc_distance(const void* a, const void* b, size_t dim, int dtype, int metric);
float orc_distance_cached(const void* a, const void* b, size_t dim, int dtype, int metric,
                          float cache_a, float cache_b);
float orc_dist_cache(const void* a, size_t dim, int dtype, int metric);

/* flat_index.rs:48-57 (+ candidate_pair.rs:43-82). ids: [nq,k] u64, dist: [nq,k] f32,
 * counts: [nq] u32 = number of valid results per query (min(k, n)). nthreads<=1 → serial,
 * otherwise a thread pool over queries (bench.rs:414-418, gen_gnd.rs:65-68). */
int orc_flat_knn(const void* base, size_t n, size_t dim, int dtype, int metric,
                 const void* queries, size_t nq, size_t k,
                 uint64_t* ids, float* dist, uint32_t* counts, int nthreads);

/* pq_table.rs:38-53. out: [m,2] (start,end). */
int orc_pq_groups(size_t dim, size_t m, uint64_t* out);

/* k_means.rs:40-57,166-170: argmin over centroids, ties → lowest id. centroids: [k, sel_hi-sel_lo]. */
uint64_t orc_find_nearest(const void* v, const void* centroids, size_t k, size_t sel_lo,
                          size_t sel_hi, int dtype, int metric);
/* k_means.rs:174-191. out: [min(n_probes,k)] centroid ids nearest first. returns count. */
size_t orc_find_n_nearest(const void* v, const void* centroids, size_t k, size_t dim, int dtype,
                          int metric, size_t n_probes, uint64_t* out);
/* k_means.rs:117-120 / ivf_index.rs:89-93: assignment of n rows (row stride = dim) */
int orc_kmeans_assign(const void* rows, size_t n, size_t dim, int dtype, int metric,
                      const void* centroids, size_t k, size_t sel_lo, size_t sel_hi,
                      uint32_t* out, int nthreads);
/* k_means.rs:108-161: Lloyd iterations from given initial centroids [k, sel_hi-sel_lo] (in/out).
 * Returns the number of iterations executed. */
int orc_kmeans_lloyd(const void* rows, size_t n, size_t dim, int dtype, int metric,
                     void* centroids, size_t k, size_t sel_lo, size_t sel_hi,
                     size_t max_iter, float tol);
/* k_means.rs:61-87 with the oracle's own RNG (splitmix64; NOT the reference's ChaCha12 stream):
 * writes [k, sel_hi-sel_lo] initial centroids. */
int orc_kmeans_pp_init(const void* rows, size_t n, size_t dim, int dtype, int metric,
                       size_t k, size_t sel_lo, size_t sel_hi, uint64_t seed, void* centroids);
/* k_means.rs:75-77: the k-means++ weight update w[i] = min(w[i], d(c, rows[i][sel_lo:sel_hi])) for i < n, c of
 * length sel_hi-sel_lo, the rows split across nthreads. kmeans_pp uses this same update. */
int orc_kmeans_pp_weights(const void* rows, size_t n, size_t dim, int dtype, int metric, const void* c,
                          size_t sel_lo, size_t sel_hi, float* w, int nthreads);

/* pq_table.rs:66-91,178-181. codebooks: m groups concatenated, group g = [kc, len_g] of dtype,
 * kc = 1<<n_bits. codes out: [n, encoded_dim]. */
int orc_pq_encode(const void* rows, size_t n, size_t dim, int dtype, int metric,
                  const void* codebooks, size_t m, size_t n_bits, uint8_t* codes, int nthreads);
/* pq_table.rs:195-224. lut: [m*kc] f32; *qcache = 0 (L2) or ||q|| (cosine). */
int orc_pq_lookup(const void* q, size_t dim, int dtype, int metric, const void* codebooks,
                  size_t m, size_t n_bits, float* lut, float* qcache);
/* pq_table.rs:165-170. out: [m*kc] (0 for L2, ||c||^2 for cosine) */
int orc_pq_dist_cache(size_t dim, int dtype, int metric, const void* codebooks, size_t m,
                      size_t n_bits, float* out);
/* pq_table.rs:239-301 */
float orc_pq_adc(const uint8_t* code, size_t m, size_t n_bits, int metric, const float* lut,
                 const float* dist_cache, float qcache);
/* flat_index.rs:84-104 + candidate_pair.rs:102-108 */
int orc_flat_knn_pq(const void* base, size_t n, size_t dim, int dtype, int metric,
                    const uint8_t* codes, const void* codebooks, size_t m, size_t n_bits,
                    const void* queries, size_t nq, size_t k, size_t ef,
                    uint64_t* ids, float* dist, uint32_t* counts, int nthreads);
/* same scan, but returns the ADC candidate list (size max(ef,k)) before the rerank */
int orc_flat_adc_topk(size_t n, int metric, const uint8_t* codes, size_t m, size_t n_bits,
                      const float* lut, const float* dist_cache, float qcache, size_t kk,
                      uint64_t* ids, float* dist, uint32_t* count);

/* ivf_index.rs:89-96: lists from assignment. offsets: [nlist+1], members: [n] (ascending in a list) */
int orc_ivf_lists(const uint32_t* assign, size_t n, size_t nlist, uint64_t* offsets, uint64_t* members);
/* ivf_index.rs:143-154 */
int orc_ivf_knn(const void* base, size_t n, size_t dim, int dtype, int metric,
                const void* centroids, size_t nlist, const uint64_t* offsets, const uint64_t* members,
                const void* queries, size_t nq, size_t k, size_t n_probes,
                uint64_t* ids, float* dist, uint32_t* counts, int nthreads);

/* hnsw_index.rs:351-358 batched: out[j] = cached-form distance between query and rows[cand[j]] */
int orc_gather_dist(const void* base, size_t dim, int dtype, int metric, const float* row_cache,
                    const void* query, float query_cache, const uint64_t* cand, size_t ncand,
                    float* out);

/* candidate_pair.rs:127-140 */
/* HNSW (hnsw_index.rs), single-thread restatement: sequential add of every row with the given levels, knn_with_ef */
void* orc_hnsw_build(const void* rows, size_t n, size_t dim, int dtype, int metric, size_t m, size_t ef_construction,
                     const uint32_t* levels);
/* the same object over a graph built elsewhere (layouts of vdb_hnsw_links0 / vdb_hnsw_upper) */
void* orc_hnsw_from_graph(const void* rows, size_t n, size_t dim, int dtype, int metric, size_t m, size_t ef_construction,
                          const uint32_t* levels, const uint32_t* links0, const uint32_t* len0, const uint32_t* ulinks,
                          const uint32_t* ulen, long enter_point, long enter_level);
/* the batch pipeline of the device build (hnsw.cu hnsw_insert_range): a build of rows [0, n0), then an append of
 * rows [n0, n) onto it; n0 = 0 is one build. max_batch = 1 gives orc_hnsw_build's graph. */
void* orc_hnsw_build_batched(const void* rows, size_t n, size_t dim, int dtype, int metric, size_t m, size_t ef_construction,
                             const uint32_t* levels, size_t max_batch, size_t n0);
/* Tie events: adds to a full ResultSet with a distance equal to its last entry's (candidate_pair.rs:61-74 keeps the
 * older entry; a k-smallest selection by (distance, id) may not). Of a whole build: */
uint64_t orc_hnsw_build_ties(const void* handle, int dtype);
int orc_hnsw_enter(const void* handle, int dtype, long* enter_point, long* enter_level);
/* ties (may be NULL): [nq] tie events of each query's walk (and, for knn_pq, of its pq_resort) */
int orc_hnsw_knn(const void* handle, int dtype, const void* queries, size_t nq, size_t k, size_t ef, uint64_t* ids,
                 float* dists, uint32_t* counts, int nthreads, uint32_t* ties);
int orc_hnsw_knn_pq(const void* handle, int dtype, const void* queries, size_t nq, size_t k, size_t ef, const uint8_t* codes,
                    const void* codebooks, size_t m, size_t n_bits, uint64_t* ids, float* dists, uint32_t* counts, int nthreads,
                    uint32_t* ties);
int orc_hnsw_links0(const void* handle, int dtype, uint32_t* links0, uint32_t* len0);
int orc_hnsw_upper(const void* handle, int dtype, uint32_t* ulinks, uint32_t* ulen);
void orc_hnsw_free(void* handle, int dtype);
float orc_recall(const uint64_t* gnd, size_t n_gnd, const uint64_t* pred, size_t n_pred);

#ifdef __cplusplus
}
#endif
#endif
