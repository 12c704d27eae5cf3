// dataset.cuh — device mirror of a VecSet<T> (reference src/vec_set.rs:15-30) and internal launchers.
#pragma once
#include "common.cuh"

struct vdb_dataset {
    int device = 0;
    void* d_rows = nullptr;   // [cap][pitch] of dtype, pad columns are zero
    bool owned = true;
    uint64_t n = 0, cap = 0;
    uint32_t dim = 0;
    uint32_t pitch = 0;       // row pitch in ELEMENTS; pitch * elem_size is a multiple of 16 bytes
    int dtype = VDB_F32;
    int metric = VDB_L2SQR;
    uint64_t id_base = 0;
    // lazily built side arrays for the tensor-core path (K2); invalidated on mutation
    float* d_lo = nullptr;    // ||x|| (fp32), [n]
    float* d_sqnorm = nullptr;  // L2Sqr: ||x||^2; cosine: 1 / ||x||  (fp32), [n]
    float* d_ex = nullptr;    // operand error norm: L2Sqr ||x - x~||, cosine ||x - x~|| / ||x||  (x~ = what the MMA consumes), [n]
    // the tensor-core operand: kind 1 = an FP16 copy [n][op_pitch] of the rows scaled by the power of two op_scale
    // (d_op); kind 0 = the fp32 rows themselves, truncated to TF32 by the hardware (d_op == nullptr, nothing is copied)
    void* d_op = nullptr;
    int op_kind = 0;
    bool op_owned = false;
    uint32_t op_pitch = 0;    // elements per operand row
    float op_scale = 1.0f;
    void* d_sample = nullptr;  // stratified random sample of the operand rows, [sample_n][op row bytes]
    float* d_sample_sq = nullptr, *d_sample_rn = nullptr, *d_sample_ex = nullptr;  // the sampled rows' scalars
    uint32_t* d_sample_row = nullptr;  // and the local row each of them was taken from
    uint32_t sample_n = 0;
    uint64_t side_n = 0;      // number of rows the side arrays cover
    float mean_norm = 0.f;    // mean ||x|| over a row sample (threshold margin of the tensor path)
    float mean_ex = 0.f;      // mean of d_ex over the same rows
    int flat_path = -1;       // vdb_dataset_set_flat_path: 0 auto, 1 scan, 2 tensor; -1 = the process default
    // row-sharded parent (vdb_init with several devices; multi.cu): the rows live in the shards' own vdb_dataset
    // handles, this handle only carries n / dim / dtype / metric and the worker pool
    struct vdb_sharded_state* sharded = nullptr;
    struct vdb_batcher* batcher = nullptr;   // coalesces concurrent single-query host calls (capi.cu), created on first use
    uint32_t elem_size() const { return dtype == VDB_F32 ? 4u : 1u; }
    size_t pitch_bytes() const { return (size_t)pitch * elem_size(); }
};

namespace vdb {

inline uint32_t vec_elems(int dtype) { return dtype == VDB_F32 ? 4u : 16u; }  // elements per 16-byte load

// ---- query preparation: T[nq][dim] -> f32 tile layout used by the scan kernels --------------
// f32 sets: per query [nit*32] float4, element e of the (zero padded) row in float4 e / 4, component e % 4.
// u8 sets: per query the row's bytes, zero padded to nit * 512 bytes (qstride counts 4-byte words in both cases).
struct QueryTile {
    DevBuf q;        // [nq][qstride] f32 (f32 sets) / [nq][qstride * 4] bytes (u8 sets)
    DevBuf qcache;   // [nq] f32: ||q|| (cosine) / ||q||^2 (l2) in plain f32
    uint32_t qstride = 0;  // floats per query
    uint32_t nvec = 0, nit = 0;
};
QueryTile prepare_queries(const vdb_dataset* ds, const void* d_queries, uint32_t nq, cudaStream_t st,
                          uint32_t* d_zero_word = nullptr);   // d_zero_word: a counter the kernel clears on the way

// ---- Flat exact scan (K1) ---------------------------------------------------------------------
// keys out: [nq][k] ascending, KEY_NONE padded. If `d_members` != nullptr the scan visits only the
// rows listed per query (IVF probe scan): see ivf.cu.
// Decoded results of a search (the SoA arrays of the C ABI). flat_scan_keys writes them itself and returns true when the
// whole batch is ONE scan launch (1-8 queries): the last CTA to finish merges the per-CTA lists and decodes, so a
// single-query call is two launches (query tile + scan) instead of four. Otherwise it returns false: decode d_keys.
struct ScanOut {
    uint64_t* ids = nullptr;
    float* dist = nullptr;
    uint32_t* counts = nullptr;
};
// True when the fused top-k of the scan holds k (its shared-memory segments and, when the per-CTA lists are merged, the
// merge's); otherwise flat_scan_keys takes the large-k path (emit every key, then select + sort in global memory).
bool fused_topk_fits(const vdb_dataset* ds, uint32_t nq, uint32_t k);
bool flat_scan_keys(const vdb_dataset* ds, const void* d_queries, uint32_t nq, uint32_t k, uint64_t* d_keys, cudaStream_t st,
                    const ScanOut* out = nullptr);
// decode [nq][k] keys into the SoA result arrays
void decode_keys(const uint64_t* d_keys, uint32_t nq, uint32_t k, uint64_t* d_ids, float* d_dist,
                 uint32_t* d_counts, cudaStream_t st);

// ---- Flat tensor-core path (K2) ----------------------------------------------------------------
bool flat_gemm_supported(const vdb_dataset* ds, uint32_t nq, uint32_t k);
void flat_gemm_keys(const vdb_dataset* ds, const void* d_queries, uint32_t nq, uint32_t k,
                    uint64_t* d_keys, cudaStream_t st);

// exact distances of listed rows: out[j] for pairs (query qidx[j], local row rid[j]); difference
// form / 3-dot cosine (mode 0) or the cached form of hnsw_index.rs:351-358 (mode 1)
void pair_distances(const vdb_dataset* ds, const float* d_qtile, uint32_t qstride, const float* d_qcache,
                    const float* d_rowcache, const uint32_t* d_qidx, const uint32_t* d_rid, uint64_t npairs,
                    int mode, float* d_out, cudaStream_t st);

void drop_side_arrays(vdb_dataset* ds);   // flat_gemm.cu: frees the lazily built side arrays (called on mutation)
extern std::atomic<bool> g_batching;
extern std::atomic<int> g_flat_path;   // process default of the Flat path selection (vdb_flat_set_path)

}  // namespace vdb
