// kmeans.cu — K4/K5: k-means assignment and Lloyd update with the reference's exact arithmetic.
//
// Replaces (reference paths):
//   find_nearest_base / KMeans::find_nearest     src/distance/k_means.rs:40-57, 166-170
//   Lloyd assignment + update + convergence      src/distance/k_means.rs:108-161
//   IVF list assignment                          src/index_algorithm/ivf_index.rs:89-96
//   k-means++ weight update                      src/distance/k_means.rs:75-77
//
// Index results (assignments, lists) must be bit-exact, so every (row, centroid) distance is one
// thread's strictly sequential f32 chain with separately rounded multiply and add (__fmul_rn /
// __fadd_rn are never contracted into FMA) — the same arithmetic rustc emits for the reference.
// Parallelism comes from the (row, centroid) pairs, not from splitting a sum:
//   lane = centroid of a 32-wide chunk held TRANSPOSED in shared memory ([d][32], conflict free),
//   each warp stages its rows in shared memory with coalesced loads and broadcasts them.
// The centroid update sums members in ascending row order (stable lists built by ballot compaction).
#include "index.cuh"
#include "topk.cuh"

namespace vdb {

constexpr int ASG_THREADS = 256;
constexpr int ASG_WARPS = ASG_THREADS / 32;

template <typename T> __device__ __forceinline__ float to_f32(T v) { return (float)v; }
__device__ __forceinline__ float from_f32_as(float v, float*) { return v; }
__device__ __forceinline__ uint8_t from_f32_as(float v, uint8_t*) {
    // Rust `as u8`: truncate toward zero, saturate, NaN -> 0 (reference src/scalar.rs:22-37)
    if (!(v == v)) return 0;
    if (v <= 0.f) return 0;
    if (v >= 255.f) return 255;
    return (uint8_t)__float2uint_rz(v);
}

struct AssignParams {
    const void* rows;
    uint64_t n;
    uint64_t pitch;        // elements between rows
    uint32_t lo, d;        // selected dimension range [lo, lo+d)
    const void* cent;      // [k][d] all centroids (dataset dtype)
    uint32_t k;
    uint32_t c_base, kc;   // this launch handles centroids [c_base, c_base+kc), kc <= cpw
    uint32_t cpw;          // lanes per row (power of two <= 32)
    uint32_t rps;          // rows per warp step (<= 32 / cpw; fewer when shared memory is tight)
    uint64_t* best;        // [n] running best key (in/out)
    uint32_t* out_assign;  // optional: written when non-null
    float* all_dist;       // optional [n][k]: every exact distance
    uint32_t iters;        // row-steps per warp
};

template <typename T, int METRIC>
__global__ void __launch_bounds__(ASG_THREADS) assign_exact_kernel(const AssignParams p) {
    extern __shared__ __align__(16) uint8_t smem[];
    const uint32_t cpw = p.cpw, rps = p.rps;
    float* centT = reinterpret_cast<float*>(smem);            // [d][cpw]
    float* cnorm = centT + (size_t)p.d * cpw;                  // [cpw]  ||c|| (cosine)
    float* rowbuf = cnorm + 32;                                // [ASG_WARPS][rps][d]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const T* cent = (const T*)p.cent;
    for (uint32_t i = threadIdx.x; i < p.d * cpw; i += blockDim.x) {
        const uint32_t j = i / cpw, c = i - j * cpw;
        centT[i] = c < p.kc ? to_f32(cent[(size_t)(p.c_base + c) * p.d + j]) : 0.f;
    }
    __syncthreads();
    if (METRIC == VDB_COSINE && threadIdx.x < cpw) {
        float s = 0.f;
        for (uint32_t j = 0; j < p.d; ++j) {
            const float c = centT[(size_t)j * cpw + threadIdx.x];
            s = __fadd_rn(s, __fmul_rn(c, c));
        }
        cnorm[threadIdx.x] = sqrtf(s);
    }
    __syncthreads();

    float* myrows = rowbuf + (size_t)warp * rps * p.d;
    const uint32_t sub = lane / cpw, ci = lane % cpw;
    const T* rows = (const T*)p.rows;
    const uint64_t total_warps = (uint64_t)gridDim.x * ASG_WARPS;
    uint64_t step = (uint64_t)blockIdx.x * ASG_WARPS + warp;
    for (uint32_t it = 0; it < p.iters; ++it, step += total_warps) {
        const uint64_t row0 = step * rps;
        __syncwarp();
        for (uint32_t i = lane; i < rps * p.d; i += 32) {
            const uint32_t r = i / p.d, j = i - r * p.d;
            const uint64_t row = row0 + r;
            myrows[i] = row < p.n ? to_f32(rows[row * p.pitch + p.lo + j]) : 0.f;
        }
        __syncwarp();
        const float* x = myrows + (size_t)(sub < rps ? sub : 0) * p.d;
        float s = 0.f, svv = 0.f;
        for (uint32_t j = 0; j < p.d; ++j) {
            const float xv = x[j];
            const float cv = centT[(size_t)j * cpw + ci];
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
            const float den = fmaxf(__fmul_rn(sqrtf(svv), cnorm[ci]), 1e-10f);
            dist = __fsub_rn(1.0f, __fdiv_rn(s, den));
        }
        const uint64_t row = row0 + sub;
        const bool valid = row < p.n && ci < p.kc && sub < rps;
        if (valid && p.all_dist) p.all_dist[row * p.k + p.c_base + ci] = dist;
        unsigned long long key = valid ? make_key(dist, p.c_base + ci) : KEY_NONE;
        for (uint32_t o = cpw >> 1; o > 0; o >>= 1) {
            const unsigned long long other = __shfl_xor_sync(0xffffffffu, key, o);
            key = other < key ? other : key;
        }
        if (ci == 0 && row < p.n && sub < rps) {
            const uint64_t prev = p.best[row];
            const uint64_t b = key < prev ? key : prev;
            p.best[row] = b;
            if (p.out_assign) p.out_assign[row] = key_id(b);
        }
    }
}

constexpr size_t ASG_SMEM_MAX = 200 * 1024;
static size_t assign_smem(uint32_t d, uint32_t cpw, uint32_t rps) {
    return ((size_t)d * cpw + 32 + (size_t)ASG_WARPS * rps * d) * 4;
}

// rows: device pointer to the first row (dataset dtype), pitch in elements
void kmeans_assign_exact(const void* d_rows, uint64_t n, uint64_t pitch, int dtype, int metric, uint32_t lo,
                         uint32_t d, const void* d_cent, uint32_t k, uint64_t* d_best, uint32_t* d_assign,
                         float* d_all_dist, cudaStream_t st) {
    VDB_REQUIRE(k > 0, "The number of centroids should be greater than 0.");
    VDB_REQUIRE(d > 0, "empty dimension range");
    if (n == 0) return;
    // lanes = (rows per warp step) x (centroid chunk); pick the combination with the most busy lanes whose
    // transposed centroid chunk + row staging fit in shared memory (ties -> wider centroid chunk)
    uint32_t cpw = 0, rps = 0;
    for (uint32_t c = std::min(32u, next_pow2(k)); c >= 1; c >>= 1)
        for (uint32_t r = 32 / c; r >= 1; r >>= 1)
            if (assign_smem(d, c, r) <= ASG_SMEM_MAX && c * r > cpw * rps) cpw = c, rps = r;
    VDB_REQUIRE(cpw > 0, "k-means assignment: dimension range %u too large for shared memory", d);
    const size_t smem = assign_smem(d, cpw, rps);
    VDB_CUDA(cudaMemsetAsync(d_best, 0xff, n * 8, st));
    AssignParams p{};
    p.rows = d_rows;
    p.n = n;
    p.pitch = pitch;
    p.lo = lo;
    p.d = d;
    p.cent = d_cent;
    p.k = k;
    p.cpw = cpw;
    p.rps = rps;
    p.best = d_best;
    p.all_dist = d_all_dist;
    const uint64_t steps = ceil_div<uint64_t>(n, rps);
    const int occ = std::max<int>(1, (int)(ASG_SMEM_MAX / std::max<size_t>(smem, 16 * 1024)));
    const uint32_t grid = (uint32_t)std::max<uint64_t>(
        1, std::min<uint64_t>((uint64_t)sm_count() * std::min(occ, 8), ceil_div<uint64_t>(steps, ASG_WARPS)));
    p.iters = (uint32_t)ceil_div<uint64_t>(steps, (uint64_t)grid * ASG_WARPS);
    auto launch = [&](auto kern) {
        if (smem > 48 * 1024)
            VDB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ASG_SMEM_MAX));
        for (uint32_t c0 = 0; c0 < k; c0 += cpw) {
            p.c_base = c0;
            p.kc = std::min(cpw, k - c0);
            p.out_assign = (c0 + cpw >= k) ? d_assign : nullptr;
            ProfScope prof("kmeans_assign", st);
            kern<<<grid, ASG_THREADS, smem, st>>>(p);
            VDB_LAUNCHED();
        }
    };
    if (dtype == VDB_F32) {
        if (metric == VDB_L2SQR) launch(assign_exact_kernel<float, VDB_L2SQR>);
        else launch(assign_exact_kernel<float, VDB_COSINE>);
    } else {
        if (metric == VDB_L2SQR) launch(assign_exact_kernel<uint8_t, VDB_L2SQR>);
        else launch(assign_exact_kernel<uint8_t, VDB_COSINE>);
    }
}

// ---- stable member lists (ascending row order inside every list) ---------------------------------
__global__ void hist_kernel(const uint32_t* __restrict__ assign, uint64_t n, uint32_t k, uint32_t* __restrict__ counts) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t c = assign[i];
        if (c < k) atomicAdd(&counts[c], 1u);
    }
}
__global__ void prefix_kernel(const uint32_t* __restrict__ counts, uint32_t k, uint64_t* __restrict__ offsets) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        uint64_t s = 0;
        for (uint32_t c = 0; c < k; ++c) {
            offsets[c] = s;
            s += counts[c];
        }
        offsets[k] = s;
    }
}
// one warp per list: scans assign[] in order, appends matching rows with ballot compaction
__global__ void fill_lists_kernel(const uint32_t* __restrict__ assign, uint64_t n, uint32_t k,
                                  const uint64_t* __restrict__ offsets, uint32_t* __restrict__ members) {
    const uint32_t c = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (c >= k) return;
    uint64_t w = offsets[c];
    for (uint64_t i0 = 0; i0 < n; i0 += 32) {
        const uint64_t i = i0 + lane;
        const bool hit = i < n && assign[i] == c;
        const uint32_t m = __ballot_sync(0xffffffffu, hit);
        if (hit) members[w + __popc(m & ((1u << lane) - 1))] = (uint32_t)i;
        w += __popc(m);
    }
}

void build_lists(const uint32_t* d_assign, uint64_t n, uint32_t k, uint64_t* d_offsets, uint32_t* d_members,
                 cudaStream_t st) {
    DevBuf counts((size_t)k * 4, st);
    VDB_CUDA(cudaMemsetAsync(counts.p, 0, (size_t)k * 4, st));
    if (n) {
        hist_kernel<<<(uint32_t)std::min<uint64_t>(ceil_div<uint64_t>(n, 256), 1024), 256, 0, st>>>(
            d_assign, n, k, counts.as<uint32_t>());
        VDB_LAUNCHED();
    }
    prefix_kernel<<<1, 32, 0, st>>>(counts.as<uint32_t>(), k, d_offsets);
    VDB_LAUNCHED();
    if (n) {
        fill_lists_kernel<<<ceil_div<uint32_t>(k * 32, 256), 256, 0, st>>>(d_assign, n, k, d_offsets, d_members);
        VDB_LAUNCHED();
    }
}

// ---- Lloyd update: per (centroid, dim) sequential f32 sum over members in ascending order -----------
template <typename T>
__global__ void update_kernel(const T* __restrict__ rows, uint64_t pitch, uint32_t lo, uint32_t d,
                              const uint64_t* __restrict__ offsets, const uint32_t* __restrict__ members,
                              const T* __restrict__ cent_old, T* __restrict__ cent_new) {
    const uint32_t c = blockIdx.x;
    const uint64_t b = offsets[c], e = offsets[c + 1];
    for (uint32_t j = threadIdx.x; j < d; j += blockDim.x) {
        float s;
        if (b == e) {
            s = to_f32(cent_old[(size_t)c * d + j]);  // empty cluster keeps its centroid (k_means.rs:131-137)
        } else {
            s = 0.f;
            for (uint64_t t = b; t < e; ++t) s = __fadd_rn(s, to_f32(rows[(uint64_t)members[t] * pitch + lo + j]));
            s = __fdiv_rn(s, (float)(e - b));
        }
        cent_new[(size_t)c * d + j] = from_f32_as(s, (T*)nullptr);
    }
}
// max over centroids of the sequential L2Sqr(old, new); f32::max fold from -inf (k_means.rs:150-154)
template <typename T>
__global__ void shift_kernel(const T* __restrict__ a, const T* __restrict__ b, uint32_t k, uint32_t d,
                             float* __restrict__ per_c, float* __restrict__ out) {
    const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c < k) {
        float s = 0.f;
        for (uint32_t j = 0; j < d; ++j) {
            const float df = __fsub_rn(to_f32(a[(size_t)c * d + j]), to_f32(b[(size_t)c * d + j]));
            s = __fadd_rn(s, __fmul_rn(df, df));
        }
        per_c[c] = s;
    }
    __threadfence();
    __syncthreads();
    // last block reduces (k is small); a second tiny launch would do as well
    __shared__ bool last;
    __shared__ uint32_t ticket;
    if (threadIdx.x == 0) {
        ticket = atomicAdd(reinterpret_cast<uint32_t*>(out + 1), 1u);
        last = ticket == gridDim.x - 1;
    }
    __syncthreads();
    if (last && threadIdx.x == 0) {
        float m = __uint_as_float(0xff800000u);  // -inf
        for (uint32_t i = 0; i < k; ++i) m = fmaxf(m, ((volatile float*)per_c)[i]);
        out[0] = m;
    }
}

template <typename T>
static uint32_t lloyd_t(const void* d_rows, uint64_t n, uint64_t pitch, int dtype, int metric, uint32_t lo,
                        uint32_t d, T* d_cent, uint32_t k, uint32_t max_iter, float tol, cudaStream_t st) {
    DevBuf best(n * 8, st), assign(n * 4, st), offsets((size_t)(k + 1) * 8, st), members(n * 4, st);
    DevBuf cent_new((size_t)k * d * sizeof(T), st), per_c((size_t)k * 4, st), shift(8, st);
    uint32_t iters = 0;
    for (uint32_t it = 0; it < max_iter; ++it) {
        ++iters;
        kmeans_assign_exact(d_rows, n, pitch, dtype, metric, lo, d, d_cent, k, best.as<uint64_t>(),
                            assign.as<uint32_t>(), nullptr, st);
        build_lists(assign.as<uint32_t>(), n, k, offsets.as<uint64_t>(), members.as<uint32_t>(), st);
        update_kernel<T><<<k, (uint32_t)std::min<uint32_t>(256, round_up(d, 32u)), 0, st>>>(
            (const T*)d_rows, pitch, lo, d, offsets.as<uint64_t>(), members.as<uint32_t>(), d_cent,
            cent_new.as<T>());
        VDB_LAUNCHED();
        VDB_CUDA(cudaMemsetAsync(shift.p, 0, 8, st));
        shift_kernel<T><<<ceil_div<uint32_t>(k, 128), 128, 0, st>>>(d_cent, cent_new.as<T>(), k, d,
                                                                   per_c.as<float>(), shift.as<float>());
        VDB_LAUNCHED();
        VDB_CUDA(cudaMemcpyAsync(d_cent, cent_new.p, (size_t)k * d * sizeof(T), cudaMemcpyDeviceToDevice, st));
        float max_diff = 0.f;
        VDB_CUDA(cudaMemcpyAsync(&max_diff, shift.p, 4, cudaMemcpyDeviceToHost, st));
        VDB_CUDA(cudaStreamSynchronize(st));
        if (max_diff < tol) break;
    }
    return iters;
}

uint32_t kmeans_lloyd(const void* d_rows, uint64_t n, uint64_t pitch, int dtype, int metric, uint32_t lo,
                      uint32_t d, void* d_cent, uint32_t k, uint32_t max_iter, float tol, cudaStream_t st) {
    VDB_REQUIRE(k > 0, "The number of clusters should be greater than 0.");
    if (dtype == VDB_F32)
        return lloyd_t<float>(d_rows, n, pitch, dtype, metric, lo, d, (float*)d_cent, k, max_iter, tol, st);
    return lloyd_t<uint8_t>(d_rows, n, pitch, dtype, metric, lo, d, (uint8_t*)d_cent, k, max_iter, tol, st);
}

// ---- k-means++ weights: w[i] = min(w[i], d(c, v_i)) ----------------------------------------------------
// d(c, v_i) must be the reference's sequential f32 chain (k_means.rs:76): every weight moves a WeightedIndex boundary, so
// a last-bit difference can change a pick. The assignment kernel with the single centroid c computes exactly that chain
// (rows staged through shared memory with coalesced loads); its all_dist output is folded into w here.
__global__ void fmin_into_kernel(const float* __restrict__ d, uint64_t n, float* __restrict__ w) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
        w[i] = fminf(w[i], d[i]);   // f32::min: a NaN operand yields the other one
}

void kmeans_pp_weights(const void* d_rows, uint64_t n, uint64_t pitch, int dtype, int metric, uint32_t lo,
                       uint32_t d, const void* d_c, float* d_w, cudaStream_t st) {
    if (n == 0) return;
    DevBuf best(n * 8, st), dist(n * 4, st);
    kmeans_assign_exact(d_rows, n, pitch, dtype, metric, lo, d, d_c, 1, best.as<uint64_t>(), nullptr, dist.as<float>(), st);
    fmin_into_kernel<<<(uint32_t)std::min<uint64_t>(ceil_div<uint64_t>(n, 256), (uint64_t)sm_count() * 8), 256, 0, st>>>(
        dist.as<float>(), n, d_w);
    VDB_LAUNCHED();
}

// ---- batched PQ training: every group's k-means (k-means++ init + Lloyd) in ONE launch --------------------------------
// PQTable::from_vec_set trains one KMeans per group on the same sample (pq_table.rs:154-172), serially. A group is tiny
// (C4: 10 000 rows x 4 dims x 16 centroids), so the per-group path is bound by launches and host round trips
// (~100 per group). Here one CTA owns one group and runs the whole k_means_init (k_means.rs:61-87) and Lloyd loop
// (:108-161) with the reference's arithmetic: sequential f32 distances, ties to the lowest centroid id, member sums in
// ascending row order, empty clusters keep their centroid, max squared shift < tol. Given the same initial centroids
// the result is bit-identical to vdb_kmeans_train (tested).
struct PqTrainParams {
    const void* rows;
    uint64_t n, pitch;
    uint32_t m, kc, max_iter;
    float tol;
    const uint32_t* groups;   // [m][3] (lo, len, codebook element offset)
    const double* uniforms;   // [m][2 kc - 1] or nullptr when init != nullptr
    const void* init;         // optional initial codebooks (same layout as out)
    void* out;                // codebooks, groups concatenated, [kc][len] each
    uint32_t* iters;          // [m]
    float* w;                 // scratch [m][n]
    uint8_t* assign;          // scratch [m][n]
};

template <typename T, int METRIC>
__device__ __forceinline__ float seq_dist(const T* __restrict__ x, const float* __restrict__ c, uint32_t len, float cnorm) {
    float s = 0.f, svv = 0.f;
    for (uint32_t j = 0; j < len; ++j) {
        const float xv = to_f32(x[j]), cv = c[j];
        if (METRIC == VDB_L2SQR) {
            const float df = __fsub_rn(xv, cv);
            s = __fadd_rn(s, __fmul_rn(df, df));
        } else {
            s = __fadd_rn(s, __fmul_rn(xv, cv));
            svv = __fadd_rn(svv, __fmul_rn(xv, xv));
        }
    }
    if (METRIC == VDB_L2SQR) return s;
    return __fsub_rn(1.0f, __fdiv_rn(s, fmaxf(__fmul_rn(sqrtf(svv), cnorm), 1e-10f)));
}

template <typename T, int METRIC>
__global__ void __launch_bounds__(256) pq_train_kernel(const PqTrainParams p) {
    extern __shared__ __align__(16) uint8_t smem[];
    const uint32_t g = blockIdx.x;
    const uint32_t lo = p.groups[3 * g], len = p.groups[3 * g + 1], off = p.groups[3 * g + 2];
    const uint32_t kc = p.kc;
    float* cent = reinterpret_cast<float*>(smem);   // [kc][len]  current centroids (T-valued)
    float* cnew = cent + (size_t)kc * len;           // [kc][len]
    float* cnorm = cnew + (size_t)kc * len;          // [kc]
    float* perc = cnorm + kc;                        // [kc]
    __shared__ double tsum[256];
    __shared__ int s_ok, s_pick_thread, s_conv;
    __shared__ unsigned long long s_pick;
    __shared__ double s_base, s_target;
    const T* rows = reinterpret_cast<const T*>(p.rows);
    T* out = reinterpret_cast<T*>(p.out) + off;
    const uint64_t n = p.n;
    float* w = p.w + (size_t)g * n;
    uint8_t* asg = p.assign + (size_t)g * n;
    const uint32_t tid = threadIdx.x;
    auto sub = [&](uint64_t i) { return rows + i * p.pitch + lo; };
    auto set_cnorm = [&]() {
        if (METRIC == VDB_COSINE)
            for (uint32_t c = tid; c < kc; c += blockDim.x) {
                float s = 0.f;
                for (uint32_t j = 0; j < len; ++j) s = __fadd_rn(s, __fmul_rn(cent[c * len + j], cent[c * len + j]));
                cnorm[c] = sqrtf(s);
            }
    };
    if (p.init) {
        const T* ini = reinterpret_cast<const T*>(p.init) + off;
        for (uint32_t e = tid; e < kc * len; e += blockDim.x) cent[e] = to_f32(ini[e]);
        __syncthreads();
    } else {
        // ---- k_means_init: first = floor(u0 n); then weighted picks with the eager uniform fallback ----
        const double* u = p.uniforms + (size_t)g * (2 * kc - 1);
        const uint64_t chunk = (n + blockDim.x - 1) / blockDim.x;
        const uint64_t i0 = min(n, (uint64_t)tid * chunk), i1 = min(n, i0 + chunk);
        for (uint64_t i = i0; i < i1; ++i) w[i] = __uint_as_float(0x7f800000u);
        uint64_t cur = (uint64_t)fmin((double)(n - 1), floor(u[0] * (double)n));
        for (uint32_t r = 0; r < kc; ++r) {
            __syncthreads();
            for (uint32_t j = tid; j < len; j += blockDim.x) cent[r * len + j] = to_f32(sub(cur)[j]);
            __syncthreads();
            if (r + 1 == kc) break;
            if (METRIC == VDB_COSINE && tid == 0) {
                float s = 0.f;
                for (uint32_t j = 0; j < len; ++j) s = __fadd_rn(s, __fmul_rn(cent[r * len + j], cent[r * len + j]));
                cnorm[r] = sqrtf(s);
            }
            if (tid == 0) s_ok = 1;
            __syncthreads();
            double acc = 0.0;
            bool ok = true;
            for (uint64_t i = i0; i < i1; ++i) {
                const float d = seq_dist<T, METRIC>(sub(i), cent + r * len, len, METRIC == VDB_COSINE ? cnorm[r] : 0.f);
                const float x = fminf(w[i], d);
                w[i] = x;
                if (!(x >= 0.f) || isinf(x)) ok = false;
                acc += (double)x;
            }
            tsum[tid] = acc;
            if (!ok) s_ok = 0;
            __syncthreads();
            if (tid == 0) {
                double total = 0.0;
                for (uint32_t t = 0; t < blockDim.x; ++t) total += tsum[t];
                s_pick = (unsigned long long)fmin((double)(n - 1), floor(u[2 * (r + 1)] * (double)n));  // fallback
                s_pick_thread = -1;
                if (s_ok && total > 0.0) {
                    const double target = u[2 * (r + 1) - 1] * total;
                    double pre = 0.0;
                    s_pick = n - 1;
                    for (uint32_t t = 0; t < blockDim.x; ++t) {
                        if (target < pre + tsum[t]) {
                            s_pick_thread = (int)t;
                            s_base = pre;
                            s_target = target;
                            break;
                        }
                        pre += tsum[t];
                    }
                }
            }
            __syncthreads();
            if ((int)tid == s_pick_thread) {
                double a = s_base;
                unsigned long long pick = i1 ? i1 - 1 : 0;
                for (uint64_t i = i0; i < i1; ++i) {
                    a += (double)w[i];
                    if (s_target < a) {
                        pick = i;
                        break;
                    }
                }
                s_pick = pick;
            }
            __syncthreads();
            cur = s_pick;
        }
        __syncthreads();
    }
    // ---- Lloyd ----
    uint32_t iters = 0;
    for (uint32_t it = 0; it < p.max_iter; ++it) {
        ++iters;
        set_cnorm();
        __syncthreads();
        for (uint64_t i = tid; i < n; i += blockDim.x) {
            const T* x = sub(i);
            unsigned long long best = KEY_NONE;
            for (uint32_t c = 0; c < kc; ++c) {
                const unsigned long long key = make_key(seq_dist<T, METRIC>(x, cent + c * len, len, METRIC == VDB_COSINE ? cnorm[c] : 0.f), c);
                best = key < best ? key : best;
            }
            asg[i] = (uint8_t)key_id(best);
        }
        __syncthreads();
        for (uint32_t slot = tid; slot < kc * len; slot += blockDim.x) {
            const uint32_t c = slot / len, j = slot - c * len;
            float s = 0.f;
            uint32_t cnt = 0;
            for (uint64_t i = 0; i < n; ++i)
                if (asg[i] == c) {
                    s = __fadd_rn(s, to_f32(sub(i)[j]));
                    ++cnt;
                }
            const float v = cnt ? __fdiv_rn(s, (float)cnt) : cent[slot];  // empty cluster keeps its centroid
            cnew[slot] = to_f32(from_f32_as(v, (T*)nullptr));
        }
        __syncthreads();
        for (uint32_t c = tid; c < kc; c += blockDim.x) {
            float s = 0.f;
            for (uint32_t j = 0; j < len; ++j) {
                const float df = __fsub_rn(cent[c * len + j], cnew[c * len + j]);
                s = __fadd_rn(s, __fmul_rn(df, df));
            }
            perc[c] = s;
        }
        __syncthreads();
        if (tid == 0) {
            float mx = __uint_as_float(0xff800000u);
            for (uint32_t c = 0; c < kc; ++c) mx = fmaxf(mx, perc[c]);
            s_conv = mx < p.tol;
        }
        for (uint32_t e = tid; e < kc * len; e += blockDim.x) cent[e] = cnew[e];
        __syncthreads();
        if (s_conv) break;
    }
    for (uint32_t e = tid; e < kc * len; e += blockDim.x) out[e] = from_f32_as(cent[e], (T*)nullptr);
    if (tid == 0) p.iters[g] = iters;
}

bool pq_train_supported(uint32_t kc, uint32_t max_len) { return kc <= 256 && (size_t)kc * max_len * 8 + kc * 8 <= 160 * 1024; }

// groups: device [m][3]; uniforms: device [m][2 kc - 1] doubles (or nullptr with d_init); d_out / d_init: device codebooks
void pq_train_groups(const void* d_rows, uint64_t n, uint64_t pitch, int dtype, int metric, uint32_t m, uint32_t kc, uint32_t max_len,
                     const uint32_t* d_groups, const double* d_uniforms, const void* d_init, uint32_t max_iter, float tol,
                     void* d_out, uint32_t* d_iters, cudaStream_t st) {
    VDB_REQUIRE(pq_train_supported(kc, max_len), "batched PQ training: k=%u x sub-dim %u does not fit in shared memory", kc, max_len);
    VDB_REQUIRE(n > 0, "cannot train on an empty vector set");
    DevBuf w((size_t)m * n * 4, st), asg((size_t)m * n, st);
    PqTrainParams p{};
    p.rows = d_rows;
    p.n = n;
    p.pitch = pitch;
    p.m = m;
    p.kc = kc;
    p.max_iter = max_iter;
    p.tol = tol;
    p.groups = d_groups;
    p.uniforms = d_uniforms;
    p.init = d_init;
    p.out = d_out;
    p.iters = d_iters;
    p.w = w.as<float>();
    p.assign = asg.as<uint8_t>();
    const size_t smem = (size_t)kc * max_len * 8 + (size_t)kc * 8;
    auto go = [&](auto kern) {
        if (smem > 48 * 1024) VDB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        ProfScope prof("pq_train", st);
        kern<<<m, 256, smem, st>>>(p);
        VDB_LAUNCHED();
    };
    if (dtype == VDB_F32) {
        if (metric == VDB_L2SQR) go(pq_train_kernel<float, VDB_L2SQR>);
        else go(pq_train_kernel<float, VDB_COSINE>);
    } else {
        if (metric == VDB_L2SQR) go(pq_train_kernel<uint8_t, VDB_L2SQR>);
        else go(pq_train_kernel<uint8_t, VDB_COSINE>);
    }
}

}  // namespace vdb
