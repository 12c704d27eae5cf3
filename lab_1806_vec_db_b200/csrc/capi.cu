// capi.cu — the extern "C" boundary declared in include/vdb_b200.h.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <limits>
#include <vector>

#include "dataset.cuh"
#include "index.cuh"
#include "topk.cuh"

#include <chrono>
#include <condition_variable>
#include <deque>
#include <functional>
#include <map>
#include <mutex>
#include <thread>

namespace vdb {
std::atomic<bool> g_batching{true};
bool g_prof_on = false;
namespace {
struct ProfEntry {
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> spans;
    std::map<cudaStream_t, cudaEvent_t> open;   // per launching stream: several devices / threads record concurrently
};
std::mutex g_prof_mu;
std::map<std::string, ProfEntry> g_prof;
}  // namespace
void prof_record(const char* name, cudaStream_t st, bool begin) {
    std::lock_guard<std::mutex> lk(g_prof_mu);
    ProfEntry& e = g_prof[name];
    cudaEvent_t ev;
    if (cudaEventCreate(&ev) != cudaSuccess) return;
    cudaEventRecord(ev, st);
    auto it = e.open.find(st);
    if (begin) {
        if (it != e.open.end()) cudaEventDestroy(it->second);
        e.open[st] = ev;
    } else if (it != e.open.end()) {
        e.spans.emplace_back(it->second, ev);
        e.open.erase(it);
    } else {
        cudaEventDestroy(ev);
    }
}
}  // namespace vdb

namespace vdb {
// multi.cu
std::vector<int> registered_devices();
void init_devices(const int* devices, uint32_t n, bool register_default);
vdb_dataset* sharded_create(const std::vector<int>& devs, uint64_t n, uint32_t dim, int dtype, int metric, uint64_t id_base,
                            const std::vector<uint64_t>* counts,
                            const std::function<vdb_dataset*(uint32_t, int, uint64_t, uint64_t)>& make_shard);
void sharded_destroy(vdb_dataset* md);
void sharded_flat_knn(const vdb_dataset* md, const void* queries, uint32_t nq, uint32_t k, uint64_t* ids, float* dist,
                      uint32_t* counts);
void sharded_flat_knn_dev(const vdb_dataset* md, const void* const* d_queries, uint32_t nq, uint32_t k, uint64_t* const* d_ids,
                          float* const* d_dist, uint32_t* const* d_counts);
uint32_t sharded_count(const vdb_dataset* md);
void sharded_info(const vdb_dataset* md, uint32_t s, int* device, uint64_t* lo, uint64_t* hi, vdb_dataset** ds);
}  // namespace vdb

namespace {
thread_local std::string t_error;
thread_local int t_device = -1;

template <class F> int guarded(F f) {
    try {
        f();
        return VDB_OK;
    } catch (const vdb::Error& e) {
        t_error = e.what();
        return e.code;
    } catch (const std::bad_alloc&) {
        t_error = "host out of memory";
        return VDB_ENOMEM;
    } catch (const std::exception& e) {
        t_error = e.what();
        return VDB_ECUDA;
    }
}

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) {
        VDB_CUDA(cudaGetDevice(&prev));
        if (dev != prev) VDB_CUDA(cudaSetDevice(dev));
        else prev = -1;
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

// per-call stream for the host-pointer entry points: re-entrant, no cross-call serialisation
// Stream of the host-pointer entry points: one per (calling thread, device), created on first use and kept for the
// life of the thread (re-entrant: concurrent callers never share a stream; no create / destroy per call).
struct ThreadStreams {
    cudaStream_t s[vdb::VDB_MAX_DEVICES] = {};
    ~ThreadStreams() {
        for (int d = 0; d < vdb::VDB_MAX_DEVICES; ++d)
            if (s[d]) {
                int prev = 0;
                if (cudaGetDevice(&prev) != cudaSuccess) break;   // the runtime is shutting down
                cudaSetDevice(d);
                cudaStreamDestroy(s[d]);
                cudaSetDevice(prev);
            }
    }
};
thread_local ThreadStreams t_streams;
struct CallStream {
    cudaStream_t s = nullptr;
    CallStream() {   // the current device is the handle's (DeviceGuard)
        int dev = 0;
        VDB_CUDA(cudaGetDevice(&dev));
        cudaStream_t& slot = t_streams.s[dev & (vdb::VDB_MAX_DEVICES - 1)];
        if (!slot) VDB_CUDA(cudaStreamCreateWithFlags(&slot, cudaStreamNonBlocking));
        s = slot;
    }
    void sync() { VDB_CUDA(cudaStreamSynchronize(s)); }
};

int current_device() {
    if (t_device >= 0) return t_device;
    int d = 0;
    VDB_CUDA(cudaGetDevice(&d));
    return d;
}

// device of an unsharded handle; entry points without a row-sharded implementation refuse a sharded parent
int dev_of(const vdb_dataset* ds) {
    if (ds->sharded) vdb::fail(VDB_EUNSUPPORTED, "this entry point has no row-sharded implementation: call it on the shards "
                                                 "(vdb_dataset_shard) or on an unsharded dataset");
    return ds->device;
}

void check_dtype_metric(int dtype, int metric) {
    VDB_REQUIRE(dtype == VDB_F32 || dtype == VDB_U8, "dtype must be VDB_F32 or VDB_U8");
    VDB_REQUIRE(metric == VDB_L2SQR || metric == VDB_COSINE, "metric must be VDB_L2SQR or VDB_COSINE");
}

void upload_rows(vdb_dataset* ds, uint64_t at, const void* rows, uint64_t n, cudaStream_t st) {
    if (n == 0) return;
    const size_t es = ds->elem_size();
    uint8_t* dst = (uint8_t*)ds->d_rows + at * ds->pitch_bytes();
    if (ds->pitch == ds->dim) {
        VDB_CUDA(cudaMemcpyAsync(dst, rows, n * ds->pitch_bytes(), cudaMemcpyHostToDevice, st));
    } else {
        VDB_CUDA(cudaMemsetAsync(dst, 0, n * ds->pitch_bytes(), st));
        VDB_CUDA(cudaMemcpy2DAsync(dst, ds->pitch_bytes(), rows, ds->dim * es, ds->dim * es, n,
                                   cudaMemcpyHostToDevice, st));
    }
}

using vdb::drop_side_arrays;

// copies nq query rows to the device, runs `body(d_queries, d_ids, d_dist, d_counts, stream)`, copies back
template <class Body>
void host_search(int device, const void* queries, uint32_t nq, size_t qbytes_per, uint32_t k, uint64_t* ids,
                 float* dist, uint32_t* counts, Body body) {
    DeviceGuard g(device);
    CallStream cs;
    vdb::DevBuf dq((size_t)nq * qbytes_per, cs.s);
    vdb::DevBuf dids((size_t)nq * k * 8, cs.s), ddist((size_t)nq * k * 4, cs.s), dcnt((size_t)nq * 4, cs.s);
    if (nq) VDB_CUDA(cudaMemcpyAsync(dq.p, queries, (size_t)nq * qbytes_per, cudaMemcpyHostToDevice, cs.s));
    body(dq.p, dids.as<uint64_t>(), ddist.as<float>(), dcnt.as<uint32_t>(), cs.s);
    if (nq && k) {
        VDB_CUDA(cudaMemcpyAsync(ids, dids.p, (size_t)nq * k * 8, cudaMemcpyDeviceToHost, cs.s));
        VDB_CUDA(cudaMemcpyAsync(dist, ddist.p, (size_t)nq * k * 4, cudaMemcpyDeviceToHost, cs.s));
    }
    if (nq) VDB_CUDA(cudaMemcpyAsync(counts, dcnt.p, (size_t)nq * 4, cudaMemcpyDeviceToHost, cs.s));
    cs.sync();
    dq.release();
    dids.release();
    ddist.release();
    dcnt.release();
    cs.sync();
}
}  // namespace

namespace vdb {
// an unsharded dataset over rows already on `device` (not owned: the caller frees them unless it sets `owned`)
vdb_dataset* adopt_dataset_on(int device, const void* d_rows, uint64_t n, uint32_t dim, uint32_t pitch, int dtype, int metric,
                              uint64_t id_base) {
    VDB_REQUIRE(((uintptr_t)d_rows & 15) == 0, "device rows must be 16-byte aligned");
    auto ds = new vdb_dataset();
    ds->device = device;
    ds->d_rows = const_cast<void*>(d_rows);
    ds->owned = false;
    ds->n = ds->cap = n;
    ds->dim = dim;
    ds->pitch = pitch;
    ds->dtype = dtype;
    ds->metric = metric;
    ds->id_base = id_base;
    return ds;
}
// the calling thread's stream on the current device (the stream of the host-pointer entry points)
cudaStream_t thread_stream() { return CallStream().s; }
}  // namespace vdb
using vdb::adopt_dataset_on;

struct vdb_batcher {
    std::mutex mu;
    std::condition_variable cv;
    struct Req {
        const void* q;
        uint32_t k;
        uint64_t* ids;
        float* dist;
        uint32_t* count;
        int state = 0;   // 0 pending, 1 done, 2 failed
        int code = 0;
        std::string err;
    };
    std::deque<Req*> pending;
    bool leader_active = false;
    uint32_t last_batch = 1;
    cudaStream_t st = nullptr;
    uint8_t* h_stage = nullptr;   // pinned: queries in, packed results out
    size_t h_cap = 0;
    uint8_t* d_stage = nullptr;
    size_t d_cap = 0;
    uint64_t batches = 0, served = 0;
};
constexpr uint32_t BATCH_MAX = 64;
constexpr uint32_t BATCH_WINDOW_US = 120;

static void batcher_free(vdb_batcher* b) {
    if (!b) return;
    if (b->st) cudaStreamSynchronize(b->st), cudaStreamDestroy(b->st);
    if (b->h_stage) cudaFreeHost(b->h_stage);
    if (b->d_stage) cudaFree(b->d_stage);
    delete b;
}


extern "C" {

const char* vdb_last_error(void) { return t_error.c_str(); }
int vdb_version(void) { return 801; /* tracks reference v0.8.1 */ }
uint64_t vdb_launch_count(void) { return vdb::g_launches.load(); }

int vdb_device_count(int* out) {
    return guarded([&] {
        VDB_REQUIRE(out, "out is NULL");
        VDB_CUDA(cudaGetDeviceCount(out));
    });
}
int vdb_set_device(int device) {
    return guarded([&] {
        int n = 0;
        VDB_CUDA(cudaGetDeviceCount(&n));
        VDB_REQUIRE(device >= 0 && device < n, "device %d out of range (have %d)", device, n);
        VDB_CUDA(cudaSetDevice(device));
        t_device = device;
    });
}

// ---- dataset -------------------------------------------------------------------------------------
static vdb_dataset* upload_dataset_on(int device, const void* rows, uint64_t n, uint32_t dim, int dtype, int metric,
                                      uint64_t id_base) {
    auto ds = new vdb_dataset();
    ds->device = device;
    DeviceGuard g(device);
    ds->dim = dim;
    ds->dtype = dtype;
    ds->metric = metric;
    ds->id_base = id_base;
    ds->pitch = vdb::round_up(dim, vdb::vec_elems(dtype));
    ds->n = n;
    ds->cap = std::max<uint64_t>(n, 1);
    try {
        VDB_CUDA(cudaMalloc(&ds->d_rows, ds->cap * ds->pitch_bytes()));
        CallStream cs;
        upload_rows(ds, 0, rows, n, cs.s);
        cs.sync();
    } catch (...) {
        if (ds->d_rows) cudaFree(ds->d_rows);
        delete ds;
        throw;
    }
    return ds;
}

int vdb_init(const int* devices, uint32_t n) {
    return guarded([&] {
        VDB_REQUIRE(devices || n == 0, "devices is NULL");
        vdb::init_devices(devices, n, true);
        if (n == 1) {
            VDB_CUDA(cudaSetDevice(devices[0]));
            t_device = devices[0];
        }
    });
}

int vdb_dataset_create(const void* rows, uint64_t n, uint32_t dim, int dtype, int metric, uint64_t id_base,
                       vdb_dataset** out) {
    return guarded([&] {
        VDB_REQUIRE(out, "out is NULL");
        VDB_REQUIRE(dim > 0, "dim must be > 0");
        VDB_REQUIRE(rows || n == 0, "rows is NULL");
        check_dtype_metric(dtype, metric);
        VDB_REQUIRE(id_base + n < 0xFFFFFFFFull, "id_base + n must be < 2^32 - 1");
        const std::vector<int> devs = vdb::registered_devices();
        if (devs.size() > 1) {
            // vdb_init registered several devices: contiguous row blocks, one per device (SURVEY.md section 8e)
            const size_t rb = (size_t)dim * (dtype == VDB_F32 ? 4 : 1);
            *out = vdb::sharded_create(devs, n, dim, dtype, metric, id_base, nullptr,
                                       [&](uint32_t, int device, uint64_t lo, uint64_t hi) {
                                           return upload_dataset_on(device, (const uint8_t*)rows + lo * rb, hi - lo, dim, dtype,
                                                                    metric, id_base + lo);
                                       });
            return;
        }
        *out = upload_dataset_on(devs.size() == 1 && t_device < 0 ? devs[0] : current_device(), rows, n, dim, dtype, metric,
                                 id_base);
    });
}

int vdb_dataset_create_dev(const void* d_rows, uint64_t n, uint32_t dim, uint32_t pitch, int dtype, int metric,
                           uint64_t id_base, vdb_dataset** out) {
    return guarded([&] {
        VDB_REQUIRE(out && (d_rows || n == 0), "NULL argument");
        VDB_REQUIRE(dim > 0 && pitch >= dim, "need 0 < dim <= pitch");
        check_dtype_metric(dtype, metric);
        VDB_REQUIRE(pitch % vdb::vec_elems(dtype) == 0, "row pitch must be a multiple of 16 bytes");
        VDB_REQUIRE(id_base + n < 0xFFFFFFFFull, "id_base + n must be < 2^32 - 1");
        *out = adopt_dataset_on(current_device(), d_rows, n, dim, pitch, dtype, metric, id_base);
    });
}

int vdb_dataset_create_sharded_dev(const void* const* d_rows, const uint64_t* counts, const int* devices, uint32_t nshards,
                                   uint32_t dim, uint32_t pitch, int dtype, int metric, uint64_t id_base, vdb_dataset** out) {
    return guarded([&] {
        VDB_REQUIRE(out && d_rows && counts && devices && nshards > 0, "NULL argument");
        VDB_REQUIRE(dim > 0 && pitch >= dim, "need 0 < dim <= pitch");
        check_dtype_metric(dtype, metric);
        VDB_REQUIRE(pitch % vdb::vec_elems(dtype) == 0, "row pitch must be a multiple of 16 bytes");
        uint64_t n = 0;
        std::vector<uint64_t> cnt(counts, counts + nshards);
        for (uint64_t c : cnt) n += c;
        VDB_REQUIRE(id_base + n < 0xFFFFFFFFull, "id_base + n must be < 2^32 - 1");
        std::vector<int> devs(devices, devices + nshards);
        vdb::init_devices(devices, nshards, false);   // peer access between the shards' devices (no global registration)
        *out = vdb::sharded_create(devs, n, dim, dtype, metric, id_base, &cnt,
                                   [&](uint32_t s, int device, uint64_t lo, uint64_t hi) {
                                       VDB_REQUIRE(d_rows[s] || hi == lo, "d_rows[%u] is NULL", s);
                                       return adopt_dataset_on(device, d_rows[s], hi - lo, dim, pitch, dtype, metric, id_base + lo);
                                   });
    });
}

int vdb_dataset_shards(const vdb_dataset* ds, uint32_t* n) {
    return guarded([&] {
        VDB_REQUIRE(ds && n, "NULL argument");
        *n = vdb::sharded_count(ds);
    });
}
int vdb_dataset_shard(const vdb_dataset* ds, uint32_t s, vdb_dataset** shard, int* device, uint64_t* row_lo, uint64_t* row_hi) {
    return guarded([&] {
        VDB_REQUIRE(ds, "NULL dataset");
        VDB_REQUIRE(ds->sharded, "not a row-sharded dataset");
        vdb::sharded_info(ds, s, device, row_lo, row_hi, shard);
    });
}
int vdb_dataset_set_flat_path(vdb_dataset* ds, int path) {
    return guarded([&] {
        VDB_REQUIRE(ds, "NULL dataset");
        VDB_REQUIRE(path >= -1 && path <= 2, "path must be -1 (process default), 0 (auto), 1 (scan) or 2 (tensor)");
        ds->flat_path = path;
    });
}
int vdb_set_batching(int on) {
    vdb::g_batching = on != 0;
    return VDB_OK;
}
int vdb_batch_stats(const vdb_dataset* ds, uint64_t* batches, uint64_t* queries) {
    return guarded([&] {
        VDB_REQUIRE(ds, "NULL dataset");
        vdb_batcher* b = ds->batcher;
        uint64_t nb = 0, nq = 0;
        if (b) {
            std::lock_guard<std::mutex> lk(b->mu);
            nb = b->batches, nq = b->served;
        }
        if (batches) *batches = nb;
        if (queries) *queries = nq;
    });
}
int vdb_debug_force_redo(uint32_t every) {
    vdb::g_debug_force_redo = every;
    return VDB_OK;
}

int vdb_dataset_append(vdb_dataset* ds, const void* rows, uint64_t n) {
    return guarded([&] {
        VDB_REQUIRE(ds && (rows || n == 0), "NULL argument");
        dev_of(ds);
        VDB_REQUIRE(ds->owned, "cannot append to an adopted device dataset");
        VDB_REQUIRE(ds->id_base + ds->n + n < 0xFFFFFFFFull, "id_base + n must be < 2^32 - 1");
        DeviceGuard g(dev_of(ds));
        drop_side_arrays(ds);
        CallStream cs;
        if (ds->n + n > ds->cap) {  // amortised growth, like Vec::push
            uint64_t cap = std::max<uint64_t>(ds->n + n, ds->cap + ds->cap / 2);
            void* p = nullptr;
            VDB_CUDA(cudaMalloc(&p, cap * ds->pitch_bytes()));
            VDB_CUDA(cudaMemcpyAsync(p, ds->d_rows, ds->n * ds->pitch_bytes(), cudaMemcpyDeviceToDevice, cs.s));
            cs.sync();
            cudaFree(ds->d_rows);
            ds->d_rows = p;
            ds->cap = cap;
        }
        upload_rows(ds, ds->n, rows, n, cs.s);
        cs.sync();
        ds->n += n;
    });
}

int vdb_dataset_swap_remove(vdb_dataset* ds, uint64_t idx) {
    return guarded([&] {
        VDB_REQUIRE(ds, "NULL dataset");
        dev_of(ds);
        VDB_REQUIRE(ds->owned, "cannot mutate an adopted device dataset");
        VDB_REQUIRE(idx < ds->n, "swap_remove index %llu out of range (len %llu)", (unsigned long long)idx,
                    (unsigned long long)ds->n);
        DeviceGuard g(dev_of(ds));
        drop_side_arrays(ds);
        if (idx != ds->n - 1) {
            uint8_t* base = (uint8_t*)ds->d_rows;
            VDB_CUDA(cudaMemcpy(base + idx * ds->pitch_bytes(), base + (ds->n - 1) * ds->pitch_bytes(),
                                ds->pitch_bytes(), cudaMemcpyDeviceToDevice));
        }
        ds->n -= 1;
    });
}
int vdb_dataset_len(const vdb_dataset* ds, uint64_t* n) {
    return guarded([&] {
        VDB_REQUIRE(ds && n, "NULL argument");
        *n = ds->n;
    });
}
int vdb_dataset_dim(const vdb_dataset* ds, uint32_t* dim) {
    return guarded([&] {
        VDB_REQUIRE(ds && dim, "NULL argument");
        *dim = ds->dim;
    });
}
int vdb_dataset_destroy(vdb_dataset* ds) {
    return guarded([&] {
        if (!ds) return;
        if (ds->sharded) {
            vdb::sharded_destroy(ds);
            return;
        }
        DeviceGuard g(ds->device);
        batcher_free(ds->batcher);
        drop_side_arrays(ds);
        if (ds->owned && ds->d_rows) cudaFree(ds->d_rows);
        delete ds;
    });
}

// ---- Flat ------------------------------------------------------------------------------------------
constexpr uint64_t LARGE_K_RESULT_BYTES = 1ull << 30;

int vdb_flat_set_path(int path) {
    return guarded([&] {
        VDB_REQUIRE(path >= 0 && path <= 2, "path must be 0 (auto), 1 (scan) or 2 (tensor)");
        vdb::g_flat_path = path;
    });
}

// returns true when `out` (optional) has already received the decoded results
static bool flat_keys_dispatch(const vdb_dataset* ds, const void* d_q, uint32_t nq, uint32_t k, uint64_t* d_keys,
                               cudaStream_t st, const vdb::ScanOut* out = nullptr) {
    const int path = ds->flat_path >= 0 ? ds->flat_path : vdb::g_flat_path.load();
    bool tensor = false;
    if (path == 2) {
        VDB_REQUIRE(vdb::flat_gemm_supported(ds, nq, k),
                    "tensor-core Flat path needs f32 rows, at least 65536 of them, and k <= 1024");
        tensor = true;
    } else if (path == 0) {
        // measured crossover (scripts/probe_parts2.py, 1M x 960 f32): the tensor pass streams the FP16 operand copy (half
        // the bytes of the rows) and costs 0.50-0.59 ms for any nq <= 128 (single CTAs, M = 128); the exact scan costs
        // 0.59 ms for 1-2 queries (99 % of the HBM roofline of the fp32 rows), 0.70 ms for 3-4, 1.04 ms for 5-8
        tensor = nq >= 3 && vdb::flat_gemm_supported(ds, nq, k);
    }
    if (tensor) {
        vdb::flat_gemm_keys(ds, d_q, nq, k, d_keys, st);
        return false;
    }
    return vdb::flat_scan_keys(ds, d_q, nq, k, d_keys, st, out);
}


// ---- coalescing of concurrent single-query calls -----------------------------------------------------------------------
// The reference's call pattern is ONE query per knn call from many threads (rayon workers: examples/bench.rs:410-416,
// src/bin/gen_gnd.rs:65-68; Python threads under a read lock: src/database/mod.rs:248-256). Every such call is a full
// pass over the rows, so concurrent callers are served together: the first caller becomes the leader of a batch, the
// requests that arrive while a batch runs (or within a <= 120 us window when the previous batch showed that several
// callers are active) form the next batch, one database pass answers them all, and results are bit-identical to the
// individual calls (the scan and the tensor path return the same bits for any batch composition). A lone caller never
// waits: its request is the whole batch. Staging buffers and the stream are owned by the dataset handle.
static std::mutex g_batcher_mu;
static vdb_batcher* batcher_of(const vdb_dataset* cds) {
    vdb_dataset* ds = const_cast<vdb_dataset*>(cds);
    std::lock_guard<std::mutex> lk(g_batcher_mu);
    if (!ds->batcher) {
        auto b = new vdb_batcher();
        DeviceGuard g(ds->device);
        VDB_CUDA(cudaStreamCreateWithFlags(&b->st, cudaStreamNonBlocking));
        ds->batcher = b;
    }
    return ds->batcher;
}

// one database pass for `reqs` (same k): stage -> H2D -> search -> decode -> one D2H -> scatter
static void batcher_run(const vdb_dataset* ds, vdb_batcher* b, std::vector<vdb_batcher::Req*>& reqs) {
    DeviceGuard g(ds->device);
    const uint32_t nb = (uint32_t)reqs.size(), k = reqs[0]->k;
    const size_t rb = (size_t)ds->dim * ds->elem_size();
    const size_t q_bytes = vdb::round_up<size_t>(nb * rb, 16);
    const size_t ids_off = q_bytes, dist_off = ids_off + (size_t)nb * k * 8, cnt_off = dist_off + vdb::round_up<size_t>((size_t)nb * k * 4, 16);
    const size_t total = cnt_off + vdb::round_up<size_t>((size_t)nb * 4, 16);
    if (total > b->h_cap) {
        if (b->h_stage) VDB_CUDA(cudaFreeHost(b->h_stage));
        b->h_stage = nullptr;
        b->h_cap = 0;
        VDB_CUDA(cudaHostAlloc((void**)&b->h_stage, total * 2, cudaHostAllocDefault));
        b->h_cap = total * 2;
    }
    if (total > b->d_cap) {
        if (b->d_stage) VDB_CUDA(cudaFree(b->d_stage));
        b->d_stage = nullptr;
        b->d_cap = 0;
        VDB_CUDA(cudaMalloc((void**)&b->d_stage, total * 2));
        b->d_cap = total * 2;
    }
    for (uint32_t i = 0; i < nb; ++i) memcpy(b->h_stage + i * rb, reqs[i]->q, rb);
    cudaStream_t st = b->st;
    VDB_CUDA(cudaMemcpyAsync(b->d_stage, b->h_stage, nb * rb, cudaMemcpyHostToDevice, st));
    uint64_t* d_ids = (uint64_t*)(b->d_stage + ids_off);
    float* d_dist = (float*)(b->d_stage + dist_off);
    uint32_t* d_cnt = (uint32_t*)(b->d_stage + cnt_off);
    {
        vdb::DevBuf keys((size_t)nb * k * 8, st);
        const vdb::ScanOut so{d_ids, d_dist, d_cnt};
        if (!flat_keys_dispatch(ds, b->d_stage, nb, k, keys.as<uint64_t>(), st, &so))
            vdb::decode_keys(keys.as<uint64_t>(), nb, k, d_ids, d_dist, d_cnt, st);
    }
    VDB_CUDA(cudaMemcpyAsync(b->h_stage + ids_off, b->d_stage + ids_off, total - ids_off, cudaMemcpyDeviceToHost, st));
    VDB_CUDA(cudaStreamSynchronize(st));
    for (uint32_t i = 0; i < nb; ++i) {
        memcpy(reqs[i]->ids, b->h_stage + ids_off + (size_t)i * k * 8, (size_t)k * 8);
        memcpy(reqs[i]->dist, b->h_stage + dist_off + (size_t)i * k * 4, (size_t)k * 4);
        *reqs[i]->count = ((const uint32_t*)(b->h_stage + cnt_off))[i];
    }
}

static void batched_single_knn(const vdb_dataset* ds, const void* query, uint32_t k, uint64_t* ids, float* dist, uint32_t* count) {
    vdb_batcher* b = batcher_of(ds);
    vdb_batcher::Req me{query, k, ids, dist, count};
    std::unique_lock<std::mutex> lk(b->mu);
    b->pending.push_back(&me);
    b->cv.notify_all();   // a leader inside its collection window counts the arrivals
    while (me.state == 0) {
        if (b->leader_active) {
            b->cv.wait(lk);
            continue;
        }
        // lead: serve batches until this thread's own request has been answered, then hand over
        b->leader_active = true;
        while (me.state == 0) {
            if (b->last_batch > 1 && b->pending.size() < b->last_batch) {
                // several callers were active a moment ago: give them a moment to line up behind this request (they are
                // waking up from the previous batch: a futex wake-up takes tens of microseconds; a database pass takes
                // >= 500 us at 1M x 960, so a fuller batch repays the wait many times over)
                const uint32_t want = b->last_batch;
                b->cv.wait_for(lk, std::chrono::microseconds(BATCH_WINDOW_US), [&] { return b->pending.size() >= want; });
            }
            std::vector<vdb_batcher::Req*> batch;
            const uint32_t bk = b->pending.front()->k;
            for (auto it = b->pending.begin(); it != b->pending.end() && batch.size() < BATCH_MAX;) {
                if ((*it)->k == bk) {
                    batch.push_back(*it);
                    it = b->pending.erase(it);
                } else {
                    ++it;
                }
            }
            lk.unlock();
            int code = 0;
            std::string err;
            try {
                batcher_run(ds, b, batch);
            } catch (const vdb::Error& e) {
                code = e.code, err = e.what();
            } catch (const std::exception& e) {
                code = VDB_ECUDA, err = e.what();
            }
            lk.lock();
            for (auto* r : batch) {
                r->state = code ? 2 : 1;
                r->code = code;
                r->err = err;
            }
            b->last_batch = (uint32_t)batch.size();
            b->batches += 1;
            b->served += batch.size();
            b->cv.notify_all();
        }
        b->leader_active = false;
        b->cv.notify_all();   // a waiting caller takes over the queue
    }
    lk.unlock();
    if (me.state == 2) throw vdb::Error(me.code, me.err);
}

int vdb_flat_knn_keys_dev(const vdb_dataset* ds, const void* d_queries, uint32_t nq, uint32_t k, uint64_t* d_keys,
                          void* stream) {
    return guarded([&] {
        VDB_REQUIRE(ds && (d_queries || nq == 0) && (d_keys || nq * (uint64_t)k == 0), "NULL argument");
        DeviceGuard g(dev_of(ds));
        flat_keys_dispatch(ds, d_queries, nq, k, d_keys, (cudaStream_t)stream);
    });
}

int vdb_flat_knn_dev(const vdb_dataset* ds, const void* d_queries, uint32_t nq, uint32_t k, uint64_t* d_ids,
                     float* d_dist, uint32_t* d_counts, void* stream) {
    return guarded([&] {
        VDB_REQUIRE(ds && (d_queries || nq == 0), "NULL argument");
        VDB_REQUIRE(nq == 0 || d_counts, "d_counts is NULL");
        VDB_REQUIRE(nq * (uint64_t)k == 0 || (d_ids && d_dist), "NULL result arrays");
        DeviceGuard g(dev_of(ds));
        cudaStream_t st = (cudaStream_t)stream;
        vdb::DevBuf keys((size_t)nq * k * 8, st);
        const vdb::ScanOut so{d_ids, d_dist, d_counts};
        if (!flat_keys_dispatch(ds, d_queries, nq, k, keys.as<uint64_t>(), st, &so))
            vdb::decode_keys(keys.as<uint64_t>(), nq, k, d_ids, d_dist, d_counts, st);
    });
}

int vdb_flat_knn(const vdb_dataset* ds, const void* queries, uint32_t nq, uint32_t k, uint64_t* ids, float* dist,
                 uint32_t* counts) {
    return guarded([&] {
        VDB_REQUIRE(ds && (queries || nq == 0), "NULL argument");
        VDB_REQUIRE(nq == 0 || counts, "counts is NULL");
        VDB_REQUIRE(nq * (uint64_t)k == 0 || (ids && dist), "NULL result arrays");
        if (ds->sharded) {   // vdb_init with several devices: the same call, spread over the shards (multi.cu)
            vdb::sharded_flat_knn(ds, queries, nq, k, ids, dist, counts);
            return;
        }
        // the trait's call: coalesced with concurrent callers, unless k is above the fused top-k (the batcher's page-locked
        // staging would grow with k, and such a call is a pass of its own)
        if (nq == 1 && k > 0 && ds->n > 0 && vdb::g_batching.load() && vdb::fused_topk_fits(ds, 1, k)) {
            batched_single_knn(ds, queries, k, ids, dist, counts);
            return;
        }
        const size_t qb = (size_t)ds->dim * ds->elem_size();
        auto search = [&](uint32_t q0, uint32_t n) {
            host_search(dev_of(ds), (const uint8_t*)queries + (size_t)q0 * qb, n, qb, k, ids + (size_t)q0 * k,
                        dist + (size_t)q0 * k, counts + q0, [&](void* dq, uint64_t* dids, float* dd, uint32_t* dc, cudaStream_t st) {
                            vdb::DevBuf keys((size_t)n * k * 8, st);
                            const vdb::ScanOut so{dids, dd, dc};
                            if (!flat_keys_dispatch(ds, dq, n, k, keys.as<uint64_t>(), st, &so))
                                vdb::decode_keys(keys.as<uint64_t>(), n, k, dids, dd, dc, st);
                        });
        };
        if (vdb::fused_topk_fits(ds, nq, k)) {
            search(0, nq);
            return;
        }
        // large k: the device copies of the results (keys, ids, distances: 20 bytes per slot) take at most
        // LARGE_K_RESULT_BYTES per pass, at least one query
        const uint32_t chunk = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(nq, LARGE_K_RESULT_BYTES / ((uint64_t)k * 20)));
        for (uint32_t q0 = 0; q0 < nq; q0 += chunk) search(q0, std::min(chunk, nq - q0));
    });
}

int vdb_flat_knn_sharded_dev(const vdb_dataset* ds, const void* const* d_queries, uint32_t nq, uint32_t k,
                             uint64_t* const* d_ids, float* const* d_dist, uint32_t* const* d_counts) {
    return guarded([&] {
        VDB_REQUIRE(ds && ds->sharded, "not a row-sharded dataset");
        VDB_REQUIRE(nq == 0 || (d_queries && d_ids && d_dist && d_counts), "NULL argument");
        vdb::sharded_flat_knn_dev(ds, d_queries, nq, k, d_ids, d_dist, d_counts);
    });
}

// The rayon loop of the reference's drivers (examples/bench.rs:410-416 `-t`, src/bin/gen_gnd.rs:65-68): nq queries, ONE
// vdb_flat_knn(nq = 1) call each, issued from `threads` native threads (query i goes to thread i % threads).
int vdb_parallel_knn(const vdb_dataset* ds, const void* queries, uint32_t nq, uint32_t k, uint32_t threads, uint64_t* ids,
                     float* dist, uint32_t* counts, double* seconds) {
    return guarded([&] {
        VDB_REQUIRE(ds && (queries || nq == 0) && threads >= 1 && threads <= 1024, "bad argument");
        VDB_REQUIRE(nq == 0 || (counts && (k == 0 || (ids && dist))), "NULL result arrays");
        const size_t rb = (size_t)ds->dim * ds->elem_size();
        std::vector<std::thread> th;
        std::vector<int> rc(threads, 0);
        std::vector<std::string> msg(threads);
        const auto t0 = std::chrono::steady_clock::now();
        for (uint32_t t = 0; t < threads; ++t)
            th.emplace_back([&, t] {
                for (uint32_t i = t; i < nq && rc[t] == 0; i += threads) {
                    rc[t] = vdb_flat_knn(ds, (const uint8_t*)queries + i * rb, 1, k, ids + (size_t)i * k, dist + (size_t)i * k, counts + i);
                    if (rc[t]) msg[t] = vdb_last_error();
                }
            });
        for (auto& x : th) x.join();
        if (seconds) *seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        for (uint32_t t = 0; t < threads; ++t)
            if (rc[t]) throw vdb::Error(rc[t], msg[t]);
    });
}

int vdb_merge_keys_dev(const uint64_t* d_keys, uint32_t nlists, uint32_t nq, uint32_t k, uint64_t* d_ids,
                       float* d_dist, uint32_t* d_counts, void* stream) {
    return guarded([&] {
        VDB_REQUIRE(nq * (uint64_t)k == 0 || (d_keys && d_ids && d_dist), "NULL argument");
        VDB_REQUIRE(nlists > 0, "nlists must be > 0");
        cudaStream_t st = (cudaStream_t)stream;
        if (k == 0) {
            if (nq && d_counts) VDB_CUDA(cudaMemsetAsync(d_counts, 0, (size_t)nq * 4, st));
            return;
        }
        vdb::launch_merge_sorted(d_keys, nlists, nq, k, k, nullptr, d_ids, d_dist, d_counts, st);
    });
}

int vdb_tq_info(const vdb_dataset* ds, uint64_t* n, uint32_t* sample_n, float* mean_norm, float* mean_ex) {
    return guarded([&] {
        VDB_REQUIRE(ds, "NULL dataset");
        DeviceGuard g(dev_of(ds));
        CallStream cs;
        vdb::tensor_info(ds, n, sample_n, mean_norm, mean_ex, cs.s);
        cs.sync();
    });
}
uint32_t vdb_tq_j0(uint32_t k, uint64_t sample_total, uint64_t n_total) {
    if (n_total == 0 || sample_total == 0) return 1;
    return vdb::tensor_j0(k, sample_total, n_total);
}
int vdb_tq_begin_dev(const vdb_dataset* ds, const void* d_queries, uint32_t nq, void* stream, vdb_tq** out) {
    return guarded([&] {
        VDB_REQUIRE(ds && d_queries && out && nq > 0, "NULL argument");
        DeviceGuard g(dev_of(ds));
        *out = vdb::tensor_begin(ds, d_queries, nq, (cudaStream_t)stream);
    });
}
int vdb_tq_sample_dev(vdb_tq* tq, uint32_t j, uint64_t* d_keys) {
    return guarded([&] {
        VDB_REQUIRE(tq && d_keys, "NULL argument");
        vdb::tensor_sample_keys(tq, j, d_keys);
    });
}
uint32_t vdb_tq_sample_j(uint32_t j0, uint64_t sample_min) { return vdb::tensor_sample_j(j0, sample_min); }
int vdb_tq_tau_dev(vdb_tq* tq, const uint64_t* d_keys_lists, uint32_t nlists, uint32_t j, uint32_t j0, float* d_tau) {
    return guarded([&] {
        VDB_REQUIRE(tq && d_keys_lists && d_tau && nlists > 0, "NULL argument");
        vdb::tensor_tau(tq, d_keys_lists, nlists, j, j0, d_tau);
    });
}
int vdb_tq_filter_dev(vdb_tq* tq, uint32_t k, const float* d_tau, uint64_t* d_keys, uint32_t* d_overflow) {
    return guarded([&] {
        VDB_REQUIRE(tq && d_tau && d_keys && d_overflow && k > 0, "NULL argument");
        vdb::tensor_filter_keys(tq, k, 0, d_tau, d_keys, d_overflow);
    });
}
int vdb_tq_check_dev(vdb_tq* tq, const uint64_t* d_merged_keys, uint32_t k, uint64_t n_total, const float* d_tau,
                     const uint32_t* d_overflow, uint32_t* d_redo, uint32_t* d_nredo) {
    return guarded([&] {
        VDB_REQUIRE(tq && d_merged_keys && d_tau && d_redo && d_nredo, "NULL argument");
        vdb::tensor_check(tq, d_merged_keys, k, n_total, d_tau, d_overflow, d_redo, d_nredo);
    });
}
int vdb_tq_end(vdb_tq* tq) {
    return guarded([&] { vdb::tensor_end(tq); });
}
int vdb_flat_scan_keys_dev(const vdb_dataset* ds, const void* d_queries, uint32_t nq, uint32_t k, uint64_t* d_keys,
                           void* stream) {
    return guarded([&] {
        VDB_REQUIRE(ds && (d_queries || nq == 0) && (d_keys || nq * (uint64_t)k == 0), "NULL argument");
        DeviceGuard g(dev_of(ds));
        vdb::flat_scan_keys(ds, d_queries, nq, k, d_keys, (cudaStream_t)stream);
    });
}
int vdb_merge_keys_to_keys_dev(const uint64_t* d_keys, uint32_t nlists, uint32_t nq, uint32_t k, uint64_t* d_out_keys,
                               void* stream) {
    return guarded([&] {
        VDB_REQUIRE(nq * (uint64_t)k == 0 || (d_keys && d_out_keys), "NULL argument");
        VDB_REQUIRE(nlists > 0, "nlists must be > 0");
        vdb::launch_merge_sorted(d_keys, nlists, nq, k, k, d_out_keys, nullptr, nullptr, nullptr, (cudaStream_t)stream);
    });
}
int vdb_decode_keys_dev(const uint64_t* d_keys, uint32_t nq, uint32_t k, uint64_t* d_ids, float* d_dist,
                        uint32_t* d_counts, void* stream) {
    return guarded([&] {
        VDB_REQUIRE(nq * (uint64_t)k == 0 || (d_keys && d_ids && d_dist), "NULL argument");
        vdb::decode_keys(d_keys, nq, k, d_ids, d_dist, d_counts, (cudaStream_t)stream);
    });
}

int vdb_debug_gemm_scores_dev(const vdb_dataset* ds, const void* d_queries, uint32_t nq, uint32_t row_stride, int kind,
                              uint64_t* d_out_keys, void* stream) {
    return guarded([&] {
        VDB_REQUIRE(ds && d_queries && d_out_keys, "NULL argument");
        DeviceGuard g(dev_of(ds));
        vdb::flat_gemm_store(ds, d_queries, nq, row_stride, kind, d_out_keys, (cudaStream_t)stream);
    });
}
int vdb_debug_pq_bounds_dev(const vdb_pq* pq, const void* d_queries, uint32_t nq, int path, float* d_lower, float* d_upper,
                            void* stream) {
    return guarded([&] {
        VDB_REQUIRE(pq && d_queries && d_lower && d_upper && nq > 0, "NULL argument");
        VDB_REQUIRE(path == 0 || path == 1, "path must be 0 (one-hot) or 1 (decoded)");
        if (!pq->shards.empty()) vdb::fail(VDB_EUNSUPPORTED, "vdb_debug_pq_bounds_dev: call it on the shards' tables");
        DeviceGuard g(pq->device);
        cudaStream_t st = (cudaStream_t)stream;
        if (path == 1) {
            vdb::pq_dec_bounds(pq, d_queries, nq, d_lower, d_upper, st);
            return;
        }
        VDB_REQUIRE(vdb::pq_tensor_supported(pq, UINT32_MAX), "one-hot PQ contraction: unsupported table");
        vdb::DevBuf lut((size_t)nq * pq->m * pq->kc * 4, st), qc((size_t)nq * 4, st);
        vdb::pq_lut(pq, d_queries, nq, lut.as<float>(), qc.as<float>(), st);
        vdb::pq_tensor_bounds(pq, lut.as<float>(), nq, d_lower, d_upper, st);
        VDB_CUDA(cudaStreamSynchronize(st));
    });
}
int vdb_dataset_operand_info(const vdb_dataset* ds, int* kind, float* scale, float* mean_norm, float* mean_ex,
                             uint64_t* side_bytes) {
    return guarded([&] {
        VDB_REQUIRE(ds, "NULL dataset");
        dev_of(ds);
        vdb::operand_info(ds, kind, scale, mean_norm, mean_ex, side_bytes);
    });
}
int vdb_dataset_drop_side_arrays(vdb_dataset* ds) {
    return guarded([&] {
        VDB_REQUIRE(ds, "NULL dataset");
        DeviceGuard g(dev_of(ds));
        VDB_CUDA(cudaDeviceSynchronize());
        drop_side_arrays(ds);
    });
}
uint64_t vdb_flat_gemm_fallbacks(void) { return vdb::g_gemm_redo.load(); }
int vdb_flat_gemm_stats(uint64_t* queries, uint64_t* candidates, uint64_t* fallbacks) {
    if (queries) *queries = vdb::g_gemm_queries.load();
    if (candidates) *candidates = vdb::g_gemm_cands.load();
    if (fallbacks) *fallbacks = vdb::g_gemm_redo.load();
    return VDB_OK;
}

int vdb_prof_enable(int on) {
    vdb::g_prof_on = on != 0;
    return VDB_OK;
}
int vdb_prof_reset(void) {
    return guarded([&] {
        std::lock_guard<std::mutex> lk(vdb::g_prof_mu);
        for (auto& kv : vdb::g_prof) {
            for (auto& sp : kv.second.spans) {
                cudaEventDestroy(sp.first);
                cudaEventDestroy(sp.second);
            }
            for (auto& o : kv.second.open) cudaEventDestroy(o.second);
        }
        vdb::g_prof.clear();
    });
}
int vdb_prof_read(const char* name, double* ms, uint64_t* launches) {
    return guarded([&] {
        VDB_REQUIRE(name && ms && launches, "NULL argument");
        VDB_CUDA(cudaDeviceSynchronize());
        std::lock_guard<std::mutex> lk(vdb::g_prof_mu);
        *ms = 0;
        *launches = 0;
        auto it = vdb::g_prof.find(name);
        if (it == vdb::g_prof.end()) return;
        for (auto& sp : it->second.spans) {
            float t = 0;
            VDB_CUDA(cudaEventElapsedTime(&t, sp.first, sp.second));
            *ms += t;
            *launches += 1;
        }
    });
}

#include "capi_index.inc"

}  // extern "C"
